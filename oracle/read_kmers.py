"""TEST INFRASTRUCTURE -- ctypes binding of the read k-mer oracle (oracle/read_kmers.c).  PARITY UNPINNED.

Only tests/ and scripts/bench_read_kmers.py import this.  The library is compiled on first use, next to liboracle.so in
oracle/_build/, or in a per-user temporary directory when the tree is read-only.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "read_kmers.c")
_LIB = None
CFLAGS = ["-O3", "-march=x86-64-v2", "-fopenmp", "-fPIC", "-fvisibility=hidden", "-Wall", "-Wextra", "-Wno-unused-parameter"]


def build() -> str:
    cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
    for d in (os.path.join(_HERE, "_build"), os.path.join(tempfile.gettempdir(), "mlg_oracle_%d" % os.getuid())):
        path = os.path.join(d, "libread_kmers.so")
        if os.path.exists(path) and os.path.getmtime(path) >= os.path.getmtime(_SRC):
            return path
        try:
            os.makedirs(d, exist_ok=True)
            tmp = "%s.%d" % (path, os.getpid())
            subprocess.check_call([cc] + CFLAGS + ["-shared", "-o", tmp, _SRC])
            os.replace(tmp, path)
            return path
        except OSError:
            continue
    raise OSError("cannot build %s: no writable directory" % _SRC)


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        vp, u64p, u8p = C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint8)
        L.orc_rk_begin.restype = vp
        L.orc_rk_begin.argtypes = [C.c_uint32]
        L.orc_rk_free.argtypes = [vp]
        L.orc_rk_push_ascii.argtypes = [vp, C.c_char_p, u64p, C.c_uint64]
        L.orc_rk_push_packed.argtypes = [vp, u8p, u8p, u64p, C.c_uint64, C.c_uint32]
        L.orc_rk_distinct.restype = C.c_uint64
        L.orc_rk_distinct.argtypes = [vp]
        L.orc_rk_result.restype = C.c_uint64
        L.orc_rk_result.argtypes = [vp, C.c_uint32, C.c_uint32, u64p, u8p, C.c_uint64]
        _LIB = L
    return _LIB


def _p(a, t):
    return a.ctypes.data_as(C.POINTER(t))


class OracleReadKmers:
    """Every canonical K-mer of the pushed reads with its count (the whole `kmc -k<K> -ci<min> -cs<max>` database, not
    only the k-mers of D); the same push forms as oracle_c.OracleQuery."""

    def __init__(self, K: int = 60):
        self.K = int(K)
        self._h = lib().orc_rk_begin(self.K)
        if not self._h:
            raise ValueError("orc_rk_begin rejected K=%d" % K)

    def push_ascii(self, text: bytes, off: np.ndarray):
        off = np.ascontiguousarray(off, dtype=np.uint64)
        lib().orc_rk_push_ascii(self._h, text, _p(off, C.c_uint64), off.size - 1)

    def push_reads(self, reads):
        off = np.zeros(len(reads) + 1, dtype=np.uint64)
        if len(reads):
            off[1:] = np.cumsum([len(r) for r in reads], dtype=np.uint64)
        self.push_ascii("".join(reads).encode(), off)

    def push_packed(self, bases: np.ndarray, nmask, off, nreads: int, read_len: int = 0):
        bases = np.ascontiguousarray(bases, dtype=np.uint8)
        nm = None if nmask is None else np.ascontiguousarray(nmask, dtype=np.uint8)
        of = None if off is None else np.ascontiguousarray(off, dtype=np.uint64)
        lib().orc_rk_push_packed(self._h, _p(bases, C.c_uint8), None if nm is None else _p(nm, C.c_uint8),
                                 None if of is None else _p(of, C.c_uint64), nreads, read_len)

    def result(self, min_count: int = 1, counter_max: int = 255):
        """(keys uint64[n, 2] ascending, counts uint8[n] saturated at counter_max) of the k-mers seen >= min_count times"""
        cap = lib().orc_rk_distinct(self._h)
        keys = np.empty((cap, 2), dtype=np.uint64)
        counts = np.empty(cap, dtype=np.uint8)
        n = lib().orc_rk_result(self._h, min_count, counter_max, _p(keys, C.c_uint64), _p(counts, C.c_uint8), cap)
        return keys[:n], counts[:n]

    def close(self):
        if self._h:
            lib().orc_rk_free(self._h)
            self._h = None

    def __del__(self):
        self.close()
