"""Read-file ingest: FASTA / FASTQ (optionally gzip) -> batches of concatenated sequence bytes + offsets for
Query.push_ascii.  In the reference this job belongs to KMC (`kmc -fq|-fa`, scripts/select_db.py:46-52):
  -fq  4-line FASTQ records, the sequence is line 2 of each record
  -fa  FASTA with one sequence line per record; here every non-header line is taken as its own record, which
       is the same thing for single-line FASTA
Symbols outside ACGTacgt are left in place: the device treats them as N (they break the k-mer run).
Two implementations of the same record rules:
  * `PackedBatches` -- the native multi-threaded reader (csrc/ingest.cpp, include/metalign_b200_ingest.h): inflates /
    reads, finds the sequence lines and packs them 2 bits per base with N as (start, length) runs, straight into
    (pinned) host buffers for `Query.push_packed_nruns`.  This is what the drop-in select_db.py uses.
  * `batches` -- the numpy version (whole file in memory, ASCII batches for `Query.push_ascii`); kept as the
    independent restatement the native reader is tested against.
"""
from __future__ import annotations

import gzip
from typing import Iterator, Tuple

import numpy as np


import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
_INGEST = None
FASTQ, FASTA = 0, 1


def ingest_lib():
    """libmlg_ingest.so (host-only C++), built on demand"""
    global _INGEST
    if _INGEST is None:
        path = os.path.join(_HERE, "libmlg_ingest.so")
        src = os.path.join(_HERE, "csrc", "ingest.cpp")
        if not os.path.exists(path) or os.path.getmtime(path) < os.path.getmtime(src):
            subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc"), "-s", "../libmlg_ingest.so"])
        L = C.CDLL(path)
        L.mlgi_last_error.restype = C.c_char_p
        L.mlgi_open.argtypes = [C.c_char_p, C.c_int, C.c_int, C.POINTER(C.c_void_p)]
        L.mlgi_open_share.argtypes = [C.c_char_p, C.c_int, C.c_int, C.c_uint64, C.c_uint64, C.POINTER(C.c_void_p)]
        L.mlgi_share_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64), C.POINTER(C.c_int)]
        L.mlgi_next.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint64, C.c_uint64,
                                C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
        L.mlgi_spilled_runs.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64]
        L.mlgi_kmc_open.argtypes = [C.c_char_p, C.POINTER(C.c_void_p)]
        L.mlgi_kmc_info.argtypes = [C.c_void_p, C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                    C.POINTER(C.c_uint64), C.POINTER(C.c_int), C.POINTER(C.c_uint32)]
        L.mlgi_kmc_read.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        L.mlgi_kmc_close.argtypes = [C.c_void_p]
        L.mlgi_kmc_close.restype = None
        L.mlgi_stats.argtypes = [C.c_void_p] + [C.POINTER(C.c_uint64)] * 3
        L.mlgi_close.argtypes = [C.c_void_p]
        L.mlgi_close.restype = None
        L.mlgi_files_open.argtypes = [C.POINTER(C.c_char_p), C.c_uint32, C.c_int, C.POINTER(C.c_void_p)]
        L.mlgi_files_next.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_void_p, C.c_uint32, C.POINTER(C.c_uint32),
                                      C.POINTER(C.c_uint64)]
        L.mlgi_files_close.argtypes = [C.c_void_p]
        L.mlgi_files_close.restype = None
        _INGEST = L
    return _INGEST


class FileBatches:
    """Whole files (gzip, BGZF or plain), inflated by `threads` workers of the native reader (mlgi_files_*) and handed
    over in the order given, as batches of consecutive files.  next_batch() fills one of two alternating buffers of
    batch_bytes (`alloc(nbytes) -> uint8 ndarray`: pinned memory from api.pinned_array for the GPU), so one batch can be
    read while the other is in use; a file larger than batch_bytes comes alone, in a buffer of its own size."""

    def __init__(self, paths, batch_bytes: int = 1 << 30, threads: int = 0, max_files: int = 1 << 16, alloc=None):
        self.L = ingest_lib()
        self.h = C.c_void_p()
        self._paths = (C.c_char_p * max(1, len(paths)))(*[os.fsencode(p) for p in paths])
        if self.L.mlgi_files_open(self._paths, len(paths), int(threads), C.byref(self.h)) != 0:
            raise IOError(self.L.mlgi_last_error().decode())
        self.alloc = alloc or (lambda nbytes: np.empty(nbytes, dtype=np.uint8))
        self.max_files = int(max_files)
        self.bufs = [self.alloc(int(batch_bytes)), self.alloc(int(batch_bytes))]
        self.offs = [np.zeros(self.max_files + 1, dtype=np.uint64) for _ in range(2)]
        self.cur = 0

    def next_batch(self):
        """-> (buf uint8 ndarray, file_off uint64[n+1]) of the next batch, or None at the end"""
        k = self.cur
        self.cur ^= 1
        n, need = C.c_uint32(), C.c_uint64()
        while True:
            b, o = self.bufs[k], self.offs[k]
            rc = self.L.mlgi_files_next(self.h, b.ctypes.data, b.size, o.ctypes.data, self.max_files, C.byref(n), C.byref(need))
            if rc != 2:
                break
            self.bufs[k] = None
            self.bufs[k] = self.alloc(int(need.value))
        if rc < 0:
            raise IOError(self.L.mlgi_last_error().decode())
        if rc == 0:
            return None
        return b, o[:n.value + 1]

    def __iter__(self):
        while True:
            r = self.next_batch()
            if r is None:
                return
            yield r

    def close(self):
        if self.h:
            self.L.mlgi_files_close(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


class PackedBatches:
    """Iterate a reads file as packed batches: yields (bases uint8[], nruns uint32[m,2], off uint64[n+1], n_reads).
    The arrays are views of two alternating buffer sets (so one batch can still be in flight to the GPU while the
    next is being filled); `alloc(nbytes) -> uint8 ndarray` supplies them (pinned memory from api.pinned_array on a
    GPU box, numpy otherwise).  share = (begin, end): only the records of that byte range of the file
    (mlgi_open_share; see share_ranges and check_share_phases)."""

    def __init__(self, path: str, input_type: str, reads_per_batch: int = 4_000_000, bases_per_batch: int = 0,
                 threads: int = 0, alloc=None, max_runs: int = 0, share=None):
        self.L = ingest_lib()
        self.h = C.c_void_p()
        t = {"fastq": FASTQ, "fasta": FASTA}[input_type]
        if share is not None:
            rc = self.L.mlgi_open_share(path.encode(), t, int(threads), int(share[0]), int(share[1]), C.byref(self.h))
        else:
            rc = self.L.mlgi_open(path.encode(), t, int(threads), C.byref(self.h))
        if rc != 0:
            raise IOError(self.L.mlgi_last_error().decode())
        self.max_reads = int(reads_per_batch)
        self.max_bases = int(bases_per_batch) or min(self.max_reads * 160, 0xFFFFFF00)
        # N runs are rare (real reads: well under one per read); a batch with more than the buffer holds comes back through
        # mlgi_spilled_runs.  (max_bases // 64 entries were 80 MB of page-locked memory per buffer set, 0.06 s of pinning each; // 256 still holds one run per 1.7 reads.)
        self.max_runs = int(max_runs) or max(1024, self.max_bases // 256)
        self._alloc = alloc or (lambda nbytes: np.zeros(nbytes, dtype=np.uint8))
        self._raw = [self._alloc(nbytes) for _ in range(2)
                     for nbytes in (self.max_bases // 4 + 64, self.max_runs * 8, (self.max_reads + 1) * 8)]
        self.sets = [(self._raw[i], self._raw[i + 1].view(np.uint32), self._raw[i + 2].view(np.uint64)) for i in (0, 3)]
        self.cur = 0

    def __iter__(self):
        return self

    def __next__(self):
        b, r, o = self.sets[self.cur]
        self.cur ^= 1
        nr, nn = C.c_uint64(), C.c_uint64()
        rc = self.L.mlgi_next(self.h, b.ctypes.data, b.size, r.ctypes.data, self.max_runs, o.ctypes.data, self.max_reads,
                              self.max_bases, C.byref(nr), C.byref(nn))
        if rc < 0:
            raise IOError(self.L.mlgi_last_error().decode())
        if rc == 0:
            raise StopIteration
        if rc == 2:          # more N runs than the (pinned) buffer holds: the reader kept them
            big = np.empty(2 * nn.value, dtype=np.uint32)
            if self.L.mlgi_spilled_runs(self.h, big.ctypes.data, nn.value) != 0:
                raise IOError(self.L.mlgi_last_error().decode())
            return b, big.reshape(-1, 2), o[:nr.value + 1], nr.value
        return b, r[:2 * nn.value].reshape(-1, 2), o[:nr.value + 1], nr.value

    def stats(self):
        a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
        self.L.mlgi_stats(self.h, C.byref(a), C.byref(b), C.byref(c))
        return dict(reads=a.value, bases=b.value, text_bytes=c.value)

    def share_info(self) -> dict:
        """after the last batch: the text offset of the share's first line, its newline count and its FASTQ phase
        (-1: empty share, -2: no record start found near it)"""
        first, nl, ph = C.c_uint64(), C.c_uint64(), C.c_int()
        if self.L.mlgi_share_info(self.h, C.byref(first), C.byref(nl), C.byref(ph)) != 0:
            raise IOError(self.L.mlgi_last_error().decode())
        return dict(first=first.value, newlines=nl.value, phase=ph.value)

    def close(self):
        if self.h:
            self.L.mlgi_close(self.h)
            self.h = C.c_void_p()
            give_back = getattr(self._alloc, "give_back", None)
            if give_back is not None:
                give_back(self._raw)
            self._raw, self.sets = [], []

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


class BufferPool:
    """An `alloc` for PackedBatches readers opened one after another (the samples of a batch): a closed reader's buffers
    go to the next reader that asks for the same sizes, so page-locked memory is pinned once per batch rather than once
    per sample (0.7 ms per MiB) and stays bounded by the readers open at one time.  The caller must not close a reader
    while a copy from its buffers may still be in flight (Query.sync first)."""

    def __init__(self, alloc):
        import threading
        self._alloc, self._free, self._lock = alloc, [], threading.Lock()

    def __call__(self, nbytes: int) -> np.ndarray:
        with self._lock:
            for i, a in enumerate(self._free):
                if a.size == nbytes:
                    return self._free.pop(i)
        return self._alloc(nbytes)

    def give_back(self, arrays) -> None:
        with self._lock:
            self._free.extend(arrays)

    def clear(self) -> None:
        with self._lock:
            self._free = []


def share_ranges(path: str, world: int):
    """balanced [begin, end) byte ranges of the file on disk, one per rank"""
    size = os.path.getsize(path)
    return [(size * r // world, size * (r + 1) // world) for r in range(world)]


def check_share_phases(infos, input_type: str = "fastq") -> None:
    """infos: share_info() of every share, in file order.  A FASTQ share parses its lines from the phase it found at its
    first record start; that is the single-reader parse only if the phase equals the number of lines before the share mod
    4 (the earlier shares' newline counts).  Raises ValueError naming the offset where they differ."""
    if input_type != "fastq":
        return
    before = 0
    for i, info in enumerate(infos):
        if info["phase"] != -1 and info["phase"] != before % 4:
            raise ValueError("reads file is not 4-line FASTQ: share %d, starting at text byte %d, took line phase %d but %d "
                             "lines come before it; read this file on one GPU" % (i, info["first"], info["phase"], before))
        before += info["newlines"]


def _read_all(path: str) -> np.ndarray:
    opener = gzip.open if path.endswith(".gz") else open
    with opener(path, "rb") as f:
        data = f.read()
    return np.frombuffer(data, dtype=np.uint8)


def _line_table(buf: np.ndarray):
    """start / end (exclusive, newline and trailing '\\r' stripped) of every line"""
    nl = np.flatnonzero(buf == 10)
    starts = np.concatenate([[0], nl + 1]).astype(np.int64)
    ends = np.concatenate([nl, [buf.size]]).astype(np.int64)
    if starts.size and starts[-1] >= buf.size:          # file ends with a newline
        starts, ends = starts[:-1], ends[:-1]
    cr = (ends > starts) & (buf[np.maximum(ends - 1, 0)] == 13)
    ends = ends - cr.astype(np.int64)
    return starts, ends


def sequence_lines(buf: np.ndarray, input_type: str):
    starts, ends = _line_table(buf)
    if input_type == "fastq":
        sel = np.arange(1, starts.size, 4)
    elif input_type == "fasta":
        nonempty = ends > starts
        first = buf[np.minimum(starts, max(buf.size - 1, 0))] if buf.size else np.zeros(0, np.uint8)
        sel = np.flatnonzero(nonempty & (first != ord(">")) & (first != ord(";")))
    else:
        raise ValueError("input_type must be 'fastq' or 'fasta'")
    return starts[sel], ends[sel]


def batches(path: str, input_type: str, reads_per_batch: int = 2_000_000) -> Iterator[Tuple[np.ndarray, np.ndarray]]:
    """yields (text uint8[total], off uint64[n+1]) per batch of reads"""
    buf = _read_all(path)
    s, e = sequence_lines(buf, input_type)
    for a in range(0, s.size, reads_per_batch):
        sb, eb = s[a:a + reads_per_batch], e[a:a + reads_per_batch]
        lens = eb - sb
        off = np.zeros(lens.size + 1, dtype=np.uint64)
        np.cumsum(lens, out=off[1:])
        total = int(off[-1])
        # gather: output position p of read i comes from input position sb[i] + (p - off[i])
        shift = np.repeat(sb - off[:-1].astype(np.int64), lens)
        text = buf[np.arange(total, dtype=np.int64) + shift]
        yield np.ascontiguousarray(text), off
    if s.size == 0:
        return


def input_type_of(reads_path: str):
    """'fastq' / 'fasta' by extension ('.gz' ignored), None when the extension says neither"""
    parts = reads_path.split(".")
    if parts[-1] == "gz":
        parts = parts[:-1]
    if parts[-1] in ("fq", "fastq"):
        return "fastq"
    if parts[-1] in ("fa", "fna", "fasta"):
        return "fasta"
    return None


def detect_input_type(reads_path: str) -> str:
    """same rule as scripts/select_db.py:144-153: by extension, '.gz' ignored"""
    kind = input_type_of(reads_path)
    if kind is None:
        raise SystemExit("Could not auto-determine file type. Use --input_type.")
    return kind


def read_kmc_database(prefix: str, with_counts: bool = False):
    """The k-mers of a KMC database (<prefix>.kmc_pre / .kmc_suf; e.g. data/cmash_db_n1000_k60_dump of the reference,
    scripts/select_db.py:44) as an (n, 2) uint64 array of (hi, lo) keys in file order, plus a dict of its header fields
    (and the counts, if asked for)."""
    L = ingest_lib()
    h = C.c_void_p()
    if L.mlgi_kmc_open(prefix.encode(), C.byref(h)) != 0:
        raise IOError(L.mlgi_last_error().decode())
    try:
        k, cs, mn, ver = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
        tot, mx, canon = C.c_uint64(), C.c_uint64(), C.c_int()
        L.mlgi_kmc_info(h, C.byref(k), C.byref(tot), C.byref(cs), C.byref(mn), C.byref(mx), C.byref(canon), C.byref(ver))
        keys = np.empty((tot.value, 2), dtype=np.uint64)
        counts = np.empty(tot.value, dtype=np.uint32) if with_counts else None
        if L.mlgi_kmc_read(h, keys.ctypes.data, counts.ctypes.data if with_counts else None) != 0:
            raise IOError(L.mlgi_last_error().decode())
    finally:
        L.mlgi_kmc_close(h)
    info = dict(k=k.value, total=tot.value, counter_size=cs.value, min_count=mn.value, max_count=mx.value,
                canonical=bool(canon.value), version=ver.value)
    return (keys, info, counts) if with_counts else (keys, info)
