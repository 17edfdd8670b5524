"""Python objects over the C ABI (include/metalign_b200.h).  Thin by design: every method is one or two
C calls; all compute is in the CUDA library.  Host arrays are numpy; device arrays are raw pointers
(e.g. ``torch_tensor.data_ptr()``)."""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from . import _lib
from ._lib import MlgError, Stats, check  # noqa: F401

GATE = {"exact": 0, "none": 1}
DEFAULT_KS = (30, 40, 50, 60)   # '30-60-10' at scripts/select_db.py:75 of the reference


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data


def pinned_array(nbytes: int) -> np.ndarray:
    """uint8 numpy view of page-locked host memory (mlg_host_alloc); freed when the array is collected"""
    import weakref
    p = C.c_void_p()
    check(_lib.lib().mlg_host_alloc(C.byref(p), int(nbytes)))
    buf = (C.c_uint8 * int(nbytes)).from_address(p.value)
    arr = np.frombuffer(buf, dtype=np.uint8)
    weakref.finalize(buf, _lib.lib().mlg_host_free, p.value)
    return arr


class Context:
    """One GPU.  One process (host thread) per context."""

    def __init__(self, device: int = 0):
        self._h = C.c_void_p()
        check(_lib.lib().mlg_ctx_create(int(device), C.byref(self._h)))
        self.device = int(device)

    def streams(self):
        """(compute, copy) cudaStream_t handles as ints, e.g. for torch.cuda.ExternalStream."""
        a, b = C.c_void_p(), C.c_void_p()
        check(_lib.lib().mlg_ctx_streams(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    def close(self):
        if self._h:
            _lib.lib().mlg_ctx_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class Database:
    """G genomes x n sketch slots of K-mers (stored in genome-strand orientation, '' = empty slot),
    queried at the prefix lengths ``ks``.  Replaces cmash_db_n1000_k60.h5 / .tst / .bf and
    cmash_db_n1000_k60_dump.kmc_* of the reference (scripts/select_db.py:44,69,70)."""

    def __init__(self, ctx: Context, handle, names=None):
        self.ctx = ctx
        self._h = handle
        G, n, K, nk = C.c_uint32(), C.c_uint32(), C.c_uint32(), C.c_uint32()
        ks = (C.c_uint32 * 8)()
        ne, nd = C.c_uint64(), C.c_uint64()
        check(_lib.lib().mlg_db_info(self._h, C.byref(G), C.byref(n), C.byref(K), C.byref(nk), C.byref(ks),
                                     C.byref(ne), C.byref(nd)))
        self.G, self.n, self.K = G.value, n.value, K.value
        self.ks = tuple(ks[i] for i in range(nk.value))
        self.n_entries, self.n_distinct = ne.value, nd.value
        self.names = list(names) if names is not None else None

    # -- constructors -------------------------------------------------------------------------
    @classmethod
    def from_keys(cls, ctx: Context, keys: np.ndarray, G: int, n: int, K: int = 60,
                  ks: Sequence[int] = DEFAULT_KS, names=None) -> "Database":
        keys = np.ascontiguousarray(keys, dtype=np.uint64).reshape(-1)
        if keys.size != 2 * G * n:
            raise ValueError("keys must hold G*n (hi, lo) pairs")
        ksa = np.asarray(ks, dtype=np.uint32)
        h = C.c_void_p()
        check(_lib.lib().mlg_db_from_keys(ctx._h, keys.ctypes.data, G, n, K, ksa.ctypes.data, ksa.size, C.byref(h)))
        return cls(ctx, h, names)

    @classmethod
    def from_device_keys(cls, ctx: Context, d_keys_ptr: int, G: int, n: int, K: int = 60,
                         ks: Sequence[int] = DEFAULT_KS, names=None) -> "Database":
        ksa = np.asarray(ks, dtype=np.uint32)
        h = C.c_void_p()
        check(_lib.lib().mlg_db_from_keys_device(ctx._h, d_keys_ptr, G, n, K, ksa.ctypes.data, ksa.size, C.byref(h)))
        return cls(ctx, h, names)

    @classmethod
    def from_device_chunks(cls, ctx: Context, chunks, G: int, n: int, K: int = 60, ks: Sequence[int] = DEFAULT_KS, names=None) -> "Database":
        """mlg_db_builder_*: `chunks` yields (device pointer, first genome, genomes) in genome order; a chunk's buffer may be
        reused as soon as the next one is asked for.  The device never holds all G*n keys beside the structures built from
        them (a 2e9-slot database builds inside 180 GB this way)."""
        ksa = np.asarray(ks, dtype=np.uint32)
        b = C.c_void_p()
        check(_lib.lib().mlg_db_builder_create(ctx._h, G, n, K, ksa.ctypes.data, ksa.size, C.byref(b)))
        h = C.c_void_p()
        try:
            for ptr, g0, count in chunks:
                check(_lib.lib().mlg_db_builder_add_device(b, ptr, g0, count))
            check(_lib.lib().mlg_db_builder_finish(b, C.byref(h)))
        except BaseException:
            _lib.lib().mlg_db_builder_destroy(b)
            raise
        return cls(ctx, h, names)

    @classmethod
    def from_sketches(cls, ctx: Context, sketches, K: int = 60, ks: Sequence[int] = DEFAULT_KS, names=None) -> "Database":
        """sketches: list of G lists of n strings ('' for an unused slot) -- what
        local_tests/dump_kmers.py:7-14 walks (`CE._kmers`).  Goes through mlg_db_from_ascii."""
        G = len(sketches)
        n = len(sketches[0])
        buf = bytearray(G * n * K)
        for g, sk in enumerate(sketches):
            if len(sk) != n:
                raise ValueError("every sketch must have the same number of slots")
            for j, s in enumerate(sk):
                if s:
                    if len(s) != K:
                        raise ValueError("sketch k-mer of length %d, expected %d" % (len(s), K))
                    o = (g * n + j) * K
                    buf[o:o + K] = s.encode()
        ksa = np.asarray(ks, dtype=np.uint32)
        h = C.c_void_p()
        check(_lib.lib().mlg_db_from_ascii(ctx._h, bytes(buf), G, n, K, ksa.ctypes.data, ksa.size, C.byref(h)))
        return cls(ctx, h, names)

    @classmethod
    def load(cls, ctx: Context, path: str) -> "Database":
        from . import dbformat
        names = dbformat.read_names(path)
        h = C.c_void_p()
        check(_lib.lib().mlg_db_load(ctx._h, path.encode(), C.byref(h)))
        return cls(ctx, h, names)

    def save(self, path: str) -> None:
        """Write the BUILT form of the database (the device structures): `Database.load` of such a file is a file read,
        not a rebuild.  Needs the genome names (a database made by `load` or given `names=`)."""
        blob = "\n".join(self.names or []).encode()
        if self.names is None or len(self.names) != self.G:
            raise ValueError("saving needs one name per genome")
        check(_lib.lib().mlg_db_save(self._h, path.encode(), blob, len(blob)))

    # -- queries ------------------------------------------------------------------------------
    def denominators(self, count_empty_in_den: bool = True) -> np.ndarray:
        den = np.zeros((self.G, len(self.ks)), dtype=np.int64)
        check(_lib.lib().mlg_db_denominators(self._h, int(count_empty_in_den), den.ctypes.data))
        return den

    def query(self, ci_min: int = 2, gate: str = "exact", count_empty_in_den: bool = True, read_kmers: bool = False,
              read_kmer_budget: int = 0, read_kmer_passes: bool = False) -> "Query":
        """read_kmers: also count every canonical K-mer of the pushed reads (K <= 60; Query.read_kmers /
        write_reads_kmc); read_kmer_budget caps that table's device bytes (0 = no cap).  read_kmer_passes: count them
        instead in key-range passes over a device copy of the reads at each output call, for read sets whose table would
        not fit; read_kmer_budget then caps the copy plus one pass (0 = the free device memory)"""
        q = Query(self, ci_min, gate, count_empty_in_den)
        if read_kmers:
            try:
                enable = _lib.lib().mlg_query_enable_read_kmer_passes if read_kmer_passes else _lib.lib().mlg_query_enable_read_kmers
                check(enable(q._h, int(read_kmer_budget)))
                q._rk_passes = bool(read_kmer_passes)
            except BaseException:
                q.close()
                raise
        return q

    def close(self):
        if self._h:
            _lib.lib().mlg_db_free(self._h)
            self._h = C.c_void_p()


class Query:
    """One read set against one database: push batches, then finish().  Replaces run_kmc_steps and the
    CMash subprocess of run_cmash_and_cutoff (scripts/select_db.py:43-76)."""

    def __init__(self, db: Database, ci_min: int = 2, gate: str = "exact", count_empty_in_den: bool = True):
        self.db = db
        self.ci_min = int(ci_min)
        self._h = C.c_void_p()
        check(_lib.lib().mlg_query_begin(db.ctx._h, db._h, int(ci_min), GATE[gate], int(count_empty_in_den),
                                         C.byref(self._h)))
        self._keep = []   # host buffers that must outlive the asynchronous copies
        self._rk_passes = False

    def push_packed(self, bases: np.ndarray, nmask: Optional[np.ndarray], off: Optional[np.ndarray],
                    n_reads: int, read_len: int = 0):
        """Host buffers (pinned for asynchronous copies).  off: uint64[n_reads+1] in bases, or None with
        fixed read_len.  Buffers must cover whole 16-byte units (see the header)."""
        if off is not None:
            off = np.ascontiguousarray(off, dtype=np.uint64)
        self._keep = self._keep[-3:] + [bases, nmask, off]
        check(_lib.lib().mlg_query_push_packed(self._h, _ptr(bases), _ptr(nmask), _ptr(off), int(n_reads), int(read_len)))

    def push_packed_nruns(self, bases: np.ndarray, nruns: Optional[np.ndarray], off: Optional[np.ndarray],
                          n_reads: int, read_len: int = 0):
        """Like push_packed, with N as sorted (start, length) uint32 runs (codec.nmask_to_runs) instead of a mask."""
        if off is not None:
            off = np.ascontiguousarray(off, dtype=np.uint64)
        n_runs = 0
        if nruns is not None:
            nruns = np.ascontiguousarray(nruns, dtype=np.uint32).reshape(-1, 2)
            n_runs = nruns.shape[0]
        self._keep = self._keep[-3:] + [bases, nruns, off]
        check(_lib.lib().mlg_query_push_packed_nruns(self._h, _ptr(bases), _ptr(nruns) if n_runs else None, n_runs,
                                                     _ptr(off), int(n_reads), int(read_len)))

    def push_packed_nruns_ptr(self, bases_ptr: int, nruns_ptr: Optional[int], n_runs: int, off_ptr: Optional[int],
                              n_reads: int, read_len: int = 0):
        check(_lib.lib().mlg_query_push_packed_nruns(self._h, bases_ptr, nruns_ptr, int(n_runs), off_ptr, int(n_reads),
                                                     int(read_len)))

    def push_packed_ptr(self, bases_ptr: int, nmask_ptr: Optional[int], off_ptr: Optional[int], n_reads: int,
                        read_len: int = 0, device: bool = False):
        """Raw-pointer variant (pinned host tensors or device tensors from torch)."""
        fn = _lib.lib().mlg_query_push_packed_device if device else _lib.lib().mlg_query_push_packed
        check(fn(self._h, bases_ptr, nmask_ptr, off_ptr, int(n_reads), int(read_len)))

    def push_ascii(self, text, off: np.ndarray):
        """text: bytes / uint8 array of concatenated reads; off: uint64[n_reads+1]."""
        if isinstance(text, (bytes, bytearray)):
            text = np.frombuffer(text, dtype=np.uint8)
        text = np.ascontiguousarray(text, dtype=np.uint8)
        off = np.ascontiguousarray(off, dtype=np.uint64)
        self._keep = self._keep[-3:] + [text, off]
        check(_lib.lib().mlg_query_push_ascii(self._h, text.ctypes.data, off.ctypes.data, off.size - 1))

    def push_reads(self, reads: Sequence[str]):
        off = np.zeros(len(reads) + 1, dtype=np.uint64)
        if len(reads):
            off[1:] = np.cumsum([len(r) for r in reads], dtype=np.uint64)
        self.push_ascii("".join(reads).encode(), off)

    def sync(self):
        check(_lib.lib().mlg_query_sync(self._h))

    def counts_export(self):
        """(device pointer, length) of the per-database-k-mer uint8 counters clamped to ci_min."""
        p, n = C.c_void_p(), C.c_uint64()
        check(_lib.lib().mlg_query_counts_export(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def counts_export_sparse(self):
        """(device pointer, n) of this rank's non-zero counters as uint64 entries: index | min(count, ci_min) << 32."""
        p, n = C.c_void_p(), C.c_uint64()
        check(_lib.lib().mlg_query_counts_export_sparse(self._h, C.byref(p), C.byref(n)))
        return p.value or 0, n.value

    def counts_merge_sparse(self, d_entries_ptr: int, n: int):
        check(_lib.lib().mlg_query_counts_merge_sparse(self._h, d_entries_ptr, int(n)))

    def counts_import(self):
        check(_lib.lib().mlg_query_counts_import(self._h))

    # -- multi-GPU exchange without a host round trip (see metalign_b200.dist) -------------------------------
    def exchange_pack(self, ex: "Exchange"):
        check(_lib.lib().mlg_query_exchange_pack(self._h, ex._h))

    def exchange_merge(self, ex: "Exchange"):
        check(_lib.lib().mlg_query_exchange_merge(self._h, ex._h))

    def exchange_p2p(self, ex: "Exchange"):
        check(_lib.lib().mlg_query_exchange_p2p(self._h, ex._h))

    def exchange_dense(self):
        """(device pointer, length) of the clamped uint8 counters; queued on the compute stream, nothing is joined"""
        p, n = C.c_void_p(), C.c_uint64()
        check(_lib.lib().mlg_query_exchange_dense(self._h, C.byref(p), C.byref(n)))
        return p.value, n.value

    def _finish_call(self, num_ptr, den_ptr, ci_ptr, sparse=None):
        """mlg_query_finish (or, with sparse = (genomes, cap, n_rows byref), mlg_query_finish_sparse); an exchange whose
        blocks turned out too small is repeated once with larger ones (self._exchange_retry is set by
        metalign_b200.dist.reduce_query)"""
        ni = C.c_uint64()

        def call():
            if sparse is None:
                return _lib.lib().mlg_query_finish(self._h, num_ptr, den_ptr, ci_ptr, C.byref(ni))
            return _lib.lib().mlg_query_finish_sparse(self._h, sparse[0], num_ptr, den_ptr, ci_ptr, sparse[1], sparse[2], C.byref(ni))
        rc = call()
        retry = getattr(self, "_exchange_retry", None)
        if rc == _lib.MLG_ERR_RETRY and retry is not None:
            msg = _lib.lib().mlg_last_error().decode(errors="replace")
            retry(int(msg.split(":")[-1].split()[0]))
            rc = call()
        check(rc)
        return ni.value

    def finish(self):
        G, nk = self.db.G, len(self.db.ks)
        num = np.zeros((G, nk), dtype=np.int64)
        den = np.zeros((G, nk), dtype=np.int64)
        ci = np.zeros((G, nk), dtype=np.float64)
        ni = self._finish_call(num.ctypes.data, den.ctypes.data, ci.ctypes.data)
        self._keep = []
        st = self.stats()
        return dict(num=num, den=den, ci=ci, n_intersect=ni, n_kmers=st["n_kmers"], stats=st)

    def finish_into(self, num_ptr: int, den_ptr: int, ci_ptr: int) -> int:
        """finish() writing into caller-provided (pinned) host buffers; returns |I|."""
        ni = self._finish_call(num_ptr, den_ptr, ci_ptr)
        self._keep = []
        return ni

    def finish_sparse(self, cap_rows: int = 1 << 16):
        """The result as rows for the genomes with a hit at any k, sorted by genome index:
        dict(genomes uint32[m], num / den int64[m, nk], ci float64[m, nk], n_intersect, n_kmers, stats)."""
        nk = len(self.db.ks)
        while True:
            g = np.empty(cap_rows, dtype=np.uint32)
            num = np.empty((cap_rows, nk), dtype=np.int64)
            den = np.empty((cap_rows, nk), dtype=np.int64)
            ci = np.empty((cap_rows, nk), dtype=np.float64)
            n = C.c_uint64()
            try:
                ni = self._finish_call(num.ctypes.data, den.ctypes.data, ci.ctypes.data, (g.ctypes.data, cap_rows, C.byref(n)))
                break
            except MlgError:
                if n.value <= cap_rows:
                    raise
                cap_rows = int(n.value)           # more rows than room: the call can simply be repeated
        self._keep = []
        m = n.value
        order = np.argsort(g[:m], kind="stable")
        st = self.stats()
        return dict(genomes=g[:m][order], num=num[:m][order], den=den[:m][order], ci=ci[:m][order], n_intersect=ni,
                    n_kmers=st["n_kmers"], stats=st)

    def finish_sparse_into(self, genomes_ptr: int, num_ptr, den_ptr, ci_ptr, cap_rows: int):
        """finish_sparse() into caller-provided (pinned) host buffers, rows in no particular order; returns (|I|, rows)"""
        n = C.c_uint64()
        ni = self._finish_call(num_ptr, den_ptr, ci_ptr, (genomes_ptr, int(cap_rows), C.byref(n)))
        self._keep = []
        return ni, n.value

    def hit_flags(self, genomes) -> np.ndarray:
        """mlg_query_hit_flags: (m, nk, n) uint8, 1 where the slot is the representative of a hit (genome, k-prefix) class"""
        g = np.ascontiguousarray(genomes, dtype=np.uint32)
        out = np.zeros((g.size, len(self.db.ks), self.db.n), dtype=np.uint8)
        if g.size:
            check(_lib.lib().mlg_query_hit_flags(self._h, g.ctypes.data, g.size, out.ctypes.data))
        return out

    def intersection(self) -> np.ndarray:
        n = C.c_uint64()
        check(_lib.lib().mlg_query_intersection(self._h, None, 0, C.byref(n)))
        out = np.empty((n.value, 2), dtype=np.uint64)
        if n.value:
            check(_lib.lib().mlg_query_intersection(self._h, out.ctypes.data, n.value, C.byref(n)))
        return out

    def dump_intersection(self, dump_path: str, fasta_path: str | None = None, counter_max: int = 3) -> None:
        """mlg_query_dump_intersection: the files `kmc_dump` and the FASTA rewrite leave behind (select_db.py:58-65);
        counter_max = the -cs3 of both KMC runs of the reference"""
        check(_lib.lib().mlg_query_dump_intersection(self._h, dump_path.encode(), fasta_path.encode() if fasta_path else None,
                                                     int(counter_max)))

    def read_kmers(self, min_count: int = 1, counter_max: int = 255):
        """(keys uint64[n, 2] as (hi, lo), ascending; counts uint8[n] saturated at counter_max) of the read k-mers seen
        >= min_count times (needs Database.query(read_kmers=True))"""
        n = C.c_uint64()
        if self._rk_passes:       # the number of records is only known after the passes have run: count them first
            check(_lib.lib().mlg_query_read_kmers(self._h, int(min_count), int(counter_max), None, None, 0, C.byref(n)))
            cap = n.value
        else:
            cap = self.read_kmer_stats()["distinct"]
        keys = np.empty((cap, 2), dtype=np.uint64)
        counts = np.empty(cap, dtype=np.uint8)
        check(_lib.lib().mlg_query_read_kmers(self._h, int(min_count), int(counter_max), keys.ctypes.data, counts.ctypes.data,
                                              cap, C.byref(n)))
        return keys[:n.value], counts[:n.value]

    def write_reads_kmc(self, prefix: str, min_count: int = 2, counter_max: int = 3) -> None:
        """<prefix>.kmc_pre / .kmc_suf: `kmc -k<K> -ci<min_count> -cs<counter_max>` of the pushed reads (select_db.py:50)"""
        check(_lib.lib().mlg_query_write_reads_kmc(self._h, prefix.encode(), int(min_count), int(counter_max)))

    def write_intersection_kmc(self, prefix: str, counter_max: int = 3) -> None:
        """after finish: <prefix>.kmc_pre / .kmc_suf of `kmc_tools simple ... intersect` (select_db.py:54-56)"""
        check(_lib.lib().mlg_query_write_intersection_kmc(self._h, prefix.encode(), int(counter_max)))

    def read_kmer_stats(self) -> dict:
        s = _lib.ReadKmerStats()
        check(_lib.lib().mlg_query_read_kmer_stats(self._h, C.byref(s)))
        return s.as_dict()

    def read_kmer_plan(self) -> dict:
        """mlg_query_read_kmer_plan: passes, refined bins, archive bytes, per-pass cap, largest pass bound, distinct keys and
        event times of the last read_kmers / write_reads_kmc call (needs Database.query(read_kmer_passes=True))"""
        s = _lib.ReadKmerPlan()
        check(_lib.lib().mlg_query_read_kmer_plan(self._h, C.byref(s)))
        return s.as_dict()

    def stats(self) -> dict:
        s = Stats()
        check(_lib.lib().mlg_query_stats(self._h, C.byref(s)))
        return s.as_dict()

    def close(self):
        if self._h:
            _lib.lib().mlg_query_free(self._h)
            self._h = C.c_void_p()
            self._keep = []

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()


class Exchange:
    """One rank's end of the multi-GPU exchange of the per-k-mer counters (mlg_exchange in the header): persistent
    device buffers for `cap_entries` non-zero counters per rank."""

    def __init__(self, ctx: Context, world: int, rank: int, cap_entries: int):
        self.ctx, self.world, self.rank, self.cap = ctx, int(world), int(rank), int(cap_entries)
        self._h = C.c_void_p()
        check(_lib.lib().mlg_exchange_create(ctx._h, self.world, self.rank, self.cap, C.byref(self._h)))
        a, b, w = C.c_void_p(), C.c_void_p(), C.c_uint64()
        check(_lib.lib().mlg_exchange_buffers(self._h, C.byref(a), C.byref(b), C.byref(w)))
        self.send_ptr, self.recv_ptr, self.block_words = a.value, b.value, w.value

    def local_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        check(_lib.lib().mlg_exchange_local_handle(self._h, buf))
        return buf.raw

    def connect(self, handles: bytes):
        if len(handles) != 64 * self.world:
            raise ValueError("need one 64-byte handle per rank")
        check(_lib.lib().mlg_exchange_connect(self._h, handles))

    def close(self):
        if self._h:
            _lib.lib().mlg_exchange_destroy(self._h)
            self._h = C.c_void_p()
