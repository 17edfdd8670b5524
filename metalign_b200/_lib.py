"""ctypes loader for libmetalign_b200.so (the C ABI in include/metalign_b200.h).

There is no CPU fallback: if the library is missing it is built with nvcc, and if that fails, or no
CUDA device is present at call time, the caller gets an exception.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MLG_LIB_PATH") or os.path.join(_HERE, "libmetalign_b200.so")   # MLG_LIB_PATH: experiment builds
_LIB = None


MLG_ERR_NOMEM = -5
MLG_ERR_RETRY = -6


class MlgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__("metalign_b200 error %d: %s" % (code, msg))
        self.code = code


class Stats(C.Structure):
    _fields_ = [("n_reads", C.c_uint64), ("n_bases", C.c_uint64), ("n_kmers", C.c_uint64),
                ("n_intersect", C.c_uint64), ("n_db_entries", C.c_uint64), ("n_db_distinct", C.c_uint64),
                ("n_buckets", C.c_uint64), ("bucket_bytes", C.c_uint32), ("gpu_launches", C.c_uint32),
                ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64), ("ms_probe", C.c_double),
                ("ms_query", C.c_double), ("probe_launches", C.c_uint32), ("filter_words", C.c_uint32),
                ("n_bucket_fetches", C.c_uint64), ("layout", C.c_uint32), ("reserved", C.c_uint32)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class ReadKmerStats(C.Structure):
    _fields_ = [("windows", C.c_uint64), ("distinct", C.c_uint64), ("slots", C.c_uint64), ("bytes", C.c_uint64),
                ("bytes_needed", C.c_uint64), ("grows", C.c_uint32), ("overflowed", C.c_uint32), ("ms_count", C.c_double),
                ("ms_rehash", C.c_double), ("out_records", C.c_uint64), ("out_bytes", C.c_uint64), ("ms_compact", C.c_double),
                ("ms_sort", C.c_double), ("ms_encode", C.c_double), ("s_write", C.c_double)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class ReadKmerPlan(C.Structure):
    _fields_ = [("passes", C.c_uint32), ("refined_bins", C.c_uint32), ("archive_bytes", C.c_uint64), ("pass_cap_bytes", C.c_uint64),
                ("max_pass_bound", C.c_uint64), ("distinct", C.c_uint64), ("ms_histogram", C.c_double), ("ms_count", C.c_double),
                ("ms_output", C.c_double), ("rank", C.c_uint32), ("world", C.c_uint32), ("peers_added", C.c_uint32),
                ("reserved", C.c_uint32), ("share_first_bin", C.c_uint64), ("share_end_bin", C.c_uint64), ("share_windows", C.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


def build(force: bool = False) -> str:
    """Compile the CUDA sources for sm_100a (nvcc cross-compiles without a GPU)."""
    src_dir = os.path.join(_HERE, "csrc")
    srcs = [os.path.join(src_dir, f) for f in os.listdir(src_dir) if f.endswith((".cu", ".cuh", ".h"))]
    srcs.append(os.path.join(_HERE, "..", "include", "metalign_b200.h"))
    stale = (not os.path.exists(LIB_PATH)) or os.path.getmtime(LIB_PATH) < max(os.path.getmtime(s) for s in srcs)
    if (force or stale) and not os.environ.get("MLG_LIB_PATH"):
        subprocess.check_call(["make", "-C", src_dir, "-s"])
    return LIB_PATH


# every exported symbol of include/metalign_b200.h: name -> (restype, argtypes)
_vp, _u8p, _u32p, _u64p, _i64p, _f64p = (C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p)
_pp = C.POINTER(C.c_void_p)
SIGNATURES = {
    "mlg_last_error": (C.c_char_p, []),
    "mlg_version": (C.c_int, []),
    "mlg_ctx_create": (C.c_int, [C.c_int, _pp]),
    "mlg_ctx_destroy": (C.c_int, [_vp]),
    "mlg_ctx_streams": (C.c_int, [_vp, _pp, _pp]),
    "mlg_host_alloc": (C.c_int, [_pp, C.c_uint64]),
    "mlg_host_free": (C.c_int, [_vp]),
    "mlg_device_memory": (C.c_int, [C.c_int, _u64p, _u64p]),
    "mlg_db_from_keys": (C.c_int, [_vp, _u64p, C.c_uint32, C.c_uint32, C.c_uint32, _u32p, C.c_uint32, _pp]),
    "mlg_db_from_keys_device": (C.c_int, [_vp, _u64p, C.c_uint32, C.c_uint32, C.c_uint32, _u32p, C.c_uint32, _pp]),
    "mlg_db_builder_create": (C.c_int, [_vp, C.c_uint32, C.c_uint32, C.c_uint32, _u32p, C.c_uint32, _pp]),
    "mlg_db_builder_add_device": (C.c_int, [_vp, _u64p, C.c_uint32, C.c_uint32]),
    "mlg_db_builder_finish": (C.c_int, [_vp, _pp]),
    "mlg_db_builder_destroy": (C.c_int, [_vp]),
    "mlg_db_from_ascii": (C.c_int, [_vp, C.c_char_p, C.c_uint32, C.c_uint32, C.c_uint32, _u32p, C.c_uint32, _pp]),
    "mlg_db_load": (C.c_int, [_vp, C.c_char_p, _pp]),
    "mlg_db_save": (C.c_int, [_vp, C.c_char_p, C.c_char_p, C.c_uint64]),
    "mlg_db_info": (C.c_int, [_vp] + [C.POINTER(C.c_uint32)] * 4 + [C.POINTER(C.c_uint32 * 8)] + [C.POINTER(C.c_uint64)] * 2),
    "mlg_db_denominators": (C.c_int, [_vp, C.c_int, _i64p]),
    "mlg_db_free": (C.c_int, [_vp]),
    "mlg_query_begin": (C.c_int, [_vp, _vp, C.c_int, C.c_int, C.c_int, _pp]),
    "mlg_query_push_packed": (C.c_int, [_vp, _u8p, _u8p, _u64p, C.c_uint64, C.c_uint32]),
    "mlg_query_push_packed_nruns": (C.c_int, [_vp, _u8p, _u32p, C.c_uint64, _u64p, C.c_uint64, C.c_uint32]),
    "mlg_query_push_packed_device": (C.c_int, [_vp, _u8p, _u8p, _u64p, C.c_uint64, C.c_uint32]),
    "mlg_query_push_ascii": (C.c_int, [_vp, _vp, _u64p, C.c_uint64]),
    "mlg_query_sync": (C.c_int, [_vp]),
    "mlg_query_counts_export": (C.c_int, [_vp, _pp, C.POINTER(C.c_uint64)]),
    "mlg_query_counts_import": (C.c_int, [_vp]),
    "mlg_query_counts_export_sparse": (C.c_int, [_vp, _pp, C.POINTER(C.c_uint64)]),
    "mlg_query_counts_merge_sparse": (C.c_int, [_vp, _u64p, C.c_uint64]),
    "mlg_exchange_create": (C.c_int, [_vp, C.c_uint32, C.c_uint32, C.c_uint64, _pp]),
    "mlg_exchange_destroy": (C.c_int, [_vp]),
    "mlg_exchange_buffers": (C.c_int, [_vp, _pp, _pp, C.POINTER(C.c_uint64)]),
    "mlg_exchange_local_handle": (C.c_int, [_vp, _vp]),
    "mlg_exchange_connect": (C.c_int, [_vp, _vp]),
    "mlg_query_exchange_pack": (C.c_int, [_vp, _vp]),
    "mlg_query_exchange_merge": (C.c_int, [_vp, _vp]),
    "mlg_query_exchange_p2p": (C.c_int, [_vp, _vp]),
    "mlg_query_exchange_dense": (C.c_int, [_vp, _pp, C.POINTER(C.c_uint64)]),
    "mlg_query_set_exchange_clamp": (C.c_int, [_vp, C.c_int]),
    "mlg_query_finish": (C.c_int, [_vp, _i64p, _i64p, _f64p, C.POINTER(C.c_uint64)]),
    "mlg_query_finish_sparse": (C.c_int, [_vp, _u32p, _i64p, _i64p, _f64p, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]),
    "mlg_query_hit_flags": (C.c_int, [_vp, _u32p, C.c_uint32, _u8p]),
    "mlg_query_intersection": (C.c_int, [_vp, _u64p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "mlg_query_dump_intersection": (C.c_int, [_vp, C.c_char_p, C.c_char_p, C.c_uint32]),
    "mlg_query_stats": (C.c_int, [_vp, C.POINTER(Stats)]),
    "mlg_query_enable_read_kmers": (C.c_int, [_vp, C.c_uint64]),
    "mlg_query_read_kmers": (C.c_int, [_vp, C.c_uint32, C.c_uint32, _u64p, _u8p, C.c_uint64, C.POINTER(C.c_uint64)]),
    "mlg_query_write_reads_kmc": (C.c_int, [_vp, C.c_char_p, C.c_uint32, C.c_uint32]),
    "mlg_query_write_intersection_kmc": (C.c_int, [_vp, C.c_char_p, C.c_uint32]),
    "mlg_query_read_kmer_stats": (C.c_int, [_vp, C.POINTER(ReadKmerStats)]),
    "mlg_query_enable_read_kmer_passes": (C.c_int, [_vp, C.c_uint64]),
    "mlg_query_read_kmer_plan": (C.c_int, [_vp, C.POINTER(ReadKmerPlan)]),
    "mlg_query_read_kmer_archive": (C.c_int, [_vp, C.c_uint32, C.c_uint32, _pp, C.POINTER(C.c_uint64)]),
    "mlg_query_read_kmer_add_archive": (C.c_int, [_vp, _vp, C.c_uint64]),
    "mlg_kmc_concat": (C.c_int, [C.c_char_p, C.POINTER(C.c_char_p), C.c_uint32]),
    "mlg_query_free": (C.c_int, [_vp]),
    "mlg_sketch_genomes": (C.c_int, [_vp, _vp, _u64p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint64, _u64p, _u32p, _vp, _vp]),
    "mlg_db_builder_add_fasta": (C.c_int, [_vp, _vp, _u64p, C.c_uint32, C.c_uint64, _vp]),
}


class SketchStats(C.Structure):
    _fields_ = [("n_windows", C.c_uint64), ("n_candidates", C.c_uint64), ("ms_kernels", C.c_double), ("passes", C.c_uint32),
                ("reserved", C.c_uint32)]


class FastaStats(C.Structure):
    _fields_ = [("files", C.c_uint64), ("file_bytes", C.c_uint64), ("text_bytes", C.c_uint64), ("n_windows", C.c_uint64),
                ("n_candidates", C.c_uint64), ("passes", C.c_uint32), ("reserved", C.c_uint32), ("ms_h2d", C.c_double),
                ("ms_cut", C.c_double), ("ms_sketch", C.c_double), ("ms_keys", C.c_double)]


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)   # AttributeError here == header and library disagree
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


def check(code: int):
    if code != 0:
        raise MlgError(code, lib().mlg_last_error().decode(errors="replace"))
