"""ctypes binding of libnohuman_gpu.so (include/nohuman_gpu.h).

This is the same stub a maintainer of the reference would write for its FFI
(see INTEGRATION.md for the Rust `extern "C"` version).  There is no fallback:
if the shared library is missing, importing callers get an ImportError that
says how to build it; if no CUDA device is present every compute call fails
with NH_ERR_CUDA.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# NH_LIB_PATH points experiments at another build of the same library (e.g. other nvcc flags)
LIB_PATH = os.environ.get("NH_LIB_PATH") or os.path.join(_PKG, "libnohuman_gpu.so")

NH_OK = 0
NH_ERR_INVALID = -1
NH_ERR_IO = -2
NH_ERR_CUDA = -3
NH_ERR_UNSUPPORTED = -4
NH_ERR_CAPACITY = -5
NH_ERR_NOMEM = -6

NH_GUNZIP_SHIFT_CANDIDATES = 1  # nh_debug_gunzip flag
# nh_debug_gunzip counts[], in order
GUNZIP_COUNTS = ("windows", "chunks", "repaired", "overflowed", "members", "carried",
                 "ns_find", "ns_decode", "ns_redecode", "ns_window", "ns_resolve")


class NhError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libnohuman_gpu error {code}: {msg}")
        self.code = code
        self.message = msg


class DbInfo(C.Structure):
    _fields_ = [
        ("k", C.c_uint64), ("l", C.c_uint64), ("spaced_seed_mask", C.c_uint64),
        ("toggle_mask", C.c_uint64), ("minimum_acceptable_hash_value", C.c_uint64),
        ("dna_db", C.c_int32), ("revcom_version", C.c_int32),
        ("capacity", C.c_uint64), ("size", C.c_uint64), ("key_bits", C.c_uint64),
        ("value_bits", C.c_uint64), ("node_count", C.c_uint64),
        ("device", C.c_int32), ("replicated_by", C.c_int32),
        ("filter_bytes", C.c_uint64),
    ]


class Params(C.Structure):
    _fields_ = [
        ("confidence", C.c_double), ("minimum_hit_groups", C.c_int32), ("paired", C.c_int32),
        ("keep_human", C.c_int32), ("threads", C.c_int32),
        ("max_batch_bases", C.c_uint64), ("max_batch_seqs", C.c_uint64),
        ("emit_runs", C.c_int32), ("gpu_gzip", C.c_int32),
    ]


class BatchStats(C.Structure):
    _fields_ = [
        ("n_units", C.c_uint64), ("n_classified", C.c_uint64), ("n_unclassified", C.c_uint64),
        ("n_kept", C.c_uint64), ("n_bases", C.c_uint64), ("n_tiles", C.c_uint64),
        ("n_lookups", C.c_uint64),
        ("ms_plan", C.c_float), ("ms_minimizer", C.c_float), ("ms_probe", C.c_float),
        ("ms_score", C.c_float), ("ms_h2d", C.c_float), ("ms_d2h", C.c_float),
        ("gpu_launches", C.c_uint32), ("fused_kernel", C.c_uint32),
        ("n_sector_reads", C.c_uint64),
    ]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_ if f != "reserved"}


class RunStats(C.Structure):
    _fields_ = [
        ("total", C.c_uint64), ("classified", C.c_uint64), ("unclassified", C.c_uint64),
        ("bases", C.c_uint64), ("seconds", C.c_double),
        ("busy_inflate_s", C.c_double), ("busy_parse_s", C.c_double), ("busy_stage_s", C.c_double),
        ("busy_classify_s", C.c_double), ("busy_serialise_s", C.c_double), ("busy_compress_s", C.c_double),
        ("busy_write_s", C.c_double), ("threads_inflate", C.c_int32), ("threads_compress", C.c_int32),
    ]


class Files(C.Structure):
    _fields_ = [
        ("in1", C.c_char_p), ("in2", C.c_char_p), ("out1", C.c_char_p), ("out2", C.c_char_p),
        ("out_format", C.c_int32), ("tag_classified", C.c_int32),
        ("kraken_output", C.c_char_p), ("kraken_report", C.c_char_p),
    ]


class BuildParams(C.Structure):
    _fields_ = [
        ("fasta", C.POINTER(C.c_char_p)), ("n_fasta", C.c_int32),
        ("nodes_dmp", C.c_char_p), ("names_dmp", C.c_char_p), ("seqid2taxid", C.c_char_p),
        ("out_dir", C.c_char_p),
        ("k", C.c_uint32), ("l", C.c_uint32), ("spaces", C.c_uint32),
        ("capacity", C.c_uint64), ("load_factor", C.c_double), ("batch_bases", C.c_uint64),
        ("threads", C.c_int32), ("device", C.c_int32),
    ]


class BuildStats(C.Structure):
    _fields_ = [
        ("sequences", C.c_uint64), ("skipped", C.c_uint64), ("bases", C.c_uint64), ("minimizers", C.c_uint64),
        ("estimate", C.c_uint64), ("estimate_slots", C.c_uint64), ("estimate_rescans", C.c_uint64),
        ("capacity", C.c_uint64), ("size", C.c_uint64), ("node_count", C.c_uint64),
        ("s_taxonomy", C.c_double), ("s_estimate", C.c_double), ("s_insert", C.c_double), ("s_write", C.c_double),
    ]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


NH_DUST_FASTA = 0
NH_DUST_INTERVAL = 1


class DustParams(C.Structure):
    _fields_ = [
        ("in_path", C.c_char_p), ("out_path", C.c_char_p), ("format", C.c_int32), ("window", C.c_int32),
        ("level", C.c_int32), ("threads", C.c_int32), ("device", C.c_int32), ("batch_bases", C.c_uint64),
    ]


class DustStats(C.Structure):
    _fields_ = [
        ("sequences", C.c_uint64), ("bases", C.c_uint64), ("masked", C.c_uint64), ("intervals", C.c_uint64),
        ("seconds", C.c_double),
    ]

    def as_dict(self):
        return {f: getattr(self, f) for f, _ in self._fields_}


# every symbol include/nohuman_gpu.h declares: name -> (restype, argtypes)
_vp, _u64, _i32 = C.c_void_p, C.c_uint64, C.c_int
SYMBOLS = {
    "nh_abi_version": (_i32, []),
    "nh_last_error": (C.c_char_p, []),
    "nh_device_count": (_i32, []),
    "nh_db_open": (_i32, [C.c_char_p, _i32, C.POINTER(_vp)]),
    "nh_db_open_memory": (_i32, [_vp, C.c_size_t, _vp, C.c_size_t, C.POINTER(_u64), _vp, _i32, _i32,
                                 C.POINTER(_vp)]),
    "nh_db_info": (_i32, [_vp, C.POINTER(DbInfo)]),
    "nh_db_open_multi": (_i32, [C.c_char_p, C.POINTER(_i32), _i32, C.POINTER(_vp)]),
    "nh_db_clone": (_i32, [_vp, _i32, C.POINTER(_vp)]),
    "nh_db_device_cells": (_vp, [_vp]),
    "nh_db_close": (None, [_vp]),
    "nh_session_create": (_i32, [_vp, C.POINTER(Params), C.POINTER(_vp)]),
    "nh_session_destroy": (None, [_vp]),
    "nh_classify_batch": (_i32, [_vp, _vp, _vp, _u64, _vp, _vp, C.POINTER(BatchStats)]),
    "nh_classify_batch_device": (_i32, [_vp, _vp, _vp, _u64, _u64, _vp, _vp]),
    "nh_packed_units": (_i32, [_vp, _u64, C.POINTER(_u64)]),
    "nh_pack_reads": (_i32, [_vp, _vp, _u64, _vp, _vp, _vp, _i32]),
    "nh_classify_batch_packed": (_i32, [_vp, _vp, _vp, _vp, _vp, _u64, _vp, _vp, C.POINTER(BatchStats)]),
    "nh_classify_batch_pack": (_i32, [_vp, _vp, _vp, _u64, _i32, _vp, _vp, C.POINTER(BatchStats)]),
    "nh_session_sync": (_i32, [_vp, C.POINTER(BatchStats)]),
    "nh_run_files": (_i32, [_vp, C.POINTER(Files), C.POINTER(RunStats)]),
    "nh_run_files_multi": (_i32, [C.POINTER(_vp), _i32, C.POINTER(Files), C.POINTER(RunStats)]),
    "nh_debug_rewrite_files": (_i32, [C.POINTER(Files), _vp, _vp, _u64, _i32, C.POINTER(RunStats)]),
    "nh_session_stream": (_vp, [_vp]),
    "nh_last_batch_runs": (_i32, [_vp, _u64, _vp, _vp, _vp, _u64, C.POINTER(_u64)]),
    "nh_bgzf_compress": (_i32, [_i32, _vp, C.c_size_t, _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
    "nh_bench_bgzf": (_i32, [_i32, _vp, C.c_size_t, _i32, C.POINTER(C.c_double)]),
    "nh_gunzip": (_i32, [_i32, _vp, C.c_size_t, _vp, C.c_size_t, C.POINTER(C.c_size_t)]),
    "nh_debug_gunzip": (_i32, [_i32, _vp, C.c_size_t, _vp, C.c_size_t, C.POINTER(C.c_size_t), C.c_size_t, C.c_size_t,
                               _i32, C.POINTER(_u64)]),
    "nh_bench_gunzip": (_i32, [_i32, _vp, C.c_size_t, _i32, C.POINTER(C.c_double)]),
    "nh_build_taxonomy": (_i32, [C.c_char_p, C.c_char_p, C.c_char_p, C.c_char_p, C.POINTER(_u64)]),
    "nh_build_db": (_i32, [C.POINTER(BuildParams), C.POINTER(BuildStats)]),
    "nh_dust_mask": (_i32, [_i32, _vp, _vp, _u64, _i32, _i32, _vp]),
    "nh_dust_fasta": (_i32, [C.POINTER(DustParams), C.POINTER(DustStats)]),
    "nh_bench_dust": (_i32, [_i32, _vp, _vp, _u64, _i32, C.POINTER(C.c_double)]),
    "nh_host_alloc": (_vp, [C.c_size_t]),
    "nh_host_free": (None, [_vp]),
    "nh_debug_minimizers": (_i32, [_vp, _vp, _vp, _u64, _vp, _vp, _vp]),
    "nh_debug_probe": (_i32, [_vp, _vp, _u64, _vp]),
    "nh_debug_last_batch": (_i32, [_vp, _vp, _vp, _vp, _u64]),
    "nh_bench_random_gather": (_i32, [_vp, _u64, _i32, C.POINTER(C.c_double)]),
    "nh_bench_probe_pattern": (_i32, [_vp, _i32, _i32, _i32, C.c_double, _u64, C.c_uint32, _i32,
                                      C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

_lib = None


def lib() -> C.CDLL:
    """Load libnohuman_gpu.so or fail loudly (no CPU fallback exists)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m nohuman_b200.build` "
            "(nvcc, sm_100a). nohuman_b200 has no CPU fallback."
        )
    L = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(L, name)  # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != NH_OK:
        raise NhError(rc, (lib().nh_last_error() or b"").decode(errors="replace"))
