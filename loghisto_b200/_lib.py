"""ctypes loader for libloghisto_b200.so (the C ABI in include/loghisto_b200.h).

There is no CPU fallback: if the shared library is missing it is built with
nvcc; if that is impossible, or no CUDA device is present when a context is
created, the error is raised to the caller.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

LIB_PATH = _build.LIB

LH_OK = 0
LH_ERR_INVALID = -1
LH_ERR_CUDA = -2
LH_ERR_NOMEM = -3
LH_ERR_NO_DEVICE = -4
LH_ERR_STATE = -5
LH_ERR_RANGE = -6
LH_MAX_PERCENTILES = 32


class lh_config(C.Structure):
    _fields_ = [
        ("struct_size", C.c_uint32), ("device", C.c_int32),
        ("max_histograms", C.c_uint32), ("max_counters", C.c_uint32),
        ("staging_bytes", C.c_uint64), ("staging_slots", C.c_uint32), ("flags", C.c_uint32),
        ("precision", C.c_uint32), ("reserved", C.c_uint32 * 3),
    ]


class lh_staging(C.Structure):
    _fields_ = [("host", C.c_void_p), ("bytes", C.c_uint64), ("slot", C.c_uint32), ("reserved", C.c_uint32)]


class lh_device_view(C.Structure):
    _fields_ = [
        ("d_buckets", C.c_void_p), ("d_counters", C.c_void_p),
        ("n_bucket_words", C.c_uint64), ("n_counter_words", C.c_uint64), ("stream", C.c_void_p),
        ("d_flags", C.c_void_p), ("n_flag_words", C.c_uint64),
    ]


LH_PEER_HANDLE_BYTES = 1024


class lh_comm_stats(C.Structure):
    _fields_ = [
        ("rank", C.c_uint32), ("world", C.c_uint32), ("status", C.c_uint32), ("reserved", C.c_uint32),
        ("allreduces", C.c_uint64), ("last_bytes_from_peers", C.c_uint64),
    ]


class lh_sparse(C.Structure):
    _fields_ = [
        ("offsets", C.POINTER(C.c_uint32)), ("keys", C.POINTER(C.c_int16)),
        ("counts", C.POINTER(C.c_uint64)), ("counter_deltas", C.POINTER(C.c_uint64)),
        ("total_entries", C.c_uint64),
    ]


class lh_window_stats(C.Structure):
    _fields_ = [
        ("intervals", C.c_uint32), ("held", C.c_uint32), ("folds", C.c_uint64),
        ("entries_held", C.c_uint64), ("device_bytes", C.c_uint64),
    ]


LH_MAX_WINDOW_INTERVALS = 1024


class lh_stats(C.Structure):
    _fields_ = [
        ("samples", C.c_uint64), ("counter_ops", C.c_uint64), ("dropped", C.c_uint64),
        ("kernel_launches", C.c_uint64), ("h2d_bytes", C.c_uint64), ("d2h_bytes", C.c_uint64),
        ("snapshots", C.c_uint64),
    ]


_vp, _sz, _u32, _u64, _i32 = C.c_void_p, C.c_size_t, C.c_uint32, C.c_uint64, C.c_int32

# name -> (restype, argtypes); every symbol include/loghisto_b200.h declares
SIGNATURES = {
    "lh_create": (_i32, [C.POINTER(lh_config), C.POINTER(_vp)]),
    "lh_destroy": (_i32, [_vp]),
    "lh_strerror": (C.c_char_p, [_i32]),
    "lh_last_error": (C.c_char_p, [_vp]),
    "lh_abi_version": (_u32, []),
    "lh_ingest_f64": (_i32, [_vp, _u32, _vp, _sz, _vp]),
    "lh_ingest_keyed_f64_u16": (_i32, [_vp, _vp, _vp, _sz, _vp]),
    "lh_ingest_keyed_f64_u32": (_i32, [_vp, _vp, _vp, _sz, _vp]),
    "lh_ingest_keyed_i64ns_u16": (_i32, [_vp, _vp, _vp, _sz, _vp]),
    "lh_ingest_keyed_pair_u16": (_i32, [_vp, _vp, _vp, _sz, _vp, _vp, _sz, _vp]),
    "lh_counter_add_u16": (_i32, [_vp, _vp, _vp, _sz, _vp]),
    "lh_counter_add_u32": (_i32, [_vp, _vp, _vp, _sz, _vp]),
    "lh_ingest_f64_host": (_i32, [_vp, _u32, _vp, _sz]),
    "lh_ingest_keyed_f64_u16_host": (_i32, [_vp, _vp, _vp, _sz]),
    "lh_ingest_keyed_i64ns_u16_host": (_i32, [_vp, _vp, _vp, _sz]),
    "lh_counter_add_u16_host": (_i32, [_vp, _vp, _vp, _sz]),
    "lh_merge_counts_host": (_i32, [_vp, _vp, _vp, _vp, _sz]),
    "lh_staging_acquire": (_i32, [_vp, C.POINTER(lh_staging)]),
    "lh_staging_commit_f64": (_i32, [_vp, C.POINTER(lh_staging), _u32, _sz]),
    "lh_staging_commit_keyed_f64_u16": (_i32, [_vp, C.POINTER(lh_staging), _sz, _u64]),
    "lh_staging_commit_counter_u16": (_i32, [_vp, C.POINTER(lh_staging), _sz, _u64]),
    "lh_staging_abandon": (_i32, [_vp, C.POINTER(lh_staging)]),
    "lh_snapshot_begin": (_i32, [_vp]),
    "lh_snapshot_device": (_i32, [_vp, C.POINTER(lh_device_view)]),
    "lh_snapshot_reduce": (_i32, [_vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp]),
    "lh_snapshot_reduce_async": (_i32, [_vp, _vp, _u32, C.POINTER(_u64)]),
    "lh_snapshot_result": (_i32, [_vp, _u64, _vp, _vp, _vp, _vp, _vp]),
    "lh_snapshot_export": (_i32, [_vp, C.POINTER(lh_sparse)]),
    "lh_snapshot_copy_histogram": (_i32, [_vp, _u32, _vp]),
    "lh_snapshot_end": (_i32, [_vp]),
    "lh_comm_export": (_i32, [_vp, _vp]),
    "lh_comm_import": (_i32, [_vp, _u32, _u32, _vp]),
    "lh_snapshot_allreduce": (_i32, [_vp, _u32, C.POINTER(_u64)]),
    "lh_comm_allreduce_ms": (_i32, [_vp, _u64, C.POINTER(C.c_float)]),
    "lh_comm_info": (_i32, [_vp, C.POINTER(lh_comm_stats)]),
    "lh_window_configure": (_i32, [_vp, _u32]),
    "lh_window_release": (_i32, [_vp]),
    "lh_window_fold": (_i32, [_vp]),
    "lh_window_reduce": (_i32, [_vp, _vp, _u32, _vp, _vp, _vp, _vp, _vp]),
    "lh_window_export": (_i32, [_vp, C.POINTER(lh_sparse)]),
    "lh_window_info": (_i32, [_vp, C.POINTER(lh_window_stats)]),
    "lh_keyed_kernel_name": (C.c_char_p, [_vp]),
    "lh_compress_f64": (_i32, [_vp, _vp, _sz, _vp, C.c_int, _vp]),
    "lh_decompress_table": (_i32, [_vp, _vp]),
    "lh_fastpath_margin": (_i32, [_vp, _vp, _sz, C.POINTER(C.c_double), C.POINTER(_u64), _vp]),
    "lh_fastpath_margin_detail": (_i32, [_vp, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
    "lh_gen_stream_f64": (_i32, [_vp, C.c_int, _u64, _u64, _sz, _vp, _vp]),
    "lh_gen_ids_u16": (_i32, [_vp, C.c_int, _u64, _u64, _sz, _u32, _vp, _vp]),
    "lh_get_stats": (_i32, [_vp, C.POINTER(lh_stats)]),
    "lh_sync": (_i32, [_vp]),
    "lh_ingest_stream": (_vp, [_vp]),
    "lh_device_alloc": (_i32, [_vp, _sz, C.POINTER(_vp)]),
    "lh_device_free": (_i32, [_vp, _vp]),
    "lh_host_alloc_pinned": (_i32, [_vp, _sz, C.POINTER(_vp)]),
    "lh_host_free_pinned": (_i32, [_vp, _vp]),
    "lh_memcpy_h2d": (_i32, [_vp, _vp, _vp, _sz]),
    "lh_memcpy_d2h": (_i32, [_vp, _vp, _vp, _sz]),
    "lh_tune": (_i32, [_vp, C.c_char_p, C.c_int64]),
    "lh_k1_variant_count": (_i32, []),
    "lh_k1_variant_current": (_i32, [_vp]),
    "lh_k1_variant_name": (C.c_char_p, [_vp, _i32]),
    "lh_last_kernel_ms": (_i32, [_vp, C.POINTER(C.c_float)]),
    "lh_ingest_seq": (_u64, [_vp]),
    "lh_kernel_ms": (_i32, [_vp, _u64, C.POINTER(C.c_float)]),
}

_lib = None


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load (building first when stale/missing) the CUDA library.  Raises on failure."""
    global _lib
    if _lib is not None:
        return _lib
    if build_if_missing and _build.needs_build():
        _build.build()
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the loghisto_b200 hot path is CUDA-only and has no CPU fallback; "
            "run `python -m loghisto_b200.build`")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)   # AttributeError if the ABI and the binding drift apart
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
