"""ctypes binding of libsvsb200.so (include/svsb200.h).  No CPU fallback: a missing library is an error."""
from __future__ import annotations

import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libsvsb200.so")

SVSB_OK = 0
SVSB_E_INVALID = -1
SVSB_E_CUDA = -2
SVSB_E_NOT_LOADED = -3
SVSB_E_SHAPE = -4
SVSB_E_STATE = -5
SVSB_E_NOMEM = -6
SVSB_E_NO_DEVICE = -7

NORM_CHECK = 0
NORM_NORMALIZE = 1

K_FAST_MAX = 2048
PAIRS_DESC_BYTES = 256       # SVSB_PAIRS_DESC_BYTES

c_float_p = C.POINTER(C.c_float)
c_i64_p = C.POINTER(C.c_int64)
c_i32_p = C.POINTER(C.c_int32)
c_u64_p = C.POINTER(C.c_uint64)

# name -> (restype, argtypes); this table is also what tests/test_abi.py checks against the header
SIGNATURES = {
    "svsb_create": (C.c_int, [c_i32_p, C.c_int, C.POINTER(C.c_void_p)]),
    "svsb_destroy": (None, [C.c_void_p]),
    "svsb_load_begin": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32]),
    "svsb_load_rows": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64]),
    "svsb_load_acquire_slab": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), c_i64_p]),
    "svsb_load_commit_slab": (C.c_int, [C.c_void_p, C.c_int64]),
    "svsb_load_end": (C.c_int, [C.c_void_p, c_u64_p]),
    "svsb_load_sqlite": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int32, C.c_int32, c_u64_p, c_i64_p, c_i32_p]),
    "svsb_sqlite_available": (C.c_int, []),
    "svsb_sqlite_read": (C.c_int, [C.c_char_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, c_i64_p, c_i32_p]),
    "svsb_load_abort": (C.c_int, [C.c_void_p]),
    "svsb_load_synthetic": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_uint64, C.c_int64, C.c_int64, c_u64_p]),
    "svsb_invalidate": (C.c_int, [C.c_void_p]),
    "svsb_is_loaded": (C.c_int, [C.c_void_p]),
    "svsb_shape": (C.c_int, [C.c_void_p, c_i64_p, c_i32_p]),
    "svsb_norm_stats": (C.c_int, [C.c_void_p, c_float_p, c_i64_p]),
    "svsb_read_rows": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p]),
    "svsb_query": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, c_i32_p]),
    "svsb_query_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.POINTER(C.c_void_p)]),
    "svsb_query_wait": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, c_i32_p]),
    "svsb_apply_mutations": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, c_u64_p]),
    "svsb_generation_rows": (C.c_int, [C.c_void_p, c_i64_p, c_i64_p]),
    "svsb_snapshot_rows": (C.c_int, [C.c_void_p, c_i64_p, c_i64_p]),
    "svsb_snapshot_acquire": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "svsb_snapshot_release": (None, [C.c_void_p]),
    "svsb_snapshot_shape": (C.c_int, [C.c_void_p, c_i64_p, c_i32_p, c_u64_p]),
    "svsb_snapshot_query": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, c_i32_p]),
    "svsb_query_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "svsb_snapshot_query_batch": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                            C.c_void_p]),
    "svsb_top_pairs": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, c_i64_p]),
    "svsb_snapshot_top_pairs": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, c_i64_p]),
    "svsb_topk_scores": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, c_i32_p]),
    "svsb_bench_set_queries": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32]),
    "svsb_bench_run": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, c_float_p, c_float_p, c_i64_p]),
    "svsb_bench_run_batch": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, c_float_p, c_float_p, c_i64_p]),
    "svsb_bench_batch_result": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, c_i32_p, c_i32_p]),
    "svsb_batch_stats": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "svsb_bench_filter_stats": (C.c_int, [C.c_void_p, c_i32_p, c_i64_p]),
    "svsb_bench_filter_route": (C.c_int, [C.c_void_p, c_i32_p]),
    "svsb_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "svsb_host_free": (C.c_int, [C.c_void_p]),
    "svsb_batch_threshold_mode": (C.c_int, [C.c_void_p]),
    "svsb_debug_select_phases": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, c_u64_p]),
    "svsb_bench_last_result": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, c_i32_p]),
    "svsb_set_shard": (C.c_int, [C.c_void_p, C.c_int64]),
    "svsb_xchg_create": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "svsb_xchg_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "svsb_xchg_connect_local": (C.c_int, [C.c_void_p, C.c_void_p]),
    "svsb_xchg_disconnect": (C.c_int, [C.c_void_p]),
    "svsb_enqueue_query_peer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "svsb_query_peer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, c_i32_p]),
    "svsb_query_peer_submit": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, c_i32_p]),
    "svsb_query_peer_wait": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, c_i32_p]),
    "svsb_xchg_read_stamps": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "svsb_enqueue_local_topk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32]),
    "svsb_batch_local_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, c_i32_p]),
    "svsb_batch_global_probe": (C.c_int, [C.c_void_p, C.c_int32, c_i32_p, c_i64_p, c_i64_p, c_float_p]),
    "svsb_batch_sample_tops": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_void_p]),
    "svsb_batch_global_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_int32,
                                            C.c_int32, C.c_void_p]),
    "svsb_enqueue_merge_batch_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                                   C.c_void_p, C.c_void_p, C.c_void_p]),
    "svsb_bxchg_create": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "svsb_bxchg_connect": (C.c_int, [C.c_void_p, C.c_void_p]),
    "svsb_bxchg_connect_local": (C.c_int, [C.c_void_p, C.c_void_p]),
    "svsb_bxchg_disconnect": (C.c_int, [C.c_void_p]),
    "svsb_batch_peer_prepare": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32]),
    "svsb_batch_peer": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_float, C.c_int32, C.c_int32,
                                  C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32]),
    "svsb_batch_peer_flush": (C.c_int, [C.c_void_p, C.c_void_p]),
    "svsb_enqueue_join": (C.c_int, [C.c_void_p, C.c_void_p]),
    "svsb_enqueue_merge_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                             C.c_void_p, C.c_void_p, C.c_void_p]),
    "svsb_enqueue_merge_sorted_records": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32,
                                                    C.c_void_p, C.c_void_p, C.c_void_p]),
    "svsb_pairs_export": (C.c_int, [C.c_void_p, c_float_p, c_i64_p, C.c_void_p]),
    "svsb_pairs_connect": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "svsb_pairs_connect_local": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "svsb_pairs_local": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_float, C.c_void_p, C.c_void_p, C.c_void_p, c_i64_p]),
    "svsb_pairs_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int64,
                                   C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "svsb_pairs_disconnect": (C.c_int, [C.c_void_p]),
    "svsb_kernel_time_collect": (C.c_int, [C.c_void_p, c_float_p]),
    "svsb_ws_create": (C.c_int, [C.c_int, C.c_int64, C.c_int32, C.POINTER(C.c_void_p)]),
    "svsb_ws_destroy": (None, [C.c_void_p]),
    "svsb_launch_local_topk": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32,
                                         C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "svsb_launch_merge": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                    C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "svsb_last_error": (C.c_char_p, []),
    "svsb_version": (C.c_char_p, []),
    "svsb_launch_count": (C.c_int64, []),
}

_lib = None
_lock = threading.Lock()


class EngineError(RuntimeError):
    """A call into libsvsb200.so failed (CUDA error, bad state, no device ...)."""

    def __init__(self, code: int, message: str):
        super().__init__(f"svs_b200 error {code}: {message}")
        self.code = code
        self.message = message


def load() -> C.CDLL:
    """Load the shared library, binding every symbol of the header.  Raises if it is not built."""
    global _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m svs_b200.build` "
                "(svs_b200 has no CPU fallback and no pure-Python path)")
        lib = C.CDLL(LIB_PATH)
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(lib, name)         # AttributeError if the symbol is not exported
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = lib
        return lib


def last_error() -> str:
    msg = load().svsb_last_error()
    return msg.decode("utf-8", "replace") if msg else ""


def check(rc: int) -> None:
    """Map the C ABI's error convention onto Python exceptions.

    SVSB_E_SHAPE -> ValueError, exactly what np.dot raises in the reference for a D mismatch or an
    empty matrix (src/svs/kb.py:1623); everything else -> EngineError.
    """
    if rc == SVSB_OK:
        return
    msg = last_error()
    if rc == SVSB_E_SHAPE:
        raise ValueError(msg)
    raise EngineError(rc, msg)
