"""ctypes binding of libmahout_b200.so (the C ABI declared in include/mahout_b200.h).

There is no fallback of any kind: if the library is missing, or the process has no sm_100
device, every entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libmahout_b200.so")

OK = 0
BAND_PENDING = 1
ERR_BAD_ARG, ERR_CUDA, ERR_OOM, ERR_INEXACT, ERR_RANGE = -1, -2, -3, -4, -5
ERR_NO_DEVICE, ERR_CM_DELTA, ERR_CM_EPSILON, ERR_UNSUPPORTED, ERR_PULL_TIMEOUT = -6, -7, -8, -9, -10
MEM_HOST, MEM_DEVICE = 0, 1
DTYPE_F16, DTYPE_BF16 = 0, 1
PRECISION_TENSOR, PRECISION_RESCORED, PRECISION_CERTIFIED = 0, 1, 2
K_UPDATE, K_NORMALIZE, K_COSINE, K_RESCORE, K_PARSE, K_PREPARE, K_GROUP, K_ROUTE, K_RECOMMEND = 0, 1, 2, 3, 4, 5, 6, 7, 8
OPT_GROUP_MIN_EVENTS, OPT_GROUP_PREFETCH, OPT_MAX_FALLBACK_ROWS = 1, 2, 4
MAX_DEPTH = 32


class NativeError(RuntimeError):
    """A non-zero status from libmahout_b200 that is not an argument error."""

    def __init__(self, code: int, msg: str):
        super().__init__(f"libmahout_b200 error {code}: {msg}")
        self.code = code


class CMException(Exception):
    """AbstractCountMinSketch.CMException (AbstractCountMinSketch.java:21-27)."""


class InexactError(NativeError):
    """An increment / counter cannot be represented exactly by the bank (MB200_ERR_INEXACT/RANGE)."""


i64, i32, f64, vp = C.c_int64, C.c_int32, C.c_double, C.c_void_p

class CosineArgs(C.Structure):
    """struct mb200_cosine_args (include/mahout_b200.h)."""
    _fields_ = [
        ("a_rows", C.c_void_p), ("a_valid", C.c_void_p), ("a_count", C.c_int64),
        ("a_id_mul", C.c_int64), ("a_id_off", C.c_int64),
        ("b_rows", C.c_void_p), ("b_valid", C.c_void_p), ("b_count", C.c_int64),
        ("b_blocks", C.c_int32), ("b_id_mul", C.c_int64), ("b_id_add", C.c_int64),
        ("depth", C.c_int32), ("width", C.c_int32), ("dtype", C.c_int32), ("precision", C.c_int32),
        ("k", C.c_int32), ("threshold", C.c_double), ("exclude_self", C.c_int32), ("block_n", C.c_int32),
        ("a_counters", C.c_void_p), ("b_counters", C.c_void_p),
        ("out_idx", C.c_void_p), ("out_sim", C.c_void_p), ("out_cnt", C.c_void_p),
        ("dense_out", C.c_void_p), ("dense_ld", C.c_int64),
        ("b_counter_blocks", C.c_void_p), ("b_counter_blocks32", C.c_void_p), ("mixed_sign", C.c_int32),
        ("defer_uncertified", C.c_int32),
    ]


class Stats(C.Structure):
    """struct mb200_stats (include/mahout_b200.h)."""
    _fields_ = [("device", C.c_int32), ("num_sms", C.c_int32), ("launches", C.c_int64),
                ("workspace_bytes", C.c_int64), ("staging_bytes", C.c_int64), ("last_fallback_rows", C.c_int64),
                ("cosine_job_active", C.c_int32), ("device_name", C.c_char * 64), ("events_updated", C.c_int64),
                ("rows_scored", C.c_int64), ("fallback_rows_total", C.c_int64), ("band_rows_total", C.c_int64),
                ("h2d_bytes", C.c_int64),
                ("d2h_bytes", C.c_int64)]


class JobParams(C.Structure):
    """struct mb200_job_params (include/mahout_b200.h)."""
    _fields_ = [("k", C.c_int32), ("threshold", C.c_double), ("width", C.c_int32), ("depth", C.c_int32),
                ("seed", C.c_int64), ("hash_a", C.c_void_p), ("hash_b", C.c_void_p), ("frac_bits", C.c_int32),
                ("dtype", C.c_int32), ("precision", C.c_int32)]


class JobStats(C.Structure):
    """struct mb200_job_stats (include/mahout_b200.h)."""
    _fields_ = [("n_gpus", C.c_int32), ("events", C.c_int64), ("rows", C.c_int64), ("similarities_kept", C.c_int64),
                ("fallback_rows", C.c_int64), ("events_busiest_gpu", C.c_int64), ("route_s", C.c_double),
                ("build_s", C.c_double), ("cosine_s", C.c_double)]


class RecommendPlan(C.Structure):
    """struct mb200_recommend_plan (include/mahout_b200.h)."""
    _fields_ = [("stream_users", C.c_int64), ("gather_users", C.c_int64), ("chunks", C.c_int64),
                ("candidates", C.c_int64), ("candidates_max", C.c_int64), ("stream_rows", C.c_int64),
                ("gather_loads", C.c_int64), ("stages", C.c_int32), ("chunk_candidates", C.c_int32)]


class ItemBasedArgs(C.Structure):
    """struct mb200_itembased_args (include/mahout_b200.h)."""
    _fields_ = [("sim_idx", C.c_void_p), ("sim_val", C.c_void_p), ("sim_cnt", C.c_void_p), ("num_items", C.c_int64),
                ("sim_ld", C.c_int32), ("user_ptr", C.c_void_p), ("pref_row", C.c_void_p), ("pref_val", C.c_void_p),
                ("num_users", C.c_int64), ("nnz", C.c_int64), ("item_ids", C.c_void_p), ("allowed", C.c_void_p),
                ("users", C.c_void_p), ("m", C.c_int64), ("how_many", C.c_int32), ("max_prefs_per_user", C.c_int32),
                ("boolean_data", C.c_int32), ("out_item", C.c_void_p), ("out_value", C.c_void_p),
                ("out_cnt", C.c_void_p), ("mem", C.c_int32)]


class ItemBasedPlan(C.Structure):
    """struct mb200_itembased_plan (include/mahout_b200.h)."""
    _fields_ = [("users", C.c_int64), ("smem_users", C.c_int64), ("dense_users", C.c_int64), ("entries", C.c_int64),
                ("entries_max", C.c_int64), ("pruned_users", C.c_int64), ("candidates_max", C.c_int64),
                ("table_slots", C.c_int32), ("dense_slices", C.c_int32)]


class SizedPlan(C.Structure):
    """struct mb200_sized_plan (include/mahout_b200.h)."""
    _fields_ = [("queries", C.c_int64), ("classes", C.c_int64), ("smem_classes", C.c_int64),
                ("global_classes", C.c_int64), ("pair_fmas", C.c_int64), ("batches", C.c_int64), ("items", C.c_int64),
                ("query_tile_max", C.c_int32), ("smem_bytes", C.c_int32)]


class SizedRecommendPlan(C.Structure):
    """struct mb200_sized_recommend_plan (include/mahout_b200.h)."""
    _fields_ = [("users", C.c_int64), ("chunks", C.c_int64), ("candidates", C.c_int64),
                ("candidates_max", C.c_int64), ("stream_visits", C.c_int64), ("row_visits", C.c_int64),
                ("gather_visits", C.c_int64),
                ("too_wide_visits", C.c_int64), ("stream_bytes", C.c_int64), ("gather_loads", C.c_int64),
                ("terms", C.c_int64), ("stages", C.c_int32), ("stage_bytes", C.c_int32),
                ("chunk_candidates", C.c_int32)]


class CosinePiece(C.Structure):
    """struct mb200_cosine_piece (include/mahout_b200.h)."""
    _fields_ = [
        ("b_rows", C.c_void_p), ("b_valid", C.c_void_p), ("b_count", C.c_int64), ("b_blocks", C.c_int32),
        ("b_id_mul", C.c_int64), ("b_id_add", C.c_int64), ("b_id_base", C.c_int64),
        ("ready_flags", C.c_void_p), ("ready_epoch", C.c_uint32), ("first_block", C.c_int32),
    ]


_PROTOS = {
    "mb200_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "mb200_destroy": (C.c_int, [vp]),
    "mb200_last_error": (C.c_char_p, [vp]),
    "mb200_set_stream": (C.c_int, [vp, vp]),
    "mb200_sync": (C.c_int, [vp]),
    "mb200_set_option": (C.c_int, [vp, C.c_int, i64]),
    "mb200_release_workspace": (C.c_int, [vp]),
    "mb200_set_profiling": (C.c_int, [vp, C.c_int]),
    "mb200_kernel_time": (C.c_int, [vp, C.c_int, C.POINTER(f64), C.POINTER(i64)]),
    "mb200_reset_profile": (C.c_int, [vp]),
    "mb200_launch_count": (C.c_int, [vp, C.POINTER(i64)]),
    "mb200_get_stats": (C.c_int, [vp, C.POINTER(Stats)]),
    "mb200_host_alloc": (C.c_int, [i64, C.POINTER(vp)]),
    "mb200_host_free": (C.c_int, [vp]),
    "mb200_host_register": (C.c_int, [vp, i64]),
    "mb200_host_unregister": (C.c_int, [vp]),
    "mb200_hash_params": (C.c_int, [i64, C.c_int, vp, vp]),
    "mb200_cm_dims": (C.c_int, [f64, f64, C.POINTER(i32), C.POINTER(i32)]),
    "mb200_hash_keys": (C.c_int, [vp, i64, i64, i32, vp, i64, vp, C.c_int]),
    "mb200_bank_create": (C.c_int, [vp, i64, i32, i32, i64, i32, C.POINTER(vp)]),
    "mb200_bank_create_params": (C.c_int, [vp, i64, i32, i32, vp, vp, i32, C.POINTER(vp)]),
    "mb200_bank_destroy": (C.c_int, [vp]),
    "mb200_bank_clear": (C.c_int, [vp]),
    "mb200_bank_ipc_handle": (C.c_int, [vp, vp]),
    "mb200_bank_narrow32": (C.c_int, [vp, vp]),
    "mb200_bank_counters": (C.c_int, [vp, C.POINTER(vp), C.POINTER(i64)]),
    "mb200_bank_dump": (C.c_int, [vp, C.c_char_p]),
    "mb200_bank_load": (C.c_int, [vp, C.c_char_p, C.POINTER(vp)]),
    "mb200_bank_update": (C.c_int, [vp, vp, vp, vp, i64, C.c_int]),
    "mb200_bank_update_f64": (C.c_int, [vp, vp, vp, vp, i64, C.c_int]),
    "mb200_bank_update_grouped": (C.c_int, [vp, vp, vp, vp, i64, C.c_int]),
    "mb200_bank_update_u8": (C.c_int, [vp, vp, vp, vp, i64, C.c_int]),
    "mb200_bank_read_i32": (C.c_int, [vp, i64, i64, vp, C.c_int]),
    "mb200_bank_check": (C.c_int, [vp]),
    "mb200_bank_read": (C.c_int, [vp, i64, i64, vp, C.c_int]),
    "mb200_bank_query": (C.c_int, [vp, vp, vp, i64, vp, C.c_int]),
    "mb200_bank_pair_cosine": (C.c_int, [vp, vp, vp, i64, vp, C.c_int]),
    "mb200_bank_cross_cosine": (C.c_int, [vp, vp, vp, vp, i64, vp, C.c_int]),
    "mb200_bank_cosine_topk": (C.c_int, [vp, i32, f64, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int]),
    "mb200_bank_estimate_prefs": (C.c_int, [vp, vp, vp, vp, i64, i32, vp, vp, vp, i64, vp, C.c_int]),
    "mb200_bank_recommend": (C.c_int, [vp, vp, vp, vp, i32, vp, vp, i64, vp, i64, vp, i64, i32, C.c_int, vp, vp, vp,
                                       C.c_int]),
    "mb200_recommend_last_plan": (C.c_int, [vp, C.POINTER(RecommendPlan)]),
    "mb200_recommend_item_based": (C.c_int, [vp, C.POINTER(ItemBasedArgs)]),
    "mb200_itembased_last_plan": (C.c_int, [vp, C.POINTER(ItemBasedPlan)]),
    "mb200_sized_bank_create": (C.c_int, [vp, i64, vp, vp, vp, vp, i32, vp, vp, vp, C.c_int, C.POINTER(vp)]),
    "mb200_sized_bank_destroy": (C.c_int, [vp]),
    "mb200_sized_bank_read": (C.c_int, [vp, i64, vp]),
    "mb200_sized_pair_cosine": (C.c_int, [vp, vp, vp, i64, vp, C.c_int]),
    "mb200_sized_neighborhood": (C.c_int, [vp, vp, i64, i32, f64, vp, vp, vp, C.c_int]),
    "mb200_sized_estimate_prefs": (C.c_int, [vp, vp, vp, vp, i64, i32, vp, vp, vp, i64, vp, C.c_int]),
    "mb200_sized_last_plan": (C.c_int, [vp, C.POINTER(SizedPlan)]),
    "mb200_sized_recommend": (C.c_int, [vp, vp, vp, vp, i32, vp, vp, i64, vp, i64, vp, i64, i32, C.c_int, vp, vp, vp,
                                        C.c_int]),
    "mb200_sized_recommend_last_plan": (C.c_int, [vp, C.POINTER(SizedRecommendPlan)]),
    "mb200_row_ld": (i64, [i32]),
    "mb200_valid_words": (i64, [i64]),
    "mb200_bank_normalize": (C.c_int, [vp, C.c_int, vp, vp]),
    "mb200_bank_sign_info": (C.c_int, [vp, C.POINTER(i32)]),
    "mb200_cosine_topk": (C.c_int, [vp, C.POINTER(CosineArgs)]),
    "mb200_events_parse": (C.c_int, [vp, vp, i64, C.c_int, C.c_int, C.c_float, C.c_int, C.POINTER(vp)]),
    "mb200_events_create": (C.c_int, [vp, vp, vp, vp, i64, C.c_int, C.POINTER(vp)]),
    "mb200_events_count": (C.c_int, [vp, C.POINTER(i64)]),
    "mb200_events_columns": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
    "mb200_events_read": (C.c_int, [vp, vp, vp, vp]),
    "mb200_events_destroy": (C.c_int, [vp]),
    "mb200_id_to_index": (C.c_int, [vp, vp, i64, vp, C.c_int]),
    "mb200_events_prepare": (C.c_int, [vp, i32, C.POINTER(vp)]),
    "mb200_prefs_info": (C.c_int, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
    "mb200_prefs_columns": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
    "mb200_prefs_user_columns": (C.c_int, [vp, C.POINTER(vp)]),
    "mb200_prefs_read": (C.c_int, [vp, vp, vp, vp, vp]),
    "mb200_prefs_tables": (C.c_int, [vp, vp, vp]),
    "mb200_prefs_destroy": (C.c_int, [vp]),
    "mb200_route_count": (C.c_int, [vp, vp, i64, i32, vp]),
    "mb200_route_scatter": (C.c_int, [vp, vp, vp, vp, i64, i32, vp, vp, vp, vp]),
    "mb200_peer_alloc": (C.c_int, [vp, i64, C.POINTER(vp), vp]),
    "mb200_peer_open": (C.c_int, [vp, vp, C.POINTER(vp)]),
    "mb200_peer_close": (C.c_int, [vp, vp]),
    "mb200_peer_free": (C.c_int, [vp, vp]),
    "mb200_gather_pull": (C.c_int, [vp, vp, vp, vp, vp, i32, i32, i64, i64, C.POINTER(vp), C.POINTER(C.c_uint32)]),
    "mb200_gather_wait": (C.c_int, [vp]),
    "mb200_gather_pull_counters": (C.c_int, [vp, vp, vp, i32, i32, i64]),
    "mb200_gather_fence": (C.c_int, [vp]),
    "mb200_cosine_begin": (C.c_int, [vp, C.POINTER(CosineArgs), C.POINTER(vp)]),
    "mb200_cosine_push": (C.c_int, [vp, C.POINTER(CosinePiece)]),
    "mb200_cosine_finish": (C.c_int, [vp, C.POINTER(CosineArgs)]),
    "mb200_cosine_abort": (C.c_int, [vp]),
    "mb200_cosine_last_fallback_rows": (C.c_int, [vp, C.POINTER(i64)]),
    "mb200_cosine_last_band_rows": (C.c_int, [vp, C.POINTER(i64)]),
    "mb200_create_multi": (C.c_int, [i32, vp, C.POINTER(vp)]),
    "mb200_multi_destroy": (C.c_int, [vp]),
    "mb200_multi_gpus": (C.c_int, [vp, C.POINTER(i32)]),
    "mb200_multi_ctx": (C.c_int, [vp, i32, C.POINTER(vp)]),
    "mb200_multi_last_error": (C.c_char_p, [vp]),
    "mb200_job_item_similarity": (C.c_int, [vp, vp, vp, vp, i64, i64, C.POINTER(JobParams), vp, vp, vp, C.POINTER(JobStats)]),
    "mb200_sized_multi_create": (C.c_int, [vp, i64, vp, vp, vp, vp, i32, vp, vp, vp, C.POINTER(vp)]),
    "mb200_sized_multi_destroy": (C.c_int, [vp]),
    "mb200_sized_multi_neighborhood": (C.c_int, [vp, vp, i64, i32, f64, vp, vp, vp]),
    "mb200_sized_multi_recommend": (C.c_int, [vp, vp, i64, i32, f64, vp, vp, i64, vp, i64, i32, C.c_int, vp, vp, vp]),
    "mb200_sized_multi_estimate_prefs": (C.c_int, [vp, vp, vp, i64, i32, f64, vp]),
    "mb200_sized_multi_last_stats": (C.c_int, [vp, vp, vp, C.POINTER(f64)]),
    "mb200_itembased_multi_create": (C.c_int, [vp, vp, vp, vp, i64, i32, vp, vp, vp, i64, i64, vp, C.POINTER(vp)]),
    "mb200_itembased_multi_recommend": (C.c_int, [vp, vp, i64, i32, i32, i32, vp, vp, vp, vp]),
    "mb200_itembased_multi_last_stats": (C.c_int, [vp, vp, vp, C.POINTER(f64)]),
    "mb200_itembased_multi_destroy": (C.c_int, [vp]),
    # bench / test support (mahout_b200/csrc/synth.h)
    "mb200_synth_events": (C.c_int, [vp, C.c_uint64, i64, i64, i64, vp, i64, vp, vp, vp, vp]),
    "mb200_bench_red64": (C.c_int, [vp, i64, i64, C.POINTER(f64), C.POINTER(f64)]),
}

_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m mahout_b200.build` "
                "(nvcc, sm_100a).  mahout_b200 has no CPU or PyTorch fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _PROTOS.items():
            fn = getattr(L, name, None)
            if fn is None:
                continue  # optional symbols are checked by tests/test_abi.py against the header
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def register(name: str, restype, argtypes) -> None:
    _PROTOS[name] = (restype, argtypes)
    if _lib is not None:
        fn = getattr(_lib, name)
        fn.restype = restype
        fn.argtypes = argtypes


def last_error(ctx=None) -> str:
    s = lib().mb200_last_error(ctx)
    return s.decode("utf-8", "replace") if s else ""


def check(rc: int, ctx=None) -> None:
    """Map a status code to the exception the reference would raise at the same place."""
    if rc == OK:
        return
    msg = last_error(ctx)
    if rc == ERR_BAD_ARG:
        raise ValueError(msg)  # IllegalArgumentException (Guava Preconditions)
    if rc in (ERR_CM_DELTA, ERR_CM_EPSILON):
        raise CMException(msg)
    if rc == ERR_OOM:
        raise MemoryError(msg)
    if rc in (ERR_INEXACT, ERR_RANGE):
        raise InexactError(rc, msg)
    raise NativeError(rc, msg)
