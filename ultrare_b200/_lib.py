"""ctypes binding of libultrare_b200.so (include/ultrare_b200.h).

There is NO fallback: if the shared library is missing and cannot be built, or a
call fails, a RuntimeError is raised.  Nothing here imports the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libultrare_b200.so")

URE_MAX_SHARDS = 256
URE_TOP_K = 10
URE_COMBINE_MAX_MODELS = 64
URE_COMBINE_GRAM_CTAS = 128

_p = C.c_void_p
_i32, _i64, _f32, _f64 = C.c_int32, C.c_int64, C.c_float, C.c_double


class MFShard(C.Structure):
    """ure_mf_shard_t"""
    _fields_ = [("inter", _p), ("perm", _p), ("P", _p), ("Q", _p), ("bufP", _p), ("bufQ", _p),
                ("gP", _p), ("gQ", _p), ("sse", _p), ("lastP", _p), ("lastQ", _p), ("touched", _p),
                ("inter_u", _p), ("inter_i", _p), ("off_u", _p), ("off_i", _p), ("perm_inv", _p),
                ("tmp_u", _p), ("tmp_i", _p),
                ("n", _i32), ("n_user", _i32), ("n_item", _i32), ("shard_id", _i32),
                ("perm_seed", C.c_uint32), ("group", _i32)]


class MFHParams(C.Structure):
    """ure_mf_hparams_t"""
    _fields_ = [("d", _i32), ("batch", _i32), ("lr0", _f32), ("lr_decay", _f32), ("lr_step", _i32),
                ("weight_decay", _f32), ("momentum", _f32), ("mode", _i32), ("decay", _p), ("decay_len", _i32),
                ("owner_cap_rows", _i32), ("owner_cap_slots", _i32), ("owner_flags", _i32),
                ("owner_spe_cap", _i32), ("owner_sched_rows", _i32), ("owner_sched", _p), ("owner_sched_off", _p),
                ("owner_sched_step0", _i64), ("owner_sched_stride", _i64),
                ("owner_cap_list", _i32), ("owner_max_n", _i32),
                ("runs", _p), ("runs_rows", _i32), ("runs_spe_cap", _i32), ("runs_step0", _i64), ("owner_plan", _p)]


class MFRuns(C.Structure):
    """ure_mf_runs_t"""
    _fields_ = [(nm, _p) for nm in ("slotP", "slotQ", "metaP", "metaQ", "list_u", "list_i", "loff_u", "loff_i")]


class EvalJob(C.Structure):
    """ure_eval_job_t"""
    _fields_ = [("P", _p), ("Q", _p), ("inter", _p), ("order", _p), ("seg", _p), ("score", _p), ("out", _p),
                ("n", _i64), ("n_seg", _i64), ("n_models", _i32), ("denom", _f32)]


class MFBatchShard(C.Structure):
    """ure_mf_batch_shard_t"""
    _fields_ = [("inter", _p), ("perm", _p), ("n", _i32), ("n_user", _i32), ("shard_id", _i32), ("group", _i32)]


class MFBatchLayout(C.Structure):
    """ure_mf_batch_layout_t"""
    _fields_ = [(nm, _i64) for nm in ("total", "table", "ws", "W", "Z", "sse", "zero_end", "rec", "off", "radix",
                                       "perm_inv", "sched", "sched_off", "rows_total", "n_total", "sched_stride")] + \
               [(nm, _i32) for nm in ("spe_cap", "max_rows", "max_n", "grid", "owner", "sched_rows")]


MF_DENSE, MF_LAZY, MF_OWNER, MF_RUNS = 0, 1, 2, 3

assert C.sizeof(MFShard) == 176 and C.sizeof(MFHParams) == 136 and C.sizeof(MFRuns) == 64
assert C.sizeof(MFBatchShard) == 32 and C.sizeof(MFBatchLayout) == 152

# name -> (restype, argtypes); every symbol include/ultrare_b200.h declares
SIGNATURES = {
    "ure_last_error": (C.c_char_p, []),
    "ure_abi_version": (C.c_int, []),
    "ure_mf_train_workspace_bytes": (_i64, []),
    "ure_mf_train": (C.c_int, [_p, C.c_int, C.POINTER(MFHParams), C.c_int, _i64, _i64, C.c_int, _p, _p]),
    "ure_mf_owner_radix_bytes": (_i64, [C.c_int]),
    "ure_mf_owner_prepare": (C.c_int, [_p, C.c_int, C.POINTER(MFHParams), C.c_int, C.c_int, _p, _p, _p]),
    "ure_mf_owner_smem_bytes": (_i64, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int]),
    "ure_mf_owner_schedule": (C.c_int, [_p, C.c_int, C.POINTER(MFHParams), C.c_int, _i64, _p]),
    "ure_mf_batch_layout": (C.c_int, [C.POINTER(MFBatchShard), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, _i64,
                                       C.POINTER(MFBatchLayout)]),
    "ure_mf_batch_setup": (C.c_int, [C.POINTER(MFBatchShard), C.c_int, C.c_int, C.POINTER(MFHParams), C.c_int, C.c_uint32,
                                      _p, C.POINTER(MFBatchLayout), _p, C.c_int, _p]),
    "ure_mf_batch_plan": (C.c_int, [_p, C.c_int, C.POINTER(MFHParams), _p, C.POINTER(MFBatchLayout), C.c_int, C.c_int,
                                     C.c_int, _p]),
    "ure_mf_runs_scratch_bytes": (_i64, [C.c_int, _i64, C.c_int, C.c_int]),
    "ure_mf_runs_init": (C.c_int, [_p, C.c_int, C.POINTER(MFHParams), _p]),
    "ure_mf_runs_schedule": (C.c_int, [_p, C.c_int, C.POINTER(MFHParams), C.c_int, _i64, _i64, _p, _p]),
    "ure_mf_runs_flush": (C.c_int, [_p, C.c_int, C.POINTER(MFHParams), C.c_int, _i64, _p]),
    "ure_mf_train_trace": (C.c_int, [_p, _p, C.c_int, _p]),
    "ure_mf_grid_size": (C.c_int, []),
    "ure_copy_to_host_async": (C.c_int, [_p, _p, _i64, _p]),
    "ure_copy_to_device_async": (C.c_int, [_p, _p, _i64, _p]),
    "ure_mf_debug_flags": (C.c_int, [_p, C.c_uint32, _p]),
    "ure_mf_flush": (C.c_int, [C.POINTER(MFShard), C.c_int, C.POINTER(MFHParams), C.c_int, _i64, _p]),
    "ure_ensemble_score": (C.c_int, [_p, _p, C.c_int, C.c_int, _p, _i64, _f32, _p, _p, _p]),
    "ure_score_finalize": (C.c_int, [_p, _p, _i64, _f32, _p, _p, _p]),
    "ure_rank_metrics": (C.c_int, [_p, _p, _p, _p, _i64, _p, _p]),
    "ure_eval_jobs": (C.c_int, [_p, C.c_int, C.c_int, _i64, _i64, _p]),
    "ure_pack_interactions_f64": (C.c_int, [_p, _i64, _i64, _p, _i32, _p, _p]),
    "ure_partition_blocks": (C.c_int, []),
    "ure_partition_interactions": (C.c_int, [_p, _i64, _i64, _i64, _f64, _p, _p, _i32, C.c_int, _p, _p, _p, _p]),
    "ure_partition_interactions_del": (C.c_int, [_p, _i64, _i64, _i64, _f64, _p, _p, _i32, C.c_int, _p, _p, _p, _p, _p,
                                                 _p]),
    "ure_remap_users": (C.c_int, [_p, _i64, _p, _i32, _p, _p]),
    "ure_host_stage_copy": (C.c_int, [_p, _p, _i64]),
    "ure_user_segments_scratch_bytes": (_i64, [_i64, C.c_int]),
    "ure_user_segments": (C.c_int, [_p, _i64, C.c_int, _p, _p, _p, _p]),
    "ure_seen_lists_scratch_bytes": (_i64, [_i64, C.c_int]),
    "ure_seen_lists": (C.c_int, [_p, _i64, C.c_int, C.c_int, _p, _p, _p, _p]),
    "ure_item_sum": (C.c_int, [_p, C.c_int, _i64, C.c_int, _p, _p]),
    "ure_split_lo": (C.c_int, [_p, _i64, _p, _p]),
    "ure_topn_scratch_bytes": (_i64, [_i64, _i64, C.c_int, C.c_int]),
    "ure_topn": (C.c_int, [_p, C.c_int, _p, _p, _i64, C.c_int, _p, _i64, _p, _p, C.c_int, _f32, _p, _p, _p, _p]),
    "ure_topn_metrics": (C.c_int, [_p, _p, _i64, C.c_int, _p, _p, _p, C.c_int, _p, _p]),
    "ure_combine_gram": (C.c_int, [_p, _p, C.c_int, C.c_int, _p, _p, C.c_int, _p, _p, _p]),
    "ure_item_wsum": (C.c_int, [_p, C.c_int, _p, C.c_int, _i64, C.c_int, _p, _p]),
    "ure_group_score": (C.c_int, [_p, _p, C.c_int, _i64, C.c_int, _p, _p, _p, _i64, _p, _p, _p]),
    "ure_route_deletions": (C.c_int, [_p, _i32, _p, _i32, _p, _i32, _p]),
    "ure_merge_user_rows": (C.c_int, [_p, _p, _p, _p, _p, _i32, C.c_int, C.c_int, _p]),
    "ure_cost_matrix": (C.c_int, [_p, _i64, C.c_int, _p, C.c_int, C.c_int, _p, _p, _p]),
    "ure_cost_matrix_simt": (C.c_int, [_p, _i64, C.c_int, _p, C.c_int, C.c_int, _p, _p, _p]),
    "ure_sinkhorn_colsum": (C.c_int, [_p, _i64, C.c_int, C.c_int, _p, _f32, _f64, _p, _p]),
    "ure_sinkhorn_update_g": (C.c_int, [_p, _p, C.c_int, _f32, _p]),
    "ure_sinkhorn_workspace_bytes": (_i64, []),
    "ure_sinkhorn": (C.c_int, [_p, _i64, C.c_int, C.c_int, _p, C.POINTER(_f32), C.POINTER(_i32), C.c_int, _f32, _p, _p]),
    "ure_sinkhorn_peer_xchg_bytes": (_i64, []),
    "ure_sinkhorn_peer": (C.c_int, [_p, _i64, _f64, C.c_int, C.c_int, _p, C.POINTER(_f32), C.POINTER(_i32), C.c_int, _f32,
                                     C.POINTER(C.c_uint64), C.c_int, C.c_int, C.c_uint64, _p, _p]),
    "ure_sinkhorn_plan": (C.c_int, [_p, _i64, C.c_int, C.c_int, _p, _f32, _f64, _p, _p]),
    "ure_assign_plan_f64": (C.c_int, [_p, _i64, C.c_int, _i64, _p, _p]),
    "ure_assign_plan_f32": (C.c_int, [_p, _i64, C.c_int, _i64, _p, _p]),
    "ure_assign_centroids": (C.c_int, [_p, _i64, C.c_int, C.c_int, _p, _p, C.c_int, _p, _p, _p, _p]),
    "ure_centroid_sums": (C.c_int, [_p, _i64, C.c_int, _p, C.c_int, _p, _p, _p]),
    "ure_balance_workspace_bytes": (_i64, [C.c_int]),
    "ure_balance_labels": (C.c_int, [_p, _i64, C.c_int, C.c_int, _p, _p, C.c_int, _p, _p]),
}

_lib = None


def lib() -> C.CDLL:
    """Load (building first if the .so is absent and nvcc is present) -- or raise."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        from . import build as _build
        _build.build()
    try:
        handle = C.CDLL(LIB_PATH)
    except OSError as e:
        raise RuntimeError(f"ultrare_b200: cannot load {LIB_PATH}: {e}. There is no CPU fallback; "
                           "run `python -m ultrare_b200.build`.") from e
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(handle, name)           # AttributeError if the .so lacks a declared symbol
        fn.restype, fn.argtypes = res, args
    if handle.ure_abi_version() != 7:
        raise RuntimeError("ultrare_b200: ABI version mismatch; rebuild the shared library")
    _lib = handle
    return handle


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().ure_last_error().decode(errors="replace")
        raise RuntimeError(f"ultrare_b200 {what} failed (code {rc}): {msg}")
