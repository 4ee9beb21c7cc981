"""ctypes binding of include/ngacf_b200.h.  There is NO CPU fallback: if the library or a CUDA device
is missing, every compute entry point raises."""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_float, c_int32, c_int64, c_size_t, c_uint32, c_uint64, c_void_p

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libngacf_b200.so")

P = c_void_p  # every device pointer crosses the boundary as a plain address

# name -> (restype, argtypes); mirrors include/ngacf_b200.h declaration by declaration
SIGNATURES = {
    "ngacf_last_error": (c_char_p, []),
    "ngacf_version": (c_int32, []),
    "ngacf_graph_build_workspace_bytes": (c_size_t, [c_int64, c_int32, c_int32]),
    "ngacf_graph_build": (c_int32, [P, P, c_int64, c_int32, c_int32, P, P, P, P, P, P, P, P, P, P, P, P, P, c_size_t, P]),
    "ngacf_feature_mask": (c_int32, [P, c_int64, c_uint64, c_uint32, P, c_uint32, c_float, P]),
    "ngacf_edge_mask": (c_int32, [P, c_int64, c_int32, c_uint64, c_uint32, P, c_uint32, c_float, P]),
    "ngacf_dropout_masks": (c_int32, [P, P, P, c_int32, c_int64, c_int64, c_uint64, c_uint32, P, c_float, P]),
    "ngacf_sample_negs": (c_int32, [P, P, P, P, P, c_int32, c_int64, c_int64, P, c_uint64, c_uint32, c_int32, c_uint32, c_int64, P, P, P]),
    "ngacf_bce_logits_loss": (c_int32, [P, c_int64, c_int32, P, P, P]),
    "ngacf_rank_metrics": (c_int32, [P, c_int64, c_int32, c_int32, P, P]),
    "ngacf_dropout_masks_ranges": (c_int32, [P, P, P, c_int32, c_int64, c_int64, c_int64, c_int64, c_int64, c_int64, c_uint64, c_uint32, P, c_float, P]),
    "ngacf_batch_rows_gather": (c_int32, [P, c_int32, P, P, c_int32, c_int64, c_int64, c_int64, c_int64, P, P]),
    "ngacf_batch_rows_scatter": (c_int32, [P, c_int32, P, P, c_int32, P, P]),
    "ngacf_memset_zero": (c_int32, [P, c_size_t, P]),
    "ngacf_spmm_sym": (c_int32, [P, c_int32, P, P, P, P, P, P, P, P, P, P, P]),
    "ngacf_node_logits": (c_int32, [P, P, c_int32, c_int64, P, P, P]),
    "ngacf_node_logits_bwd": (c_int32, [P, P, P, c_int32, c_int64, P, c_int32, P]),
    "ngacf_spgat_aggregate_fwd": (c_int32, [P, c_int32, P, P, P, P, P, P, P, P, c_int32, P, c_float, c_int32, c_int32, P, P, P]),
    "ngacf_spgat_bwd": (c_int32, [P, c_int32, P, P, P, P, P, P, P, P, P, P, P, P, c_int32, P, c_float, c_int32, c_int32, P, P, P, P, P, P, P]),
    "ngacf_counter_add": (c_int32, [P, c_int64, P]),
    "ngacf_step_counters": (c_int32, [P, P, P, c_int64, P]),
    "ngacf_mark_active": (c_int32, [P, P, P, c_int32, c_int32, c_int32, P, P, P]),
    "ngacf_active_plan": (c_int32, [P, c_int32, P, P, c_int32, c_int32, P, c_int64, P, P, P, P]),
    "ngacf_aggregate_fwd_active": (c_int32, [P, c_int32, P, P, P, P, P, P, P, P, P, P, c_int32, P, c_float, P, P, P]),
    "ngacf_stage_bwd_prep_active": (c_int32, [P, c_int32, P, P, P, P, P, P, c_int32, P, P, P]),
    "ngacf_stage_bwd_edges_active": (c_int32, [c_int32, P, c_int32, c_int32, P, P, P, P, P, P, P, P, P, P, P, P, P, c_int32, P, c_float, P,
                                               c_int32, P, c_int32, P, P, P, P, P, P]),
    "ngacf_transform_fwd": (c_int32, [P, P, c_int32, P, c_float, P, c_int32, c_int32, c_int32, P, P, P]),
    "ngacf_aggregate_fwd": (c_int32, [P, c_int32, P, P, P, P, P, P, P, P, c_int32, P, c_float, P, P, c_int32, P]),
    "ngacf_aggregate_finalize": (c_int32, [P, P, P, c_int32, c_int64, P]),
    "ngacf_stage_bwd_finalize": (c_int32, [P, P, P, P, c_int32, c_int32, c_int64, P]),
    "ngacf_bpr_loss_owned": (c_int32, [P, P, c_int32, c_float, P, P, P, P, c_int64, c_int64, P]),
    "ngacf_score_pairs": (c_int32, [P, c_int32, P, P, c_int32, P, P]),
    "ngacf_score_pairs_bwd": (c_int32, [P, c_int32, P, P, P, c_int32, P, c_int32, P]),
    "ngacf_final_features": (c_int32, [P, c_int64, P, P]),
    "ngacf_bpr_loss": (c_int32, [P, P, c_int32, c_float, P, P, P, P]),
    "ngacf_stage_bwd_prep": (c_int32, [P, P, P, P, c_int32, c_int64, P, P, P]),
    "ngacf_stage_bwd_edges": (c_int32, [c_int32, P, c_int32, c_int32, P, P, P, P, P, P, P, P, P, P, P, c_int32, P, c_float, P,
                                        c_int32, P, P, P, c_int32, P]),
    "ngacf_transform_bwd_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "ngacf_transform_bwd": (c_int32, [P, P, P, P, P, c_int32, P, c_float, P, P, c_int32, c_int32, c_int32, P, P, c_int32, c_int32,
                                      P, c_size_t, P]),
    "ngacf_transform_bwd_dx": (c_int32, [P, P, P, c_int32, P, c_float, P, c_int32, c_int32, c_int32, P, P, c_int32, P]),
    "ngacf_transform_bwd_dw_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "ngacf_transform_bwd_dw": (c_int32, [P, P, P, P, c_int32, P, c_float, P, P, c_int32, c_int32, c_int32, c_int32, P, c_size_t, P]),
    "ngacf_adam_step": (c_int32, [P, c_int32, c_int64, c_float, c_float, c_float, c_float, c_float, c_int64, P]),
    "ngacf_adam_step_dev": (c_int32, [P, c_int32, c_int64, c_float, c_float, c_float, c_float, c_float, P, P]),
    "ngacf_sample_pairs": (c_int32, [P, P, P, P, P, c_int32, c_int64, c_int64, P, c_uint64, c_uint32, P, P, P, P]),
    "ngacf_score_topk_exact": (c_int32, [P, c_int32, c_int32, P, c_int32, P, P, P, P, P, P]),
    "ngacf_score_topk_exact_split_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "ngacf_score_topk_exact_split": (c_int32, [P, c_int32, c_int32, P, c_int32, P, P, P, P, P, P, c_size_t, P]),
    "ngacf_score_topk_tc_workspace_bytes": (c_size_t, [c_int32, c_int32]),
    "ngacf_score_topk_tc": (c_int32, [P, c_int32, c_int32, P, c_int32, P, P, P, P, P, P, c_int32, P, c_size_t, P]),
    "ngacf_eval_metrics_workspace_bytes": (c_size_t, [c_int32]),
    "ngacf_eval_metrics": (c_int32, [P, P, c_int32, P, P, P, P, P, c_size_t, P]),
    # width-carrying variants (embedSize 128)
    "ngacf_dropout_masks_w": (c_int32, [P, P, P, P, c_int32, c_int64, c_int64, c_uint64, c_uint32, P, c_float, P]),
    "ngacf_transform_fwd_w": (c_int32, [P, P, c_int32, P, c_float, P, c_int32, c_int32, c_int32, c_int32, c_int32, P, P, P]),
    "ngacf_transform_bwd_workspace_bytes_w": (c_size_t, [c_int32, c_int32, c_int32, c_int32]),
    "ngacf_transform_bwd_w": (c_int32, [P, P, P, P, P, c_int32, P, c_float, P, P, c_int32, c_int32, c_int32, c_int32, c_int32, P, P, c_int32,
                                        c_int32, P, c_size_t, P]),
    "ngacf_aggregate_fwd_w": (c_int32, [P, c_int32, P, P, P, P, P, P, P, P, c_int32, c_int32, P, c_float, P, P, c_int32, P]),
    "ngacf_stage_bwd_prep_w": (c_int32, [P, P, P, P, c_int32, c_int32, c_int64, P, P, P]),
    "ngacf_stage_bwd_edges_w": (c_int32, [c_int32, P, c_int32, c_int32, P, P, P, P, P, P, P, P, P, P, P, c_int32, c_int32, P, c_float, P,
                                          c_int32, P, P, P, c_int32, P]),
    "ngacf_score_pairs_w": (c_int32, [P, c_int32, c_int32, P, P, c_int32, P, P]),
    "ngacf_score_pairs_bwd_w": (c_int32, [P, c_int32, c_int32, P, P, P, c_int32, P, c_int32, P]),
    "ngacf_final_features_w": (c_int32, [P, c_int64, c_int32, P, P]),
    "ngacf_score_topk_exact_w": (c_int32, [P, c_int32, c_int32, c_int32, P, c_int32, P, P, P, P, P, P]),
    "ngacf_score_topk_exact_split_w": (c_int32, [P, c_int32, c_int32, c_int32, P, c_int32, P, P, P, P, P, P, c_size_t, P]),
    # top-K recommendation lists
    "ngacf_recommend_topk_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32, c_int32]),
    "ngacf_recommend_topk": (c_int32, [P, c_int32, c_int32, c_int32, P, c_int32, c_int32, P, P, P, P, P, P, c_size_t, P]),
    # similar-item lists
    "ngacf_similar_items_topk_workspace_bytes": (c_size_t, [c_int32, c_int32, c_int32, c_int32]),
    "ngacf_similar_items_topk": (c_int32, [P, c_int32, c_int32, c_int32, P, c_int32, c_int32, P, P, P, P, c_size_t, P]),
}

_lib = None
PROFILE = None      # bench.py sets this to a list: every call is then bracketed with CUDA events on its stream


class NgacfError(RuntimeError):
    pass


def load(required: bool = True):
    """Loads the shared library (no CUDA call is made).  Raises if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if required:
            raise NgacfError("%s is missing: run `python -m ngacf_b200.build` (nvcc, sm_100a). "
                             "ngacf_b200 has no CPU fallback." % LIB_PATH)
        return None
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError:
            continue      # declared in the header but not built yet -> calling it raises below
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def exported_symbols():
    lib = load()
    return [n for n in SIGNATURES if hasattr(lib, n)]


def call(name: str, *args):
    """Calls an int-returning entry point and turns a negative code into an exception."""
    lib = load()
    fn = getattr(lib, name, None)
    if fn is None:
        raise NgacfError("entry point %s is not in %s" % (name, LIB_PATH))
    if PROFILE is not None:
        import torch
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        rc = fn(*args)
        e1.record()
        PROFILE.append((name, args, e0, e1))
    else:
        rc = fn(*args)
    if rc != 0:
        raise NgacfError("%s failed (%d): %s" % (name, rc, lib.ngacf_last_error().decode()))
    return rc


def require_cuda(t):
    if not t.is_cuda:
        raise NgacfError("ngacf_b200 kernels need CUDA tensors (got device %s); there is no CPU path" % t.device)
