"""ctypes binding of ``libcoper_sm100.so`` (the C ABI declared in ``include/coper.h``).

The library is the product: there is NO fallback.  If it is missing, or a call returns a
non-zero status, this module raises — it never routes to PyTorch or the CPU oracle.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcoper_sm100.so")

PREC = {"fp32": 0, "bf16": 1, "tf32x3": 2, "fp16x3": 3}
# flags of coper_cpg_fc_bwd (include/coper.h)
CPG_BWD_REUSE_FWD, CPG_BWD_INPUT_GRADS_ONLY, CPG_BWD_WEIGHT_GRADS_ONLY, CPG_BWD_DCB_ACCUMULATE = 1, 2, 4, 8

vp, i32, i64, u64, f32, sz = C.c_void_p, C.c_int, C.c_int64, C.c_uint64, C.c_float, C.c_size_t

# name -> (restype, argtypes); mirrors include/coper.h one to one (tests check the two stay in sync)
SIGNATURES = {
    "coper_version": (i32, []),
    "coper_status_string": (C.c_char_p, [i32]),
    "coper_last_cuda_error": (i32, []),
    "coper_launch_count": (C.c_longlong, []),
    "coper_device_is_sm100": (i32, []),
    "coper_set_pdl": (i32, [i32]),
    "coper_gather_rows": (i32, [vp, i64, i64, i32, vp, i32, vp, vp]),
    "coper_gather_rows2": (i32, [vp, i64, i64, i32, vp, i32, vp, vp, i64, i64, i32, vp, i32, vp, vp, vp, f32, f32, f32, vp]),
    "coper_conv_fwd": (i32, [vp, i32, i32, i32, vp, vp, i32, i32, i32, i32, vp, vp]),
    "coper_conv_bwd_slabs": (i32, [i32, i32, i32, i32, i32, i32, i32]),
    "coper_conv_bwd": (i32, [vp, vp, i32, i32, i32, vp, i32, i32, i32, i32, vp, vp, vp, vp]),
    "coper_conv_bwd_bn": (i32, [vp, vp, vp, i32, i32, i32, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, i32, f32, vp, u64,
                                vp, vp, vp, vp, vp]),
    "coper_colstats_chunks": (i32, [i64]),
    "coper_colstats": (i32, [vp, i64, i32, vp, vp]),
    "coper_bn_finalize": (i32, [vp, i32, i64, i32, vp, vp, vp, vp, f32, f32, i32, i32, i32, vp, vp, vp, vp, vp]),
    "coper_bn_stats_finalize": (i32, [vp, i64, i32, vp, vp, vp, vp, vp, vp, f32, f32, i32, i32, vp, vp, vp, vp, vp]),
    "coper_bn_act_fwd": (i32, [vp, i64, i32, vp, vp, i32, f32, vp, u64, vp, vp]),
    "coper_bn_act_fwd_moving": (i32, [vp, i64, i32, vp, vp, vp, vp, f32, i32, vp, vp]),
    "coper_bn_act_bwd_stats": (i32, [vp, vp, i64, i32, vp, vp, vp, vp, i32, f32, vp, u64, vp, vp]),
    "coper_bn_act_bwd_stats_finalize": (i32, [vp, vp, i64, i32, vp, vp, vp, vp, i32, f32, vp, u64, vp, vp, i32, vp, vp, vp, vp,
                                              vp]),
    "coper_bn_act_bwd_finalize": (i32, [vp, i32, i64, i32, i32, vp, vp, vp, vp, vp]),
    "coper_bn_act_bwd_apply": (i32, [vp, vp, i64, i32, vp, vp, vp, vp, vp, vp, i32, f32, vp, u64, f32, u64, vp, vp]),
    "coper_dropout_mask": (i32, [i64, f32, vp, u64, vp, vp]),
    "coper_dropout_apply": (i32, [vp, i64, f32, vp, u64, vp]),
    "coper_cpg_fc_fwd_workspace_bytes": (sz, [i32, i32, i32, i32, i32]),
    "coper_cpg_fc_fwd": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, f32, vp, u64, vp, vp, sz, i32, vp]),
    "coper_cpg_fc_bwd_workspace_bytes": (sz, [i32, i32, i32, i32, i32]),
    "coper_cpg_fc_bwd": (i32, [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, sz, i32, i32,
                               vp]),
    "coper_sgemm": (i32, [i32, i32, i32, i32, i32, vp, i32, vp, i32, vp, i32, i32, vp]),
    "coper_score1n_workspace_bytes": (sz, [i32, i64, i32, i32]),
    "coper_score1n_fwd": (i32, [vp, vp, vp, i32, i64, i32, vp, i64, vp, sz, i32, vp]),
    "coper_prepared_bytes": (sz, [i64, i32, i32]),
    "coper_prepare_operand": (i32, [vp, i64, i32, i64, i32, vp, vp]),
    "coper_score1n_fwd_prepared": (i32, [vp, vp, vp, i32, i64, i32, vp, i64, i32, vp]),
    "coper_tc_gemm_workspace_bytes": (sz, [i32, i32, i32, i32]),
    "coper_tc_gemm": (i32, [i32, i32, i32, i32, i32, vp, i32, vp, i32, vp, i32, i32, vp, sz, vp]),
    "coper_score1n_bce_workspace_bytes": (sz, [i32, i64, i32, i32]),
    "coper_score1n_bce_G_bytes": (sz, [i32, i64, i32]),
    "coper_score1n_bce_fwd_bwd": (i32, [vp, vp, vp, vp, vp, i32, i64, i32, f32, f32, f32, vp, vp, i64, vp, vp, vp, vp,
                                        sz, i32, vp]),
    "coper_score1n_bce_fwd_bwd_norm": (i32, [vp, vp, vp, vp, vp, i32, i64, i32, f32, f32, f32, vp, vp, i64, vp, vp, vp, vp,
                                             vp, sz, i32, vp]),
    "coper_score1n_bce_dE": (i32, [vp, i32, i64, i32, f32, vp, vp, vp, vp, sz, i32, vp]),
    "coper_sample_labels": (i32, [vp, vp, i32, i64, i32, i32, vp, u64, vp, vp, vp]),
    "coper_score_sampled_workspace_bytes": (sz, [i32, i32]),
    "coper_score_sampled_bce_fwd_bwd": (i32, [vp, vp, vp, vp, vp, i32, i32, i64, i32, f32, f32, f32, vp, vp, vp, vp, vp,
                                              vp, vp, vp, vp, sz, vp]),
    "coper_score_sampled_sharded_workspace_bytes": (sz, [i32, i32]),
    "coper_score_sampled_bce_fwd_bwd_sharded": (i32, [vp, vp, vp, vp, vp, i32, i32, i64, i32, f32, f32, f32, vp, vp, vp,
                                                      vp, vp, vp, vp, vp, i64, i64, vp, sz, vp]),
    "coper_score_candidates": (i32, [vp, vp, vp, vp, i32, i32, i32, i64, i64, vp, vp]),
    "coper_candidate_rank": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i64, i64, vp, vp, i32, vp, vp, vp]),
    "coper_csr_to_bits": (i32, [vp, vp, i32, i64, i64, vp, vp]),
    "coper_dense_to_bits": (i32, [vp, i32, i64, vp, vp]),
    "coper_gold_scores": (i32, [vp, i64, i32, i64, vp, i64, vp, vp]),
    "coper_filtered_rank": (i32, [vp, i64, i32, i64, vp, i64, vp, vp, vp, vp, vp]),
    "coper_score1n_rank_workspace_bytes": (sz, [i32, i32, i32]),
    "coper_score1n_gold_prepared": (i32, [vp, vp, vp, i32, i64, i32, vp, i64, vp, vp, sz, i32, vp]),
    "coper_score1n_rank_prepared": (i32, [vp, vp, vp, i32, i64, i32, vp, vp, vp, vp, i32, vp]),
    "coper_score1n_topk_workspace_bytes": (sz, [i32, i64, i32, i32, i32]),
    "coper_score1n_topk_prepared": (i32, [vp, vp, vp, i32, i64, i32, vp, i64, i32, vp, vp, vp, sz, i32, vp]),
    "coper_topk_scores_workspace_bytes": (sz, [i32, i64, i32]),
    "coper_topk_scores": (i32, [vp, i64, i32, i64, vp, i64, i32, vp, vp, vp, sz, vp]),
    "coper_topk_merge": (i32, [vp, vp, i32, i32, i32, vp, vp, vp]),
    "coper_csr_to_bits_t": (i32, [vp, vp, i32, i64, i64, vp, vp]),
    "coper_dense_to_bits_t": (i32, [vp, i32, i64, i64, vp, vp]),
    "coper_bits_t_set": (i32, [vp, i32, i64, i64, vp, vp]),
    "coper_segscatter_workspace_bytes": (sz, [i32]),
    "coper_segscatter_add_sq": (i32, [vp, i32, vp, i32, vp, vp, i64, i64, vp]),
    "coper_segscatter_add_pair": (i32, [vp, i32, vp, i32, vp, vp, i64, i64, vp, vp, i32, vp, i32, vp, vp, i64, i64, vp]),
    "coper_segscatter_add": (i32, [vp, i32, vp, i32, vp, i64, i64, vp, sz, vp]),
    "coper_reduce_partials": (i32, [vp, i32, i64, f32, i32, vp, vp]),
    "coper_reduce_partials2": (i32, [vp, i64, vp, vp, i64, vp, i32, f32, i32, vp]),
    "coper_sumsq": (i32, [vp, i64, i32, vp, vp]),
    "coper_clip_scale": (i32, [vp, i32, f32, vp, vp]),
    "coper_step_state_advance": (i32, [vp, vp, f32, f32, f32, vp]),
    "coper_sumsq_combine": (i32, [vp, i32, vp, i32, vp, vp]),
    "coper_mt_sumsq": (i32, [vp, i32, vp, i32, vp, vp, vp, vp]),
    "coper_clip_scale_n": (i32, [vp, i32, f32, vp, vp]),
    "coper_mt_sumsq_clip": (i32, [vp, i32, vp, i32, vp, vp, vp, i32, vp, i32, vp, i32, f32, vp, vp]),
    "coper_mt_amsgrad": (i32, [vp, vp, i32, vp, f32, f32, f32, vp, i32, vp]),
    "coper_amsgrad_step": (i32, [vp, vp, vp, vp, vp, i64, vp, f32, f32, f32, vp, i32, vp]),
}
SUMSQ_BLOCKS = 256
TOPK_MAX = 128  # COPER_TOPK_MAX
MT_CHUNK = 16384
# mirrors coper_param_desc (include/coper.h): one record per tensor of the multi-tensor clip / AMSGrad launches
PARAM_DESC = np.dtype([("theta", "<u8"), ("grad", "<u8"), ("m", "<u8"), ("v", "<u8"), ("vhat", "<u8"), ("prepared", "<u8"),
                       ("grad_sq", "<u8"), ("n", "<i8"), ("prepared_prec", "<i4"), ("mode", "<i4")])

_lib = None
launch_count = 0  # number of C-ABI compute calls issued by this process (bench.py reports it)


class CoperError(RuntimeError):
    pass


def load():
    """Load the shared library (once). Raises CoperError if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CoperError(
            "libcoper_sm100.so not found at %s — build it with `python -m coper_b200.build` "
            "(there is no CPU/PyTorch fallback for the CoPER hot path)" % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header/library drift
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        lib = load()
        msg = lib.coper_status_string(rc).decode()
        raise CoperError("%s failed: %s (status %d, cudaError %d)" % (what, msg, rc, lib.coper_last_cuda_error()))


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


def stream_ptr():
    import torch
    return torch.cuda.current_stream().cuda_stream


def call_plain(name, *args):
    """Invoke a status-returning entry point that takes no stream."""
    check(getattr(load(), name)(*args), name)


def call(name, *args):
    """Invoke a status-returning entry point on the current torch CUDA stream (appended as last arg)."""
    global launch_count
    lib = load()
    launch_count += 1
    check(getattr(lib, name)(*args, stream_ptr()), name)
