"""ctypes binding of librtucker_b200.so (the C ABI declared in include/rtucker.h).

There is NO fallback: if the shared library is missing or a call fails, an exception is raised.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librtucker_b200.so")

_lib = None

vp, i32, i64, f32, f64, sz = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double, C.c_size_t

class ApplyJob(C.Structure):
    """struct rt_apply_job of include/rtucker.h"""
    _fields_ = [("Y", vp), ("ldy", i64), ("n", i32), ("X0", vp), ("ldx0", i64), ("a0_dev", vp), ("nk", i32),
                ("X", vp * 4), ("ldx", i64 * 4), ("rk", i32 * 4), ("K", vp * 4), ("copy_out", vp * 4),
                ("ldcopy", i64 * 4)]


# name -> (restype, argtypes); mirrors include/rtucker.h one to one
PROTOTYPES = {
    "rt_abi_version": (i32, []),
    "rt_last_error": (C.c_char_p, []),
    "rt_device_info": (i32, [C.POINTER(i32)] * 3),
    "rt_launch_count": (C.c_ulonglong, []),
    "rt_small_flop_count": (C.c_double, []),
    "rt_rank_filtered": (i32, [vp, i64, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
    "rt_target_prob": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp]),
    "rt_score_rank_ws_bytes": (sz, [i32, i32, i32]),
    "rt_score_rank_fused": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "rt_score_topk_ws_bytes": (sz, [i32, i32, i32, i32]),
    "rt_score_topk": (i32, [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
    "rt_score_dense": (i32, [vp, vp, i32, i32, i32, vp, i64, vp]),
    "rt_score_dense_logits": (i32, [vp, vp, i32, i32, i32, vp, i64, vp]),
    "rt_target_logit": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp]),
    "rt_score_rank_logit_ws_bytes": (sz, [i32, i32, i32]),
    "rt_score_rank_logit": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]),
    "rt_score_topk_logit": (i32, [vp, vp, i32, i32, i32, i32, i32, vp, vp, vp, vp, vp, vp, vp]),
    "rt_filter_dense": (i32, [vp, i64, vp, i64, i32, i32, vp, vp]),
    "rt_gather_rows": (i32, [vp, i32, i32, i32, vp, i32, vp, vp]),
    "rt_scatter_rows_add": (i32, [vp, i32, i32, i32, vp, i32, vp, vp]),
    "rt_query_ws_bytes": (sz, [i32, i32, i32, i32]),
    "rt_query_fwd": (i32, [vp, vp, vp, i32, i32, i32, i32, vp, vp, vp]),
    "rt_query_bwd": (i32, [vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp, vp]),
    "rt_score_bce_ws_bytes": (sz, [i32, i32, i32, i32]),
    "rt_score_bce_fwd_bwd": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, f32, vp, vp, vp,
                                   i32, vp, vp]),
    "rt_gram_ws_bytes": (sz, [i32, i32, i32]),
    "rt_gram": (i32, [vp, i64, vp, i64, i32, i32, i32, vp, i32, vp, vp]),
    "rt_apply": (i32, [vp, i64, i32, i32, vp, i64, vp, i32, C.POINTER(vp), C.POINTER(i64),
                       C.POINTER(i32), C.POINTER(vp), vp]),
    "rt_apply_tc_supported": (i32, [i32, i32, C.POINTER(i32)]),
    "rt_apply_tc_ws_bytes": (sz, [i32, i32, C.POINTER(i32)]),
    "rt_apply_tc": (i32, [vp, i64, i32, i32, vp, i64, vp, i32, C.POINTER(vp), C.POINTER(i64), C.POINTER(i32),
                          C.POINTER(vp), vp, vp]),
    "rt_apply_multi_ws_bytes": (sz, [i32, C.POINTER(ApplyJob), i32]),
    "rt_apply_multi": (i32, [i32, C.POINTER(ApplyJob), i32, vp, vp]),
    "rt_small_ws_bytes": (sz, [i32, i32, i32, i32]),
    "rt_small_prepare": (i32, [vp, i32, i32, i32, i32, vp, vp]),
    "rt_small_ainv_offset": (sz, [i32, i32, i32, i32]),
    "rt_rows_times_ainv": (i32, [vp, i32, i32, i32, i32, i32, vp, vp, vp]),
    "rt_small_grad": (i32, [vp] * 9 + [f64, vp, i32, i32, i32, i32, i32] + [vp] * 9),
    "rt_small_norm": (i32, [vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp]),
    "rt_small_norm_adam": (i32, [vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, vp]),
    "rt_small_project": (i32, [vp] * 7 + [i32, i32, i32, i32] + [vp] * 9),
    "rt_core_axpby": (i32, [vp, vp, vp, i32, vp, vp]),
    "rt_small_retract": (i32, [vp] * 6 + [i32, i32, i32, i32] + [vp] * 12),
    "rt_epoch_batch": (i32, [vp, i32, i32, vp, i32, vp, vp, vp, vp, vp, i32, vp]),
    "rt_eigh_ws_bytes": (sz, [i32]),
    "rt_eigh": (i32, [vp, i32, vp, vp, vp, vp]),
    "rt_dominant_subspace_ws_bytes": (sz, [i32, i32]),
    "rt_dominant_subspace": (i32, [vp, i32, i32, vp, vp, vp, vp]),
    "rt_fill_normal": (i32, [vp, i32, i32, i64, C.c_uint64, C.c_uint32, vp]),
    "rt_tc_selftest": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "rt_tc_selftest16": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, vp]),
    "rt_bulk_reduce_selftest": (i32, [vp, vp, vp, i32, vp]),
    "rt_mma_probe": (i32, [i32, i32, i32, i32, i32, vp, vp]),
    "rt_score_bce_tc3_supported": (i32, [i32, i32, i32]),
    "rt_score_bce_tc3_ws_bytes": (sz, [i32, i32, i32]),
    "rt_score_bce_tc3": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, f32, vp, vp, vp, vp, vp]),
    "rt_score_lse_ws_bytes": (sz, [i32, i32, i32, i32]),
    "rt_score_lse": (i32, [vp, vp, i32, i32, i32, i32, vp, vp, vp]),
    "rt_score_ce_ws_bytes": (sz, [i32, i32, i32, i32]),
    "rt_score_ce_fwd_bwd": (i32, [vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, f32, vp, i32, vp, vp, vp, i32, vp,
                                  vp]),
    "rt_score_bce_v3_supported": (i32, [i32]),
    "rt_score_bce_v3_ws_bytes": (sz, [i32, i32, i32]),
    "rt_score_v3_set_profile": (i32, [vp]),
    "rt_score_tc_set_profile": (i32, [vp]),
    "rt_eigh_set_profile": (i32, [vp]),
    "rt_score_bce_v3_phases": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, f32, f32, vp, vp, vp, vp, vp, vp, i32]),
    "rt_score_bce_v3": (i32, [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, f32, f32, vp, vp, vp, vp, vp, vp]),
}


class RTuckerError(RuntimeError):
    pass


def lib():
    """Load the shared library once; raise loudly if it is absent (no CPU fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.isfile(LIB_PATH):
            raise RTuckerError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). rtucker_b200 has no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)  # AttributeError if the .so does not export the symbol
            fn.restype, fn.argtypes = res, args
        if handle.rt_abi_version() != 1:
            raise RTuckerError("librtucker_b200.so ABI version mismatch")
        _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().rt_last_error().decode(errors="replace")
        raise RTuckerError(f"{what} failed (code {rc}): {msg}")


def stream_ptr():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise RTuckerError("rtucker_b200 ops need CUDA tensors: there is no CPU path")
