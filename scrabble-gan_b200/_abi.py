"""ctypes binding of libsgan.so (the C ABI declared in include/sgan.h).

There is NO fallback: if the shared library is missing or a call fails, a SganError is raised.  Every wrapper
takes raw device pointers (ints); `ptr(t)` extracts one from a torch tensor, and `from_dlpack(x)` accepts any
DLPack producer (e.g. a TF2 tensor via tf.experimental.dlpack.to_dlpack) for the drop-in use described in
INTEGRATION.md."""
from __future__ import annotations

import ctypes as C
import os

SG_OK, SG_ERR_ARG, SG_ERR_CUDA, SG_ERR_UNSUPPORTED = 0, -1, -2, -3
SG_F32, SG_BF16 = 0, 1
SG_MAX_TAPS = 16
SG_LOSS_NSUMS = 16
SG_LOSS_NSTATS = 16
SG_LOSS_HINGE, SG_LOSS_NOT_SATURATING = 0, 1

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libsgan.so")


class SganError(RuntimeError):
    pass


class ConvDesc(C.Structure):
    """Mirror of struct sg_conv_desc (include/sgan.h)."""
    _fields_ = [
        ("n", C.c_int), ("in_h", C.c_int), ("in_w", C.c_int), ("c_in", C.c_int),
        ("out_h", C.c_int), ("out_w", C.c_int), ("c_out", C.c_int),
        ("grid_h", C.c_int), ("grid_w", C.c_int),
        ("in_sy", C.c_int), ("in_sx", C.c_int),
        ("out_sy", C.c_int), ("out_sx", C.c_int), ("out_py", C.c_int), ("out_px", C.c_int),
        ("ntaps", C.c_int),
        ("tap_dy", C.c_int * SG_MAX_TAPS), ("tap_dx", C.c_int * SG_MAX_TAPS),
        ("tap_w_off", C.c_longlong * SG_MAX_TAPS),
        ("w_ci_stride", C.c_longlong), ("w_co_stride", C.c_longlong),
        ("in_dt", C.c_int), ("out_dt", C.c_int), ("relu", C.c_int), ("accumulate", C.c_int), ("mask_dt", C.c_int),
    ]


_P, _I, _L, _F, _D, _Z = C.c_void_p, C.c_int, C.c_longlong, C.c_float, C.c_double, C.c_size_t
_DP = C.POINTER(ConvDesc)

# name -> (restype, argtypes).  ctx is always the first argument of the int-returning entry points.
_PROTOS = {
    "sg_version": (_I, []),
    "sg_last_error": (C.c_char_p, []),
    "sg_ctx_create": (_I, [_I, _P, C.POINTER(_P)]),
    "sg_ctx_destroy": (_I, [_P]),
    "sg_ctx_set_stream": (_I, [_P, _P]),
    "sg_ctx_sync": (_I, [_P]),
    "sg_ctx_launch_count": (_L, [_P]),
    "sg_zero": (_I, [_P, _P, _Z]),
    "sg_ctx_set_speed_mode": (_I, [_P, _I]),
    "sg_ctx_set_conv_split_tail": (_I, [_P, _I]),
    "sg_ctx_set_sm_limit": (_I, [_P, _I]),
    "sg_sizeof_conv_desc": (_I, []),
    "sg_crc32c": (C.c_uint, [_P, _Z, C.c_uint]),
    "sg_random": (_I, [_P, _P, _L, C.c_ulonglong, C.c_ulonglong, _P, _I]),
    "sg_conv_fwd_simt": (_I, [_P, _DP, _P, _P, _P, _P, _P]),
    "sg_conv_wgrad_simt": (_I, [_P, _DP, _P, _P, _P]),
    "sg_conv_tc_supported": (_I, [_DP]),
    "sg_conv_packed_weight_elems": (_Z, [_DP]),
    "sg_conv_pack_weights": (_I, [_P, _DP, _P, _P]),
    "sg_conv_pack_multi_supported": (_I, [_DP, _P]),
    "sg_conv_pack_weights_multi": (_I, [_P, _I, C.POINTER(_DP), C.POINTER(_P), C.POINTER(_P)]),
    "sg_conv_fwd_tc": (_I, [_P, _DP, _P, _P, _P, _P, _P]),
    "sg_conv_fwd_tc_rank1": (_I, [_P, _DP, _P, _P, _P, _P, _P, _P, _P]),
    "sg_conv_tc_plan": (_I, [_DP, _I, _I, C.POINTER(_I), C.POINTER(_I), C.POINTER(_I)]),
    "sg_conv_fwd_tc_phases": (_I, [_P, _I, C.POINTER(_DP), _P, _P, _P, _P]),
    "sg_conv_fwd_tc_dual": (_I, [_P, _DP, _P, _P, _DP, _P, _P, _P, _P, _P]),
    "sg_conv_tc_direct_supported": (_I, [_DP]),
    "sg_conv_fwd_tc_direct": (_I, [_P, _DP, _P, _P, _P, _P, _P]),
    "sg_conv_wgrad_tc_workspace": (_Z, [_DP, _I]),
    "sg_conv_wgrad_tc": (_I, [_P, _DP, _P, _P, _P, _P, _Z]),
    "sg_conv_wgrad_tc_bias": (_I, [_P, _DP, _P, _P, _P, _P, _P]),
    "sg_conv_wgrad_tc_bias_fits": (_I, [_P, _DP]),
    "sg_act_prep": (_I, [_P, _P, _L, _P, _P, _I]),
    "sg_mask_mul": (_I, [_P, _P, _P, _I, _P, _I, _L, _I]),
    "sg_axpby": (_I, [_P, _F, _P, _F, _P, _P, _L]),
    "sg_scale_add": (_I, [_P, _P, _P, _P, _P, _L]),
    "sg_tanh_fwd": (_I, [_P, _P, _P, _L]),
    "sg_tanh_bwd": (_I, [_P, _P, _P, _P, _L]),
    "sg_scale_rows": (_I, [_P, _P, _P, _I, _L]),
    "sg_scale_samples": (_I, [_P, _P, _I, _I, _L, _P, _F]),
    "sg_dot": (_I, [_P, _P, _P, _L, _P, _I]),
    "sg_colsum": (_I, [_P, _P, _I, _L, _I, _P, _I]),
    "sg_cast": (_I, [_P, _P, _P, _I, _L]),
    "sg_avgpool2_fwd": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "sg_avgpool2_bwd": (_I, [_P, _P, _I, _I, _I, _I, _P, _I]),
    "sg_maxpool_fwd": (_I, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _P]),
    "sg_maxpool_bwd": (_I, [_P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _P, _I]),
    "sg_gap_relu_fwd": (_I, [_P, _P, _I, _L, _I, _P]),
    "sg_gap_relu_bwd": (_I, [_P, _P, _P, _I, _L, _I, _P]),
    "sg_bn_stats_scratch_bytes": (_Z, [_L, _I]),
    "sg_bn_stats": (_I, [_P, _P, _L, _I, _P, _P, _Z]),
    "sg_bn_finalize": (_I, [_P, _P, _D, _I, _F, _F, _P, _P, _P, _P]),
    "sg_bn_infer_prepare": (_I, [_P, _P, _P, _I, _F, _P, _P]),
    "sg_bn_apply": (_I, [_P, _P, _I, _L, _I, _P, _P, _P, _P, _L, _I, _P, _I]),
    "sg_bn_bwd_reduce": (_I, [_P, _P, _P, _I, _P, _I, _L, _I, _P, _P, _P, _P]),
    "sg_bn_bwd_combine": (_I, [_P, _P, _P, _P, _L, _I, _I, _P]),
    "sg_bn_bwd_apply": (_I, [_P, _P, _P, _I, _P, _I, _L, _I, _P, _P, _P, _L, _P, _D, _I, _I, _P, _I, _I]),
    "sg_peer_buffer_bytes": (_Z, []),
    "sg_peer_max_payload_bytes": (_Z, []),
    "sg_peer_allreduce_sum": (_I, [_P, _P, _I, _I, C.POINTER(C.c_ulonglong), _I, _I]),
    "sg_peer_bucket_shard": (_L, [_L, _I]),
    "sg_peer_barrier": (_I, [_P, C.POINTER(C.c_ulonglong), _I, _I]),
    "sg_peer_bucket_allreduce": (_I, [_P, _P, _L, _P, C.POINTER(C.c_ulonglong), C.POINTER(C.c_ulonglong), _I, _I, _I]),
    "sg_bn_stats_partial": (_I, [_P, _P, _L, _I, _P, _Z, C.POINTER(_I)]),
    "sg_bn_finalize_peer": (_I, [_P, _P, _I, _I, _D, _F, _F, _P, _P, _P, _P, _P, C.POINTER(C.c_ulonglong), _I, _I]),
    "sg_gemm": (_I, [_P, _I, _I, _I, _I, _I, _P, _I, _P, _I, _P, _I, _P, _I]),
    "sg_label_lengths": (_I, [_P, _P, _I, _I, _P]),
    "sg_mask_width": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _I]),
    "sg_attn_fwd_masked": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "sg_attn_fwd_tc_masked": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "sg_cbn_dense_fwd": (_I, [_P, _P, _I, _I, _I, C.POINTER(_I), C.POINTER(_I), C.POINTER(_L), _P, _P]),
    "sg_cbn_dense_wgrad": (_I, [_P, _P, _I, _I, _I, C.POINTER(_I), C.POINTER(_I), C.POINTER(_L), C.POINTER(_P), _P]),
    "sg_filterbank_fwd": (_I, [_P, _P, _I, _P, _I, _I, _I, _P, _P]),
    "sg_filterbank_bwd": (_I, [_P, _P, _P, _I, _P, _I, _I, _I, _P, _P, _P, _I]),
    "sg_attn_fwd": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "sg_attn_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P]),
    "sg_attn_tc_supported": (_I, [_I, _I, _I, _I]),
    "sg_attn_fwd_tc": (_I, [_P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P]),
    "sg_attn_bwd_tc": (_I, [_P, _P, _P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P]),
    "sg_nonlocal_proj_fwd": (_I, [_P, _P, _L, _P, _P, _P, _P, _P, _P]),
    "sg_nonlocal_out_fwd": (_I, [_P, _P, _L, _P, _P, _P, _P, _P]),
    "sg_nonlocal_out_bwd": (_I, [_P, _P, _P, _L, _P, _P, _P, _P]),
    "sg_nonlocal_proj_bwd": (_I, [_P, _P, _P, _P, _P, _L, _P, _P, _P, _P, _P, _P, _P]),
    "sg_ctc": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P]),
    "sg_ctc_ragged": (_I, [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _P]),
    "sg_softmax_rows": (_I, [_P, _P, _L, _I, _P]),
    "sg_ctc_greedy_decode": (_I, [_P, _P, _I, _I, _I, _P, _P, _P, _P]),
    "sg_edit_distance": (_I, [_P, _P, _P, _I, _P, _P, _I, _I, _P, _P]),
    "sg_loss_sums": (_I, [_P, _I, _I, _P, _P, _P, _P, _P, _P, _P, _I, _P]),
    "sg_loss_finish": (_I, [_P, _I, _I, _I, _F, _P, _P, _P, _P, _P, _P, _I, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "sg_loss_terms": (_I, [_P, _I, _P, _P, _P, _P, _P, _I, _P]),
    "sg_grad_balance": (_I, [_P, _P, _P, _I, _F, _P, _P, _P]),
    "sg_image_grad_balance_sums": (_I, [_P, _P, _P, _L, _P]),
    "sg_image_grad_balance_apply": (_I, [_P, _P, _P, _L, _F, _P, _P, _P]),
    "sg_spectral_norm_bwd": (_I, [_P, _P, _P, _I, _I, _P, _P, _P, _P]),
    "sg_adam": (_I, [_P, _P, _P, _P, _P, _L, _F, _F, _F, _F]),
    "sg_adam_mirror": (_I, [_P, _P, _P, _P, _P, _P, _L, _F, _F, _F, _F]),
    "sg_adam_prepare": (_I, [_P, _P, _P, _I, _F, _F, _F]),
    "sg_adam_dev": (_I, [_P, _P, _P, _P, _P, _P, _L, _P, _F, _F, _F]),
    "sg_adam_fused": (_I, [_P, _P, _P, _P, _P, _P, _L, _P, _F, _F, _F, _I]),
    "sg_rmsprop": (_I, [_P, _P, _P, _P, _L, _F, _F, _F]),
    "sg_spectral_norm": (_I, [_P, _P, _I, _I, _P, _I, _P, _P, _P, _P]),
}

EXPORTED_SYMBOLS = tuple(_PROTOS.keys())

_lib = None


def load():
    """dlopen libsgan.so (once).  Raises SganError if the CUDA extension has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise SganError("libsgan.so is missing at {}: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(there is no CPU fallback)".format(LIB_PATH))
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().sg_last_error().decode("utf-8", "replace")


def check(rc: int, what: str = "") -> None:
    if rc != SG_OK:
        raise SganError("{} failed (rc={}): {}".format(what or "libsgan call", rc, last_error()))


def ptr(t) -> int:
    """Device pointer of a torch tensor (None -> NULL)."""
    if t is None:
        return None
    return t.data_ptr()


def from_dlpack(x):
    """Accept any DLPack producer (TF2 tensor capsule, torch tensor, cupy array ...) -> torch CUDA tensor view."""
    import torch
    if isinstance(x, torch.Tensor):
        return x
    return torch.utils.dlpack.from_dlpack(x)


class Call:
    """Callable proxy: abi.call.sg_xxx(ctx, ...) raises on a non-zero status."""

    def __getattr__(self, name):
        fn = getattr(load(), name)

        def wrapped(*args):
            rc = fn(*args)
            if rc != SG_OK:
                raise SganError("{} failed (rc={}): {}".format(name, rc, last_error()))
            return rc
        wrapped.__name__ = name
        setattr(self, name, wrapped)
        return wrapped


call = Call()
