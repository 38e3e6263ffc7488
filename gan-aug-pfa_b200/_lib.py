"""ctypes binding of libgap_b200.so (include/gap_b200.h).

The product path has no CPU fallback: if the shared library is missing or a call fails this module
raises — it never routes around the CUDA kernels.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "lib" / "libgap_b200.so"

ACT_NONE, ACT_LRELU, ACT_RELU, ACT_TANH, ACT_SIGMOID = 0, 1, 2, 3, 4


class ConvGemmArgs(C.Structure):
    """Mirror of ``gap_conv_gemm_args``."""

    _fields_ = [
        ("src", C.c_void_p * 2),
        ("src_c", C.c_int * 2),
        ("src_ld", C.c_int64 * 2),
        ("n", C.c_int), ("ih", C.c_int), ("iw", C.c_int),
        ("gh", C.c_int), ("gw", C.c_int),
        ("n_phase", C.c_int),
        ("taps_h", C.c_int), ("taps_w", C.c_int),
        ("in_stride", C.c_int),
        ("in_off_h", C.c_int * 2), ("in_off_w", C.c_int * 2),
        ("out_stride", C.c_int),
        ("wpk", C.c_void_p),
        ("w_rows", C.c_int),
        ("n_out", C.c_int),
        ("oh", C.c_int), ("ow", C.c_int),
        ("out", C.c_void_p),
        ("out_ld", C.c_int64),
        ("act", C.c_int),
        ("out2", C.c_void_p),
        ("out2_ld", C.c_int64),
        ("act2", C.c_int),
        ("bias", C.c_void_p),
        ("stats", C.c_void_p),
        ("out_f32", C.c_int),
        ("bwd_y", C.c_void_p), ("bwd_y_ld", C.c_int64),
        ("bwd_scale", C.c_void_p), ("bwd_shift", C.c_void_p),
        ("bwd_g2", C.c_void_p), ("bwd_g2_ld", C.c_int64),
        ("bwd_slope", C.c_float), ("bwd_c0", C.c_int),
        ("scale", C.c_void_p),
        ("accumulate", C.c_int),
    ]


class WgradArgs(C.Structure):
    """Mirror of ``gap_wgrad_args``."""

    _fields_ = [
        ("mop", C.c_void_p), ("m_c", C.c_int), ("m_rows", C.c_int), ("m_ld", C.c_int64),
        ("nop", C.c_void_p), ("n_c", C.c_int), ("n_ld", C.c_int64),
        ("n", C.c_int), ("gh", C.c_int), ("gw", C.c_int), ("nh", C.c_int), ("nw", C.c_int),
        ("taps_h", C.c_int), ("taps_w", C.c_int), ("stride", C.c_int),
        ("off_h", C.c_int), ("off_w", C.c_int),
        ("out", C.c_void_p), ("ld_m", C.c_int64), ("ld_tap", C.c_int64),
    ]


class PackEntry(C.Structure):
    """Mirror of ``gap_pack_entry``."""

    _fields_ = [
        ("w", C.c_void_p), ("out", C.c_void_p),
        ("mode", C.c_int), ("n_phase", C.c_int), ("rows", C.c_int), ("rows_pad", C.c_int),
        ("taps_h", C.c_int), ("taps_w", C.c_int), ("c", C.c_int), ("c_pad", C.c_int), ("krow", C.c_int),
        ("tile_begin", C.c_int), ("tiles_r", C.c_int), ("tiles_c", C.c_int),
        ("s_r", C.c_int64), ("s_c", C.c_int64), ("s_kh", C.c_int64), ("s_kw", C.c_int64),
    ]


_lib = None
_P, _I, _L, _F, _D = C.c_void_p, C.c_int, C.c_int64, C.c_float, C.c_double

# name -> (restype, argtypes); every symbol include/gap_b200.h declares is listed here, and
# tests/test_abi.py checks the two stay in sync.
_SIGNATURES = {
    "gap_last_error_string": (C.c_char_p, []),
    "gap_version": (C.c_int, []),
    "gap_sm_count": (C.c_int, []),
    "gap_debug_set": (C.c_int, [C.c_char_p, C.c_int]),
    "gap_conv_gemm": (C.c_int, [C.POINTER(ConvGemmArgs), C.c_void_p]),
    "gap_conv_wgrad": (C.c_int, [C.POINTER(WgradArgs), C.c_void_p]),
    "gap_nchw_f32_to_nhwc_bf16": (C.c_int, [_P, _P, _I, _I, _I, _I, _L, _P]),
    "gap_nhwc_to_nchw_f32": (C.c_int, [_P, _I, _P, _I, _I, _I, _I, _L, _I, _I, _P]),
    "gap_tanh_bwd": (C.c_int, [_P, _P, _L, _P, _L, _I, _I, _I, _I, _P]),
    "gap_gen_out_bwd": (C.c_int, [_P, _L, _P, _L, _P, _L, _F, _P, _L, _L, _I, _P, _P]),
    "gap_gen_out_bwd_u8": (C.c_int, [_P, _L, _P, _L, _P, _L, _F, _P, _L, _L, _I, _P, _P]),
    "gap_bce_logits_const": (C.c_int, [_P, _L, _F, _F, _P, _L, _P, _P]),
    "gap_bce_logits_const_f32": (C.c_int, [_P, _L, _F, _F, _P, _P, _P, _P]),
    "gap_sum_f32": (C.c_int, [_P, _L, _P, _P]),
    "gap_cout1_conv_fwd": (C.c_int, [_P, _L, _I, _I, _I, _I, _P, _P, _I, _I, _P, _P, _P, _P, _F, _P]),
    "gap_cout1_conv_dgrad": (C.c_int, [_P, _I, _I, _I, _P, _I, _I, _I, _P, _L, _I, _I, _P]),
    "gap_cout1_conv_dgrad_bwd": (C.c_int, [_P, _I, _I, _I, _P, _I, _I, _I, _P, _L, _I, _I, _P, _L, _P, _P, _F, _P, _P]),
    "gap_cout1_conv_wgrad": (C.c_int, [_P, _I, _I, _I, _P, _L, _I, _I, _I, _I, _I, _P, _P, _P, _F, _P]),
    "gap_thin_conv_fwd": (C.c_int, [_P, _L, _P, _L, _I, _I, _I, _P, _P, _I, _P, _L, _I, _P, _L, _I, _P]),
    "gap_thin_conv_wgrad": (C.c_int, [_P, _L, _P, _L, _P, _L, _I, _I, _I, _I, _P, _L, _P, _P]),
    "gap_thin_conv_wgrad_c": (C.c_int, [_P, _L, _P, _L, _I, _P, _L, _I, _I, _I, _I, _I, _P, _L, _P, _P]),
    "gap_thin_convT_fwd": (C.c_int, [_P, _L, _I, _I, _I, _I, _P, _P, _I, _P, _L, _P, _L, _P, _P]),
    "gap_thin_convT_fwd_c": (C.c_int, [_P, _L, _I, _I, _I, _I, _I, _P, _P, _I, _P, _L, _P, _L, _P, _P]),
    "gap_u8_hwc_to_nhwc_bf16": (C.c_int, [_P, _P, _L, _L, _P]),
    "gap_u8_hwc_to_nhwc_bf16_c": (C.c_int, [_P, _I, _P, _L, _L, _P]),
    "gap_resize_u8_to_nhwc_bf16": (C.c_int, [_P, _I, _I, _I, _I, _I, _P, _L, _P, _P]),
    "gap_resize_u8_to_nhwc_bf16_c": (C.c_int, [_P, _I, _I, _I, _I, _I, _I, _P, _L, _P, _P]),
    "gap_resize_nearest_i64": (C.c_int, [_P, _I, _I, _I, _I, _I, _P, _P]),
    "gap_im2col_k3s1p1_c3": (C.c_int, [_P, _L, _P, _I, _I, _I, _P]),
    "gap_im2col_k3s1p1_c": (C.c_int, [_P, _L, _I, _P, _I, _I, _I, _P]),
    "gap_maxpool2x2_fwd": (C.c_int, [_P, _L, _P, _L, _I, _I, _I, _I, _P]),
    "gap_maxpool2x2_bwd": (C.c_int, [_P, _L, _P, _L, _P, _L, _I, _I, _I, _I, _I, _P]),
    "gap_upsample_bilinear2x_fwd": (C.c_int, [_P, _L, _P, _L, _I, _I, _I, _I, _P]),
    "gap_upsample_bilinear2x_bwd": (C.c_int, [_P, _L, _P, _L, _I, _I, _I, _I, _I, _P]),
    "gap_dropout_bf16": (C.c_int, [_P, _L, _L, _I, _F, C.c_uint64, C.c_uint64, _P]),
    "gap_att_add_relu_fwd": (C.c_int, [_P, _P, _P, _P, _P, _P, _P, _L, _I, _P]),
    "gap_relu_bwd": (C.c_int, [_P, _P, _P, _L, _P]),
    "gap_lrelu_bwd_bf16": (C.c_int, [_P, _L, _P, _L, _F, _P, _L, _L, _I, _I, _P]),
    "gap_att_gate_fwd": (C.c_int, [_P, _P, _P, _P, _P, _L, _P, _L, _L, _I, _P]),
    "gap_att_gate_bwd": (C.c_int, [_P, _L, _P, _L, _P, _P, _L, _I, _P, _L, _I, _P]),
    "gap_vec_stats": (C.c_int, [_P, _L, _P, _P]),
    "gap_vec_bn_bwd": (C.c_int, [_P, _P, _L, _P, _P, _P, _P, _P, _P]),
    "gap_conv1x1_cout1_fwd": (C.c_int, [_P, _L, _P, _P, _P, _L, _I, _P]),
    "gap_conv1x1_cout1_dgrad": (C.c_int, [_P, _P, _P, _L, _L, _I, _P]),
    "gap_conv1x1_cout1_wgrad": (C.c_int, [_P, _P, _L, _L, _I, _P, _P, _P]),
    "gap_seg_loss": (C.c_int, [_P, _P, _L, _I, _F, _F, _F, _F, _F, _F, _P, _P, _F, _P, _P]),
    "gap_seg_confusion": (C.c_int, [_P, _P, _I, _I, _L, _P, _P]),
    "gap_conv1x1_ck_fwd": (C.c_int, [_P, _L, _P, _P, _I, _I, _L, _P, _P, _P]),
    "gap_conv1x1_ck_dgrad": (C.c_int, [_P, _P, _I, _I, _L, _P, _L, _P]),
    "gap_conv1x1_ck_wgrad": (C.c_int, [_P, _P, _L, _I, _I, _L, _P, _P, _P]),
    "gap_seg_ce_loss": (C.c_int, [_P, _P, _I, _I, _L, _P, _L, _P, _P, _P, _F, _P, _P]),
    "gap_seg_softmax_dice": (C.c_int, [_P, _P, _I, _I, _L, _I, _F, _F, _F, _P, _L, _P, _P, _P, _F, _P, _P]),
    "gap_seg_confusion_ck": (C.c_int, [_P, _P, _I, _I, _L, _L, _P, _P]),
    "gap_scene_gather": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "gap_scene_blend": (C.c_int, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "gap_scene_finalize": (C.c_int, [_P, _P, _I, _L, _P, _I, _P, _L, _P, _P]),
    "gap_scene_gather_one": (C.c_int, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P]),
    "gap_scene_blend_image": (C.c_int, [_P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P]),
    "gap_scene_finalize_image": (C.c_int, [_P, _P, _I, _L, _P, _I, _P]),
    "gap_bn_finalize": (C.c_int, [_P, _I, _D, _P, _P, _F, _F, _I, _P, _P, _P, _P, _P, _P, _P, _P]),
    "gap_bn_eval_scale_shift": (C.c_int, [_I, _P, _P, _P, _P, _F, _P, _P, _P]),
    "gap_bn_act": (C.c_int, [_P, _L, _P, _P, _L, _I, _P, _L, _I, _P, _L, _I, _P]),
    "gap_bn_bwd_reduce": (C.c_int, [_P, _L, _P, _L, _P, _L, _F, _P, _P, _P, _P, _L, _I, _P, _P]),
    "gap_bn_bwd_apply": (C.c_int, [_P, _L, _P, _L, _P, _L, _F, _P, _P, _P, _P, _L, _I, _P, _D, _P, _L, _P]),
    "gap_bn_param_grads": (C.c_int, [_P, _I, _P, _P, _P]),
    "gap_bn_bwd_finalize": (C.c_int, [_P, _P, _P, _I, _P, _P, _P, _P]),
    "gap_colsum_bf16": (C.c_int, [_P, _L, _L, _I, _P, _P]),
    "gap_in_stats": (C.c_int, [_P, _L, _I, _L, _I, _P, _P]),
    "gap_in_act": (C.c_int, [_P, _L, _I, _L, _I, _P, _P, _P, _L, _I, _P, _L, _I, _P]),
    "gap_in_bwd_reduce": (C.c_int, [_P, _L, _P, _L, _P, _L, _F, _P, _P, _I, _L, _I, _P, _P]),
    "gap_in_bwd_apply": (C.c_int, [_P, _L, _P, _L, _P, _L, _F, _P, _P, _I, _L, _I, _P, _P, _L, _P, _P]),
    "gap_adam_flat": (C.c_int, [_P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _I, _I, _F, _P]),
    "gap_adam_flat_devstep": (C.c_int, [_P, _P, _P, _P, _L, _F, _F, _F, _F, _F, _I, _P, _F, _P]),
    "gap_gan_losses": (C.c_int, [_P, _D, _D, _D, _P, _P]),
    "gap_pack_weights": (C.c_int, [_P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _L, _L, _L, _L, _I, _P]),
    "gap_pack_weights_multi": (C.c_int, [_P, _I, _I, _P]),
}


def lib() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python gan-aug-pfa_b200/build.py` "
                "(there is no CPU fallback for the gap_* kernels)")
        handle = C.CDLL(str(LIB_PATH))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        _lib = handle
        # bring-up A/B runs: GAP_DEBUG="knob=value,knob=value" presets gap_debug_set knobs (none are set in production)
        for item in filter(None, os.environ.get("GAP_DEBUG", "").split(",")):
            k, _, v = item.partition("=")
            DEBUG_KNOBS[k.strip()] = int(v)
            handle.gap_debug_set(k.strip().encode(), int(v))
    return _lib


LAUNCHES = 0  # gap_* kernel launches issued through this module (bench.py reports it)


def check(rc: int, what: str = "gap call") -> None:
    global LAUNCHES
    LAUNCHES += 1
    if rc != 0:
        msg = lib().gap_last_error_string().decode(errors="replace")
        raise RuntimeError(f"{what} failed (status {rc}): {msg}")


DEBUG_KNOBS: dict = {}      # what was set through debug_set (read back by tools and tests)


def debug_set(key: str, value: int) -> None:
    DEBUG_KNOBS[key] = int(value)
    lib().gap_debug_set(key.encode(), int(value))
