"""ctypes binding of libb200seg.so (the C ABI declared in include/b200seg.h).

The library is the product: there is no Python/ATen fallback.  If the shared object is missing or a call fails,
this module raises — loudly — instead of computing the result some other way.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

_PKG_DIR = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("B200SEG_LIB", _PKG_DIR.parent / "lib" / "libb200seg.so"))

B2_OK = 0
ERR_NAMES = {-1: "B2_ERR_SHAPE", -2: "B2_ERR_ALIGN", -3: "B2_ERR_ARCH", -4: "B2_ERR_CUDA", -5: "B2_ERR_NCCL",
             -6: "B2_ERR_WORKSPACE"}

_vp, _i32, _i64, _f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class ConvArgs(C.Structure):
    """struct b2_conv_args"""
    _fields_ = [("n", _i32), ("h", _i32), ("w", _i32), ("ksize", _i32),
                ("x0", _vp), ("c0", _i32), ("ldx0", _i32),
                ("x1", _vp), ("c1", _i32), ("ldx1", _i32),
                ("wpk", _vp), ("ktot", _i32), ("w_tap_stride", _i64),
                ("cout", _i32), ("y", _vp), ("ldy", _i32),
                ("bias", _vp), ("addend", _vp), ("ldadd", _i32),
                ("stats", _vp), ("relu", _i32),
                ("stride", _i32), ("out_mul", _i32), ("out_off_h", _i32), ("out_off_w", _i32),
                ("in_mul", _i32), ("in_off_h", _i32), ("in_off_w", _i32),
                ("custom_pad", _i32), ("pad_h", _i32), ("pad_w", _i32), ("add_after_act", _i32),
                ("fold_mode", _i32)]


class WgradArgs(C.Structure):
    """struct b2_wgrad_args"""
    _fields_ = [("n", _i32), ("h", _i32), ("w", _i32), ("ksize", _i32),
                ("dy", _vp), ("cout", _i32), ("lddy", _i32),
                ("x0", _vp), ("c0", _i32), ("ldx0", _i32),
                ("x1", _vp), ("c1", _i32), ("ldx1", _i32),
                ("dw", _vp), ("accumulate", _i32),
                ("workspace", _vp), ("workspace_bytes", _i64), ("x_stride", _i32),
                ("dy_mul", _i32), ("dy_off_h", _i32), ("dy_off_w", _i32),
                ("custom_pad", _i32), ("pad_h", _i32), ("pad_w", _i32), ("fold", _i32)]


class BnRunRef(C.Structure):
    """struct b2_bn_run_ref"""
    _fields_ = [("stats", _vp), ("running_mean", _vp), ("running_var", _vp), ("num_batches_tracked", _vp),
                ("count", _i64), ("c", _i32), ("momentum", C.c_float)]


class F32ConvArgs(C.Structure):
    """struct b2_f32_conv_args"""
    _fields_ = [("x0", _vp), ("x1", _vp), ("c0", _i32), ("c1", _i32), ("ldx0", _i32), ("ldx1", _i32),
                ("n", _i32), ("hi", _i32), ("wi", _i32), ("ho", _i32), ("wo", _i32),
                ("ksize", _i32), ("stride", _i32), ("pad_h", _i32), ("pad_w", _i32),
                ("w", _vp), ("bias", _vp), ("addend", _vp),
                ("ldadd", _i32), ("add_after_act", _i32), ("relu", _i32), ("cout", _i32),
                ("y", _vp), ("ldy", _i32), ("out_mul", _i32), ("out_off_h", _i32), ("out_off_w", _i32)]


class GateArgs(C.Structure):
    """struct b2_gate_args"""
    _fields_ = [("n", _i32), ("h", _i32), ("w", _i32), ("c", _i32), ("fint", _i32),
                ("g", _vp), ("ldg", _i32), ("x", _vp), ("ldx", _i32),
                ("wpk", _vp), ("bias", _vp), ("wpsi", _vp), ("bpsi", _vp), ("scale1", _vp), ("shift1", _vp),
                ("out", _vp), ("ldo", _i32)]


class GateCoef(C.Structure):
    """struct b2_gate_coef"""
    _fields_ = [(k, _vp) for k in (
        "scale_g", "shift_g", "mean_g", "invstd_g", "gamma_g",
        "scale_x", "shift_x", "mean_x", "invstd_x", "gamma_x",
        "gamma1", "mean1", "invstd1", "wpsi")]


# name -> (restype, argtypes); every symbol include/b200seg.h declares
SIGNATURES = {
    "b2_last_error": (C.c_char_p, []),
    "b2_abi_version": (C.c_int, []),
    "b2_arch_check": (C.c_int, []),
    "b2_num_sms": (C.c_int, []),
    "b2_set_deterministic": (C.c_int, [_vp, _i64]),
    "b2_det_finish": (C.c_int, [_vp, _i64, _i32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "b2_get_deterministic": (C.c_int, []),
    "b2_reload_env": (C.c_int, []),
    "b2_conv_fprop": (C.c_int, [C.POINTER(ConvArgs), _vp]),
    "b2_conv_dgrad": (C.c_int, [C.POINTER(ConvArgs), _vp]),
    "b2_conv_wgrad_workspace": (_i64, [C.POINTER(WgradArgs)]),
    "b2_conv_wgrad": (C.c_int, [C.POINTER(WgradArgs), _vp]),
    "b2_pack_weights": (C.c_int, [_vp, _i32, _i32, _i32, _i64, _i64, _i64, _i64, _vp, _vp, _vp]),
    "b2_pack_weights_folded": (C.c_int, [_vp, _i32, _i32, _i32, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _i32, _vp, _vp,
                                         _vp]),
    "b2_pack_weights_upfold": (C.c_int, [_vp, _i32, _i32, _i64, _i64, _i64, _i64, _vp, _vp, _vp]),
    "b2_fold_upconv_wgrad": (C.c_int, [_vp, _i32, _i32, _vp, _vp]),
    "b2_conv_smallc_fprop": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _vp, _i32, _vp, _i32, _i32, _vp]),
    "b2_conv_smallc_wgrad": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "b2_head_fwd": (C.c_int, [_vp, _i32, _i64, _i32, _i32, _vp, _vp, _i32, _vp, _vp]),
    "b2_head_bwd": (C.c_int, [_vp, _vp, _i32, _i64, _i32, _i32, _vp, _i32, _vp, _i32, _vp, _vp, _vp]),
    "b2_channel_stats": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _vp]),
    "b2_bn_finalize": (C.c_int, [_vp, _i32, _i64, _vp, _vp, _f32, _f32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b2_bn_update_running_multi": (C.c_int, [_vp, _i32, _i32, _vp]),
    "b2_bn_eval_coeffs": (C.c_int, [_vp, _vp, _vp, _vp, _f32, _i32, _vp, _vp, _vp, _vp, _vp]),
    "b2_bn_apply": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _vp, _i32, _vp, _i32, _vp, _i32, _vp, _i32, _vp]),
    "b2_bn_bwd_reduce": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _i32, _vp, _vp]),
    "b2_bn_bwd_apply": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _vp,
                                  _vp, _i32, _vp, _vp, _vp, _vp]),
    "b2_channel_sum": (C.c_int, [_vp, _i32, _i64, _i32, _vp, _vp]),
    "b2_maxpool2x2_fwd": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2_maxpool2x2_bwd": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2_maxpool2x2_bwd_add": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp, _i32, _vp]),
    "b2_upsample2x_fwd": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2_upsample2x_bwd": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2_add": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i32, _vp, _i32, _vp]),
    "b2_nchw_f32_to_nhwc_bf16": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2_stem_im2col3x3": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "b2_layout_nchw_to_nhwc": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2_layout_nhwc_to_nchw": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "b2_stem7x7_fprop": (C.c_int, [_vp, _i32, _i32, _i32, _vp, _i32, _vp, _i32, _vp]),
    "b2_maxpool3x3s2_fwd": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2_gate_psi_fwd": (C.c_int, [_vp, _vp, _i32, _i64, _i32, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b2_gate_apply_fwd": (C.c_int, [_vp, _i32, _vp, _i64, _i32, _vp, _vp, _vp, _vp, _i32, _vp]),
    "b2_gate_apply_bwd": (C.c_int, [_vp, _i32, _vp, _i32, _vp, _vp, _i64, _i32, _vp, _vp, _vp, _i32, _vp, _vp,
                                    _vp]),
    "b2_gate_psi_bwd_reduce": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _i32, C.POINTER(GateCoef), _vp, _i32,
                                         _vp, _vp, _vp, _vp]),
    "b2_gate_psi_bwd_apply": (C.c_int, [_vp, _vp, _vp, _vp, _i32, _i64, _i32, C.POINTER(GateCoef), _vp, _i32,
                                        _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b2_grad_sqnorm_multi": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _vp, _vp, _vp]),
    "b2_adamw_multi": (C.c_int, [_vp, _vp, _vp, _i32, _i32, _vp, _f32, _vp, _f32, _f32, _f32, _f32, _vp, _vp, _vp]),
    "b2_pack_weights_multi": (C.c_int, [_vp, _i32, _i32, _vp]),
    "b2_seg_augment": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp, C.POINTER(_f32), C.POINTER(_f32), _i32, _vp, _vp,
                                 _vp]),
    "b2_gate_fused": (C.c_int, [C.POINTER(GateArgs), _vp]),
    "b2_stem_im2col": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "b2_maxpool3x3s2_bwd": (C.c_int, [_vp, _i32, _vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2_zero_insert2x": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _vp, _i32, _vp]),
    "b2_relu_mask": (C.c_int, [_vp, _i32, _vp, _i32, _i64, _i32, _vp, _i32, _vp]),
    "b2_f32_conv": (C.c_int, [C.POINTER(F32ConvArgs), _vp]),
    "b2_f32_pack_weights": (C.c_int, [_vp, _i32, _i32, _i32, _i64, _i64, _i64, _i64, _vp, _vp, _vp, _vp, _vp, _vp]),
    "b2_f32_gate_tail": (C.c_int, [_vp, _vp, _i32, _vp, _vp, _vp, _vp, _vp, _i32, _i32, _i64, _vp, _i32, _vp]),
    "b2_f32_maxpool": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _i32, _i32, _i32, _vp, _vp]),
    "b2_f32_upsample2x": (C.c_int, [_vp, _i32, _i32, _i32, _i32, _vp, _vp]),
    "b2_f32_layout": (C.c_int, [_vp, _i32, _i32, _i64, _i32, _vp, _vp]),
    "b2_loss_fwd": (C.c_int, [_vp, _vp, _i64, _vp, _vp]),
    "b2_loss_finalize": (C.c_int, [_vp, _i64, _f32, _f32, _f32, _vp, _vp]),
    "b2_loss_bwd": (C.c_int, [_vp, _vp, _i64, _vp, _f32, _f32, _f32, _vp, _vp, _vp]),
    "b2_seg_counts": (C.c_int, [_vp, _vp, _i32, _i64, _f32, _f32, _vp, _vp]),
    "b2_logits_to_mask": (C.c_int, [_vp, _i64, _f32, _vp, _vp]),
    "b2_ce_loss_fwd": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i64, _vp, _i64, _vp, _vp]),
    "b2_ce_loss_finalize": (C.c_int, [_vp, _i32, _f32, _f32, _f32, _vp, _vp]),
    "b2_ce_loss_bwd": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i64, _vp, _i64, _vp, _f32, _f32, _f32, _vp, _vp, _vp]),
    "b2_seg_counts_mc": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i64, _i64, _vp, _vp]),
    "b2_logits_to_labels": (C.c_int, [_vp, _i32, _i32, _i64, _vp, _vp]),
    "b2_seg_augment_labels": (C.c_int, [_vp, _vp, _i32, _i32, _i32, _i32, _vp, C.POINTER(_f32), C.POINTER(_f32), _vp,
                                        _vp, _vp]),
}

_lib = None


class B2Error(RuntimeError):
    pass


def load():
    """dlopen libb200seg.so and bind every declared symbol.  Raises if the library or a symbol is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise B2Error(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                      f"or `make -C {_PKG_DIR.parent / 'csrc'}` — there is no fallback path")
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != B2_OK:
        msg = load().b2_last_error()
        raise B2Error(f"{what or 'libb200seg'} failed with {ERR_NAMES.get(rc, rc)}: "
                      f"{msg.decode() if msg else ''}")


# kernels launched per entry point (for bench.py's `gpu_launches` claim); entries not listed launch one kernel
LAUNCHES_PER_CALL = {"b2_conv_wgrad": 2, "b2_channel_sum": 1, "b2_pack_weights_folded": 2,
                     "b2_grad_sqnorm_multi": 1}
launch_count = 0


# B200SEG_NVTX=1: an NVTX range named after the entry point around every library call (SURVEY.md §5, tracing) — gives
# `ncu --nvtx --nvtx-include "b2_conv_fprop/"` and timeline tools a per-op handle; read once at import
_NVTX = os.environ.get("B200SEG_NVTX", "0") not in ("", "0")


def call(name: str, *args):
    """Call an int-returning entry point and raise on a non-zero code."""
    global launch_count
    if _NVTX:
        from torch.cuda import nvtx
        nvtx.range_push(name)
        try:
            rc = getattr(load(), name)(*args)
        finally:
            nvtx.range_pop()
    else:
        rc = getattr(load(), name)(*args)
    check(rc, name)
    launch_count += LAUNCHES_PER_CALL.get(name, 1)
