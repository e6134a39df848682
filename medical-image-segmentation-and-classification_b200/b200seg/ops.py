"""torch.library custom ops (namespace `b200seg`) with autograd, built on the C ABI wrappers in kernels.py.

Internal activation format: NHWC bf16 tensors [N, H, W, C].  Parameters stay ordinary fp32 nn.Parameters in the
reference's shapes; their bf16 MMA-layout copies are cached per parameter (kernels.packed) and refreshed by the fused
optimizer in one multi-tensor launch per step.

Each op cites the reference lines whose ATen dispatch it replaces.  There is no fallback: every op launches
kernels of libb200seg.so or raises.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import torch
from torch import Tensor
from torch.library import custom_op

from . import kernels as K

_F64 = torch.float64


def _c(t: Optional[Tensor]) -> Optional[Tensor]:
    return t if t is None or t.is_contiguous() else t.contiguous()


def _dw_as_param_grad(dw: Tensor, weight: Tensor) -> Tensor:
    """[Cout, taps, Cin] fp32 -> logical [Cout, Cin, k, k] (channels_last memory, zero copy)."""
    cout, cin, k, _ = weight.shape
    return dw.view(cout, k, k, cin).permute(0, 3, 1, 2)


# ----------------------------------------------------------------------------------------------------------
# layout adapters (module boundary; helpers.py:318 hands the model an NCHW fp32 batch)
# ----------------------------------------------------------------------------------------------------------
@custom_op("b200seg::to_nhwc", mutates_args=())
def to_nhwc(x: Tensor) -> Tensor:
    return K.to_nhwc_bf16(_c(x))


@custom_op("b200seg::to_nchw", mutates_args=())
def to_nchw(x: Tensor) -> Tensor:
    return K.to_nchw_f32(_c(x))


to_nhwc.register_autograd(lambda ctx, g: to_nchw(_c(g)))
to_nchw.register_autograd(lambda ctx, g: to_nhwc(_c(g)))


@to_nhwc.register_fake
def _(x):
    n, c, h, w = x.shape
    return x.new_empty((n, h, w, c), dtype=torch.bfloat16)


@to_nchw.register_fake
def _(x):
    n, h, w, c = x.shape
    return x.new_empty((n, c, h, w), dtype=torch.float32)


# ----------------------------------------------------------------------------------------------------------
# convolution (tcgen05 implicit GEMM): nn.Conv2d 3x3 p1 / 1x1, stride 1
#   AttentionUNet.py:6,9,20,33,37  R2U_Net.py:10,27,43  ResnetUnet.py:7,10,54 ; x1 = elided torch.cat partner
# ----------------------------------------------------------------------------------------------------------
@custom_op("b200seg::conv2d", mutates_args=())
def conv2d(x0: Tensor, x1: Optional[Tensor], weight: Tensor, bias: Optional[Tensor],
           want_stats: bool) -> Tuple[Tensor, Tensor]:
    cout, cin, k, _ = weight.shape
    wf, _ = K.packed(weight)
    stats = torch.zeros((2, cout), dtype=_F64, device=x0.device) if want_stats else \
        torch.empty((0,), dtype=_F64, device=x0.device)
    y = K.conv_igemm(_c(x0), wf, cout, k, x1=_c(x1), bias=bias, stats=stats if want_stats else None)
    return y, stats


@conv2d.register_fake
def _(x0, x1, weight, bias, want_stats):
    n, h, w, _ = x0.shape
    cout = weight.shape[0]
    return (x0.new_empty((n, h, w, cout)),
            x0.new_empty((2, cout) if want_stats else (0,), dtype=_F64))


@custom_op("b200seg::conv2d_bwd", mutates_args=())
def conv2d_bwd(dy: Tensor, x0: Tensor, x1: Optional[Tensor], weight: Tensor, need_dx0: bool, need_dx1: bool,
               need_dw: bool, need_db: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    """aten::convolution_backward: dgrad (same kernel, flipped/transposed packing), wgrad, bias grad."""
    cout, cin, k, _ = weight.shape
    dev = dy.device
    dy = _c(dy)
    c0 = x0.shape[3]
    dx0 = torch.empty((0,), dtype=torch.bfloat16, device=dev)
    dx1 = torch.empty((0,), dtype=torch.bfloat16, device=dev)
    if need_dx0 or need_dx1:
        _, wd = K.packed(weight, want_dgrad=True)
        if need_dx0:
            dx0 = K.conv_igemm(dy, wd, c0, k, row_offset=0, dgrad=True)
        if need_dx1 and x1 is not None:
            dx1 = K.conv_igemm(dy, wd, x1.shape[3], k, row_offset=c0, dgrad=True)
    if need_dw:
        x0c, x1c = _c(x0), _c(x1)
        with K.wgrad_stream(dy, x0c, x1c, allow=K.grad_is_stolen(weight)):
            dw = K.conv_wgrad(dy, x0c, k, x1=x1c, out=K.grad_slot(weight, (cout, k * k, cin)))
    else:
        dw = torch.empty((0,), device=dev)
    db = K.channel_sum(dy) if need_db else torch.empty((0,), device=dev)
    return dx0, dx1, dw, db


def _conv2d_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)      # unused outputs (z, coef, stats, ...) must not get zero-filled grads
    x0, x1, weight, bias, _ = inputs
    ctx.save_for_backward(x0, x1, weight)
    ctx.has_bias = bias is not None


def _conv2d_backward(ctx, dy, _dstats):
    x0, x1, weight = ctx.saved_tensors
    need = ctx.needs_input_grad
    dx0, dx1, dw, db = conv2d_bwd(dy, x0, x1, weight, need[0], bool(need[1]) and x1 is not None, need[2],
                                  bool(need[3]) and ctx.has_bias)
    return (dx0 if need[0] else None,
            dx1 if (need[1] and x1 is not None) else None,
            _dw_as_param_grad(dw, weight) if need[2] else None,
            db if (need[3] and ctx.has_bias) else None,
            None)


conv2d.register_autograd(_conv2d_backward, setup_context=_conv2d_setup)


# ----------------------------------------------------------------------------------------------------------
# image stem: Cin <= 4 direct convolution from the NCHW fp32 batch
#   AttentionUNet.py:6 (basic_block(3,64) first conv), R2U_Net.py:43 (RRCNN1.conv_1x1, 3 -> 64)
# ----------------------------------------------------------------------------------------------------------
_STEM_GEMM = os.environ.get("B200SEG_STEM_GEMM", "1") != "0"     # 0: CUDA-core stem kernels (A/B switch)


def _stem_as_gemm(weight) -> bool:
    """3x3 stem with <= 3 input channels and a tensor-core-sized Cout: im2col (K = 32) + the tcgen05 1x1 kernels."""
    cout, cin, k, _ = weight.shape
    return k == 3 and cin <= 3 and cout % 32 == 0 and _STEM_GEMM


@custom_op("b200seg::stem_conv", mutates_args=())
def stem_conv(x: Tensor, weight: Tensor, bias: Optional[Tensor], want_stats: bool) -> Tuple[Tensor, Tensor, Tensor]:
    cout, cin, k, _ = weight.shape
    stats = (torch.zeros((2, cout), dtype=_F64, device=x.device) if want_stats
             else torch.empty((0,), dtype=_F64, device=x.device))
    if _stem_as_gemm(weight):
        x4 = K.stem_im2col3x3(_c(x))
        wf, _ = K.packed(weight, "stem")
        y = K.conv_igemm(x4, wf, cout, 1, bias=bias, stats=stats if want_stats else None)
        return y, stats, x4
    x4 = K.image_to_nhwc4(_c(x))
    y = K.conv_smallc_fprop(x4, K.pack_small_weight(weight), bias, k)
    if want_stats:
        K.channel_stats(y, stats)
    return y, stats, x4


@custom_op("b200seg::stem_conv_bwd", mutates_args=())
def stem_conv_bwd(dy: Tensor, x4: Tensor, weight: Tensor, need_db: bool) -> Tuple[Tensor, Tensor]:
    cout, cin, k, _ = weight.shape
    dy = _c(dy)
    if x4.shape[-1] == K.STEM_COLS:
        dwk = K.stem_weight_grad(K.conv_wgrad(dy, x4, 1), cin)     # [cout, taps, cin]
    else:
        dwk = K.conv_smallc_wgrad(dy, x4, k)                       # [cout, taps, 4]
    dw = dwk[:, :, :cin].reshape(cout, k, k, cin).permute(0, 3, 1, 2).contiguous()
    db = K.channel_sum(dy) if need_db else torch.empty((0,), device=dy.device)
    return dw, db


def _stem_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)      # unused outputs (z, coef, stats, ...) must not get zero-filled grads
    _, weight, bias, _ = inputs
    ctx.save_for_backward(output[2], weight)
    ctx.has_bias = bias is not None


def _stem_backward(ctx, dy, _ds, _dx4):
    x4, weight = ctx.saved_tensors
    dw, db = stem_conv_bwd(dy, x4, weight, ctx.has_bias)
    return None, dw, (db if ctx.has_bias else None), None


stem_conv.register_autograd(_stem_backward, setup_context=_stem_setup)


@stem_conv.register_fake
def _(x, weight, bias, want_stats):
    n, _, h, w = x.shape
    cout = weight.shape[0]
    return (x.new_empty((n, h, w, cout), dtype=torch.bfloat16),
            x.new_empty((2, cout) if want_stats else (0,), dtype=_F64),
            x.new_empty((n, h, w, K.STEM_COLS if _stem_as_gemm(weight) else 4), dtype=torch.bfloat16))


# ----------------------------------------------------------------------------------------------------------
# BatchNorm2d (+ReLU): AttentionUNet.py:7-8,10-11,21-22  R2U_Net.py:11-12,28-29  ResnetUnet.py:8-9,11-12,55-56
#   bn_finalize_ : statistics -> (mean, invstd, scale, shift); the ONLY op that mutates the running buffers
#   bn_apply     : functional normalise(+ReLU) with the full BatchNorm backward (dz, dgamma, dbeta)
# ----------------------------------------------------------------------------------------------------------
@custom_op("b200seg::bn_finalize_", mutates_args=("running_mean", "running_var", "num_batches_tracked"))
def bn_finalize_(stats: Tensor, count: int, gamma: Tensor, beta: Tensor, running_mean: Tensor, running_var: Tensor,
                 num_batches_tracked: Tensor, training: bool, momentum: float, eps: float) -> Tensor:
    if training:
        return K.bn_finalize(stats, count, gamma, beta, eps, momentum, running_mean, running_var,
                             num_batches_tracked)
    return K.bn_eval_coeffs(gamma, beta, running_mean, running_var, eps)


@bn_finalize_.register_fake
def _(stats, count, gamma, beta, rm, rv, nbt, training, momentum, eps):
    return gamma.new_empty((4, gamma.shape[0]), dtype=torch.float32)


@custom_op("b200seg::bn_apply", mutates_args=())
def bn_apply(z: Tensor, coef: Tensor, gamma: Tensor, beta: Tensor, relu: bool, training: bool) -> Tensor:
    return K.bn_apply(_c(z), coef, relu=relu)


@bn_apply.register_fake
def _(z, coef, gamma, beta, relu, training):
    return torch.empty_like(z)


@custom_op("b200seg::bn_apply_bwd", mutates_args=())
def bn_apply_bwd(dy: Tensor, z: Tensor, coef: Tensor, gamma: Tensor, relu: bool,
                 training: bool) -> Tuple[Tensor, Tensor, Tensor]:
    return K.bn_bwd(_c(dy), z, coef, gamma, relu=relu, training=training)


def _bn_setup(ctx, inputs, output):
    z, coef, gamma, _beta, ctx.relu, ctx.training = inputs
    ctx.save_for_backward(_c(z), coef, gamma)


def _bn_backward(ctx, dy):
    z, coef, gamma = ctx.saved_tensors
    dz, dgamma, dbeta = bn_apply_bwd(dy, z, coef, gamma, ctx.relu, ctx.training)
    return dz, None, dgamma, dbeta, None, None


bn_apply.register_autograd(_bn_backward, setup_context=_bn_setup)


def batch_norm_act(z: Tensor, stats: Tensor, bn: torch.nn.BatchNorm2d, relu: bool) -> Tensor:
    """nn.BatchNorm2d(+ReLU) on a conv output whose epilogue already produced `stats`."""
    n, h, w, _ = z.shape
    training = bn.training or bn.running_mean is None
    coef = bn_finalize_(stats.detach(), n * h * w, bn.weight.detach(), bn.bias.detach(), bn.running_mean, bn.running_var,
                        bn.num_batches_tracked, training, float(bn.momentum), float(bn.eps))
    return bn_apply(z, coef, bn.weight, bn.bias, relu, training)


# ----------------------------------------------------------------------------------------------------------
# fused conv -> BatchNorm -> (ReLU): one autograd node for [Conv2d, BatchNorm2d, ReLU] of basic_block / UpConv /
# Recurrent_block (AttentionUNet.py:6-8,9-11,20-22; R2U_Net.py:10-12,27-29; ResnetUnet.py:7-12,54-56).
# Functional: batch statistics come back as `stats`; the caller applies the running-stat momentum update with
# bn_update_running_.  Backward = BN backward (2 passes, the second also yields the conv bias gradient) -> dgrad
# -> wgrad.  x0 may be the fp32 NCHW image (<= 4 channels): the CUDA-core stem kernels are used then.
# ----------------------------------------------------------------------------------------------------------
@custom_op("b200seg::conv_bn_act", mutates_args=())
def conv_bn_act(x0: Tensor, x1: Optional[Tensor], weight: Tensor, bias: Optional[Tensor], gamma: Tensor,
                beta: Tensor, running_mean: Tensor, running_var: Tensor, training: bool, eps: float,
                relu: bool, addend: Optional[Tensor] = None, share_index: int = 0,
                share_count: int = 1) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    """`addend`: the first output becomes act(bn(conv(x))) + addend (Recurrent_block's x + x1, R2U_Net.py:19); the
    un-summed activation is then never written.  `share_index` / `share_count`: this is application number
    share_index of share_count sequentially dependent applications of the SAME conv weight (Recurrent_block's t+1 uses,
    R2U_Net.py:15-20): their weight gradients are accumulated by the wgrad kernel into one buffer that the node of
    application 0 — the last to run in backward — hands to autograd, the others return no weight gradient."""
    cout, cin, k, _ = weight.shape
    dev = x0.device
    stats = K.zeros_scratch((2, cout), _F64, dev) if training else torch.empty((0,), dtype=_F64, device=dev)
    if x0.dtype != torch.bfloat16 and _stem_as_gemm(weight):   # image stem on the tensor cores (im2col, K = 32)
        x4 = K.stem_im2col3x3(_c(x0))
        wf, _ = K.packed(weight, "stem")
        z = K.conv_igemm(x4, wf, cout, 1, bias=bias, stats=stats if training else None)
    elif x0.dtype != torch.bfloat16:                      # other small-channel stems: CUDA-core kernels
        x4 = K.image_to_nhwc4(_c(x0))
        z = K.conv_smallc_fprop(x4, K.pack_small_weight(weight), bias, k)
        if training:
            K.channel_stats(z, stats)
    else:
        x4 = torch.empty((0,), dtype=torch.bfloat16, device=dev)
        wf, _ = K.packed(weight)
        z = K.conv_igemm(_c(x0), wf, cout, k, x1=_c(x1), bias=bias, stats=stats if training else None)
    n, h, w, _ = z.shape
    if training:
        coef = K.bn_finalize(stats, n * h * w, gamma, beta, eps, 0.0, None, None, None)
    else:
        coef = K.bn_eval_coeffs(gamma, beta, running_mean, running_var, eps)
    if addend is not None:
        return K.bn_apply(z, coef, relu=relu, addend=_c(addend), sum_only=True), z, coef, stats, x4
    return K.bn_apply(z, coef, relu=relu), z, coef, stats, x4


@conv_bn_act.register_fake
def _(x0, x1, weight, bias, gamma, beta, rm, rv, training, eps, relu, addend=None, share_index=0, share_count=1):
    cout = weight.shape[0]
    if x0.dtype != torch.bfloat16:
        n, _, h, w = x0.shape
        x4 = x0.new_empty((n, h, w, K.STEM_COLS if _stem_as_gemm(weight) else 4), dtype=torch.bfloat16)
    else:
        n, h, w, _ = x0.shape
        x4 = x0.new_empty((0,), dtype=torch.bfloat16)
    y = x0.new_empty((n, h, w, cout), dtype=torch.bfloat16)
    return (y, torch.empty_like(y), x0.new_empty((4, cout), dtype=torch.float32),
            x0.new_empty((2, cout) if training else (0,), dtype=_F64), x4)


_SHARED_DW = {}      # (weight address, device) -> fp32 gradient buffer of a shared conv weight, alive within one backward


@custom_op("b200seg::conv_bn_act_bwd", mutates_args=())
def conv_bn_act_bwd(dy: Tensor, x0: Tensor, x1: Optional[Tensor], x4: Tensor, weight: Tensor, z: Tensor,
                    coef: Tensor, gamma: Tensor, relu: bool, training: bool, need_dx0: bool, need_dx1: bool,
                    has_bias: bool, share_index: int = 0,
                    share_count: int = 1) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    cout, cin, k, _ = weight.shape
    dev = dy.device
    res = K.bn_bwd(_c(dy), z, coef, gamma, relu=relu, training=training, want_dbias=has_bias)
    dz, dgamma, dbeta = res[0], res[1], res[2]
    db = res[3] if has_bias else torch.empty((0,), device=dev)
    dx0 = torch.empty((0,), dtype=torch.bfloat16, device=dev)
    dx1 = torch.empty((0,), dtype=torch.bfloat16, device=dev)
    if x4.numel() > 0 and x4.shape[-1] == K.STEM_COLS:    # stem as a GEMM: no input gradient
        dw = K.stem_weight_grad(K.conv_wgrad(dz, x4, 1), cin)
    elif x4.numel() > 0:                                  # stem: no input gradient
        dwk = K.conv_smallc_wgrad(dz, x4, k)
        dw = dwk[:, :, :cin].reshape(cout, k * k, cin).contiguous()
    else:
        c0 = x0.shape[3]
        if need_dx0 or need_dx1:
            _, wd = K.packed(weight, want_dgrad=True)
            if need_dx0:
                dx0 = K.conv_igemm(dz, wd, c0, k, row_offset=0, dgrad=True)
            if need_dx1 and x1 is not None:
                dx1 = K.conv_igemm(dz, wd, x1.shape[3], k, row_offset=c0, dgrad=True)
        with K.wgrad_stream(dz, x0, x1, allow=K.grad_is_stolen(weight)):
            if share_count <= 1:
                dw = K.conv_wgrad(dz, x0, k, x1=x1, out=K.grad_slot(weight, (cout, k * k, cin)))
            else:
                # shared weight: backward visits the applications in reverse order (each consumes the previous one's
                # output), so the last application opens the buffer, the others add to it, application 0 returns it
                key = (weight.data_ptr(), dz.device.index)
                buf = None if share_index == share_count - 1 else _SHARED_DW.get(key)
                if buf is None:
                    buf = K.conv_wgrad(dz, x0, k, x1=x1, out=K.grad_slot(weight, (cout, k * k, cin)))
                else:
                    K.conv_wgrad(dz, x0, k, x1=x1, out=buf, accumulate=True)
                if share_index == 0:
                    _SHARED_DW.pop(key, None)
                    dw = buf
                else:
                    _SHARED_DW[key] = buf
                    dw = torch.empty((0,), device=dev)
    return dx0, dx1, dw, db, dgamma, dbeta


def _cba_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)      # unused outputs (z, coef, stats, ...) must not get zero-filled grads
    (x0, x1, weight, bias, gamma, _beta, _rm, _rv, ctx.training, _eps, ctx.relu, addend, ctx.share_index,
     ctx.share_count) = inputs
    ctx.has_addend = addend is not None
    _y, z, coef, _stats, x4 = output
    stem = x0.dtype != torch.bfloat16
    ctx.save_for_backward(None if stem else _c(x0), _c(x1), x4, weight, z, coef, gamma)
    ctx.has_bias = bias is not None
    ctx.stem = stem


def _cba_backward(ctx, dy, *_unused):
    x0, x1, x4, weight, z, coef, gamma = ctx.saved_tensors
    need = ctx.needs_input_grad
    need0 = bool(need[0]) and not ctx.stem
    need1 = bool(need[1]) and x1 is not None
    dx0, dx1, dw, db, dgamma, dbeta = conv_bn_act_bwd(dy, x0 if x0 is not None else x4, x1, x4, weight, z, coef,
                                                      gamma, ctx.relu, ctx.training, need0, need1, ctx.has_bias,
                                                      ctx.share_index, ctx.share_count)
    return (dx0 if need0 else None, dx1 if need1 else None,
            _dw_as_param_grad(dw, weight) if dw.numel() > 0 else None,
            db if ctx.has_bias else None, dgamma, dbeta, None, None, None, None, None,
            dy if (ctx.has_addend and need[11]) else None, None, None)   # d(addend) = d(output): the sum is linear


conv_bn_act.register_autograd(_cba_backward, setup_context=_cba_setup)


@custom_op("b200seg::bn_update_running_", mutates_args=("running_mean", "running_var", "num_batches_tracked"))
def bn_update_running_(stats: Tensor, count: int, momentum: float, running_mean: Tensor, running_var: Tensor,
                       num_batches_tracked: Tensor) -> None:
    """running_mean/var momentum update (unbiased variance) + num_batches_tracked += 1, from epilogue statistics"""
    K.bn_update_running(stats, count, momentum, running_mean, running_var, num_batches_tracked)


def conv_bn_act_module(x, conv: torch.nn.Conv2d, bn: torch.nn.BatchNorm2d, relu: bool = True,
                       addend: Optional[Tensor] = None, share_index: int = 0, share_count: int = 1) -> Tensor:
    """[Conv2d -> BatchNorm2d -> ReLU] (+ addend) on module objects; x: image | activation | (activation, activation)."""
    x0, x1 = x if isinstance(x, tuple) else (x, None)
    training = bn.training or bn.running_mean is None
    if x0.dtype == torch.bfloat16 and os.environ.get("B200SEG_FOLD_BN", "1") != "0":
        from . import ops_infer
        if ops_infer.inference_mode(bn):       # eval + no_grad: conv with folded BN, bias/ReLU in the epilogue
            return ops_infer.conv_bn_act_infer(x0, x1, conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean,
                                               bn.running_var, float(bn.eps), relu, addend)
    y, _z, _coef, stats, _x4 = conv_bn_act(x0, x1, conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean,
                                           bn.running_var, training, float(bn.eps), relu, addend, share_index,
                                           share_count)
    if training:
        n, h, w, _ = y.shape
        bn_update_running_(stats.detach(), n * h * w, float(bn.momentum), bn.running_mean, bn.running_var,
                           bn.num_batches_tracked)
    return y


# ----------------------------------------------------------------------------------------------------------
# UpConv = Upsample(x2, nearest) -> Conv3x3 -> BN -> ReLU (AttentionUNet.py:15-27, R2U_Net.py:22-34), folded:
# phase (a,b) of the 2x grid is a 2x2 convolution of the LOW-resolution input with summed weights, so the upsampled
# tensor is never built and the three GEMMs (fprop, dgrad, wgrad) do 16/36 of the reference's FLOPs.  Exact algebra;
# the only numerical difference is that the 3x3 taps are summed in fp32 before the bf16 rounding of the weights.
# ----------------------------------------------------------------------------------------------------------
_PHASES = ((0, 0), (0, 1), (1, 0), (1, 1))


@custom_op("b200seg::upconv_bn_act", mutates_args=())
def upconv_bn_act(x: Tensor, weight: Tensor, bias: Optional[Tensor], gamma: Tensor, beta: Tensor,
                  running_mean: Tensor, running_var: Tensor, training: bool, eps: float,
                  relu: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    cout, cin, _, _ = weight.shape
    x = _c(x)
    n, h, w, _ = x.shape
    dev = x.device
    stats = K.zeros_scratch((2, cout), _F64, dev) if training else torch.empty((0,), dtype=_F64, device=dev)
    wf, _ = K.packed(weight, "upfold")
    z = K.new_act(n, 2 * h, 2 * w, cout, dev)
    if cout % 64 == 0 and cin % 64 == 0:
        # all four phase convolutions in ONE launch (the phase is an extra tile dimension, pixel-shuffle TMA stores)
        K.conv_igemm(x, wf.view(16, cout, cin), cout, 2, bias=bias, stats=stats if training else None, out=z, fold=1,
                     alg_scale=2.25)
    else:
        for ph, (a, b) in enumerate(_PHASES):
            K.conv_igemm(x, wf[ph], cout, 2, bias=bias, stats=stats if training else None, out=z, out_mul=2,
                         out_off=(a, b), pad=(1 - a, 1 - b), alg_scale=2.25)
    if training:
        coef = K.bn_finalize(stats, n * 4 * h * w, gamma, beta, eps, 0.0, None, None, None)
    else:
        coef = K.bn_eval_coeffs(gamma, beta, running_mean, running_var, eps)
    return K.bn_apply(z, coef, relu=relu), z, coef, stats


@upconv_bn_act.register_fake
def _(x, weight, bias, gamma, beta, rm, rv, training, eps, relu):
    n, h, w, _ = x.shape
    cout = weight.shape[0]
    y = x.new_empty((n, 2 * h, 2 * w, cout))
    return (y, torch.empty_like(y), x.new_empty((4, cout), dtype=torch.float32),
            x.new_empty((2, cout) if training else (0,), dtype=_F64))


@custom_op("b200seg::upconv_bn_act_bwd", mutates_args=())
def upconv_bn_act_bwd(dy: Tensor, x: Tensor, weight: Tensor, z: Tensor, coef: Tensor, gamma: Tensor, relu: bool,
                      training: bool, need_dx: bool, has_bias: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    cout, cin, _, _ = weight.shape
    dev = dy.device
    res = K.bn_bwd(_c(dy), z, coef, gamma, relu=relu, training=training, want_dbias=has_bias)
    dz, dgamma, dbeta = res[0], res[1], res[2]
    db = res[3] if has_bias else torch.empty((0,), device=dev)
    n, h, w, _ = x.shape
    if need_dx:
        _, wd = K.packed(weight, "upfold", want_dgrad=True)
        dx = K.new_act(n, h, w, cin, dev)
        if cout % 64 == 0 and cin % 64 == 0:
            # the four phases as ONE K loop of 16 taps over the sub-lattices of dz: one launch, one epilogue per tile
            K.conv_igemm(dz, wd.view(16, cin, cout), cin, 2, out=dx, dgrad=True, fold=2, alg_scale=2.25)
        else:
            for ph, (a, b) in enumerate(_PHASES):
                # 2x2 conv of the (a,b) sub-lattice of dz with the flipped/transposed phase weights, chained through
                # the epilogue's addend so the four phases sum into one dx
                K.conv_igemm(dz, wd[ph], cin, 2, addend=dx if ph > 0 else None, out=dx, dgrad=True, in_mul=2,
                             in_off=(a, b), pad=(a, b), alg_scale=2.25)
    else:
        dx = torch.empty((0,), dtype=torch.bfloat16, device=dev)
    with K.wgrad_stream(dz, x, allow=K.grad_is_stolen(weight)):
        dweff = torch.empty((4, cout, 4, cin), dtype=torch.float32, device=dev)
        # all four phases in ONE launch (every X row fetched once per filter row, the two column phases share it)
        merged = (cout == 64 or cout % 128 == 0) and cin % 64 == 0 and \
            K.conv_wgrad(dz, x, 2, out=dweff, dy_mul=2, fold=True, alg_scale=2.25) is not None
        if not merged:
            for ph, (a, b) in enumerate(_PHASES):
                K.conv_wgrad(dz, x, 2, out=dweff[ph], dy_mul=2, dy_off=(a, b), pad=(1 - a, 1 - b), alg_scale=2.25)
        dw = K.fold_upconv_wgrad(dweff, out=K.grad_slot(weight, (cout, 9, cin)))
    return dx, dw, db, dgamma, dbeta


def _ucba_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)
    x, weight, bias, gamma, _beta, _rm, _rv, ctx.training, _eps, ctx.relu = inputs
    _y, z, coef, _stats = output
    ctx.save_for_backward(_c(x), weight, z, coef, gamma)
    ctx.has_bias = bias is not None


def _ucba_backward(ctx, dy, *_unused):
    x, weight, z, coef, gamma = ctx.saved_tensors
    need_dx = bool(ctx.needs_input_grad[0])
    dx, dw, db, dgamma, dbeta = upconv_bn_act_bwd(dy, x, weight, z, coef, gamma, ctx.relu, ctx.training, need_dx,
                                                  ctx.has_bias)
    return (dx if need_dx else None, _dw_as_param_grad(dw, weight), db if ctx.has_bias else None, dgamma, dbeta,
            None, None, None, None, None)


upconv_bn_act.register_autograd(_ucba_backward, setup_context=_ucba_setup)


def upconv_bn_act_module(x: Tensor, conv: torch.nn.Conv2d, bn: torch.nn.BatchNorm2d, relu: bool = True) -> Tensor:
    training = bn.training or bn.running_mean is None
    if os.environ.get("B200SEG_FOLD_BN", "1") != "0":
        from . import ops_infer
        if ops_infer.inference_mode(bn):
            return ops_infer.upconv_bn_act_infer(x, conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean,
                                                 bn.running_var, float(bn.eps), relu)
    y, _z, _coef, stats = upconv_bn_act(x, conv.weight, conv.bias, bn.weight, bn.bias, bn.running_mean,
                                        bn.running_var, training, float(bn.eps), relu)
    if training:
        n, h, w, _ = y.shape
        bn_update_running_(stats.detach(), n * h * w, float(bn.momentum), bn.running_mean, bn.running_var,
                           bn.num_batches_tracked)
    return y


# ----------------------------------------------------------------------------------------------------------
# pooling / upsampling / add
# ----------------------------------------------------------------------------------------------------------
@custom_op("b200seg::maxpool2x2", mutates_args=())
def maxpool2x2(x: Tensor) -> Tensor:
    """nn.MaxPool2d(2, 2): AttentionUNet.py:61, R2U_Net.py:54"""
    return K.maxpool_fwd(_c(x))


@custom_op("b200seg::maxpool2x2_bwd", mutates_args=())
def maxpool2x2_bwd(dy: Tensor, x: Tensor) -> Tensor:
    return K.maxpool_bwd(_c(dy), x)


maxpool2x2.register_autograd(lambda ctx, dy: maxpool2x2_bwd(dy, ctx.saved_tensors[0]),
                             setup_context=lambda ctx, inputs, output: ctx.save_for_backward(_c(inputs[0])))


@maxpool2x2.register_fake
def _(x):
    n, h, w, c = x.shape
    return x.new_empty((n, h // 2, w // 2, c))


class _MaxPoolPass(torch.autograd.Function):
    """(pool(x), x): the skip tensor of a U-Net level feeds the pool AND the decoder (gate / concat).  Handing the
    decoder the pass-through output makes this node x's only consumer, so the decoder-side gradient arrives here and
    is added inside the pool-backward kernel (b2_maxpool2x2_bwd_add) instead of autograd's separate accumulation
    pass over the full-size tensor (AttentionUNet.py:88-101; R2U_Net.py:78-95)."""

    @staticmethod
    def forward(ctx, x):
        xc = _c(x)
        ctx.save_for_backward(xc)
        ctx.set_materialize_grads(False)
        return K.maxpool_fwd(xc), x

    @staticmethod
    def backward(ctx, dy, dpass):
        (x,) = ctx.saved_tensors
        if dy is None:
            return dpass
        return K.maxpool_bwd(_c(dy), x, addend=_c(dpass) if dpass is not None else None)


_POOL_PASS = os.environ.get("B200SEG_POOL_PASS", "1") != "0"      # 0: plain pool, autograd accumulates (A/B switch)


def maxpool2x2_pass(x: Tensor) -> Tuple[Tensor, Tensor]:
    """-> (MaxPool2d(2, 2)(x), x as the tensor the decoder should consume)"""
    if not _POOL_PASS or not (torch.is_grad_enabled() and x.requires_grad):
        return maxpool2x2(x), x
    return _MaxPoolPass.apply(x)


@custom_op("b200seg::upsample2x", mutates_args=())
def upsample2x(x: Tensor) -> Tensor:
    """nn.Upsample(scale_factor=2) (nearest): AttentionUNet.py:18, R2U_Net.py:25"""
    return K.upsample_fwd(_c(x))


@custom_op("b200seg::upsample2x_bwd", mutates_args=())
def upsample2x_bwd(dy: Tensor) -> Tensor:
    return K.upsample_bwd(_c(dy))


upsample2x.register_autograd(lambda ctx, dy: upsample2x_bwd(dy))


@upsample2x.register_fake
def _(x):
    n, h, w, c = x.shape
    return x.new_empty((n, 2 * h, 2 * w, c))


@custom_op("b200seg::add", mutates_args=())
def add(a: Tensor, b: Tensor) -> Tensor:
    """x + x1 on activations: R2U_Net.py:19,48"""
    return K.add(_c(a), _c(b))


add.register_autograd(lambda ctx, g: (g, g))


@add.register_fake
def _(a, b):
    return torch.empty_like(a)


# ----------------------------------------------------------------------------------------------------------
# attention gate, everything after the two 1x1 GEMMs: AttentionUNet.py:48-54 / R2AttU_Net.py:80-86
# (functional: psi.1's running statistics are updated by the caller from the returned qstats)
# ----------------------------------------------------------------------------------------------------------
@custom_op("b200seg::gate_mid", mutates_args=())
def gate_mid(g1p: Tensor, x1p: Tensor, x: Tensor, coef_g: Tensor, coef_x: Tensor,
             gamma_g: Tensor, beta_g: Tensor, gamma_x: Tensor, beta_x: Tensor,
             wpsi: Tensor, bpsi: Tensor, gamma_1: Tensor, beta_1: Tensor, rm_1: Tensor, rv_1: Tensor,
             training: bool, eps: float) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor]:
    n, h, w, fint = g1p.shape
    q, qstats = K.gate_psi_fwd(_c(g1p), _c(x1p), coef_g, coef_x, wpsi, bpsi)
    if training:
        coef_1 = K.bn_finalize(qstats, n * h * w, gamma_1, beta_1, eps, 0.0, None, None, None)
    else:
        coef_1 = K.bn_eval_coeffs(gamma_1, beta_1, rm_1, rv_1, eps)
    out, psi = K.gate_apply_fwd(_c(x), q, coef_1)
    return out, q, psi, coef_1, qstats


@gate_mid.register_fake
def _(g1p, x1p, x, *rest):
    n, h, w, fint = g1p.shape
    return (torch.empty_like(x), x.new_empty((n, h, w)), x.new_empty((n, h, w)),
            x.new_empty((4, 1), dtype=torch.float32), x.new_empty((2,), dtype=_F64))


@custom_op("b200seg::gate_mid_bwd", mutates_args=())
def gate_mid_bwd(dout: Tensor, x: Tensor, psi: Tensor, q: Tensor, g1p: Tensor, x1p: Tensor, coef_g: Tensor,
                 gamma_g: Tensor, coef_x: Tensor, gamma_x: Tensor, coef_1: Tensor, gamma_1: Tensor, wpsi: Tensor,
                 training: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    dx, dsig, sums1 = K.gate_apply_bwd(_c(dout), x, psi, q, coef_1)
    dg1p, dx1p, dgb, dbn1, dwpsi, dbpsi, _dbias = K.gate_psi_bwd(dsig, sums1, q, g1p, x1p, coef_g, gamma_g, coef_x, gamma_x,
                                                         coef_1, gamma_1, wpsi, training=training)
    return dg1p, dx1p, dx, dgb, dbn1, dwpsi, dbpsi


def _gate_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)      # unused outputs (z, coef, stats, ...) must not get zero-filled grads
    (g1p, x1p, x, coef_g, coef_x, gamma_g, _bg, gamma_x, _bx, wpsi, _bpsi, gamma_1, _b1, _rm1, _rv1, training,
     _eps) = inputs
    out, q, psi, coef_1, _qstats = output
    ctx.save_for_backward(_c(x), psi, q, _c(g1p), _c(x1p), coef_g, gamma_g, coef_x, gamma_x, coef_1, gamma_1, wpsi)
    ctx.training = training


def _gate_backward(ctx, dout, *_unused):
    x, psi, q, g1p, x1p, coef_g, gamma_g, coef_x, gamma_x, coef_1, gamma_1, wpsi = ctx.saved_tensors
    dg1p, dx1p, dx, dgb, dbn1, dwpsi, dbpsi = gate_mid_bwd(dout, x, psi, q, g1p, x1p, coef_g, gamma_g, coef_x,
                                                           gamma_x, coef_1, gamma_1, wpsi, ctx.training)
    return (dg1p, dx1p, dx, None, None,
            dgb[0], dgb[1], dgb[2], dgb[3],
            dwpsi.view_as(wpsi), dbpsi, dbn1[0:1], dbn1[1:2], None, None,
            None, None)


gate_mid.register_autograd(_gate_backward, setup_context=_gate_setup)


# ----------------------------------------------------------------------------------------------------------
# 1x1 heads -> fp32 NCHW logits: AttentionUNet.py:84,119  R2U_Net.py:76,109  ResnetUnet.py:58,81
# ----------------------------------------------------------------------------------------------------------
@custom_op("b200seg::head", mutates_args=())
def head(x: Tensor, weight: Tensor, bias: Optional[Tensor]) -> Tensor:
    cout, cin = weight.shape[0], weight.shape[1]
    return K.head_fwd(_c(x), weight.reshape(cout, cin).contiguous(), bias)


@head.register_fake
def _(x, weight, bias):
    n, h, w, _ = x.shape
    return x.new_empty((n, weight.shape[0], h, w), dtype=torch.float32)


@custom_op("b200seg::head_bwd", mutates_args=())
def head_bwd(dy: Tensor, x: Tensor, weight: Tensor, need_dx: bool) -> Tuple[Tensor, Tensor, Tensor]:
    cout, cin = weight.shape[0], weight.shape[1]
    dx, dw, db = K.head_bwd(_c(dy), _c(x), weight.reshape(cout, cin).contiguous(), need_dx=need_dx)
    if dx is None:
        dx = torch.empty((0,), dtype=torch.bfloat16, device=dy.device)
    return dx, dw.view(weight.shape), db


def _head_setup(ctx, inputs, output):
    x, weight, bias = inputs
    ctx.save_for_backward(x, weight)
    ctx.has_bias = bias is not None


def _head_backward(ctx, dy):
    x, weight = ctx.saved_tensors
    dx, dw, db = head_bwd(dy, x, weight, ctx.needs_input_grad[0])
    return (dx if ctx.needs_input_grad[0] else None), dw, (db if ctx.has_bias else None)


head.register_autograd(_head_backward, setup_context=_head_setup)


# ----------------------------------------------------------------------------------------------------------
# loss: BCEWithLogits (helpers.py:245,327) and w_bce*BCE + w_dice*Dice (clip_seg_finetuner.py:61-74)
# ----------------------------------------------------------------------------------------------------------
@custom_op("b200seg::seg_loss", mutates_args=())
def seg_loss(logits: Tensor, target: Tensor, w_bce: float, w_dice: float, smooth: float) -> Tuple[Tensor, Tensor]:
    """-> (scalar loss fp32, sums fp64[6]); sums[4], sums[5] are the IoU intersection / union counts."""
    return K.loss_fwd(_c(logits.float()), _c(target.float()), w_bce, w_dice, smooth)


@seg_loss.register_fake
def _(logits, target, w_bce, w_dice, smooth):
    return logits.new_empty((), dtype=torch.float32), logits.new_empty((6,), dtype=_F64)


@custom_op("b200seg::seg_loss_bwd", mutates_args=())
def seg_loss_bwd(grad_out: Tensor, logits: Tensor, target: Tensor, sums: Tensor, w_bce: float, w_dice: float,
                 smooth: float) -> Tensor:
    return K.loss_bwd(_c(logits.float()), _c(target.float()), sums, _c(grad_out.float()), w_bce, w_dice, smooth)


def _loss_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)      # unused outputs (z, coef, stats, ...) must not get zero-filled grads
    logits, target, ctx.w_bce, ctx.w_dice, ctx.smooth = inputs
    ctx.save_for_backward(logits, target, output[1])


def _loss_backward(ctx, g, _gs):
    logits, target, sums = ctx.saved_tensors
    dz = seg_loss_bwd(g, logits, target, sums, ctx.w_bce, ctx.w_dice, ctx.smooth)
    return dz.view_as(logits), None, None, None, None


seg_loss.register_autograd(_loss_backward, setup_context=_loss_setup)


# ----------------------------------------------------------------------------------------------------------
# multi-class loss: w_ce * CrossEntropy(weight, ignore_index) + w_dice * (1 - mean foreground soft Dice)
# (nn.CrossEntropyLoss semantics; w_ce = w_dice = 0.5 mirrors CombinedLoss, clip_seg_finetuner.py:61-74)
# ----------------------------------------------------------------------------------------------------------
@custom_op("b200seg::seg_loss_ce", mutates_args=())
def seg_loss_ce(logits: Tensor, labels: Tensor, weight: Optional[Tensor], ignore_index: int, w_ce: float,
                w_dice: float, smooth: float) -> Tuple[Tensor, Tensor]:
    """logits fp32 [N, K, H, W], labels uint8 / int64 [N, H, W] (or [N, 1, H, W]) -> (scalar loss fp32, sums fp64
    [3 + 5K], layout kernels.ce_sums_fields).  The loss is NaN when a label is neither in [0, K) nor ignore_index."""
    return K.ce_loss_fwd(_c(logits.float()), _c(labels), _c(weight), ignore_index, w_ce, w_dice, smooth)


@seg_loss_ce.register_fake
def _(logits, labels, weight, ignore_index, w_ce, w_dice, smooth):
    return logits.new_empty((), dtype=torch.float32), logits.new_empty((K.ce_nsums(logits.shape[1]),), dtype=_F64)


@custom_op("b200seg::seg_loss_ce_bwd", mutates_args=())
def seg_loss_ce_bwd(grad_out: Tensor, logits: Tensor, labels: Tensor, weight: Optional[Tensor], ignore_index: int,
                    sums: Tensor, w_ce: float, w_dice: float, smooth: float) -> Tensor:
    return K.ce_loss_bwd(_c(logits.float()), _c(labels), _c(weight), ignore_index, sums, _c(grad_out.float()), w_ce,
                         w_dice, smooth)


@seg_loss_ce_bwd.register_fake
def _(grad_out, logits, labels, weight, ignore_index, sums, w_ce, w_dice, smooth):
    return torch.empty_like(logits, dtype=torch.float32)


def _loss_ce_setup(ctx, inputs, output):
    ctx.set_materialize_grads(False)
    logits, labels, weight, ctx.ignore_index, ctx.w_ce, ctx.w_dice, ctx.smooth = inputs
    ctx.save_for_backward(logits, labels, weight, output[1])


def _loss_ce_backward(ctx, g, _gs):
    logits, labels, weight, sums = ctx.saved_tensors
    dz = seg_loss_ce_bwd(g, logits, labels, weight, ctx.ignore_index, sums, ctx.w_ce, ctx.w_dice, ctx.smooth)
    return dz.view_as(logits), None, None, None, None, None, None


seg_loss_ce.register_autograd(_loss_ce_backward, setup_context=_loss_ce_setup)
