"""Inference fast path (SURVEY.md §8f N2; reference callers utils/pipeline.py:340-357, utils/tester.py:264-289,
validation loop utils/helpers.py:345-360): with BatchNorm in eval mode and autograd off, every
[Conv2d -> BatchNorm2d -> ReLU] collapses into ONE tcgen05 convolution whose weights carry gamma/sqrt(var+eps) and
whose epilogue adds the folded bias and applies the ReLU (Appendix D.3).  UpConv uses the 16-tap folded weights, so
the up-sampled tensor is never built either.  Forward-only ops: no autograd formula.
"""
from __future__ import annotations

from typing import Optional

import torch
from torch import Tensor
from torch.library import custom_op

import weakref

from . import kernels as K
from .ops import _PHASES, _c

# BN-folded weights are a pure function of (conv weight, conv bias, BN affine, BN running statistics): they are cached
# per conv weight and rebuilt only when one of those tensors changed — torch writers bump Tensor._version, the fused
# optimizer (raw-pointer writes) bumps kernels.param_epoch().  Batch-1 inference no longer re-folds and re-packs every
# conv on every call (pipeline.py:340-357 runs one image per call).
_FOLDED = {}


def _folded(weight, bias, gamma, beta, rm, rv, eps, upfold):
    tensors = (weight, bias, gamma, beta, rm, rv)
    stamp = tuple((t.data_ptr(), t._version) if t is not None else None for t in tensors) + (K.param_epoch(), float(eps))
    key = (weight.data_ptr(), bool(upfold))
    hit = _FOLDED.get(key)
    if hit is not None and hit[0]() is weight and hit[1] == stamp:
        return hit[2], hit[3]
    coef = K.bn_eval_coeffs(gamma, beta, rm, rv, eps)
    wf, bf = K.pack_weights_folded(weight, bias, coef, upfold=upfold)
    if len(_FOLDED) > 4096:
        for k in [k for k, v in _FOLDED.items() if v[0]() is None]:
            del _FOLDED[k]
    _FOLDED[key] = (weakref.ref(weight), stamp, wf, bf)
    return wf, bf


@custom_op("b200seg::conv_bn_act_infer", mutates_args=())
def conv_bn_act_infer(x0: Tensor, x1: Optional[Tensor], weight: Tensor, bias: Optional[Tensor], gamma: Tensor,
                      beta: Tensor, running_mean: Tensor, running_var: Tensor, eps: float, relu: bool,
                      addend: Optional[Tensor]) -> Tensor:
    """y = act(conv(x; W*s) + (b*s + t)) [+ addend]  with s = gamma/sqrt(running_var+eps), t = beta - running_mean*s"""
    cout, cin, k, _ = weight.shape
    wf, bf = _folded(weight, bias, gamma, beta, running_mean, running_var, eps, False)
    return K.conv_igemm(_c(x0), wf, cout, k, x1=_c(x1), bias=bf, relu=relu, addend=_c(addend),
                        add_after_act=addend is not None)


@conv_bn_act_infer.register_fake
def _(x0, x1, weight, bias, gamma, beta, rm, rv, eps, relu, addend):
    n, h, w, _ = x0.shape
    return x0.new_empty((n, h, w, weight.shape[0]))


@custom_op("b200seg::upconv_bn_act_infer", mutates_args=())
def upconv_bn_act_infer(x: Tensor, weight: Tensor, bias: Optional[Tensor], gamma: Tensor, beta: Tensor,
                        running_mean: Tensor, running_var: Tensor, eps: float, relu: bool) -> Tensor:
    cout = weight.shape[0]
    x = _c(x)
    n, h, w, _ = x.shape
    wf, bf = _folded(weight, bias, gamma, beta, running_mean, running_var, eps, True)
    y = K.new_act(n, 2 * h, 2 * w, cout, x.device)
    cin = x.shape[3]
    if cout % 64 == 0 and cin % 64 == 0:
        K.conv_igemm(x, wf.view(16, cout, cin), cout, 2, bias=bf, relu=relu, out=y, fold=1)
    else:
        for ph, (a, b) in enumerate(_PHASES):
            K.conv_igemm(x, wf[ph], cout, 2, bias=bf, relu=relu, out=y, out_mul=2, out_off=(a, b), pad=(1 - a, 1 - b))
    return y


@upconv_bn_act_infer.register_fake
def _(x, weight, bias, gamma, beta, rm, rv, eps, relu):
    n, h, w, _ = x.shape
    return x.new_empty((n, 2 * h, 2 * w, weight.shape[0]))


# ----------------------------------------------------------------------------------------------------------
# attention gate, eval mode, ONE kernel (north_star (2); AttentionUNet.py:29-54): the three BatchNorms fold into the
# weights / biases / two scalars, the GEMM runs over K = [g | x] and its epilogue reduces each accumulator row to psi and
# writes x * psi (b2_gate_fused, csrc/conv_igemm.cu) — g1, x1, q and psi never exist in HBM.
# ----------------------------------------------------------------------------------------------------------
_GATE_FOLDED = {}


def _gate_folded(gate):
    """(wpk bf16 [1, fint, 2C], bias fp32 [fint], wpsi fp32 [fint], coef_1 fp32 [4, 1]) cached per gate module"""
    cg, bng, cx, bnx, cp, bn1 = gate.W_g[0], gate.W_g[1], gate.W_x[0], gate.W_x[1], gate.psi[0], gate.psi[1]
    tensors = [cg.weight, cg.bias, cx.weight, cx.bias, cp.weight, cp.bias]
    for bn in (bng, bnx, bn1):
        tensors += [bn.weight, bn.bias, bn.running_mean, bn.running_var]
    stamp = tuple((t.data_ptr(), t._version) if t is not None else None for t in tensors) + (K.param_epoch(),)
    key = cg.weight.data_ptr()
    hit = _GATE_FOLDED.get(key)
    if hit is not None and hit[0]() is cg.weight and hit[1] == stamp:
        return hit[2]
    wgf, bgf = _folded(cg.weight, cg.bias, bng.weight, bng.bias, bng.running_mean, bng.running_var, float(bng.eps), False)
    wxf, bxf = _folded(cx.weight, cx.bias, bnx.weight, bnx.bias, bnx.running_mean, bnx.running_var, float(bnx.eps), False)
    wpk = torch.cat((wgf, wxf), dim=2).contiguous()            # [1, fint, C_g + C_x]   (tiny; cached)
    bias = (bgf + bxf).contiguous()
    wpsi = cp.weight.detach().reshape(-1).to(torch.bfloat16).float().contiguous()   # the unfused path multiplies in bf16
    coef1 = K.bn_eval_coeffs(bn1.weight, bn1.bias, bn1.running_mean, bn1.running_var, float(bn1.eps))
    out = (wpk, bias, wpsi, coef1)
    if len(_GATE_FOLDED) > 1024:
        for k in [k for k, v in _GATE_FOLDED.items() if v[0]() is None]:
            del _GATE_FOLDED[k]
    _GATE_FOLDED[key] = (weakref.ref(cg.weight), stamp, out)
    return out


def gate_fusable(gate, g: Tensor, x: Tensor) -> bool:
    c, fint = x.shape[3], gate.W_g[0].out_channels
    return (g.shape[3] == c and c % 64 == 0 and fint in (32, 64, 128, 256) and gate.psi[0].out_channels == 1)


@custom_op("b200seg::attention_gate_infer", mutates_args=())
def attention_gate_infer(g: Tensor, x: Tensor, wpk: Tensor, bias: Tensor, wpsi: Tensor, bpsi: Tensor,
                         coef1: Tensor) -> Tensor:
    import ctypes as C
    from ._lib import GateArgs, call
    g, x = _c(g), _c(x)
    n, h, w, c = x.shape
    out = K.new_act(n, h, w, c, x.device)
    a = GateArgs()
    a.n, a.h, a.w, a.c, a.fint = n, h, w, c, wpk.shape[1]
    a.g, a.ldg, a.x, a.ldx = g.data_ptr(), g.stride(2), x.data_ptr(), x.stride(2)
    a.wpk, a.bias, a.wpsi, a.bpsi = wpk.data_ptr(), bias.data_ptr(), wpsi.data_ptr(), bpsi.data_ptr()
    a.scale1, a.shift1 = coef1[2].data_ptr(), coef1[3].data_ptr()
    a.out, a.ldo = out.data_ptr(), c
    call("b2_gate_fused", C.byref(a), K._stream())
    return out


@attention_gate_infer.register_fake
def _(g, x, wpk, bias, wpsi, bpsi, coef1):
    return torch.empty_like(x)


def attention_gate_fused(gate, g: Tensor, x: Tensor) -> Tensor:
    wpk, bias, wpsi, coef1 = _gate_folded(gate)
    return attention_gate_infer(g, x, wpk, bias, wpsi, gate.psi[0].bias.detach(), coef1)


def inference_mode(bn: torch.nn.BatchNorm2d) -> bool:
    """folded path applies: eval-mode BN with running statistics and no autograd recording"""
    return (not bn.training) and bn.running_mean is not None and not torch.is_grad_enabled()
