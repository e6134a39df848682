"""Building blocks shared by the drop-in models.  Same constructor signatures, submodule names and therefore the
same state_dict keys as the reference blocks; forward() runs the b200seg custom ops on NHWC bf16 activations.

Calling convention
  * inside a model, activations are bf16 tensors [N, H, W, C] ("internal");
  * a block called directly with an fp32 NCHW tensor (the reference's convention) converts on the way in and out,
    so blocks are drop-ins on their own as well;
  * `(a, b)` tuples stand for torch.cat((a, b), dim=1) — the concat is never materialised, the consuming
    convolution reads its K dimension from both tensors.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn

from . import ops

BF16 = torch.bfloat16
UPFOLD = os.environ.get("B200SEG_UPFOLD", "1") != "0"


def _is_external(x) -> bool:
    t = x[0] if isinstance(x, tuple) else x
    return t.dtype != BF16


def check_image(x: torch.Tensor) -> torch.Tensor:
    if not x.is_cuda:
        raise RuntimeError("b200seg modules run on a CUDA (sm_100) device only; there is no CPU fallback — "
                           "move the model and the input to the GPU")
    if x.dim() != 4:
        raise ValueError(f"expected a 4-D NCHW tensor, got shape {tuple(x.shape)}")
    return x.float().contiguous()


def to_internal(x):
    if isinstance(x, tuple):
        return tuple(to_internal(t) for t in x)
    return ops.to_nhwc(check_image(x)) if x.dtype != BF16 else x


def conv_bn_act(x, conv: nn.Conv2d, bn: nn.BatchNorm2d, relu: bool = True, addend=None, share_index=0,
                share_count=1):
    """conv (3x3 p1 or 1x1) -> BatchNorm -> optional ReLU as ONE fused autograd node.  `x` may be an fp32 NCHW image
    with <= 4 channels (stem), an internal activation, or a tuple of two internal activations (virtual concat)."""
    return ops.conv_bn_act_module(x, conv, bn, relu, addend, share_index, share_count)


def conv_plain(x, conv: nn.Conv2d):
    """conv without BN/ReLU (RRCNN_block.conv_1x1, R2U_Net.py:43,46)."""
    if not isinstance(x, tuple) and x.dtype != BF16:
        return ops.stem_conv(x, conv.weight, conv.bias, False)[0]
    x0, x1 = x if isinstance(x, tuple) else (x, None)
    return ops.conv2d(x0, x1, conv.weight, conv.bias, False)[0]


def _stem_ok(x, conv) -> bool:
    return (not isinstance(x, tuple)) and x.dtype != BF16 and conv.in_channels <= 4


class BasicBlock(nn.Sequential):
    """basic_block(cin, cout): [Conv3x3 p1, BN, ReLU] x 2 — AttentionUNet.py:4-13, ResnetUnet.py:5-14."""

    def __init__(self, in_channels, out_channels):
        super().__init__(
            nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(inplace=True),
            nn.Conv2d(out_channels, out_channels, kernel_size=3, padding=1),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(inplace=True),
        )

    def _internal(self, x):
        """returns the internal activation whatever the input convention (used by the models' stems)"""
        y = conv_bn_act(x, self[0], self[1])
        return conv_bn_act(y, self[3], self[4])

    def forward(self, x):
        ext = _is_external(x)
        if ext and not _stem_ok(x, self[0]):
            x = to_internal(x)
        elif ext:
            x = check_image(x)
        y = self._internal(x)
        return ops.to_nchw(y) if ext else y


def basic_block(in_channels, out_channels):
    return BasicBlock(in_channels, out_channels)


class UpConv(nn.Module):
    """Upsample(x2, nearest) -> Conv3x3 -> BN -> ReLU — AttentionUNet.py:15-27, R2U_Net.py:22-34."""

    def __init__(self, in_channels, out_channels):
        super().__init__()
        self.up = nn.Sequential(
            nn.Upsample(scale_factor=2),
            nn.Conv2d(in_channels, out_channels, kernel_size=3, stride=1, padding=1, bias=True),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(inplace=True),
        )

    def forward(self, x):
        ext = _is_external(x)
        x = to_internal(x)
        if UPFOLD:     # folded: four 2x2 phase convolutions on the low-resolution input (see ops.upconv_bn_act)
            y = ops.upconv_bn_act_module(x, self.up[1], self.up[2])
        else:          # literal: materialise the upsampled tensor, then conv3x3
            y = conv_bn_act(ops.upsample2x(x), self.up[1], self.up[2])
        return ops.to_nchw(y) if ext else y


class AttentionGate(nn.Module):
    """x * sigmoid(BN(psi(relu(BN(W_g g) + BN(W_x x))))) — AttentionUNet.py:29-54, R2AttU_Net.py:61-86."""

    def __init__(self, F_g, F_l, F_int):
        super().__init__()
        self.W_g = nn.Sequential(nn.Conv2d(F_g, F_int, kernel_size=1, stride=1, padding=0, bias=True),
                                 nn.BatchNorm2d(F_int))
        self.W_x = nn.Sequential(nn.Conv2d(F_l, F_int, kernel_size=1, stride=1, padding=0, bias=True),
                                 nn.BatchNorm2d(F_int))
        self.psi = nn.Sequential(nn.Conv2d(F_int, 1, kernel_size=1, stride=1, padding=0, bias=True),
                                 nn.BatchNorm2d(1), nn.Sigmoid())
        self.relu = nn.ReLU(inplace=True)

    def forward(self, g, x):
        ext = _is_external(x)
        g, x = to_internal(g), to_internal(x)
        from .ops_gate import attention_gate_module
        out = attention_gate_module(self, g, x)
        return ops.to_nchw(out) if ext else out

    def gate_pass(self, g, x):
        """(forward(g, x), g) on internal activations — the second value is g as the tensor the decoder's concat should
        consume, so that g's concat-side gradient is added inside the gate's backward (ops_gate._GatePass)."""
        from .ops_gate import attention_gate_module
        return attention_gate_module(self, g, x, with_pass=True)


class Recurrent_block(nn.Module):
    """One shared conv3x3+BN+ReLU applied t+1 times with x + x1 re-injection — R2U_Net.py:4-20."""

    def __init__(self, in_channels, out_channels, t=2):
        super().__init__()
        self.t = t
        self.out_channels = out_channels
        self.conv = nn.Sequential(
            nn.Conv2d(out_channels, out_channels, kernel_size=3, stride=1, padding=1, bias=True),
            nn.BatchNorm2d(out_channels),
            nn.ReLU(inplace=True),
        )

    def forward(self, x):
        ext = _is_external(x)
        x = to_internal(x)
        # t+1 applications of the shared conv+BN+ReLU; every application but the last emits x + f(.) directly from the
        # BatchNorm pass (the un-summed activation is never needed), the last one emits f(.) itself
        n_uses = self.t + 1               # sequentially dependent applications of the one shared conv weight
        f = lambda v, add, i: conv_bn_act(v, self.conv[0], self.conv[1], addend=add, share_index=i,
                                          share_count=n_uses)
        if self.t == 0:
            raise ValueError("Recurrent_block needs t >= 1 (the reference leaves x1 undefined for t = 0)")
        s = f(x, x, 0)                        # x + f(x)
        for i in range(self.t - 1):
            s = f(s, x, i + 1)                # x + f(x + x1)
        x1 = f(s, None, self.t)
        return ops.to_nchw(x1) if ext else x1


class RRCNN_block(nn.Module):
    """x0 = conv1x1(x); x0 + RB(RB(x0)) — R2U_Net.py:36-48."""

    def __init__(self, in_channels, out_channels, t=2):
        super().__init__()
        self.RCNN = nn.Sequential(Recurrent_block(in_channels, out_channels, t=t),
                                  Recurrent_block(in_channels, out_channels, t=t))
        self.conv_1x1 = nn.Conv2d(in_channels, out_channels, kernel_size=1, stride=1, padding=0)

    def _internal(self, x):
        x0 = conv_plain(x, self.conv_1x1)
        return ops.add(x0, self.RCNN(x0))

    def forward(self, x):
        ext = _is_external(x)
        if ext and not _stem_ok(x, self.conv_1x1):
            x = to_internal(x)
        elif ext:
            x = check_image(x)
        y = self._internal(x)
        return ops.to_nchw(y) if ext else y
