"""Seed-stable synthetic inputs and weights (SURVEY.md §8d) — the data generator of bench.py, tools/ and the tests.
Pure torch, no kernels: it only manufactures the batch the hot path is then run on (there is no dataset offline).

* xray_batch: smooth chest-X-ray-shaped field (super-Gaussian torso minus two elliptical lung Gaussians + noise),
  replicated to 3 channels and ImageNet-normalised (reference utils/trainer.py:48-49 mean/std), with the lung mask
  as the binary target (shape of utils/dataset.py:100-134 samples: img [3,H,W] f32, mask [1,H,W] in {0,1}).
* fill_state_dict_: deterministic parameter/buffer values that do not depend on module construction order, so the
  reference modules (in the build container), the oracle and the CUDA modules all see identical weights.
"""
from __future__ import annotations

import math

import torch

IMAGENET_MEAN = (0.485, 0.456, 0.406)
IMAGENET_STD = (0.229, 0.224, 0.225)


def xray_batch(n, h=256, w=256, seed=0, device="cpu", dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    ys = torch.linspace(-1, 1, h).view(1, h, 1)
    xs = torch.linspace(-1, 1, w).view(1, 1, w)
    torso = torch.exp(-((xs / 0.9) ** 4 + (ys / 0.95) ** 4)) * 0.75
    jit = (torch.rand(n, 2, 2, generator=g) - 0.5) * 0.12          # centre jitter +-0.06 per lung
    lungs = torch.zeros(n, h, w)
    for side, cx in enumerate((-0.4, 0.4)):
        cxj = (cx + jit[:, side, 0]).view(n, 1, 1)
        cyj = jit[:, side, 1].view(n, 1, 1)
        lungs = lungs + torch.exp(-(((xs - cxj) / 0.28) ** 2 + ((ys - cyj) / 0.55) ** 2) / 2)
    img = (torso - 0.55 * lungs + 0.03 * torch.randn(n, h, w, generator=g)).clamp(0, 1)
    mean = torch.tensor(IMAGENET_MEAN).view(1, 3, 1, 1)
    std = torch.tensor(IMAGENET_STD).view(1, 3, 1, 1)
    x = (img.unsqueeze(1).expand(n, 3, h, w) - mean) / std
    mask = (lungs > 0.5).float().unsqueeze(1)
    return x.contiguous().to(device=device, dtype=dtype), mask.contiguous().to(device=device, dtype=dtype)


def xray_batch_multiclass(n, h=256, w=256, seed=0, device="cpu", dtype=torch.float32):
    """xray_batch's image with a 3-class label map uint8 [N, H, W]: 0 background, 1 lung, 2 a lesion — a seeded
    ellipse around a point of one lung's mask, clipped to that mask (the background / lung / infection maps of the
    reference's dataset family)."""
    x, mask = xray_batch(n, h, w, seed=seed, device="cpu", dtype=torch.float32)
    lung = mask[:, 0] > 0.5
    labels = lung.to(torch.uint8)
    g = torch.Generator().manual_seed(seed + 7919)
    ys = torch.linspace(-1, 1, h).view(h, 1)
    xs = torch.linspace(-1, 1, w).view(1, w)
    for i in range(n):
        idx = lung[i].flatten().nonzero()[:, 0]
        if idx.numel() == 0:
            continue
        c = int(idx[int(torch.randint(idx.numel(), (1,), generator=g))])
        cy, cx = float(ys[c // w, 0]), float(xs[0, c % w])
        ry, rx = (0.1 + 0.1 * torch.rand(2, generator=g)).tolist()
        lesion = ((ys - cy) / ry) ** 2 + ((xs - cx) / rx) ** 2 <= 1.0
        labels[i][lesion & lung[i]] = 2
    return x.to(device=device, dtype=dtype), labels.contiguous().to(device)


def noise_batch(n, h=256, w=256, seed=1234, device="cpu", dtype=torch.float32):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, 3, h, w, generator=g)
    t = (torch.rand(n, 1, h, w, generator=g) > 0.7).float()
    return x.to(device=device, dtype=dtype), t.to(device=device, dtype=dtype)


def fill_state_dict_(sd, seed=0, conv_gain=1.0):
    """In-place deterministic fill of a state_dict (keys visited in sorted order; each key has its own stream).
    conv_gain scales the He-normal convolution weights (< 1 keeps eval-mode activations of the recurrent models, whose
    x + x1 re-injection doubles the variance at every application, in range)."""
    for idx, k in enumerate(sorted(sd.keys())):
        v = sd[k]
        g = torch.Generator().manual_seed(seed * 100003 + idx)
        if k.endswith("num_batches_tracked"):
            v.zero_()
        elif k.endswith("running_mean"):
            v.copy_(0.1 * torch.randn(v.shape, generator=g))
        elif k.endswith("running_var"):
            v.copy_(1.0 + 0.2 * torch.rand(v.shape, generator=g))
        elif v.dim() == 4:                                          # conv / conv-transpose weight
            fan_in = v.shape[1] * v.shape[2] * v.shape[3]
            v.copy_(torch.randn(v.shape, generator=g) * (conv_gain * math.sqrt(2.0 / fan_in)))
        elif k.endswith("weight"):                                  # BatchNorm gamma
            v.copy_(1.0 + 0.1 * torch.randn(v.shape, generator=g))
        else:                                                       # conv bias / BatchNorm beta
            v.copy_(0.1 * torch.randn(v.shape, generator=g))
    return sd
