"""GPU input pipeline (SURVEY.md §8f N4): the reference's segmentation transforms (utils/trainer.py:88-115) and sample
format (utils/dataset.py:100-134) on the device, feeding the training step without a CPU augmentation bottleneck.

    aug = GpuSegAugment(size=256, train=True, seed=0)          # train_seg_transform; train=False = val_seg_transform
    for img_u8, mask_u8 in loader:                             # uint8 [N,Hs,Ws,3] / [N,Hs,Ws] batches (pinned host)
        x, t = aug(img_u8, mask_u8)                            # fp32 [N,3,256,256] normalised, fp32 [N,1,256,256]
        loss = stepper(x, t)

    # or, with the prefetcher (H2D of the raw uint8 batch — 4x fewer bytes than fp32 — on the copy stream):
    for x, t in PinnedPrefetcher(loader, device, device_transform=aug): ...

One kernel per batch (b2_seg_augment, csrc/augment.cu) reproduces Resize -> ShiftScaleRotate -> HorizontalFlip ->
RandomBrightnessContrast -> Normalize with the uint8 rounding points of the OpenCV / Albumentations implementation; the
random draw (same distributions and probabilities as the reference's A.Compose) stays on the host.  The pipeline is pinned
against OpenCV itself: tests/golden/augment.npz is produced by oracle/make_golden_aug.py with cv2.resize / cv2.warpAffine /
cv2.flip / cv2.LUT on fixed parameters.
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np
import torch

from ._lib import _f32, call
from .kernels import _p, _stream
from .utils.synthetic import IMAGENET_MEAN, IMAGENET_STD

PARAM_FLOATS = 12          # sizeof(b2_aug_params) / 4


def affine_matrix(size, angle_deg, scale, dx, dy):
    """forward 2x3 matrix of A.ShiftScaleRotate as OpenCV builds it: cv2.getRotationMatrix2D(centre, angle, scale) with
    the translation (dx, dy) given as fractions of the image size; centre = (size / 2 - 0.5, size / 2 - 0.5)"""
    c = size / 2.0 - 0.5
    a = math.radians(angle_deg)
    al, be = scale * math.cos(a), scale * math.sin(a)
    return np.array([[al, be, (1 - al) * c - be * c + dx * size],
                     [-be, al, be * c + (1 - al) * c + dy * size]], dtype=np.float64)


def invert_affine(m):
    """cv2.invertAffineTransform"""
    a = m[:, :2]
    d = a[0, 0] * a[1, 1] - a[0, 1] * a[1, 0]
    ia = np.array([[a[1, 1], -a[0, 1]], [-a[1, 0], a[0, 0]]]) / d
    return np.concatenate([ia, -(ia @ m[:, 2:3])], axis=1)


def pack_params(size, samples, border="constant"):
    """samples: list of dicts {angle, scale, dx, dy (or warp=False), flip, alpha, beta (or adjust=False)} ->
    float32 [N, 12] array with the memory layout of b2_aug_params"""
    out = np.zeros((len(samples), PARAM_FLOATS), dtype=np.float32)
    iv = out.view(np.int32)
    for i, s in enumerate(samples):
        warp = s.get("warp", True) and "angle" in s
        inv = invert_affine(affine_matrix(size, s["angle"], s["scale"], s["dx"], s["dy"])) if warp else np.eye(2, 3)
        out[i, 0:6] = inv.reshape(-1)
        adjust = s.get("adjust", True) and "alpha" in s
        out[i, 6] = s.get("alpha", 1.0) if adjust else 1.0
        out[i, 7] = s.get("beta", 0.0) if adjust else 0.0
        iv[i, 8], iv[i, 9], iv[i, 10] = int(bool(s.get("flip", False))), int(warp), int(adjust)
        iv[i, 11] = 0 if border == "constant" else 1
    return out


class GpuSegAugment:
    """The reference's train_seg_transform / val_seg_transform (utils/trainer.py:88-115) on the GPU.

    Defaults are the reference's: Resize(256), ShiftScaleRotate(shift 0.05, scale 0.05, rotate 15 deg, p 0.7),
    HorizontalFlip(p 0.5), RandomBrightnessContrast(0.1, 0.1, p 0.5), ImageNet Normalize.  `border`: 'constant' (fill 0,
    the Albumentations 2.0.8 default the reference pins) or 'reflect101' (the 1.x default)."""

    def __init__(self, size=256, train=True, shift_limit=0.05, scale_limit=0.05, rotate_limit=15.0, p_ssr=0.7,
                 p_flip=0.5, brightness_limit=0.1, contrast_limit=0.1, p_bc=0.5, mean=IMAGENET_MEAN, std=IMAGENET_STD,
                 border="constant", mask_nearest_resize=True, seed=None, labels=False):
        """labels=True: the masks are multi-class label maps (class index per pixel); they are resized and warped
        nearest-neighbour and returned as uint8 [N, S, S] class indices instead of fp32 [N, 1, S, S] in {0, 1}"""
        if labels and not mask_nearest_resize:
            raise ValueError("label maps are resized nearest-neighbour: labels=True needs mask_nearest_resize=True")
        self.labels = bool(labels)
        self.size, self.train = int(size), bool(train)
        self.shift_limit, self.scale_limit, self.rotate_limit, self.p_ssr = shift_limit, scale_limit, rotate_limit, p_ssr
        self.p_flip, self.brightness_limit, self.contrast_limit, self.p_bc = p_flip, brightness_limit, contrast_limit, p_bc
        self.mean = (_f32 * 3)(*[float(v) for v in mean])
        self.std = (_f32 * 3)(*[float(v) for v in std])
        self.border, self.mask_nearest_resize = border, bool(mask_nearest_resize)
        self.rng = np.random.default_rng(seed)

    def sample(self, n):
        """per-image random parameters, drawn like the reference's A.Compose draws them"""
        out = []
        for _ in range(n):
            s = {}
            if self.train and self.rng.random() < self.p_ssr:
                s.update(angle=self.rng.uniform(-self.rotate_limit, self.rotate_limit),
                         scale=1.0 + self.rng.uniform(-self.scale_limit, self.scale_limit),
                         dx=self.rng.uniform(-self.shift_limit, self.shift_limit),
                         dy=self.rng.uniform(-self.shift_limit, self.shift_limit))
            s["flip"] = bool(self.train and self.rng.random() < self.p_flip)
            if self.train and self.rng.random() < self.p_bc:
                s.update(alpha=1.0 + self.rng.uniform(-self.contrast_limit, self.contrast_limit),
                         beta=self.rng.uniform(-self.brightness_limit, self.brightness_limit))
            out.append(s)
        return out

    def __call__(self, img_u8, mask_u8, samples=None, device=None):
        """img_u8 uint8 [N, Hs, Ws, 3], mask_u8 uint8 [N, Hs, Ws] (or [N, Hs, Ws, 1]); host or device tensors.
        Returns (x fp32 [N, 3, S, S], t fp32 [N, 1, S, S]) on the device; with labels=True t is uint8 [N, S, S]."""
        assert img_u8.dtype == torch.uint8 and mask_u8.dtype == torch.uint8 and img_u8.dim() == 4 and img_u8.shape[3] == 3
        if mask_u8.dim() == 4:
            mask_u8 = mask_u8[..., 0]
        dev = torch.device(device) if device is not None else (img_u8.device if img_u8.is_cuda else torch.device("cuda"))
        img_d = img_u8.to(dev, non_blocking=True).contiguous()
        msk_d = mask_u8.to(dev, non_blocking=True).contiguous()
        n, hs, ws, _ = img_d.shape
        assert msk_d.shape == (n, hs, ws)
        samples = self.sample(n) if samples is None else samples
        prm = torch.from_numpy(pack_params(self.size, samples, self.border)).to(dev, non_blocking=True)
        S = self.size
        x = torch.empty((n, 3, S, S), dtype=torch.float32, device=dev)
        if self.labels:
            y = torch.empty((n, S, S), dtype=torch.uint8, device=dev)
            call("b2_seg_augment_labels", _p(img_d), _p(msk_d), n, hs, ws, S, _p(prm), self.mean, self.std, _p(x), _p(y),
                 _stream())
            return x, y
        t = torch.empty((n, 1, S, S), dtype=torch.float32, device=dev)
        call("b2_seg_augment", _p(img_d), _p(msk_d), n, hs, ws, S, _p(prm), self.mean, self.std,
             int(self.mask_nearest_resize), _p(x), _p(t), _stream())
        return x, t
