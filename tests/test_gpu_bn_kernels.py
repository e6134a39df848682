"""The BatchNorm kernels of csrc/bn.cu (and relu_mask of csrc/resnet.cu), one at a time, at every launch geometry they
select, against an fp64 reference that rounds where they round.

b2_channel_stats -> b2_bn_finalize / b2_bn_eval_coeffs -> b2_bn_apply -> b2_bn_bwd_reduce + b2_bn_bwd_apply, plus
b2_channel_sum (a conv bias gradient), b2_bn_update_running_multi and b2_relu_mask.  The reference forward rounds to
bf16 exactly where bn.cu does, with straight-through gradients (the gate kernels' scheme, tests/test_gpu_gate_kernels.py):
y = bf16(act(fp32 fma(z, scale, shift))), ysum = bf16(y + addend), residual y = bf16(act(bf16(fma) + addend)); the
backward ReLU mask is that fp32 fma > 0 with the kernel's own coefficients.  In train mode the batch mean and invstd
carry the values the kernel was given and the gradients of the fp64 batch statistics of z; dz, dgamma and dbeta are
torch autograd of that forward, not a copy of the collapsed A*dy*mask + B*z + C of the kernels.

Bounds: 1e-5 (fp32 accumulation) of the sum of the absolute values of the terms a kernel adds, plus one bf16 ulp where
it rounds its output; bit equality where the kernel's arithmetic is emulated exactly (bn_apply, bn_finalize,
bn_eval_coeffs, the running statistics, relu_mask).  The unmarked tests check the reference against torch's own
BatchNorm with rounding off, and check that seven plausible kernel bugs move some checked output by at least 10x its
bound at every shape of the GPU matrix, under an upstream gradient correlated with the output (with a random one the
batch terms of the BatchNorm backward are O(1/sqrt(npix)) of dz and a wrong backward hides inside the bound).
"""
import math
import os
import subprocess
import sys
from fractions import Fraction

import numpy as np
import pytest
import torch

from test_gpu_gate_kernels import _bits, _nhwc, _r, _st, _worst, correlated, ulp_bf16

EPS = 1e-5
EPS32 = float(np.float32(EPS))     # what the kernels receive (a C float)
MOMENTUM = 0.1
TOL = 1e-5                         # fp32 accumulation: relative to the sum of the absolute values of the terms
SMS_B200 = 148

C_LIST = [8, 24, 64, 96, 128, 200, 512, 1024, 1032, 2048]
PIX = ["1", "126", "2x48x80", "sweep"]
MATRIX = [(c, kind) for c in C_LIST for kind in PIX]
MUTANTS = ["mean", "xhat", "swap", "eval_batch", "shift", "dbias_dy", "biased"]


# ----------------------------------------------------------------------------------------------------------
# launch geometry, mirrored from bn.cu: make_map / light_map (threads per pixel, pixels per block iteration), the
# 64-channel slice rule of b2_channel_sum / b2_bn_bwd_*, chan_grid(npix, map, waves) and each kernel's pixels in flight
# ----------------------------------------------------------------------------------------------------------
def _rows8(c):
    """pixels per block iteration of make_map: C / 8 threads per pixel in a 256-thread block"""
    return 256 // (c // 8)


def _switch(name):
    v = os.environ.get(name)
    return not (v is not None and v.strip() and int(v) == 0)


def loops(c, light=None, slices=None):
    """kernel -> (rows, waves, channel slices, pixels in flight per thread) of each grid-stride pixel loop at C"""
    light = _switch("B200SEG_BN_LIGHT") if light is None else light
    slices = _switch("B200SEG_BN_SLICE") if slices is None else slices
    out = {"channel_stats": (_rows8(c), 8, 1, 1)}
    out["channel_sum"] = (32, 4, -(-c // 64), 2) if c > 64 and slices else (_rows8(c), 4, 1, 2)
    if light and c % 4 == 0 and c // 4 <= 256:
        if c % 64 == 0 and c > 64 and slices:
            out["bn_bwd"] = (16, 8, c // 64, 4)              # light, 64-channel slices
        else:
            out["bn_bwd"] = (256 // (c // 4), 8, 1, 4)      # light, unsliced
    else:
        out["bn_bwd"] = (_rows8(c), 4, 1, 2)                # 8-channel kernels
    return out


def apply_loops(c):
    """the three pixel loops of bn_apply_kernel: plain (4 in flight), y + ysum (2), residual (1)"""
    return {"plain": (_rows8(c), 16, 1, 4), "sum": (_rows8(c), 16, 1, 2), "residual": (_rows8(c), 16, 1, 1)}


def _step(npix, rows, waves, slices, sms):
    grid = max(1, min(-(-npix // rows), sms * waves))
    return max(1, -(-grid // slices)) * rows


def reaches_last_lane(npix, loop, sms):
    """npix gives the loop U + 1 full grid-stride sweeps and a last iteration whose last in-flight lane is partly
    filled (U = pixels in flight per thread)"""
    rows, waves, slices, u = loop
    step = _step(npix, rows, waves, slices, sms)
    return npix >= (u + 1) * step and (u - 1) * step < npix % (u * step)


def sweep_count(ls, sms):
    """the smallest pixel count that reaches the last lane of every loop in `ls`"""
    lo = max((u + 1) * _step(1 << 40, r, w, s, sms) for r, w, s, u in ls.values())
    span = 4 * max(u * _step(1 << 40, r, w, s, sms) for r, w, s, u in ls.values())
    n = np.arange(lo, lo + span, dtype=np.int64)
    ok = np.ones_like(n, dtype=bool)
    for r, w, s, u in ls.values():
        step = _step(1 << 40, r, w, s, sms)        # at these counts every grid is at its cap
        ok &= (n % (u * step)) > (u - 1) * step
    assert ok.any(), ls
    npix = int(n[ok][0])
    for name, loop in ls.items():
        assert reaches_last_lane(npix, loop, sms), (name, loop, npix)
    return npix


def npix_of(kind, c, sms):
    if kind == "sweep":
        return sweep_count(loops(c), sms)
    return math.prod(int(v) for v in kind.split("x"))


def test_geometry_reaches_every_lane():
    """the sweep counts reach the last lane of every loop (with both switch settings), and the matrix selects the
    paths it is meant to: tpp 2 / 128 rows at C = 8, idle threads at 24 / 96 / 200 / 1032, 64-channel slices"""
    for c in C_LIST:
        for light in (True, False):
            for sl in (True, False):
                ls = loops(c, light, sl)
                sweep_count(ls, SMS_B200)
        sweep_count(apply_loops(c), SMS_B200)
    assert loops(8, True, True)["bn_bwd"] == (128, 8, 1, 4)
    assert loops(24, True, True)["bn_bwd"] == (42, 8, 1, 4)           # 6 x 42 = 252 of 256 threads
    assert loops(96, True, True)["bn_bwd"] == (10, 8, 1, 4)           # 24 x 10 = 240
    assert loops(200, True, True)["bn_bwd"] == (5, 8, 1, 4)           # tpp 50, 250
    assert apply_loops(200)["plain"][0] == 10                         # 25 tpp x 10 rows
    assert loops(200, True, True)["channel_sum"] == (32, 4, 4, 2)     # the 4th slice has 8 channels
    assert loops(96, True, True)["channel_sum"][2] == 2
    assert loops(1024, True, True)["bn_bwd"] == (16, 8, 16, 4)
    assert loops(1032, True, True)["bn_bwd"] == (1, 4, 1, 2)          # tpp 129, 127 idle threads
    assert loops(2048, True, True)["bn_bwd"] == (1, 4, 1, 2)


# ----------------------------------------------------------------------------------------------------------
# exact emulation of the fp32 / fp64 arithmetic of the coefficient kernels
# ----------------------------------------------------------------------------------------------------------
def fma32(a, b, c):
    """fp32 fma(a, b, c) rounded once, for fp32-valued fp64 tensors: a * b is exact in fp64, the sum is an exact
    two-sum s + e, and a tie of s between two fp32 neighbours is broken by the sign of e"""
    p = a * b
    s = p + c
    bb = s - p
    e = (p - (s - bb)) + (c - bb)
    r = s.float()
    rd = r.double()
    d = s - rd
    other = torch.nextafter(r, torch.where(d > 0, torch.full_like(r, math.inf), torch.full_like(r, -math.inf))).double()
    tie = (d != 0) & (2 * d == other - rd)
    take = tie & (e != 0) & ((e > 0) == (d > 0))
    return torch.where(take, other, rd)


def _f32(v):
    return v.float().double()


def finalize_emu(stats, count, gamma, beta, momentum, rm, rv, biased=False):
    """bn_finalize_kernel on the CPU: -> coefficient rows (mean, invstd, scale, shift) fp32 [4, C] and the updated running
    statistics (None without running buffers).  var = fma(-m, m, q) in fp64 is taken exactly (fractions)."""
    stats = stats.detach().double().cpu()
    c = stats.shape[-1] // 2 if stats.dim() == 1 else stats.shape[1]
    s, q = stats.reshape(2, c)[0] / count, stats.reshape(2, c)[1] / count
    var = torch.tensor([float(Fraction(b) - Fraction(a) * Fraction(a)) for a, b in zip(s.tolist(), q.tolist())],
                       dtype=torch.float64).clamp_min(0.0)
    fm = _f32(s)
    inv = _f32(1.0 / torch.sqrt(var + EPS32))
    g = _f32(gamma.detach().cpu().double()) if gamma is not None else torch.ones(c, dtype=torch.float64)
    b = _f32(beta.detach().cpu().double()) if beta is not None else torch.zeros(c, dtype=torch.float64)
    sc = _f32(g * inv)
    coef = torch.stack([fm, inv, sc, fma32(-fm, sc, b)]).float()
    if rm is None:
        return coef, None, None
    unb = var if biased or count <= 1 else var * count / (count - 1)
    m32 = float(np.float32(momentum))
    om = _f32(torch.tensor(1.0, dtype=torch.float64) - m32)
    rm_new = fma32(torch.full_like(fm, m32), fm, _f32(om * _f32(rm.detach().cpu().double())))
    rv_new = fma32(torch.full_like(fm, m32), _f32(unb), _f32(om * _f32(rv.detach().cpu().double())))
    return coef, rm_new.float(), rv_new.float()


def eval_coeffs_emu(gamma, beta, rm, rv):
    """bn_eval_coeffs_kernel on the CPU"""
    rm, rv = _f32(rm.detach().cpu().double()), _f32(rv.detach().cpu().double())
    inv = _f32(1.0 / torch.sqrt(rv + EPS32))
    sc = _f32(_f32(gamma.detach().cpu().double()) * inv)
    return torch.stack([rm, inv, sc, fma32(-rm, sc, _f32(beta.detach().cpu().double()))]).float()


def exact_stats(v):
    vd = v.double()
    return torch.stack([vd.sum(0), (vd * vd).sum(0)])


# ----------------------------------------------------------------------------------------------------------
# the reference (fp64, torch, any device)
# ----------------------------------------------------------------------------------------------------------
def bn_ref(t, training, relu, mode="plain", rounding=True, mutant=None):
    """t: fp64 z [P, C] (leaf), gamma, beta [C] (leaves), addend [P, C], coef [4, C] = the kernel's fp32 (mean, invstd,
    scale, shift), rm / rv.  mode: 'plain', 'sum' (also ysum = y + addend) or 'residual' (act(bn(z) + addend)).
    mutant: 'mean' / 'xhat' drop the mean / x-hat term of the train-mode backward, 'eval_batch' takes the batch terms
    in eval mode, 'shift' takes the ReLU mask from z * scale > 0.  -> {'y', 'ysum'}"""
    z, gamma, beta = t["z"], t["gamma"], t["beta"]
    coef = t.get("coef")
    if training or mutant == "eval_batch":
        mean, inv = z.mean(0), (z.var(0, unbiased=False) + EPS).rsqrt()
        if rounding:
            mean, inv = _st(mean, coef[0]), _st(inv, coef[1])
        if mutant == "mean":
            mean = mean.detach()
        if mutant == "xhat":
            inv = inv.detach()
    elif rounding:
        mean, inv = coef[0], coef[1]
    else:
        mean, inv = t["rm"], (t["rv"] + EPS).rsqrt()
    pre = (z - mean) * inv * gamma + beta
    if rounding:
        with torch.no_grad():
            v = fma32(z.detach(), coef[2], coef[3])
        pre = _st(pre, v)
    out = {}
    if mode == "residual":
        s = (_st(pre, _r(pre)) if rounding else pre) + t["addend"]
        y = torch.relu(s) if relu else s
    else:
        y = torch.relu(pre) if relu else pre
        if mutant == "shift":
            with torch.no_grad():
                mask = fma32(z.detach(), coef[2], torch.zeros_like(coef[3])) > 0
            y = _st(torch.where(mask, pre, torch.zeros_like(pre)), y)
    if rounding:
        y = _st(y, _r(y))
    out["y"] = y
    if mode == "sum":
        ys = y + t["addend"]
        out["ysum"] = _st(ys, _r(ys)) if rounding else ys
    return out


def bwd_ref(t, training, relu, dy, mutant=None):
    """reference dz, dgamma, dbeta, dbias (the column sums of the bf16-rounded dz) under the upstream dy"""
    y = bn_ref(t, training, relu, mutant=mutant)["y"]
    dz, dg, db = torch.autograd.grad([y], [t["z"], t["gamma"], t["beta"]], [dy])
    if mutant == "swap":
        dg, db = db, dg
    dbias = dy.sum(0) if mutant == "dbias_dy" else _r(dz).sum(0)
    return {"dz": dz.detach(), "dgamma": dg.detach(), "dbeta": db.detach(), "dbias": dbias.detach()}


def bwd_tolerances(t, training, relu, dy, dz_kernel=None):
    """TOL x the sum of |terms| each kernel adds, per checked output.  dbeta: sum dd (dd = dy * mask); dgamma:
    invstd * (sum dd * z - mean * sum dd), both sums fp32; dz = A dd + B z + C with |B z| + |C| <= |A| (mean|dd| + invstd
    (|z| + |mean|) mean|dd x-hat|) in train mode; dbias: the sum of the kernel's own (or the reference's) rounded dz.
    dgamma_centred: TOL x sum |dd x-hat|, the bound of a centred sum.  Where |mean| / sigma ~ 250 the uncentred bound
    is ~500x wider and would pass an fp32 accumulation that loses a few 1e-3 of dgamma; the GPU test holds those
    channels to the centred bound as well (today's kernels add dd * z products that are exact in fp32, over short
    per-thread and per-block chains, and stay far inside it)."""
    if dz_kernel is None:
        dz_kernel = bwd_ref(t, training, relu, dy)["dz"]
    with torch.no_grad():
        z, coef = t["z"].detach(), t["coef"]
        mask = fma32(z, coef[2], coef[3]) > 0 if relu else torch.ones_like(z, dtype=torch.bool)
        mda = dy.abs() * mask
        inv, mu = coef[1], coef[0]
        ka = (t["gamma"].detach() * inv).abs()
        xh = (z - mu) * inv
        if training:
            mdz = ka * (mda + mda.mean(0) + inv * (z.abs() + mu.abs()) * (mda * xh.abs()).mean(0))
        else:
            mdz = ka * mda
        dgam = inv * ((mda * z.abs()).sum(0) + mu.abs() * mda.sum(0))
        return {"dz": TOL * mdz, "dgamma": TOL * dgam, "dbeta": TOL * mda.sum(0),
                "dbias": TOL * _r(dz_kernel).abs().sum(0), "dgamma_centred": TOL * (mda * xh.abs()).sum(0)}


# ----------------------------------------------------------------------------------------------------------
# inputs
# ----------------------------------------------------------------------------------------------------------
def hi_mean_channels(c):
    return [1, c // 2 + 1]


def make_inputs(npix, c, seed, device, ld_pad=0, off=0):
    """bf16 z, addend and noise [P, C] (z and addend channel slices of [P, C + ld_pad] buffers at channel offset
    `off` when ld_pad > 0), fp32 gamma, beta, rm, rv.  Channels 1 and C/2 + 1 have |mean| / sigma ~ 250 (bf16 values
    near +-256, spread about 1); channel C - 1 is constant (sigma = 0: invstd = 1 / sqrt(eps))."""
    gen = torch.Generator(device="cpu").manual_seed(seed)

    def rn(*s):
        return torch.randn(*s, generator=gen, dtype=torch.float64)

    mu, sig = 0.3 * rn(c), 0.5 + torch.rand(c, generator=gen, dtype=torch.float64)
    zf = mu + sig * rn(npix, c)
    hi = hi_mean_channels(c)
    zf[:, hi[0]] = 256.0 + rn(npix)
    zf[:, hi[1]] = -256.0 + rn(npix)
    zf[:, c - 1] = 0.75
    p = {"gamma": 0.5 + torch.rand(c, generator=gen, dtype=torch.float64), "beta": 0.2 * rn(c),
         "rm": 0.2 * rn(c), "rv": 0.01 + 0.04 * torch.rand(c, generator=gen, dtype=torch.float64)}
    p = {k: v.float().to(device) for k, v in p.items()}

    def act(v):
        v = v.float().bfloat16()
        if not ld_pad:
            return v.to(device)
        buf = rn(npix, c + ld_pad).float().bfloat16()
        buf[:, off:off + c] = v
        return buf.to(device)[:, off:off + c]

    z, addend = act(zf), act(rn(npix, c))
    noise = rn(npix, c).float().to(device)
    return z, addend, noise, p


def ref_tensors(z, p, coef, addend=None):
    t = {"z": z.double().requires_grad_(True), "gamma": p["gamma"].double().requires_grad_(True),
         "beta": p["beta"].double().requires_grad_(True), "rm": p["rm"].double(), "rv": p["rv"].double(),
         "coef": coef.double().to(z.device)}
    if addend is not None:
        t["addend"] = addend.double()
    return t


# ----------------------------------------------------------------------------------------------------------
# §1 the reference on its own (CPU)
# ----------------------------------------------------------------------------------------------------------
def _close(a, b, what):
    a, b = a.detach(), b.detach()
    assert float((a - b).abs().max()) <= 1e-10 * max(1.0, float(b.abs().max())), what


@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("mode", ["plain", "sum", "residual"])
def test_reference_without_rounding_is_torch(mode, relu, training):
    """rounding off, the reference is torch's BatchNorm (+ ReLU), (+ addend after / before the activation) with its
    autograd gradients; in train mode the running statistics (unbiased variance) and num_batches_tracked of
    nn.BatchNorm2d follow the momentum update the emulation rounds"""
    n, h, w, c = 2, 5, 6, 16
    z, addend, _, p = make_inputs(n * h * w, c, 3, "cpu")
    t = ref_tensors(z, p, torch.zeros(4, c), addend)
    nchw = lambda v: v.reshape(n, h, w, c).permute(0, 3, 1, 2)              # [P, C] -> NCHW
    bn = torch.nn.BatchNorm2d(c, eps=EPS, momentum=MOMENTUM).double().train(training)
    with torch.no_grad():
        bn.weight.copy_(t["gamma"])
        bn.bias.copy_(t["beta"])
        bn.running_mean.copy_(t["rm"])
        bn.running_var.copy_(t["rv"])
    zo = nchw(t["z"].detach()).clone().requires_grad_(True)
    a = nchw(t["addend"])
    if mode == "residual":
        yo = bn(zo) + a
        yo = torch.relu(yo) if relu else yo
    else:
        yo = torch.relu(bn(zo)) if relu else bn(zo)
    out = bn_ref(t, training, relu, mode, rounding=False)
    y = out["y"]
    if mode == "sum":
        _close(out["ysum"], (yo + a).permute(0, 2, 3, 1).reshape(-1, c), "ysum")
    dy = torch.randn(n * h * w, c, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    _close(y, yo.permute(0, 2, 3, 1).reshape(-1, c), "y")
    yo.backward(nchw(dy))
    gz, gg, gb = torch.autograd.grad([y], [t["z"], t["gamma"], t["beta"]], [dy])
    _close(gz, zo.grad.permute(0, 2, 3, 1).reshape(-1, c), "dz")
    _close(gg, bn.weight.grad, "dgamma")
    _close(gb, bn.bias.grad, "dbeta")
    if training:
        zd = t["z"].detach()
        P = zd.shape[0]
        _close(bn.running_mean, 0.9 * t["rm"] + 0.1 * zd.mean(0), "running_mean")
        _close(bn.running_var, 0.9 * t["rv"] + 0.1 * zd.var(0, unbiased=False) * P / (P - 1), "running_var")
        assert int(bn.num_batches_tracked) == 1
        # the emulation rounds that same update: within fp32 rounding of it
        coef, rm, rv = finalize_emu(exact_stats(zd), P, p["gamma"], p["beta"], MOMENTUM, p["rm"], p["rv"])
        assert torch.allclose(rm.double(), bn.running_mean, rtol=1e-6, atol=1e-7)
        assert torch.allclose(rv.double(), bn.running_var, rtol=1e-6, atol=1e-7)
        assert torch.allclose(coef[0].double(), zd.mean(0), rtol=1e-6, atol=1e-7)


def test_fma32_is_a_single_rounding():
    """fma32 against exact rational arithmetic on values that land on and near fp32 ties"""
    g = torch.Generator().manual_seed(1)
    a = torch.randn(4000, generator=g).double()
    b = torch.randn(4000, generator=g).double()
    c = torch.randn(4000, generator=g).double() * torch.exp2(torch.randint(-30, 30, (4000,), generator=g).double())
    c[:1000] = -_f32(a[:1000] * b[:1000])                  # cancellation
    c[1000:2000] = _f32(c[1000:2000]) + torch.ldexp(torch.ones(1000, dtype=torch.float64), torch.full((1000,), -70))
    got = fma32(a, b, c)
    for i in range(0, 4000, 7):
        exact = Fraction(float(a[i])) * Fraction(float(b[i])) + Fraction(float(c[i]))
        lo = float(np.float32(float(exact)))
        cands = [np.nextafter(np.float32(lo), np.float32(-np.inf)), np.float32(lo),
                 np.nextafter(np.float32(lo), np.float32(np.inf))]
        best = min(cands, key=lambda v: (abs(Fraction(float(v)) - exact), int(np.float32(v).view(np.int32)) & 1))
        assert float(got[i]) == float(best), (i, float(got[i]), float(best))


def _cpu_case(c, kind, training, seed=5):
    npix = npix_of(kind, c, SMS_B200)
    z, _, noise, p = make_inputs(npix, c, seed, "cpu")
    st = exact_stats(z)
    if training:
        coef, rm, rv = finalize_emu(st, npix, p["gamma"], p["beta"], MOMENTUM, p["rm"], p["rv"])
    else:
        coef, rm, rv = eval_coeffs_emu(p["gamma"], p["beta"], p["rm"], p["rv"]), None, None
    t = ref_tensors(z, p, coef)
    with torch.no_grad():
        y = bn_ref(t, training, True)["y"]
    dy = correlated(y, noise).double()
    return t, dy, st, npix, p, rv


def _units(got, ref, tols):
    out = {}
    for k, v in ref.items():
        tol = tols[k] + (ulp_bf16(v) if k == "dz" else 0)
        out[k] = _worst(got[k] - v, tol)
    return max(out.values())


@pytest.mark.parametrize("c,kind", MATRIX)
def test_tolerances_see_the_mutants(c, kind):
    """each mutant moves some checked output by >= 10x the GPU test's bound for it (the running variance, which the
    GPU test holds bit-exact, by at least one fp32 ulp).  One pixel: the train-mode dz is identically 0 and x-hat is
    0, so dropping the x-hat term changes nothing, and the biased and unbiased variance of one sample are the same
    (bn.cu takes var for count 1): those two mutants are exempt there."""
    units = {}
    for training in (True, False):
        t, dy, st, npix, p, rv = _cpu_case(c, kind, training)
        ref = bwd_ref(t, training, True, dy)
        tols = bwd_tolerances(t, training, True, dy)
        for m in MUTANTS:
            if (m == "eval_batch") == training or m == "biased":
                continue
            units[m] = _units(bwd_ref(t, training, True, dy, mutant=m), ref, tols)
        if training:
            _, _, rv_b = finalize_emu(st, npix, p["gamma"], p["beta"], MOMENTUM, p["rm"], p["rv"], biased=True)
            ulp = (torch.nextafter(rv, torch.full_like(rv, math.inf)) - rv).double()
            units["biased"] = _worst((rv_b - rv).double(), ulp)
    print(f"C={c} {kind}: mutants in bound units {units}")
    for m in MUTANTS:
        if kind == "1" and m in ("xhat", "biased"):
            continue
        assert units[m] >= (1 if m == "biased" else 10), (m, units)


# ----------------------------------------------------------------------------------------------------------
# §2 the kernels one at a time, each fed the previous kernel's outputs (GPU)
# ----------------------------------------------------------------------------------------------------------
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _check_sums(got, v, label):
    """fp64 column sums of v (and of v^2 when got has two rows) within 1e-5 of the sum of |terms|"""
    vd = v.double()
    if got.dim() == 2:
        want = torch.stack([vd.sum(0), (vd * vd).sum(0)])
        tol = TOL * torch.stack([vd.abs().sum(0), (vd * vd).sum(0)])
    else:
        want, tol = vd.sum(0), TOL * vd.abs().sum(0)
    u = _worst(got.double() - want, tol)
    assert u <= 1, (label, u)
    return u


def _check_coef(coef, want, label):
    assert torch.equal(_bits(coef.cpu().contiguous()), _bits(want.contiguous())), (
        label, (coef.cpu() != want).nonzero()[:8].tolist())


def _check_apply(z, addend, coef, relu, label):
    """the four bn_apply modes, bit for bit against the reference evaluated from the kernel's own scale / shift"""
    from b200seg import kernels as K
    npix, c = z.shape
    t = {"z": z.double(), "gamma": torch.ones(c, dtype=torch.float64, device=z.device),
         "beta": torch.zeros(c, dtype=torch.float64, device=z.device), "coef": coef.double(), "addend": addend.double()}
    with torch.no_grad():
        ref = bn_ref(t, False, relu, "sum")
        res = bn_ref(t, False, relu, "residual")["y"]
    y = K.bn_apply(_nhwc(z), coef, relu=relu).view(npix, c)
    y2, ysum = K.bn_apply(_nhwc(z), coef, relu=relu, addend=_nhwc(addend), want_sum=True)
    ysum_only = K.bn_apply(_nhwc(z), coef, relu=relu, addend=_nhwc(addend), sum_only=True)
    yres = K.bn_apply(_nhwc(z), coef, relu=relu, addend=_nhwc(addend))
    want_y = ref["y"].float().bfloat16()
    for name, got, want in (("plain", y, want_y), ("sum: y", y2, want_y), ("sum: ysum", ysum, ref["ysum"].float().bfloat16()),
                            ("sum only", ysum_only, ref["ysum"].float().bfloat16()),
                            ("residual", yres, res.float().bfloat16())):
        got = got.reshape(npix, c)
        bad = (_bits(got) != _bits(want)).nonzero()
        assert bad.numel() == 0, (label, name, relu, bad[:8].tolist())
    return y


def _check_bwd(t, k, dy, training, relu, label):
    """bn_bwd against autograd of the reference under the same dy: dgamma, dbeta within 1e-5 of sum |terms|, dz within
    one bf16 ulp + 1e-5 of sum |terms|, dbias the column sums of the kernel's own dz; in the |mean| / sigma ~ 250
    channels dgamma also within the centred bound (see bwd_tolerances)"""
    npix, c = dy.shape
    ref = bwd_ref(t, training, relu, dy.double())
    tols = bwd_tolerances(t, training, relu, dy.double(), k["dz"].double())
    units = {}
    for key in ("dz", "dgamma", "dbeta"):
        tol = tols[key] + (ulp_bf16(ref[key]) if key == "dz" else 0)
        units[key] = _worst(k[key].double() - ref[key], tol)
    hi = hi_mean_channels(c)
    units["dgamma centred"] = _worst(k["dgamma"].double()[hi] - ref["dgamma"][hi], tols["dgamma_centred"][hi])
    if k.get("dbias") is not None:
        units["dbias"] = _worst(k["dbias"].double() - k["dz"].double().sum(0), tols["dbias"])
    worst = max(units, key=units.get)
    assert units[worst] <= 1, (label, units)
    return units


def _run_bwd(dy, z, coef, gamma, relu, training):
    """bn_bwd with and without the bias gradient: the same dz / dgamma / dbeta bits either way"""
    from b200seg import kernels as K
    npix, c = dy.shape
    dz, dg, db, dbias = K.bn_bwd(_nhwc(dy), _nhwc(z), coef, gamma, relu=relu, training=training, want_dbias=True)
    dz2, dg2, db2 = K.bn_bwd(_nhwc(dy), _nhwc(z), coef, gamma, relu=relu, training=training)
    for a, b in ((dz, dz2), (dg, dg2), (db, db2)):
        assert torch.equal(_bits(a), _bits(b))
    return {"dz": dz.view(npix, c), "dgamma": dg, "dbeta": db, "dbias": dbias}


def run_stages(z, addend, noise, p, training, label, relus=(True, False)):
    """the BatchNorm pipeline of one layer, each stage checked and fed the previous kernel's outputs; -> every output"""
    from b200seg import kernels as K
    npix, c = z.shape
    dev = z.device
    out = []
    # channel_stats: fp32 per thread and per block, fp64 across blocks
    stats = torch.zeros(2, c, dtype=torch.float64, device=dev)
    K.channel_stats(_nhwc(z), stats)
    _check_sums(stats, z, label + " channel_stats")
    out.append(stats)
    if training:
        # bn_finalize on the kernel's statistics, with the running buffers: every output bit-exact
        rm, rv = p["rm"].clone(), p["rv"].clone()
        nbt = torch.full((), 7, dtype=torch.int64, device=dev)
        coef_k = K.bn_finalize(stats, npix, p["gamma"], p["beta"], EPS, MOMENTUM, rm, rv, nbt)
        want, rm_w, rv_w = finalize_emu(stats, npix, p["gamma"], p["beta"], MOMENTUM, p["rm"], p["rv"])
        _check_coef(coef_k, want, label + " bn_finalize")
        _check_coef(rm, rm_w, label + " running_mean")
        _check_coef(rv, rv_w, label + " running_var")
        assert int(nbt) == 8, label
        out += [coef_k, rm, rv]
        # the backward's reference takes the batch statistics of z in fp64, so the later stages run on the coefficients
        # of the exact statistics (the ops' NULL-running call, momentum 0): with |mean| / sigma ~ 250 the one-pass
        # sum of squares of any fp32 accumulation loses ~1e-3 of the variance, which is not the backward's error
        coef = K.bn_finalize(exact_stats(z), npix, p["gamma"], p["beta"], EPS, 0.0, None, None, None)
        _check_coef(coef, finalize_emu(exact_stats(z), npix, p["gamma"], p["beta"], 0.0, None, None)[0],
                    label + " bn_finalize (no running buffers)")
    else:
        coef = K.bn_eval_coeffs(p["gamma"], p["beta"], p["rm"], p["rv"], EPS)
        _check_coef(coef, eval_coeffs_emu(p["gamma"], p["beta"], p["rm"], p["rv"]), label + " bn_eval_coeffs")
    out.append(coef)
    t = ref_tensors(z, p, coef)
    gen = torch.Generator(device=dev).manual_seed(npix + c)
    worst = {}
    for relu in relus:
        y = _check_apply(z, addend, coef, relu, label)
        out.append(y)
        for kind in ("random", "correlated"):
            if kind == "random":
                dy = torch.randn((npix, c), device=dev, generator=gen).bfloat16()
            else:
                dy = correlated(y, noise)
            db = K.channel_sum(_nhwc(dy))
            _check_sums(db, dy, f"{label} channel_sum {kind}")
            k = _run_bwd(dy, z, coef, p["gamma"], relu, training)
            units = _check_bwd(t, k, dy, training, relu, f"{label} relu={relu} dy={kind}")
            worst = {key: max(v, worst.get(key, 0.0)) for key, v in units.items()}
            out += [db] + list(k.values())
    print(f"{label}: bn_bwd worst in bound units " + ", ".join(f"{key} {v:.3g}" for key, v in worst.items()))
    return out


def _label(c, npix, training, extra=""):
    return f"C={c} npix={npix}{extra} {'train' if training else 'eval'}"


@pytest.mark.gpu
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("c,kind", MATRIX)
def test_bn_stages(c, kind, training):
    npix = npix_of(kind, c, _sms())
    z, addend, noise, p = make_inputs(npix, c, seed=c + npix, device="cuda")
    run_stages(z, addend, noise, p, training, _label(c, npix, training))


@pytest.mark.gpu
@pytest.mark.parametrize("off", [8, 64])
@pytest.mark.parametrize("c", [24, 128, 200, 1032])
def test_bn_stages_channel_slices(c, off):
    """z, dy and the addend as channel slices of wider buffers (ld = C + 64), as when a BatchNorm reads part of a
    concatenation"""
    npix = 2 * 48 * 80
    z, addend, noise, p = make_inputs(npix, c, seed=c + off, device="cuda", ld_pad=64, off=off)
    assert z.stride(0) == c + 64 and addend.stride(0) == c + 64
    for training in (True, False):
        out = run_stages(z, addend, noise, p, training, _label(c, npix, training, f" ld=C+64 at {off}"), relus=(True,))
        # and dy as a slice too
        from b200seg import kernels as K
        coef = out[4] if training else out[1]
        gen = torch.Generator(device="cuda").manual_seed(c + off + int(training))
        buf = torch.randn((npix, c + 64), device="cuda", generator=gen).bfloat16()
        dy = buf[:, off:off + c]
        k = _run_bwd(dy, z, coef, p["gamma"], True, training)
        _check_bwd(ref_tensors(z, p, coef), k, dy, training, True, f"C={c} dy slice at {off}")
        _check_sums(K.channel_sum(_nhwc(dy)), dy, f"C={c} channel_sum of a slice at {off}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["1", "126", "sweep"])
@pytest.mark.parametrize("c", C_LIST)
def test_bn_apply_modes(c, kind):
    """bn_apply's three pixel loops (4, 2 and 1 pixels in flight) past U + 1 sweeps with a partly filled last lane,
    all four modes, ReLU on and off, bit for bit"""
    sms = _sms()
    npix = sweep_count(apply_loops(c), sms) if kind == "sweep" else int(kind)
    z, addend, _, p = make_inputs(npix, c, seed=3 * c + npix, device="cuda")
    coef = torch.stack([p["rm"], p["rv"], p["gamma"] * 1.7, p["beta"]])
    for relu in (True, False):
        _check_apply(z, addend, coef, relu, f"C={c} npix={npix}")


@pytest.mark.gpu
@pytest.mark.parametrize("c,npix,off", [(8, 1, 0), (64, 126, 8), (200, 7680, 64), (2048, 1000, 8), (96, 300000, 0)])
def test_relu_mask(c, npix, off):
    """relu_mask (the ReLU of the residual BatchNorm, resnet.cu): g = out > 0 ? dy : 0 bit for bit, dy and out read as
    channel slices"""
    from b200seg import kernels as K
    gen = torch.Generator(device="cuda").manual_seed(c + npix)
    pad = 64 if off else 0
    dyb = torch.randn((npix, c + pad), device="cuda", generator=gen).bfloat16()
    outb = torch.relu(torch.randn((npix, c + pad), device="cuda", generator=gen)).bfloat16()
    outb[::3, ::5] = -outb[::3, ::5].abs() - 1
    dy, out = dyb[:, off:off + c], outb[:, off:off + c]
    g = K.relu_mask(_nhwc(dy), _nhwc(out)).view(npix, c)
    want = torch.where(out.float() > 0, dy.float(), torch.zeros_like(dy.float())).bfloat16()
    assert torch.equal(_bits(g), _bits(want))


@pytest.mark.gpu
def test_bn_update_running_multi(monkeypatch):
    """70 BatchNorms in one deferred flush (two launches of up to 64 layers, C from 8 to 2048, so blockIdx.y reaches 7
    and most layers have c < max_c): every running statistic bit-identical to bn_finalize's NULL-output call on the
    same statistics and to the emulation, every num_batches_tracked + 1"""
    from b200seg import kernels as K
    monkeypatch.delenv("B200SEG_DEFER_RUNNING", raising=False)      # its A/B switch would turn deferral off
    calls = []
    inner = K.call

    def recording_call(name, *args):
        calls.append((name, args))
        return inner(name, *args)

    monkeypatch.setattr(K, "call", recording_call)
    layers = []
    gen = torch.Generator(device="cuda").manual_seed(70)
    for i in range(70):
        c = C_LIST[(3 * i) % len(C_LIST)]
        count = [1, 126, 7680, 1 << 17][i % 4]
        mean = torch.randn(c, device="cuda", generator=gen, dtype=torch.float64)
        var = torch.rand(c, device="cuda", generator=gen, dtype=torch.float64) + 0.1
        if i % 9 == 0:
            var[0] = -1e-9                                    # clamps to 0
        stats = torch.stack([mean * count, (var + mean * mean) * count])
        rm = torch.randn(c, device="cuda", generator=gen)
        rv = torch.rand(c, device="cuda", generator=gen) + 0.5
        nbt = torch.full((), i, dtype=torch.int64, device="cuda")
        mom = 0.1 if i % 5 else 0.3
        layers.append((stats, count, mom, rm, rv, nbt))
    before = [(rm.clone(), rv.clone()) for _, _, _, rm, rv, _ in layers]
    ones = [(rm.clone(), rv.clone(), nbt.clone()) for _, _, _, rm, rv, nbt in layers]
    with K.deferred_running_updates():
        for stats, count, mom, rm, rv, nbt in layers:
            K.bn_update_running(stats, count, mom, rm, rv, nbt)
    # the whole queue went through ONE b2_bn_update_running_multi call of 70 layers, and through nothing else
    assert [(name, args[1]) for name, args in calls] == [("b2_bn_update_running_multi", 70)], calls
    for i, ((stats, count, mom, rm, rv, nbt), (rm1, rv1, nbt1), (rm0, rv0)) in enumerate(zip(layers, ones, before)):
        K.bn_update_running(stats, count, mom, rm1, rv1, nbt1)          # not deferred: bn_finalize, NULL outputs
        assert torch.equal(_bits(rm), _bits(rm1)) and torch.equal(_bits(rv), _bits(rv1)), i
        assert int(nbt) == i + 1 and int(nbt1) == i + 1, i
        _, rm_w, rv_w = finalize_emu(stats, count, None, None, mom, rm0, rv0)
        _check_coef(rm, rm_w, f"layer {i} running_mean")
        _check_coef(rv, rv_w, f"layer {i} running_var")


# ----------------------------------------------------------------------------------------------------------
# §3 the A/B switches: read once per process, so the matrix runs again in a child process
# ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("switch", ["B200SEG_BN_LIGHT", "B200SEG_BN_SLICE"])
def test_bn_stages_switched_off(switch):
    """B200SEG_BN_LIGHT=0: the 8-channel backward kernels at every C; B200SEG_BN_SLICE=0: the unsliced light kernels
    and channel_sum at C > 64.  The child recomputes its sweep counts for that geometry."""
    env = dict(os.environ, **{switch: "0"})
    here = os.path.abspath(__file__)
    r = subprocess.run([sys.executable, "-m", "pytest", f"{here}::test_bn_stages", "-q", "-x", "-p", "no:cacheprovider"],
                       env=env, cwd=os.path.dirname(os.path.dirname(here)), capture_output=True, text=True,
                       timeout=1800)
    assert r.returncode == 0, (switch, r.stdout[-4000:], r.stderr[-2000:])


# ----------------------------------------------------------------------------------------------------------
# §4 deterministic mode (GPU)
# ----------------------------------------------------------------------------------------------------------
@pytest.fixture()
def filled_workspace(monkeypatch):
    """deterministic mode on; fill(value) sets what the workspace holds before every library call from then on"""
    from b200seg import kernels as K, optim
    K.set_deterministic(True)
    state = {"value": 0.0}
    inner = K._stream

    def stream_after_fill():
        s = inner()
        buf = K._DET["bufs"][torch.cuda.current_device()]
        buf.view(torch.float64).fill_(state["value"])            # on the current stream, ahead of the call
        return s

    monkeypatch.setattr(K, "_stream", stream_after_fill)
    monkeypatch.setattr(optim, "_stream", stream_after_fill)      # (imported by name there: the gradient norm)

    def fill(value):
        state["value"] = value

    try:
        yield fill
    finally:
        monkeypatch.undo()
        K.set_deterministic(False)


@pytest.mark.gpu
@pytest.mark.parametrize("c", [24, 200, 2048])
def test_bn_stages_deterministic(filled_workspace, c):
    """every stage bit-identical over two runs and between a NaN- and a zero-filled workspace (no partial slot, also of
    a partly filled last channel slice, is left unwritten), and within the §2 bounds"""
    npix = npix_of("sweep", c, _sms())
    z, addend, noise, p = make_inputs(npix, c, seed=c, device="cuda")
    runs = []
    for v in (float("nan"), 0.0, 0.0):
        filled_workspace(v)
        runs.append(run_stages(z, addend, noise, p, True, _label(c, npix, True, " deterministic")))
        torch.cuda.synchronize()
    for i, (a, b, zz) in enumerate(zip(*runs)):
        assert torch.isfinite(b.float()).all(), (c, i)
        assert torch.equal(_bits(b), _bits(zz)), (c, i, "two runs differ")
        assert torch.equal(_bits(a), _bits(b)), (c, i, "differs when the workspace starts as NaN")


# ----------------------------------------------------------------------------------------------------------
# §5 wiring: ops.batch_norm_act with a real nn.BatchNorm2d
# ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("relu", [True, False])
@pytest.mark.parametrize("training", [True, False])
def test_batch_norm_act_wiring(training, relu):
    """the training flag, the ReLU flag and the running buffers of the module reach the kernels: z, gamma and beta
    gradients as the stage reference gives them, running statistics and num_batches_tracked updated in train mode
    (bit-exact) and untouched in eval mode"""
    from b200seg import kernels as K, ops
    n, h, w, c = 2, 24, 20, 96
    npix = n * h * w
    z, _, noise, p = make_inputs(npix, c, seed=17, device="cuda")
    bn = torch.nn.BatchNorm2d(c).cuda().train(training)
    with torch.no_grad():
        for k, v in (("weight", "gamma"), ("bias", "beta"), ("running_mean", "rm"), ("running_var", "rv")):
            getattr(bn, k).copy_(p[v])
        bn.num_batches_tracked.fill_(3)
    stats = exact_stats(z)
    zi = z.reshape(n, h, w, c).clone().requires_grad_(True)
    y = ops.batch_norm_act(zi, stats, bn, relu)
    if training:
        coef = K.bn_finalize(stats, npix, p["gamma"], p["beta"], EPS, 0.0, None, None, None)
        _, rm_w, rv_w = finalize_emu(stats, npix, p["gamma"], p["beta"], MOMENTUM, p["rm"], p["rv"])
        _check_coef(bn.running_mean, rm_w, "running_mean")
        _check_coef(bn.running_var, rv_w, "running_var")
        assert int(bn.num_batches_tracked) == 4
    else:
        coef = K.bn_eval_coeffs(p["gamma"], p["beta"], p["rm"], p["rv"], EPS)
        assert torch.equal(bn.running_mean, p["rm"]) and torch.equal(bn.running_var, p["rv"])
        assert int(bn.num_batches_tracked) == 3
    t = ref_tensors(z, p, coef)
    with torch.no_grad():
        want = bn_ref(t, training, relu)["y"].float().bfloat16()
    assert torch.equal(_bits(y.detach().reshape(npix, c)), _bits(want))
    dy = correlated(y.detach().reshape(npix, c), noise)
    y.backward(dy.reshape(n, h, w, c))
    k = {"dz": zi.grad.reshape(npix, c), "dgamma": bn.weight.grad, "dbeta": bn.bias.grad}
    _check_bwd(t, k, dy, training, relu, f"batch_norm_act {'train' if training else 'eval'} relu={relu}")
