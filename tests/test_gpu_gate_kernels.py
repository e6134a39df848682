"""The train-mode attention-gate kernels of csrc/gate.cu, one at a time and as one autograd node, against an fp64
reference that rounds where the kernels round.

Everything in a gate after its two 1x1 GEMMs is five kernels: b2_gate_psi_fwd, b2_gate_apply_fwd, b2_gate_apply_bwd,
b2_gate_psi_bwd_reduce and b2_gate_psi_bwd_apply.  They hold three BatchNorms (BN_g, BN_x and BN1 on the psi
pre-activation) whose backward is written in a collapsed form.  A reference without bf16 rounding flips ReLU masks
against the kernels, which forces tolerances loose enough to hide whole BatchNorm-backward terms.  So the reference
here is a forward with straight-through rounding at exactly the kernels' rounding points (gate.cu: every BN output,
g1 + x1, the psi dot, the BN1 output, sigmoid, x * psi): each rounded node has the rounded value and the gradient of
the unrounded one, and the masks are bit-identical to the kernels'.  Its backward is torch autograd, never a
transcription of the kernels' formulas.

Every tolerance is 1e-5 (fp32 accumulation) of the sum of the absolute values of the terms the kernel adds, plus one
bf16 ulp where the kernel rounds its output.  The unmarked tests check the reference against the oracle and check that
four plausible kernel bugs move some checked output by at least 10x its tolerance under an upstream gradient
correlated with the output (the gradient of sum(out^2)), at every shape of the GPU matrix.  With a random upstream
gradient the BatchNorm batch terms are O(1/sqrt(npix)); with a correlated one they are O(1).
"""
import math

import pytest
import torch

EPS = 1e-5
TOL = 1e-5              # fp32 accumulation: relative to the sum of the absolute values of the terms
SMS_B200 = 148

FINTS = [8, 24, 32, 64, 96, 128, 200, 256]          # <= 64 unsliced U=4; 72..128 sliced U=4; 136..256 sliced U=2
PIX = ["1", "2x7x9", "2x48x80", "sweep"]
C_LIST = [8, 64, 256, 320, 512, 1024]
MUTANTS = ["bn1", "bngx", "swap", "relu"]


def _pow2ceil(v):
    p = 1
    while p < v:
        p <<= 1
    return p


def _sweep(fint, c, sms):
    """pixels of one full grid-stride sweep (grid at its cap x pixels per block x pixels in flight) of the gate kernels
    at this F_int and C, as the launchers in gate.cu size them; the largest of the five"""
    cap8, cap16 = sms * 8, sms * 16
    sliced = fint > 64
    slices = -(-fint // 64) if sliced else 1
    u = 4 if fint <= 128 else 2
    psi_fwd = cap8 * (256 // _pow2ceil(fint // 8))
    reduce = -(-cap8 // slices) * (256 // _pow2ceil((64 if sliced else fint) // 4)) * u
    apply = -(-cap8 // slices) * (256 // (16 if sliced else fint // 4)) * u
    apply_fwd = cap16 * (256 // (c // 8))
    apply_bwd = cap8 * (256 // min(_pow2ceil(c // 8), 32)) * 2
    return max(psi_fwd, reduce, apply, apply_fwd, apply_bwd)


def _npix(kind, fint, c, sms):
    if kind == "sweep":
        s = _sweep(fint, c, sms)
        return s + s // 7 + 37           # past one full sweep, not a multiple of it: every tail runs
    return math.prod(int(v) for v in kind.split("x"))


def _matrix():
    out = []
    for i, fint in enumerate(FINTS):
        for j, kind in enumerate(PIX):
            c = C_LIST[(i + j) % len(C_LIST)]
            if kind == "sweep" and fint <= 64:
                c = min(c, 64)           # these sweeps are ~10^5 - 10^6 pixels: keep x small
            out.append((fint, kind, c))
    return out


MATRIX = _matrix()


# ----------------------------------------------------------------------------------------------------------
# the reference (fp64, torch, any device)
# ----------------------------------------------------------------------------------------------------------
def _r(v):
    """fp64 -> fp32 -> bf16, as fp64: the kernels round fp32 results (fp64 straight to bf16 can round differently)"""
    return v.detach().float().bfloat16().double()


def _st(v, value):
    """the value `value` (exactly), the gradient of v"""
    return value.detach() + (v - v.detach())


def _bn(v, coef, gamma, beta, rm, rv, training, rounding, detach_stats):
    """BatchNorm over dim 0 of v [P, C] as y = v * scale + shift.  Rounding: y has the value bf16(fp32(v * scale +
    shift)) with scale / shift the fp32 coefficient rows the kernel received; its gradient flows through the fp64
    batch statistics (train) or the running statistics (eval)."""
    if training:
        mean, var = v.mean(0), v.var(0, unbiased=False)
        if detach_stats:                  # a mutant: the batch statistics treated as constants
            mean, var = mean.detach(), var.detach()
        invstd = (var + EPS).rsqrt()
    elif rounding:
        mean, invstd = coef[0], coef[1]
    else:
        mean, invstd = rm, (rv + EPS).rsqrt()
    scale = gamma * invstd
    y = v * scale + (beta - mean * scale)
    if not rounding:
        return y
    return _st(y, _r(v.detach() * coef[2] + coef[3]))


def gate_ref(t, training, rounding=True, mutant=None, q=None, psi=None):
    """The gate after its two GEMMs.  t: fp64 tensors g1p, x1p [P, F], x [P, C]; gamma_g, beta_g, gamma_x, beta_x,
    wpsi [F]; bpsi, gamma_1, beta_1 [1]; running statistics rm_*, rv_*; fp32-valued coefficient rows coef_g, coef_x
    [4, F], coef_1 [4, 1] = (mean, invstd, scale, shift).  q / psi: evaluate at these values (the kernel's own) instead
    of the reference's.  mutant: 'bn1' / 'bngx' drop the batch-statistics terms of BN1 / BN_g and BN_x, 'relu' takes
    the ReLU mask from the unrounded g1 + x1 ('swap' is applied to the gradients, see grads()).
    -> dict of graph nodes."""
    g1 = _bn(t["g1p"], t.get("coef_g"), t["gamma_g"], t["beta_g"], t["rm_g"], t["rv_g"], training, rounding,
             mutant == "bngx")
    x1 = _bn(t["x1p"], t.get("coef_x"), t["gamma_x"], t["beta_x"], t["rm_x"], t["rv_x"], training, rounding,
             mutant == "bngx")
    s = g1 + x1
    if rounding:
        s = _st(s, _r(s))
    a = torch.relu(s)
    if mutant == "relu":
        with torch.no_grad():
            g1u = t["g1p"] * t["coef_g"][2] + t["coef_g"][3]
            x1u = t["x1p"] * t["coef_x"][2] + t["coef_x"][3]
        a = _st(torch.where(g1u + x1u > 0, s, torch.zeros_like(s)), a)
    wp = _st(t["wpsi"], _r(t["wpsi"])) if rounding else t["wpsi"]
    qn = a @ wp + t["bpsi"]
    if rounding:
        qn = _st(qn, q if q is not None else _r(qn))
    z = _bn(qn[:, None], t.get("coef_1"), t["gamma_1"], t["beta_1"], t["rm_1"], t["rv_1"], training, rounding,
            mutant == "bn1")[:, 0]
    if rounding:
        # sigmoid whose backward uses its saved (rounded) output, as torch's own sigmoid backward does
        pv = psi if psi is not None else _r(torch.sigmoid(z))
        p = pv + pv * (1 - pv) * (z - z.detach())
        out = t["x"] * p[:, None]
        out = _st(out, _r(out))
    else:
        p = torch.sigmoid(z)
        out = t["x"] * p[:, None]
    return {"g1": g1, "x1": x1, "a": a, "wp": wp, "q": qn, "z": z, "psi": p, "out": out}


PARAMS = ["gamma_g", "beta_g", "gamma_x", "beta_x", "wpsi", "bpsi", "gamma_1", "beta_1"]


def grads(t, nodes, root, upstream, mutant=None):
    """autograd of nodes[root] under `upstream` -> gradients of g1p, x1p, x and PARAMS, and of the nodes z and q"""
    keys = ["g1p", "x1p", "x"] + PARAMS
    ins = [t[k] for k in keys] + [nodes["z"], nodes["q"]]
    gs = torch.autograd.grad([nodes[root]], ins, [upstream], retain_graph=True, allow_unused=True)
    out = {k: (g if g is not None else torch.zeros_like(i)) for k, g, i in zip(keys + ["dz", "dq"], gs, ins)}
    if mutant == "swap":
        out["gamma_g"], out["gamma_x"] = out["gamma_x"], out["gamma_g"]
    return out


def psi_bwd_tolerances(t, nodes, dz, training):
    """per checked output of the psi backward, TOL x the sum of the absolute values of the terms the kernels add
    (gate_dq, the reduce kernel's sums, and the collapsed dg1p = Wg*dq*[a>0] + Bg*g + Cg), plus one bf16 ulp of the
    reference for the rounded dg1p / dx1p (added by the caller)"""
    with torch.no_grad():
        c1, c_g, c_x = t["coef_1"], t["coef_g"], t["coef_x"]
        qh = (nodes["q"] - c1[0, 0]) * c1[1, 0]
        gh = (t["g1p"] - c_g[0]) * c_g[1]
        xh = (t["x1p"] - c_x[0]) * c_x[1]
        k1 = (t["gamma_1"] * c1[1]).abs()
        adz = dz.abs()
        mdq = k1 * (adz + adz.mean() + qh.abs() * (dz * qh).abs().mean()) if training else k1 * adz
        a = nodes["a"].detach()
        mda = mdq[:, None] * nodes["wp"].detach().abs() * (a > 0)
        mag = {"gamma_g": (mda * gh.abs()).sum(0), "gamma_x": (mda * xh.abs()).sum(0), "beta_g": mda.sum(0),
               "beta_x": mda.sum(0), "wpsi": (mdq[:, None] * a).sum(0), "bpsi": mdq.sum().reshape(1),
               "gamma_1": (dz * qh).abs().sum().reshape(1), "beta_1": adz.sum().reshape(1)}
        for key, v, c, hat in (("g1p", t["g1p"], c_g, gh), ("x1p", t["x1p"], c_x, xh)):
            gam = (t["gamma_" + key[0]] * c[1]).abs()
            if training:
                mag[key] = gam * (mda + mda.mean(0) + c[1] * (v.abs() + c[0].abs()) * (mda * hat.abs()).mean(0))
            else:
                mag[key] = gam * mda
    return {k: TOL * v for k, v in mag.items()}


def ulp_bf16(v):
    """one bf16 ulp of |v| (0 where v is 0)"""
    a = v.detach().abs()
    e = torch.floor(torch.log2(torch.where(a > 0, a, torch.ones_like(a))))
    return torch.where(a > 0, torch.exp2(e - 7), torch.zeros_like(a))


def _worst(err, tol):
    """max of |err| / tol (tol 0 where err 0 counts as 0)"""
    err = err.abs()
    r = torch.where(err > 0, err / tol.clamp_min(1e-300), torch.zeros_like(err))
    return float(r.max()) if r.numel() else 0.0


def psi_bwd_checked(t, nodes, dz, training, mutant=None):
    """reference gradients of the outputs of b2_gate_psi_bwd_* under the upstream dz at the BN1 output"""
    g = grads(t, nodes, "z", dz, mutant)
    return {k: g[k] for k in ["g1p", "x1p"] + PARAMS}


def mutant_units(t, training, dz, tols, ref, q, psi):
    """for each mutant: the largest deviation of a checked psi-backward output from the true reference, in units of the
    tolerance the GPU test uses for it"""
    out = {}
    for m in MUTANTS:
        nodes = gate_ref(t, training, mutant=m, q=q, psi=psi)
        mg = psi_bwd_checked(t, nodes, dz, training, mutant=m)
        out[m] = max(_worst(mg[k] - ref[k], tols[k] + (ulp_bf16(ref[k]) if k in ("g1p", "x1p") else 0))
                     for k in ref)
    return out


# ----------------------------------------------------------------------------------------------------------
# inputs
# ----------------------------------------------------------------------------------------------------------
def make_inputs(npix, fint, c, seed, device, ld_pad=0):
    """bf16 g1p, x1p [P, F], x [P, C] (x a channel slice of a wider buffer when ld_pad > 0), fp32 parameters and
    running statistics.  Every eighth channel (f % 8 == 5) is a cancellation channel: x1p = -g1p and BN_x the negated
    BN_g up to beta_x = -beta_g + 2^-14, so g1 + x1 = 2^-14 before rounding and the bf16 sum is (mostly) exactly 0 —
    the ReLU mask there depends on where the kernel rounds."""
    gen = torch.Generator(device="cpu").manual_seed(seed)

    def rn(*s):
        return torch.randn(*s, generator=gen, dtype=torch.float64)

    def ru(*s):
        return torch.rand(*s, generator=gen, dtype=torch.float64)

    tie = torch.arange(fint) % 8 == 5
    g1p = (rn(npix, fint) * 0.7 + 0.3).float().bfloat16()
    x1p = (rn(npix, fint) * 1.3 - 0.2).float().bfloat16()
    x1p[:, tie] = -g1p[:, tie]
    p = {"gamma_g": 0.5 + ru(fint), "beta_g": 0.2 * rn(fint), "gamma_x": 0.5 + ru(fint), "beta_x": 0.2 * rn(fint),
         "wpsi": rn(fint) / fint ** 0.5, "bpsi": 0.1 * rn(1), "gamma_1": 0.8 + 0.6 * ru(1), "beta_1": 0.2 * rn(1),
         "rm_g": 0.3 + 0.1 * rn(fint), "rv_g": 0.4 + ru(fint), "rm_x": -0.2 + 0.2 * rn(fint), "rv_x": 1.2 + ru(fint),
         "rm_1": 0.1 * rn(1), "rv_1": 0.3 + ru(1)}
    p["gamma_x"][tie] = p["gamma_g"][tie]
    p["beta_x"][tie] = -p["beta_g"][tie] + 2.0 ** -14
    p["rm_x"][tie] = -p["rm_g"][tie]
    p["rv_x"][tie] = p["rv_g"][tie]
    p = {k: v.float().to(device) for k, v in p.items()}
    xb = rn(npix, c + ld_pad).float().bfloat16().to(device)
    x = xb[:, ld_pad // 2: ld_pad // 2 + c] if ld_pad else xb
    noise = rn(npix, c).float().to(device)
    return g1p.to(device), x1p.to(device), x, p, noise


def bn_coef_torch(v, gamma, beta, rm, rv, training):
    """fp32 coefficient rows (mean, invstd, scale, shift) computed as b2_bn_finalize / b2_bn_eval_coeffs do"""
    if training:
        vd = v.double()
        m = vd.mean(0)
        var = ((vd * vd).mean(0) - m * m).clamp_min(0)
        fm, inv = m.float(), (1.0 / (var + EPS).sqrt()).float()
    else:
        fm, inv = rm, (1.0 / (rv.double() + EPS).sqrt()).float()
    sc = gamma * inv
    return torch.stack([fm, inv, sc, beta - fm * sc])


def ref_tensors(g1p, x1p, x, p, coef_g, coef_x, coef_1, requires_grad=True):
    """fp64 leaves for gate_ref from the kernel-side tensors"""
    t = {"g1p": g1p.double(), "x1p": x1p.double(), "x": x.double()}
    for k in PARAMS:
        t[k] = p[k].double()
    t = {k: v.clone().requires_grad_(requires_grad) for k, v in t.items()}
    for k in ("rm_g", "rv_g", "rm_x", "rv_x", "rm_1", "rv_1"):
        t[k] = p[k].double()
    t["coef_g"], t["coef_x"] = coef_g.double(), coef_x.double()
    if coef_1 is not None:
        t["coef_1"] = coef_1.double()
    return t


def correlated(out, noise):
    """the upstream gradient of sum(out^2), plus a little noise"""
    return (2 * out.double() + 0.1 * noise.double()).float().bfloat16()


# ----------------------------------------------------------------------------------------------------------
# §1 the reference on its own (CPU)
# ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("c,fint", [(16, 8), (24, 24)])
def test_reference_without_rounding_is_the_oracle(c, fint, training):
    """rounding off, the reference (from the two GEMM outputs on) has the oracle's value and autograd gradients"""
    from oracle import unet_oracle as O
    n, h, w = 2, 5, 6
    g1p, x1p, _x, p, _ = make_inputs(n * h * w, fint, c, 3, "cpu")
    gen = torch.Generator().manual_seed(9)
    sd = {"att.W_g.0.weight": torch.randn(fint, c, 1, 1, generator=gen, dtype=torch.float64) / c ** 0.5,
          "att.W_g.0.bias": 0.1 * torch.randn(fint, generator=gen, dtype=torch.float64),
          "att.W_x.0.weight": torch.randn(fint, c, 1, 1, generator=gen, dtype=torch.float64) / c ** 0.5,
          "att.W_x.0.bias": 0.1 * torch.randn(fint, generator=gen, dtype=torch.float64),
          "att.psi.0.weight": p["wpsi"].double().view(1, fint, 1, 1), "att.psi.0.bias": p["bpsi"].double()}
    for br, key in (("W_g.1", "g"), ("W_x.1", "x"), ("psi.1", "1")):
        sd[f"att.{br}.weight"] = p["gamma_" + key].double()
        sd[f"att.{br}.bias"] = p["beta_" + key].double()
        sd[f"att.{br}.running_mean"] = p["rm_" + key].double()
        sd[f"att.{br}.running_var"] = p["rv_" + key].double()
        sd[f"att.{br}.num_batches_tracked"] = torch.tensor(0)
    g = torch.randn(n, c, h, w, generator=gen, dtype=torch.float64)
    x = torch.randn(n, c, h, w, generator=gen, dtype=torch.float64)
    dy = torch.randn(n, c, h, w, generator=gen, dtype=torch.float64)

    leaves = {k: v.clone().requires_grad_(True) for k, v in sd.items() if v.is_floating_point() and "running" not in k}
    go, xo = g.clone().requires_grad_(True), x.clone().requires_grad_(True)
    yo, _ = O.attention_gate({**sd, **leaves}, go, xo, "att", training=training)
    yo.backward(dy)

    gr, xr = g.clone().requires_grad_(True), x.clone().requires_grad_(True)
    lw = {k: v.clone().requires_grad_(True) for k, v in sd.items() if k.endswith(".0.weight") or k.endswith(".0.bias")}
    flat = lambda v: v.permute(0, 2, 3, 1).reshape(-1, v.shape[1])           # NCHW -> [P, C]
    t = {"g1p": flat(gr) @ lw["att.W_g.0.weight"][:, :, 0, 0].T + lw["att.W_g.0.bias"],
         "x1p": flat(xr) @ lw["att.W_x.0.weight"][:, :, 0, 0].T + lw["att.W_x.0.bias"], "x": flat(xr)}
    names = {"gamma_g": "W_g.1.weight", "beta_g": "W_g.1.bias", "gamma_x": "W_x.1.weight", "beta_x": "W_x.1.bias",
             "gamma_1": "psi.1.weight", "beta_1": "psi.1.bias"}
    for k, s in names.items():
        t[k] = sd["att." + s].clone().requires_grad_(True)
    t["wpsi"] = lw["att.psi.0.weight"].view(-1)
    t["bpsi"] = lw["att.psi.0.bias"]
    for k in ("rm_g", "rv_g", "rm_x", "rv_x", "rm_1", "rv_1"):
        t[k] = p[k].double()
    nodes = gate_ref(t, training, rounding=False)
    y = nodes["out"].reshape(n, h, w, c).permute(0, 3, 1, 2)
    y.backward(dy)

    def close(a, b, what):
        a, b = a.detach(), b.detach()
        assert float((a - b).abs().max()) <= 1e-10 * max(1.0, float(b.abs().max())), what

    close(y, yo, "out")
    close(gr.grad, go.grad, "dg")
    close(xr.grad, xo.grad, "dx")
    for k, v in lw.items():
        close(v.grad, leaves[k].grad, k)
    for k, s in names.items():
        close(t[k].grad, leaves["att." + s].grad, s)


def _cpu_case(fint, kind, c, training, seed=5):
    """the reference pipeline on the CPU: inputs, coefficient rows, rounded forward, correlated upstream, dsig"""
    npix = _npix(kind, fint, c, SMS_B200)
    g1p, x1p, _x, p, _ = make_inputs(npix, fint, 8, seed, "cpu")     # C only enters through x: keep it small here
    x = _x
    noise = torch.randn(npix, 8, generator=torch.Generator().manual_seed(seed + 1))
    coef_g = bn_coef_torch(g1p, p["gamma_g"], p["beta_g"], p["rm_g"], p["rv_g"], training)
    coef_x = bn_coef_torch(x1p, p["gamma_x"], p["beta_x"], p["rm_x"], p["rv_x"], training)
    t = ref_tensors(g1p, x1p, x, p, coef_g, coef_x, None)
    # BN1's rows come from the reference's own rounded q
    with torch.no_grad():
        pre = gate_ref({**t, "coef_1": torch.zeros(4, 1, dtype=torch.float64)}, False)
    qv = pre["q"].detach()
    t["coef_1"] = bn_coef_torch(qv[:, None].float(), p["gamma_1"], p["beta_1"], p["rm_1"], p["rv_1"],
                                training).double()
    nodes = gate_ref(t, training)
    dout = correlated(nodes["out"].detach(), noise).double()
    dz = grads(t, nodes, "out", dout)["dz"].detach()
    return t, nodes, dz, qv, nodes["psi"].detach()


@pytest.mark.parametrize("fint,kind,c", MATRIX)
def test_tolerances_see_the_mutants(fint, kind, c):
    """each mutant moves some checked output of the psi backward by >= 10x the GPU test's tolerance for it.
    At one pixel the train-mode gradient below BN1 is identically zero (q - mean = 0, so dq = 0), which no mutant of
    BN_g / BN_x, the mask or dgamma can change: there the mask and dgamma mutants are checked in eval mode and the
    BN_g / BN_x one is exempt (eval mode has no batch terms)."""
    units = {}
    for training in (True, False):
        t, nodes, dz, qv, pv = _cpu_case(fint, kind, c, training)
        ref = psi_bwd_checked(t, nodes, dz, training)
        tols = psi_bwd_tolerances(t, nodes, dz, training)
        units[training] = mutant_units(t, training, dz, tols, ref, qv, pv)
    print(f"F_int={fint} {kind}: mutants in tolerance units, train {units[True]}, eval {units[False]}")
    if kind != "1":
        need = [(m, True) for m in MUTANTS]
    else:
        need = [("bn1", True), ("swap", False), ("relu", False)]
    for m, training in need:
        assert units[training][m] >= 10, (m, "train" if training else "eval", units)


# ----------------------------------------------------------------------------------------------------------
# §2 the five kernels one at a time, each fed the kernel's own upstream tensors (GPU)
# ----------------------------------------------------------------------------------------------------------
def _nhwc(t):
    """[P, C] (possibly a channel slice of a wider row) -> the [1, 1, P, C] view the kernel wrappers take"""
    return t.as_strided((1, 1) + tuple(t.shape), (t.shape[0] * t.stride(0), t.shape[0] * t.stride(0)) + t.stride())


def _gpu_case(fint, npix, c, training, seed, ld_pad=0):
    from b200seg import kernels as K
    g1p, x1p, x, p, noise = make_inputs(npix, fint, c, seed, "cuda", ld_pad)
    if training:
        def coef(v, key):
            vd = v.double()
            stats = torch.stack([vd.sum(0), (vd * vd).sum(0)])
            return K.bn_finalize(stats, npix, p["gamma_" + key], p["beta_" + key], EPS, 0.0, None, None, None)
    else:
        def coef(v, key):
            return K.bn_eval_coeffs(p["gamma_" + key], p["beta_" + key], p["rm_" + key], p["rv_" + key], EPS)
    return {"g1p": g1p, "x1p": x1p, "x": x, "p": p, "noise": noise, "coef_g": coef(g1p, "g"),
            "coef_x": coef(x1p, "x"), "training": training, "npix": npix}


def _run_kernels(cs, dout_kinds=("random", "correlated")):
    """the gate's five kernels in pipeline order; every stage takes the previous stage's kernel outputs"""
    from b200seg import kernels as K
    p, npix, training = cs["p"], cs["npix"], cs["training"]
    r = {}
    q, qstats = K.gate_psi_fwd(_nhwc(cs["g1p"]), _nhwc(cs["x1p"]), cs["coef_g"], cs["coef_x"], p["wpsi"], p["bpsi"])
    if training:
        coef_1 = K.bn_finalize(qstats, npix, p["gamma_1"], p["beta_1"], EPS, 0.0, None, None, None)
    else:
        coef_1 = K.bn_eval_coeffs(p["gamma_1"], p["beta_1"], p["rm_1"], p["rv_1"], EPS)
    out, psi = K.gate_apply_fwd(_nhwc(cs["x"]), q, coef_1)
    r.update(q=q.view(npix), qstats=qstats.clone(), coef_1=coef_1, out=out.view(npix, -1), psi=psi.view(npix))
    gen = torch.Generator(device="cuda").manual_seed(npix)
    for kind in dout_kinds:
        if kind == "random":
            dout = torch.randn(r["out"].shape, device="cuda", generator=gen).bfloat16()
        else:
            dout = correlated(r["out"], cs["noise"])
        dx, dsig, sums1 = K.gate_apply_bwd(_nhwc(dout), _nhwc(cs["x"]), psi, q, coef_1)
        sums1 = sums1.clone()
        dg1p, dx1p, dgb, dbn1, dwpsi, dbpsi, dbias = K.gate_psi_bwd(
            dsig, sums1, q, _nhwc(cs["g1p"]), _nhwc(cs["x1p"]), cs["coef_g"], p["gamma_g"], cs["coef_x"],
            p["gamma_x"], coef_1, p["gamma_1"], p["wpsi"], training=training)
        r[kind] = {"dout": dout, "dx": dx.view(npix, -1), "dsig": dsig.view(npix), "sums1": sums1,
                   "dg1p": dg1p.view(npix, -1), "dx1p": dx1p.view(npix, -1), "dgb": dgb, "dbn1": dbn1,
                   "dwpsi": dwpsi, "dbpsi": dbpsi, "dbias": dbias}
    return r


def _bits(t):
    return t.view(torch.int16) if t.dtype == torch.bfloat16 else t.view(torch.int32 if t.element_size() == 4
                                                                        else torch.int64)


def _psi_bwd_outputs(b):
    """the kernels' psi-backward outputs under the reference's names"""
    return {"g1p": b["dg1p"], "x1p": b["dx1p"], "gamma_g": b["dgb"][0], "beta_g": b["dgb"][1],
            "gamma_x": b["dgb"][2], "beta_x": b["dgb"][3], "wpsi": b["dwpsi"], "bpsi": b["dbpsi"],
            "gamma_1": b["dbn1"][0:1], "beta_1": b["dbn1"][1:2]}


def _check_psi_bwd(t, nodes, b, training, label, with_mutants=True):
    """b2_gate_psi_bwd_reduce + _apply against autograd of the reference from the BN1 output, under the kernel's dsig.
    dwpsi, dbpsi, dgamma / dbeta of both branches, dbn1: |err| <= TOL x (sum of |terms|); dg1p / dx1p: one bf16 ulp
    plus TOL x (sum of |terms|).  dbias: the column sums of the kernel's own rounded dg1p / dx1p, TOL x sum |dg1p|
    (fp32 per-thread and per-block sums, fp32 atomics across blocks)."""
    dz = b["dsig"].double()
    ref = psi_bwd_checked(t, nodes, dz, training)
    tols = psi_bwd_tolerances(t, nodes, dz, training)
    got = _psi_bwd_outputs(b)
    units = {}
    for k, v in ref.items():
        tol = tols[k] + (ulp_bf16(v) if k in ("g1p", "x1p") else 0)
        units[k] = _worst(got[k].double() - v, tol)
    for i, k in enumerate(("dg1p", "dx1p")):
        v = b[k].double()
        units["bias_" + k] = _worst(b["dbias"][i].double() - v.sum(0), TOL * v.abs().sum(0))
    worst = max(units, key=units.get)
    mut = mutant_units(t, training, dz, tols, ref, nodes["q"].detach(), nodes["psi"].detach()) if with_mutants else {}
    print(f"{label} psi_bwd: worst {units[worst]:.3f} tol ({worst}); mutants "
          + ", ".join(f"{m} {u:.3g}" for m, u in mut.items()))
    assert units[worst] <= 1, (label, units)


def _check_stages(cs, r, label, with_mutants=True):
    p, training, npix = cs["p"], cs["training"], cs["npix"]
    t = ref_tensors(cs["g1p"], cs["x1p"], cs["x"], p, cs["coef_g"], cs["coef_x"], r["coef_1"])
    rep = {}
    with torch.no_grad():
        # gate_psi_fwd: q within one bf16 ulp + the fp32 error of the psi dot (<= 14 fp32 roundings deep: 8-channel
        # fma chains and the <= 32-lane shuffle tree) and bit-equal on >= 99.9 % of the pixels
        n0 = gate_ref(t, training)
        qk, qr = r["q"].double(), n0["q"]
        mag = (n0["a"] * n0["wp"].abs()).sum(1) + t["bpsi"].abs()
        rep["q"] = _worst(qk - qr, ulp_bf16(qr) + 1e-6 * mag)
        off = int((qk != qr).sum())
        assert off <= max(1, npix // 1000), (label, "q bit-equal on too few pixels", off, npix)
        # qstats: the fp64 (sum q, sum q^2) of the kernel's own q; per-thread, warp and block sums are fp32
        want = torch.stack([qk.sum(), (qk * qk).sum()])
        rep["qstats"] = _worst(r["qstats"] - want, 1e-6 * torch.stack([qk.abs().sum(), (qk * qk).sum()]))
        # gate_apply_fwd: out = bf16(x * psi) bit for bit (an exact product, rounded once); psi within one ulp
        x = cs["x"].double()
        assert torch.equal(_bits(r["out"]), _bits(_r(x * r["psi"].double()[:, None]).bfloat16())), label
        n1 = gate_ref(t, training, q=qk)
        rep["psi"] = _worst(r["psi"].double() - n1["psi"], ulp_bf16(n1["psi"]))
    nodes = gate_ref(t, training, q=qk, psi=r["psi"].double())
    for kind in ("random", "correlated"):
        if kind not in r:
            continue
        b = r[kind]
        dout = b["dout"].double()
        with torch.no_grad():
            psi = r["psi"].double()
            # gate_apply_bwd: dx = bf16(dout * psi) bit for bit
            assert torch.equal(_bits(b["dx"]), _bits(_r(dout * psi[:, None]).bfloat16())), (label, kind, "dx")
        # dsig: fp32 sum over C of dout * x, times psi (1 - psi)
        dz = grads(t, nodes, "out", dout)["dz"].detach()
        with torch.no_grad():
            tol = 1e-5 * psi * (1 - psi) * (dout * x).abs().sum(1)
            rep[kind + " dsig"] = _worst(b["dsig"].double() - dz, tol)
            # sums1 = (sum dsig, sum dsig * qhat) of the kernel's own dsig, fp32 within a block
            c1 = r["coef_1"].double()
            ds = b["dsig"].double()
            qh = (qk - c1[0, 0]) * c1[1, 0]
            rep[kind + " sums1"] = _worst(b["sums1"] - torch.stack([ds.sum(), (ds * qh).sum()]),
                                          1e-5 * torch.stack([ds.abs().sum(), (ds * qh).abs().sum()]))
        _check_psi_bwd(t, nodes, b, training, f"{label} dout={kind}", with_mutants)
    worst = max(rep, key=rep.get)
    print(f"{label} fwd / apply_bwd: worst {rep[worst]:.3f} tol ({worst})")
    assert rep[worst] <= 1, (label, rep)


def _label(fint, npix, c, training, extra=""):
    return f"F_int={fint} npix={npix} C={c}{extra} {'train' if training else 'eval'}"


@pytest.mark.gpu
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("fint,kind,c", MATRIX)
def test_gate_stages(fint, kind, c, training):
    npix = _npix(kind, fint, c, torch.cuda.get_device_properties(0).multi_processor_count)
    cs = _gpu_case(fint, npix, c, training, seed=fint + npix)
    r = _run_kernels(cs)
    _check_stages(cs, r, _label(fint, npix, c, training))


@pytest.mark.gpu
@pytest.mark.parametrize("training", [True, False])
def test_gate_stages_strided_x(training):
    """x a channel slice of a wider buffer (ldx > C), as when the gate reads part of a concatenation"""
    fint, npix, c = 64, 2 * 48 * 80, 320
    cs = _gpu_case(fint, npix, c, training, seed=11, ld_pad=16)
    assert cs["x"].stride(0) == c + 16
    _check_stages(cs, _run_kernels(cs), _label(fint, npix, c, training, " ldx=C+16"))


@pytest.mark.gpu
@pytest.mark.parametrize("npix", [1, 2 * 7 * 9, 2 * 48 * 80, 7001])
def test_gate_apply_fwd_c2048(npix):
    """the widest C the forward apply takes: one pixel per block"""
    from b200seg import kernels as K
    c = 2048
    g = torch.Generator(device="cuda").manual_seed(npix)
    x = torch.randn((npix, c), device="cuda", generator=g).bfloat16()
    q = torch.randn((1, 1, npix), device="cuda", generator=g).bfloat16()
    coef_1 = torch.tensor([[0.1], [1.3], [0.9], [-0.2]], device="cuda")
    out, psi = K.gate_apply_fwd(_nhwc(x), q, coef_1)
    c1 = coef_1.double()
    psi_ref = _r(torch.sigmoid(_r(q.double().view(-1) * c1[2, 0] + c1[3, 0])))
    assert _worst(psi.double().view(-1) - psi_ref, ulp_bf16(psi_ref)) <= 1
    assert torch.equal(_bits(out.view(npix, c)), _bits(_r(x.double() * psi.double().view(-1, 1)).bfloat16()))


# ----------------------------------------------------------------------------------------------------------
# §3 the gate as one autograd node (GPU)
# ----------------------------------------------------------------------------------------------------------
MODULE_SHAPES = [(64, 32, 2, 48, 80), (256, 128, 2, 9, 7), (512, 256, 1, 16, 16)]


def _gate_module(c, fint, seed):
    from b200seg import blocks
    torch.manual_seed(seed)
    m = blocks.AttentionGate(c, c, fint).cuda()
    gen = torch.Generator(device="cuda").manual_seed(seed)
    with torch.no_grad():
        for bn in (m.W_g[1], m.W_x[1], m.psi[1]):      # non-trivial affine parameters and running statistics
            sh = bn.weight.shape
            bn.weight.copy_(0.5 + torch.rand(sh, device="cuda", generator=gen))
            bn.bias.copy_(0.2 * torch.randn(sh, device="cuda", generator=gen))
            bn.running_mean.copy_(0.2 * torch.randn(sh, device="cuda", generator=gen))
            bn.running_var.copy_(0.5 + torch.rand(sh, device="cuda", generator=gen))
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("dout_kind", ["random", "correlated"])
@pytest.mark.parametrize("mode", ["train", "eval", "pass", "no_dg"])
@pytest.mark.parametrize("c,fint,n,h,w", MODULE_SHAPES)
def test_attention_gate_node(c, fint, n, h, w, mode, dout_kind):
    """AttentionGate in train mode, in eval mode with gradients (the unfused path with training=False), through
    gate_pass (attention_gate_module(with_pass=True): the pass-through gradient rides the W_g dgrad as its addend) and
    with g not requiring a gradient.  Deterministic mode makes the node's kernels reproducible, so the test recomputes
    the node's dsig / dg1p / dx1p with the same calls and checks them against the §1 reference; the 1x1 GEMM parts are
    fp64 products of those bf16 tensors with the bf16-rounded weights."""
    from b200seg import kernels as K
    K.set_deterministic(True)
    try:
        _gate_node(c, fint, n, h, w, mode, dout_kind)
    finally:
        K.set_deterministic(False)


def _gate_node(c, fint, n, h, w, mode, dout_kind):
    from b200seg import kernels as K, ops_gate
    m = _gate_module(c, fint, seed=c + fint)
    training = mode != "eval"
    m.train(training)
    before = {k: v.detach().clone() for k, v in m.state_dict().items()}
    P = n * h * w
    gen = torch.Generator(device="cuda").manual_seed(P + c)
    g = torch.randn((n, h, w, c), device="cuda", generator=gen).bfloat16()
    x = torch.randn((n, h, w, c), device="cuda", generator=gen).bfloat16()
    noise = torch.randn((P, c), device="cuda", generator=gen)
    bn_g, bn_x, bn_1 = m.W_g[1], m.W_x[1], m.psi[1]
    with torch.no_grad():                              # the op's own forward outputs (bit-identical to the node's)
        res = ops_gate.attention_gate(
            g, x, m.W_g[0].weight, m.W_g[0].bias, m.W_x[0].weight, m.W_x[0].bias, bn_g.weight, bn_g.bias,
            before["W_g.1.running_mean"], before["W_g.1.running_var"], bn_x.weight, bn_x.bias,
            before["W_x.1.running_mean"], before["W_x.1.running_var"], m.psi[0].weight, m.psi[0].bias, bn_1.weight,
            bn_1.bias, before["psi.1.running_mean"], before["psi.1.running_var"], training, float(bn_1.eps))
    out_k, q_k, psi_k, g1p_k, x1p_k, coef_g, coef_x, coef_1 = res[:8]

    gi, xi = g.clone().requires_grad_(mode != "no_dg"), x.clone().requires_grad_(True)
    if mode == "pass":
        out, g_pass = m.gate_pass(gi, xi)
    else:
        out = m(g=gi, x=xi)
    assert torch.equal(_bits(out), _bits(out_k)), "the node's forward differs from the op's"
    if dout_kind == "random":
        dout = torch.randn((n, h, w, c), device="cuda", generator=gen).bfloat16()
    else:
        dout = correlated(out.detach().view(P, c), noise).view(n, h, w, c)
    if mode == "pass":
        dpass = torch.randn((n, h, w, c), device="cuda", generator=gen).bfloat16()
        torch.autograd.backward([out, g_pass], [dout, dpass])
    else:
        out.backward(dout)

    # the node's intermediate gradients, recomputed with the same calls
    dx_d, dsig, sums1 = K.gate_apply_bwd(dout, x, psi_k, q_k, coef_1)
    sums1 = sums1.clone()
    dg1p, dx1p, dgb, dbn1, dwpsi, dbpsi, dbias = K.gate_psi_bwd(
        dsig, sums1, q_k, g1p_k, x1p_k, coef_g, bn_g.weight, coef_x, bn_x.weight, coef_1, bn_1.weight,
        m.psi[0].weight, training=training)
    p = {"gamma_g": bn_g.weight, "beta_g": bn_g.bias, "gamma_x": bn_x.weight, "beta_x": bn_x.bias,
         "wpsi": m.psi[0].weight.view(-1), "bpsi": m.psi[0].bias, "gamma_1": bn_1.weight, "beta_1": bn_1.bias}
    p = {k: v.detach() for k, v in p.items()}
    for br, key in (("W_g.1", "g"), ("W_x.1", "x"), ("psi.1", "1")):
        p["rm_" + key], p["rv_" + key] = before[br + ".running_mean"], before[br + ".running_var"]
    t = ref_tensors(g1p_k.view(P, fint), x1p_k.view(P, fint), x.view(P, c), p, coef_g, coef_x, coef_1)
    nodes = gate_ref(t, training, q=q_k.view(P).double(), psi=psi_k.view(P).double())
    label = f"node C={c} F_int={fint} {n}x{h}x{w} {mode} dout={dout_kind}"
    b = {"dsig": dsig.view(P), "dg1p": dg1p.view(P, fint), "dx1p": dx1p.view(P, fint), "dgb": dgb, "dbn1": dbn1,
         "dwpsi": dwpsi, "dbpsi": dbpsi, "dbias": dbias}
    _check_psi_bwd(t, nodes, b, training, label, with_mutants=False)

    # every parameter gradient lands on its parameter, with the kernels' bits
    grads_of = dict(m.named_parameters())
    tail = {"W_g.1.weight": dgb[0], "W_g.1.bias": dgb[1], "W_x.1.weight": dgb[2], "W_x.1.bias": dgb[3],
            "psi.0.weight": dwpsi.view(1, fint, 1, 1), "psi.0.bias": dbpsi, "psi.1.weight": dbn1[0:1],
            "psi.1.bias": dbn1[1:2], "W_g.0.bias": dbias[0], "W_x.0.bias": dbias[1]}
    for k, v in tail.items():
        assert torch.equal(grads_of[k].grad.reshape(v.shape), v), (label, k)
    with torch.no_grad():
        dg1, dx1 = dg1p.view(P, fint).double(), dx1p.view(P, fint).double()
        wg = m.W_g[0].weight.view(fint, c).bfloat16().double()
        wx = m.W_x[0].weight.view(fint, c).bfloat16().double()
        rep = {}
        # 1x1 dgrads: fp32 accumulation over F_int, the direct dx / pass-through gradient added before the bf16 rounding
        if mode == "no_dg":
            assert gi.grad is None
        else:
            add = dpass.view(P, c).double() if mode == "pass" else torch.zeros((P, c), device="cuda",
                                                                                 dtype=torch.float64)
            ref = dg1 @ wg + add
            rep["dg"] = _worst(gi.grad.view(P, c).double() - ref,
                               ulp_bf16(ref) + TOL * (dg1.abs() @ wg.abs() + add.abs()))
        dxd = dx_d.view(P, c).double()
        ref = dxd + dx1 @ wx
        rep["dx"] = _worst(xi.grad.view(P, c).double() - ref, ulp_bf16(ref) + TOL * (dxd.abs() + dx1.abs() @ wx.abs()))
        # 1x1 wgrads: fp32 (1e-4 of the sum of |terms| over the pixels)
        for key, d1, inp in (("W_g.0.weight", dg1, g), ("W_x.0.weight", dx1, x)):
            a = inp.view(P, c).double()
            rep[key] = _worst(grads_of[key].grad.reshape(fint, c).double() - d1.T @ a, 1e-4 * (d1.abs().T @ a.abs()))
        # running statistics: momentum 0.1 with the batch statistics of the kernel's g1p / x1p / q (unbiased variance);
        # the GEMM epilogue may take its statistics before the bf16 rounding of g1p / x1p: half a bf16 ulp of slack
        msd = m.state_dict()
        for br, v in (("W_g.1", g1p_k.view(P, fint)), ("W_x.1", x1p_k.view(P, fint)), ("psi.1", q_k.view(P, 1))):
            nbt_old = int(before[br + ".num_batches_tracked"])
            if not training:
                for s in ("running_mean", "running_var"):
                    assert torch.equal(msd[f"{br}.{s}"], before[f"{br}.{s}"]), (label, br, s)
                assert int(msd[br + ".num_batches_tracked"]) == nbt_old
                continue
            vd = v.double()
            mean, var = vd.mean(0), vd.var(0, unbiased=True)
            rm = 0.9 * before[br + ".running_mean"].double() + 0.1 * mean
            rv = 0.9 * before[br + ".running_var"].double() + 0.1 * var
            rep[br + " running_mean"] = _worst(msd[br + ".running_mean"].double() - rm,
                                               1e-6 * rm.abs() + 0.1 * 2.0 ** -9 * vd.abs().mean(0))
            rep[br + " running_var"] = _worst(msd[br + ".running_var"].double() - rv,
                                              1e-6 * rv + 0.1 * 2.0 ** -7 * (vd * vd).mean(0) * P / (P - 1))
            assert int(msd[br + ".num_batches_tracked"]) == nbt_old + 1, (label, br)
    worst = max(rep, key=rep.get)
    print(f"{label}: worst {rep[worst]:.3f} tol ({worst})")
    assert rep[worst] <= 1, (label, rep)


# ----------------------------------------------------------------------------------------------------------
# §5 deterministic mode (GPU): every F_int at a pixel count past one full grid-stride sweep
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


def _flat(r):
    out = [r[k] for k in ("q", "qstats", "coef_1", "out", "psi")]
    for kind in ("random", "correlated"):
        out += [r[kind][k] for k in ("dx", "dsig", "sums1", "dg1p", "dx1p", "dgb", "dbn1", "dwpsi", "dbpsi", "dbias")]
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("fint", FINTS)
def test_gate_stages_deterministic(filled_workspace, fint):
    """every stage bit-identical over two runs and between a NaN- and a zero-filled workspace (no partial slot, also
    of a partial last channel slice, is left unwritten), and within the §2 tolerances of the reference"""
    c = 64
    npix = _npix("sweep", fint, c, torch.cuda.get_device_properties(0).multi_processor_count)
    cs = _gpu_case(fint, npix, c, True, seed=fint)
    runs = []
    for v in (float("nan"), 0.0, 0.0):
        filled_workspace(v)
        r = _run_kernels(cs)
        torch.cuda.synchronize()
        runs.append(r)
    for i, (a, b, z) in enumerate(zip(*[_flat(r) for r in runs])):
        assert torch.isfinite(b.float()).all(), (fint, i)
        assert torch.equal(_bits(b), _bits(z)), (fint, i, "two runs differ")
        assert torch.equal(_bits(a), _bits(b)), (fint, i, "differs when the workspace starts as NaN")
    _check_stages(cs, runs[1], _label(fint, npix, c, True, " deterministic"), with_mutants=False)
