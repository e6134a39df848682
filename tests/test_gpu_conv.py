"""GPU parity: tcgen05 implicit-GEMM convolution (fprop / dgrad / wgrad) vs torch fp32 on identical bf16-rounded
operands.  Tolerance: bf16 output rounding only (rel-L2 <= 4e-3; north_star allows 1e-2 fwd / 2e-2 grads)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def rel(a, b):
    a = a.double()
    b = b.double()
    return float((a - b).norm() / (b.norm() + 1e-30))


def nhwc(x):  # NCHW fp32 -> NHWC bf16
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def nchw(x):  # NHWC bf16 -> NCHW fp32
    return x.float().permute(0, 3, 1, 2).contiguous()


SHAPES = [
    # n, h, w, cin, cout, k
    (2, 256, 256, 64, 64, 3),
    (2, 128, 128, 64, 128, 3),
    (2, 64, 64, 128, 256, 3),
    (3, 32, 32, 256, 512, 3),
    (2, 16, 16, 512, 1024, 3),
    (1, 8, 8, 128, 128, 3),
    (3, 8, 8, 64, 64, 3),
    (2, 64, 64, 256, 128, 1),
    (2, 256, 256, 64, 32, 1),
    (2, 32, 32, 32, 64, 1),
    (1, 512, 512, 64, 64, 3),
    (2, 128, 128, 128, 64, 3),      # Cout = 64 weight gradient: row-pair mode, two channel blocks
    (3, 64, 64, 64, 64, 3),         # ... at the narrowest width it applies to
]


@pytest.fixture(autouse=True)
def _fp32_reference():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False


@pytest.mark.parametrize("n,h,w,cin,cout,k", SHAPES)
def test_fprop(n, h, w, cin, cout, k):
    from b200seg import kernels as K
    g = torch.Generator(device="cuda").manual_seed(1)
    x = torch.randn(n, cin, h, w, device="cuda", generator=g)
    wt = torch.randn(cout, cin, k, k, device="cuda", generator=g) / (cin * k * k) ** 0.5
    b = torch.randn(cout, device="cuda", generator=g)
    xb = nhwc(x)
    wf, wd = K.pack_weights(wt)
    stats = torch.zeros(2, cout, dtype=torch.float64, device="cuda")
    y = K.conv_igemm(xb, wf, cout, k, bias=b, stats=stats)
    ref = F.conv2d(nchw(xb), wt.to(torch.bfloat16).float(), b, padding=k // 2)
    e = rel(nchw(y), ref)
    print(f"fprop {n}x{h}x{w} {cin}->{cout} k{k}: rel {e:.2e}")
    assert e < 4e-3
    yf = y.float().reshape(-1, cout)
    assert rel(stats[0], yf.double().sum(0)) < 1e-5
    assert rel(stats[1], (yf.double() ** 2).sum(0)) < 1e-5


@pytest.mark.parametrize("n,h,w,cin,cout,k", SHAPES[:8])
def test_dgrad(n, h, w, cin, cout, k):
    from b200seg import kernels as K
    g = torch.Generator(device="cuda").manual_seed(2)
    dy = torch.randn(n, cout, h, w, device="cuda", generator=g)
    wt = torch.randn(cout, cin, k, k, device="cuda", generator=g) / (cout * k * k) ** 0.5
    dyb = nhwc(dy)
    wf, wd = K.pack_weights(wt)
    dx = K.conv_igemm(dyb, wd, cin, k, dgrad=True)
    ref = F.conv_transpose2d(nchw(dyb), wt.to(torch.bfloat16).float(), padding=k // 2)
    e = rel(nchw(dx), ref)
    print(f"dgrad {n}x{h}x{w} {cin}<-{cout} k{k}: rel {e:.2e}")
    assert e < 4e-3


@pytest.mark.parametrize("n,h,w,cin,cout,k", SHAPES)
def test_wgrad(n, h, w, cin, cout, k):
    from b200seg import kernels as K
    g = torch.Generator(device="cuda").manual_seed(3)
    x = torch.randn(n, cin, h, w, device="cuda", generator=g)
    dy = torch.randn(n, cout, h, w, device="cuda", generator=g)
    xb, dyb = nhwc(x), nhwc(dy)
    dw = K.conv_wgrad(dyb, xb, k)                      # [cout, taps, cin]
    ref = torch.nn.grad.conv2d_weight(nchw(xb), (cout, cin, k, k), nchw(dyb), padding=k // 2)
    got = dw.reshape(cout, k, k, cin).permute(0, 3, 1, 2)
    e = rel(got, ref)
    print(f"wgrad {n}x{h}x{w} {cin}->{cout} k{k}: rel {e:.2e}")
    assert e < 1e-3
    # accumulate mode (shared weights)
    dw2 = K.conv_wgrad(dyb, xb, k, out=dw.clone(), accumulate=True)
    assert rel(dw2, 2 * dw) < 1e-6


def test_fprop_two_sources_addend_relu():
    from b200seg import kernels as K
    g = torch.Generator(device="cuda").manual_seed(4)
    n, h, w, c0, c1, cout = 2, 64, 64, 128, 128, 128
    xa = torch.randn(n, c0, h, w, device="cuda", generator=g)
    xb_ = torch.randn(n, c1, h, w, device="cuda", generator=g)
    add = torch.randn(n, cout, h, w, device="cuda", generator=g)
    wt = torch.randn(cout, c0 + c1, 3, 3, device="cuda", generator=g) / ((c0 + c1) * 9) ** 0.5
    # sources live as channel slices of wider buffers (ld > c)
    buf = torch.zeros(n, h, w, c0 + 64, dtype=torch.bfloat16, device="cuda")
    buf[..., :c0] = nhwc(xa)
    a0 = buf[..., :c0]
    a1 = nhwc(xb_)
    wf, wd = K.pack_weights(wt)
    y = K.conv_igemm(a0, wf, cout, 3, x1=a1, addend=nhwc(add), relu=True)
    ref = F.conv2d(torch.cat([nchw(a0), nchw(a1)], 1), wt.to(torch.bfloat16).float(), None, padding=1)
    ref = torch.relu(ref + nchw(nhwc(add)))
    e = rel(nchw(y), ref)
    print(f"two-source fprop: rel {e:.2e}")
    assert e < 4e-3
    # wgrad with two sources
    dy = nhwc(torch.randn(n, cout, h, w, device="cuda", generator=g))
    dw = K.conv_wgrad(dy, a0, 3, x1=a1)
    refw = torch.nn.grad.conv2d_weight(torch.cat([nchw(a0), nchw(a1)], 1), (cout, c0 + c1, 3, 3), nchw(dy), padding=1)
    e2 = rel(dw.reshape(cout, 3, 3, c0 + c1).permute(0, 3, 1, 2), refw)
    print(f"two-source wgrad: rel {e2:.2e}")
    assert e2 < 1e-3
    # dgrad into the second source only (row offset into the dgrad packing)
    dx1 = K.conv_igemm(dy, wd, c1, 3, row_offset=c0, dgrad=True)
    refd = F.conv_transpose2d(nchw(dy), wt.to(torch.bfloat16).float(), padding=1)[:, c0:]
    e3 = rel(nchw(dx1), refd)
    print(f"two-source dgrad(src1): rel {e3:.2e}")
    assert e3 < 4e-3


@pytest.mark.parametrize("cin", [128, 64, 192])
def test_wgrad_rowpair_2x2_phase_matches_plain(cin):
    """Cout = 64 weight gradient of a folded-UpConv phase (2x2 taps, dY read as a sub-lattice): the row-pair layout
    must reproduce the plain layout (B200SEG_WG_ROWPAIR=0) and the fp32 reference."""
    import os
    from b200seg import kernels as K
    g = torch.Generator(device="cuda").manual_seed(11)
    n, h, w, cout = 2, 64, 128, 64                 # coarse grid; dY lives on the 2x finer grid
    x = nhwc(torch.randn(n, cin, h, w, device="cuda", generator=g))
    dz = nhwc(torch.randn(n, cout, 2 * h, 2 * w, device="cuda", generator=g))
    for a, b in ((0, 0), (0, 1), (1, 0), (1, 1)):
        os.environ["B200SEG_WG_ROWPAIR"] = "0"
        K.reload_switches()              # the library caches its environment switches
        plain = K.conv_wgrad(dz, x, 2, dy_mul=2, dy_off=(a, b), pad=(1 - a, 1 - b))
        os.environ["B200SEG_WG_ROWPAIR"] = "1"
        K.reload_switches()
        try:
            pair = K.conv_wgrad(dz, x, 2, dy_mul=2, dy_off=(a, b), pad=(1 - a, 1 - b))
        finally:
            del os.environ["B200SEG_WG_ROWPAIR"]
            K.reload_switches()
        # fp32 reference: dW[co, r, s, ci] = sum_p dY[p, co] * X[p + (r - pad_h, s - pad_w), ci]
        dys = nchw(dz)[:, :, a::2, b::2]
        xp = F.pad(nchw(x), (1 - b, b, 1 - a, a))       # (left, right, top, bottom)
        ref = torch.nn.grad.conv2d_weight(xp, (cout, cin, 2, 2), dys)
        got = pair.reshape(cout, 2, 2, cin).permute(0, 3, 1, 2)
        assert rel(got, ref) < 1e-3, (a, b, rel(got, ref))
        assert rel(pair, plain) < 1e-5


@pytest.mark.parametrize("n,h,w,cin,cout", [
    (2, 64, 128, 128, 64),       # fold 2 (Cout = 64: the column phases are the two halves of the M operand)
    (2, 64, 64, 256, 128),       # fold 1, one row per chunk
    (3, 32, 32, 512, 256),       # two rows per chunk, two Cout tiles
    (2, 16, 16, 1024, 512),      # four rows per chunk
    (2, 16, 16, 64, 128),        # a single X channel block
    (1, 20, 28, 128, 128),       # clipped chunks (general extents)
    (1, 12, 20, 192, 64),        # ... with an odd number of X blocks, Cout = 64
])
def test_wgrad_folded_upconv_merged_matches_phases(n, h, w, cin, cout):
    """b2_wgrad_args::fold — the four phase weight gradients of a folded UpConv (AttentionUNet.py:15-27) from ONE
    launch must equal the four dy_off launches and the fp32 reference."""
    from b200seg import kernels as K
    g = torch.Generator(device="cuda").manual_seed(31)
    x = nhwc(torch.randn(n, cin, h, w, device="cuda", generator=g))
    dz = nhwc(torch.randn(n, cout, 2 * h, 2 * w, device="cuda", generator=g))
    merged = K.conv_wgrad(dz, x, 2, dy_mul=2, fold=True)
    assert merged is not None and merged.shape == (cout, 16, cin)
    merged = merged.view(4, cout, 4, cin)
    for ph, (a, b) in enumerate(((0, 0), (0, 1), (1, 0), (1, 1))):
        plain = K.conv_wgrad(dz, x, 2, dy_mul=2, dy_off=(a, b), pad=(1 - a, 1 - b))
        dys = nchw(dz)[:, :, a::2, b::2]
        xp = F.pad(nchw(x), (1 - b, b, 1 - a, a))
        ref = torch.nn.grad.conv2d_weight(xp, (cout, cin, 2, 2), dys)
        got = merged[ph].reshape(cout, 2, 2, cin).permute(0, 3, 1, 2)
        assert rel(got, ref) < 1e-3, (a, b, rel(got, ref))
        assert rel(merged[ph], plain) < 1e-5, (a, b, rel(merged[ph], plain))


def test_wgrad_folded_upconv_merged_rejects_narrow_images():
    """coarse images narrower than 16 pixels are not taken in merged mode: the wrapper reports it (None) and the
    caller launches the phases"""
    from b200seg import kernels as K
    x = torch.zeros(1, 8, 8, 64, device="cuda", dtype=torch.bfloat16)
    dz = torch.zeros(1, 16, 16, 64, device="cuda", dtype=torch.bfloat16)
    assert K.conv_wgrad(dz, x, 2, dy_mul=2, fold=True) is None


@pytest.mark.parametrize("n,h,w,cin", [(2, 256, 256, 64), (2, 128, 128, 128), (1, 6, 128, 64)])
def test_fprop_dgrad_cout64_matches_fp32(n, h, w, cin):
    """Cout = 64 3x3 fprop with bias, ReLU and the BatchNorm-statistics epilogue, and a dgrad into 64 channels, against
    the fp32 reference; the statistics against fp64 sums of the stored output."""
    from b200seg import kernels as K
    g = torch.Generator(device="cuda").manual_seed(21)
    cout = 64
    x = nhwc(torch.randn(n, cin, h, w, device="cuda", generator=g))
    wt = torch.randn(cout, cin, 3, 3, device="cuda", generator=g) / (cin * 9) ** 0.5
    b = torch.randn(cout, device="cuda", generator=g)
    wf, wd = K.pack_weights(wt)
    wt2 = torch.randn(cin, cout, 3, 3, device="cuda", generator=g) / (cout * 9) ** 0.5       # a conv whose dgrad has 64 ch
    _, wd2 = K.pack_weights(wt2)
    dy2 = nhwc(torch.randn(n, cin, h, w, device="cuda", generator=g))
    st = torch.zeros(2, cout, dtype=torch.float64, device="cuda")
    y = K.conv_igemm(x, wf, cout, 3, bias=b, stats=st, relu=True)
    dx = K.conv_igemm(dy2, wd2, cout, 3, dgrad=True)
    ref = torch.relu(F.conv2d(nchw(x), wt.to(torch.bfloat16).float(), b, padding=1))
    assert rel(nchw(y), ref) < 4e-3
    refd = F.conv_transpose2d(nchw(dy2), wt2.to(torch.bfloat16).float(), padding=1)
    assert rel(nchw(dx), refd) < 4e-3
    yf = y.float().reshape(-1, cout)
    assert rel(st[0], yf.double().sum(0)) < 1e-5 and rel(st[1], (yf.double() ** 2).sum(0)) < 1e-5
