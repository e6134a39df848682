"""GPU: the finish of the deterministic-reduction mode (C ABI b2_det_finish) and the partial rows it reads.

The finish must add every column's partial rows in row order, r = 0, 1, ..., rows-1, in fp64 — that order is what
makes two runs bit-identical and what every earlier build computed.  np.cumsum is a strictly sequential fp64 sum
(np.sum is pairwise), so its last row is the bitwise reference.

The partial rows are not cleared before a reducing kernel runs: each producer writes every slot of its rows itself.
A slot some block skipped would be read as whatever the workspace held.  The second group of tests fills the registered
workspace with NaN before every library call, runs the reducing ops and whole training steps, and compares bitwise with
the same calls after a zero fill: a skipped slot turns the NaN run's results into NaN."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _finish(partial, segs, row_stride):
    """segs: [(offset, count, dst tensor)] -> b2_det_finish on the current stream"""
    from b200seg import _lib
    n = len(segs)
    offs = (C.c_int32 * n)(*[s[0] for s in segs])
    cnts = (C.c_int32 * n)(*[s[1] for s in segs])
    dsts = (C.c_void_p * n)(*[s[2].data_ptr() for s in segs])
    f64 = (C.c_int32 * n)(*[1 if s[2].dtype == torch.float64 else 0 for s in segs])
    rc = _lib.load().b2_det_finish(C.c_void_p(partial.data_ptr()), partial.shape[0], row_stride, n, offs, cnts, dsts,
                                   f64, C.c_void_p(torch.cuda.current_stream().cuda_stream))
    _lib.check(rc, "b2_det_finish")


def _reference(part, off, count, dst0):
    s = np.cumsum(part[:, off:off + count], axis=0)[-1]          # sequential over the rows, fp64
    if dst0.dtype == np.float64:
        return dst0 + s
    return (dst0.astype(np.float64) + s).astype(np.float32)


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


@pytest.mark.parametrize("rows", [1, 7, 64, 296, 1184, 5000])
@pytest.mark.parametrize("count", [1, 2, 6, 33, 128, 2049])
def test_finish_is_the_sequential_row_sum(rows, count):
    rng = np.random.default_rng(rows * 7919 + count)
    row_stride = count + 3                                       # row_stride > count: the columns after are not read
    # magnitudes spread over many binades, so that any other summation order changes the last bits
    part = rng.standard_normal((rows, row_stride)) * np.exp2(rng.integers(-20, 20, (rows, row_stride)))
    for dtype in (np.float64, np.float32):
        dst0 = rng.standard_normal(count).astype(dtype)
        dev = torch.device("cuda")
        p = torch.from_numpy(part).to(dev)
        d = torch.from_numpy(dst0.copy()).to(dev)
        _finish(p, [(0, count, d)], row_stride)
        got = d.cpu().numpy()
        want = _reference(part, 0, count, dst0)
        assert np.array_equal(_bits(got), _bits(want)), f"rows {rows} count {count} {dtype.__name__}"


@pytest.mark.parametrize("rows", [5, 1184])
def test_finish_segments_in_one_call(rows):
    """the gate backward's layout: [0, 4F) -> sums (fp64), [4F, 5F) -> dwpsi, [5F] -> dbpsi (fp32); one launch"""
    rng = np.random.default_rng(rows)
    F = 64
    stride = 5 * F + 1
    part = rng.standard_normal((rows, stride)) * np.exp2(rng.integers(-16, 16, (rows, stride)))
    segs_np = [(0, 4 * F, rng.standard_normal(4 * F)), (4 * F, F, rng.standard_normal(F).astype(np.float32)),
               (5 * F, 1, rng.standard_normal(1).astype(np.float32))]
    p = torch.from_numpy(part).cuda()
    dsts = [torch.from_numpy(d.copy()).cuda() for _, _, d in segs_np]
    _finish(p, [(o, c, d) for (o, c, _), d in zip(segs_np, dsts)], stride)
    for (o, c, d0), d in zip(segs_np, dsts):
        assert np.array_equal(_bits(d.cpu().numpy()), _bits(_reference(part, o, c, d0))), f"segment at {o}"


# ----------------------------------------------------------------------------------------------------------
# no slot of the partial rows is left unwritten
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


def _both(fill, fn):
    """fn() under a NaN-filled and a zero-filled workspace -> the two results (tensors, cloned)"""
    out = []
    for v in (float("nan"), 0.0):
        fill(v)
        torch.manual_seed(0)
        r = fn()
        torch.cuda.synchronize()
        out.append([t.detach().clone() if t is not None else None for t in r])
    return out


def _assert_same(a, b, what):
    assert len(a) == len(b)
    for i, (x, y) in enumerate(zip(a, b)):
        if x is None:
            assert y is None
            continue
        assert torch.isfinite(y.float()).all(), f"{what}[{i}]: zero-fill run not finite"
        assert torch.equal(x.view(torch.uint8) if x.dtype == torch.bfloat16 else x,
                           y.view(torch.uint8) if y.dtype == torch.bfloat16 else y), \
            f"{what}[{i}]: differs when the workspace starts as NaN (a partial slot is never written)"


def _act(n, h, w, c, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn((n, h, w, c), generator=g, device="cuda").to(torch.bfloat16)


@pytest.mark.parametrize("c", [64, 128, 512])
@pytest.mark.parametrize("hw", [(16, 16), (24, 40), (64, 64)])
def test_batchnorm_reductions_write_every_slot(filled_workspace, c, hw):
    from b200seg import kernels as K
    h, w = hw
    z = _act(2, h, w, c, 1)
    dy = _act(2, h, w, c, 2)
    gamma = torch.rand(c, device="cuda") + 0.5
    beta = torch.randn(c, device="cuda")

    def run():
        stats = torch.zeros((2, c), dtype=torch.float64, device="cuda")
        K.channel_stats(z, stats)
        db = K.channel_sum(dy)
        rm, rv = torch.zeros(c, device="cuda"), torch.ones(c, device="cuda")
        nbt = torch.zeros((), dtype=torch.int64, device="cuda")
        coef = K.bn_finalize(stats, 2 * h * w, gamma, beta, 1e-5, 0.1, rm, rv, nbt)
        dz, dgamma, dbeta, dbias = K.bn_bwd(dy, z, coef, gamma, relu=True, training=True, want_dbias=True)
        return [stats, db, dz, dgamma, dbeta, dbias]

    a, b = _both(filled_workspace, run)
    _assert_same(a, b, f"BatchNorm C={c} {h}x{w}")


@pytest.mark.parametrize("model_name,n,h,w", [
    ("AttentionUNet", 2, 256, 256),      # conv_igemm plain / pair / double-M, conv_c64, folded UpConv, gate, head
    ("AttentionUNet", 1, 224, 224),      # clipped tiles
    ("AttentionUNet", 2, 48, 80),        # clipped extents (four 2x2 pools: sides divisible by 16), few blocks
    ("R2AttU_Net", 2, 64, 64),
])
def test_training_step_writes_every_slot(filled_workspace, model_name, n, h, w):
    """every reducing call of a training step — conv statistics, BatchNorm and gate backward, bias / head / stem
    gradients, the loss and the gradient norm of the fused clip + AdamW — under a NaN-filled workspace"""
    from b200seg import kernels as K, ops
    from b200seg.models import segmentation_models as M
    from b200seg.optim import FusedClipAdamW
    from b200seg.utils.synthetic import xray_batch
    kw = {"t": 2} if model_name.startswith("R2") else {}
    torch.manual_seed(0)
    model = getattr(M, model_name)(**kw).cuda().to(memory_format=torch.channels_last)
    model.train()
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    x, t = xray_batch(n, h, w, seed=3, device=torch.device("cuda"))

    def run():
        model.load_state_dict(state)
        model.zero_grad(set_to_none=True)
        opt = FusedClipAdamW(model.parameters(), lr=1e-3, weight_decay=5e-4, max_norm=1.0)
        K.step_begin()
        logits = model(x)
        loss, sums = ops.seg_loss(logits, t, 0.5, 0.5, 1.0)
        loss.backward()
        grads = [p.grad for p in model.parameters()]
        grads = [g.clone() if g is not None else None for g in grads]
        opt.step()
        return [logits, loss, sums, *grads, *[v for v in model.state_dict().values()]]

    a, b = _both(filled_workspace, run)
    _assert_same(a, b, f"{model_name} {n}x{h}x{w}")
