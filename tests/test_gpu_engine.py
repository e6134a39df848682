"""GPU: the fast step is a package component (b200seg.engine) — train() replays a CUDA graph, the graphed step computes
what the eager step computes, cached packed weights follow every kind of parameter update, and the pinned prefetcher
delivers the loader's batches unchanged."""
import pytest
import torch
from torch.utils.data import DataLoader, TensorDataset

pytestmark = pytest.mark.gpu


def test_train_replays_a_cuda_graph(tmp_path):
    from b200seg.utils.helpers import get_seg_model, train
    from b200seg.utils.synthetic import xray_batch
    torch.manual_seed(0)
    x, t = xray_batch(14, 64, 64, seed=31)
    train_dl = DataLoader(TensorDataset(x[:12], t[:12]), batch_size=2, shuffle=False)       # 6 steps per epoch
    val_dl = DataLoader(TensorDataset(x[12:], t[12:]), batch_size=2)
    model = get_seg_model("attentionunet")
    logs = []
    train(model, train_dl, val_dl, torch.device("cuda"), epochs=2, lr=1e-3, name="AttentionUNet",
          save_dir=str(tmp_path), seg=True, log=logs.append)
    st = train.last_stepper
    assert st.capture_error is None, st.capture_error
    assert st.eager_steps == 3 and st.replays == 9, (st.eager_steps, st.replays)
    losses = [float(l.split("TrainLoss ")[1].split(" ")[0]) for l in logs if "TrainLoss" in l]
    assert len(losses) == 2 and losses[1] < losses[0], losses


@pytest.mark.parametrize("name,kw", [("AttentionUNet", {}), ("R2U_Net", {"t": 2})])
def test_graphed_step_matches_eager_step(name, kw):
    """deterministic mode: the parameters after 6 steps through GraphedTrainStep (3 eager + capture + replays) are
    bit-identical to 6 eager steps — graph capture, the static buffers, the cached packed weights and the multi-tensor
    re-pack change nothing"""
    from b200seg import kernels as K
    from b200seg.engine import GraphedTrainStep
    from b200seg.models import segmentation_models as M
    from b200seg.optim import FusedClipAdamW
    from b200seg.utils.synthetic import xray_batch
    batches = [xray_batch(2, 64, 64, seed=40 + i, device="cuda") for i in range(6)]

    def run(graph):
        torch.manual_seed(0)
        model = getattr(M, name)(**kw).cuda().to(memory_format=torch.channels_last).train()
        opt = FusedClipAdamW(model.parameters(), lr=1e-3, weight_decay=5e-4, max_norm=1.0)
        st = GraphedTrainStep(model, opt, graph=graph, warmup=3, wgrad_overlap=True)
        losses = [float(st(x, t)) for x, t in batches]
        torch.cuda.synchronize()
        assert st.replays == (3 if graph else 0)
        return losses, {k: v.detach().clone() for k, v in model.state_dict().items()}

    K.set_deterministic(True)
    try:
        l_eager, sd_eager = run(False)
        l_graph, sd_graph = run(True)
    finally:
        K.set_deterministic(False)
    assert l_eager == l_graph, (l_eager, l_graph)
    bad = [k for k in sd_eager if not torch.equal(sd_eager[k], sd_graph[k])]
    assert not bad, bad[:5]


def test_packed_weights_follow_parameter_updates():
    """the cached bf16 copies must track: the fused optimizer (raw-pointer writes + multi-tensor re-pack), a torch
    optimizer / in-place update (version bump), load_state_dict, and a re-created parameter at a reused address"""
    from b200seg import kernels as K
    from b200seg.optim import FusedClipAdamW
    g = torch.Generator(device="cuda").manual_seed(1)

    def fresh(w, kind="plain"):
        if kind == "upfold":
            return K.pack_weights_upfold(w, want_dgrad=True)
        return K.pack_weights(w, want_dgrad=True)

    for kind, shape in (("plain", (64, 32, 3, 3)), ("plain", (40, 24, 1, 1)), ("upfold", (64, 128, 3, 3))):
        w = torch.nn.Parameter(torch.randn(shape, device="cuda", generator=g).contiguous(memory_format=torch.channels_last))
        wf, wd = K.packed(w, kind, want_dgrad=True)
        rf, rd = fresh(w, kind)
        assert torch.equal(wf, rf) and torch.equal(wd, rd)
        assert K.packed(w, kind, want_dgrad=True)[0] is wf                  # cache hit: same buffers
        opt = FusedClipAdamW([w], lr=1e-1, weight_decay=0.0, max_norm=0.0)
        w.grad = torch.randn(shape, device="cuda", generator=g).contiguous(memory_format=torch.channels_last)
        before = w.detach().clone()
        opt.step()                                                          # raw-pointer update + multi-tensor re-pack
        assert not torch.equal(before, w.detach())
        wf2, wd2 = K.packed(w, kind, want_dgrad=True)
        assert wf2 is wf                                                    # refreshed in place by the optimizer
        rf, rd = fresh(w, kind)
        assert torch.equal(wf2, rf) and torch.equal(wd2, rd), kind
        with torch.no_grad():
            w.mul_(0.5)                                                     # torch writer: version bump
        wf3, wd3 = K.packed(w, kind, want_dgrad=True)
        rf, rd = fresh(w, kind)
        assert torch.equal(wf3, rf) and torch.equal(wd3, rd)
    # stem matrix
    w = torch.nn.Parameter(torch.randn(64, 3, 3, 3, device="cuda", generator=g))
    wf, _ = K.packed(w, "stem")
    ref, _ = K.pack_weights(K.stem_weight_matrix(w), want_dgrad=False)
    assert torch.equal(wf, ref)
    opt = FusedClipAdamW([w], lr=1e-1, weight_decay=0.0, max_norm=0.0)
    w.grad = torch.randn_like(w)
    opt.step()
    ref, _ = K.pack_weights(K.stem_weight_matrix(w), want_dgrad=False)
    assert torch.equal(K.packed(w, "stem")[0], ref)
    # a new parameter at a recycled address never sees the old entry
    ptr = w.data_ptr()
    del w, opt, wf
    torch.cuda.empty_cache()
    for _ in range(4):
        w2 = torch.nn.Parameter(torch.randn(64, 3, 3, 3, device="cuda", generator=g))
        ref, _ = K.pack_weights(K.stem_weight_matrix(w2), want_dgrad=False)
        assert torch.equal(K.packed(w2, "stem")[0], ref), w2.data_ptr() == ptr


def test_inference_fold_cache_tracks_updates():
    from b200seg.models.segmentation_models import AttentionUNet
    from b200seg.optim import FusedClipAdamW
    from b200seg import ops, ops_infer
    from b200seg.utils.synthetic import xray_batch
    torch.manual_seed(0)
    m = AttentionUNet().cuda()
    x, t = xray_batch(2, 64, 64, seed=3, device="cuda")
    m.eval()
    with torch.no_grad():
        y0 = m(x)
        n_fold = len(ops_infer._FOLDED)
        y0b = m(x)
        assert torch.equal(y0, y0b) and len(ops_infer._FOLDED) == n_fold
    m.train()
    opt = FusedClipAdamW(m.parameters(), lr=1e-2, weight_decay=5e-4, max_norm=1.0)
    loss, _ = ops.seg_loss(m(x), t, 1.0, 0.0, 1.0)
    loss.backward()
    opt.step()
    m.eval()
    with torch.no_grad():
        y1 = m(x)
        import os
        os.environ["B200SEG_FOLD_BN"] = "0"
        try:
            y1_plain = m(x)
        finally:
            os.environ["B200SEG_FOLD_BN"] = "1"
    assert not torch.equal(y0, y1)
    assert float((y1 - y1_plain).norm() / y1_plain.norm()) < 1e-2


def test_pinned_prefetcher_delivers_batches_in_order():
    from b200seg.engine import PinnedPrefetcher
    g = torch.Generator().manual_seed(0)
    data = torch.randn(10, 3, 16, 16, generator=g)
    tgt = (torch.rand(10, 1, 16, 16, generator=g) > 0.5).float()
    for pin in (False, True):
        dl = DataLoader(TensorDataset(data, tgt), batch_size=3, shuffle=False, pin_memory=pin)    # ragged last batch
        got_x, got_t = [], []
        for xb, tb in PinnedPrefetcher(dl, "cuda"):
            assert xb.is_cuda
            got_x.append(xb.clone())
            got_t.append(tb.clone())
        assert torch.equal(torch.cat(got_x).cpu(), data) and torch.equal(torch.cat(got_t).cpu(), tgt)


def test_deferred_running_updates_match_immediate_ones():
    """kernels.deferred_running_updates (one b2_bn_update_running_multi launch per round instead of one launch per
    BatchNorm call): running_mean / running_var / num_batches_tracked after a train-mode forward must be BIT-identical to
    the immediate updates — including a Recurrent_block's shared BatchNorm, whose t + 1 sequential updates go to t + 1
    rounds (R2U_Net.py:15-20)."""
    from b200seg import kernels as K
    from b200seg.models.segmentation_models import R2AttU_Net
    from b200seg.utils.synthetic import xray_batch
    torch.manual_seed(0)
    model = R2AttU_Net(t=2).cuda().train()
    x, _ = xray_batch(2, 64, 64, seed=2, device=torch.device("cuda"))
    state = {k: v.clone() for k, v in model.state_dict().items()}
    K.set_deterministic(True)
    try:
        with torch.no_grad():
            model(x)
        torch.cuda.synchronize()
        ref = {k: v.clone() for k, v in model.state_dict().items() if "running" in k or "num_batches" in k}
        model.load_state_dict(state)
        with torch.no_grad(), K.deferred_running_updates():
            model(x)
        torch.cuda.synchronize()
    finally:
        K.set_deterministic(False)
    got = model.state_dict()
    assert any(int(v) == 3 for k, v in ref.items() if "num_batches" in k)        # the shared BatchNorms: t + 1 = 3
    bad = [k for k in ref if not torch.equal(ref[k], got[k])]
    assert not bad, bad[:5]


def test_bench_dumps_the_state_the_timed_steps_left(tmp_path):
    """bench.py --steps K --dump-outputs DIR: K steps are timed, and DIR holds the loss and every state_dict entry the
    last of them left; each BatchNorm has counted 3 eager warm-up steps + the capture step + the K timed steps, and a
    second run with the same arguments dumps the same bits"""
    import json
    import subprocess
    import sys
    from pathlib import Path

    import numpy as np
    root = Path(__file__).resolve().parent.parent

    def run(out):
        cmd = [sys.executable, str(root / "bench.py"), "--steps", "5", "--warmup", "1", "--batch", "2", "--side", "64",
               "--no-cpu-baseline", "--dump-outputs", str(out)]
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-3000:]
        lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
        assert len(lines) == 1
        d = json.loads(lines[0])
        assert d["steps"] == 5 and d["config"]["cuda_graph"] and d["config"]["deterministic_reductions"]
        return {p.stem: np.load(p) for p in out.glob("*.npy")}

    arrays, again = run(tmp_path / "a"), run(tmp_path / "b")
    gold = np.load(root / "tests" / "golden" / "AttentionUNet.npz")
    assert set(arrays) == {"loss"} | {str(k) for k in gold["keys"]}
    assert all(a.dtype in (np.float32, np.float64) and np.isfinite(a).all() for a in arrays.values())
    assert 0.0 < float(arrays["loss"]) < 10.0
    counts = [float(a) for k, a in arrays.items() if k.endswith("num_batches_tracked")]
    assert counts and set(counts) == {3 + 1 + 5}
    assert set(again) == set(arrays) and all(np.array_equal(arrays[k], again[k]) for k in arrays)
