"""GPU: multi-class segmentation — the fused softmax cross-entropy + soft Dice loss and its gradient against fp64 torch,
invalid / ignored labels, exact per-class counts and argmax (ties included), deterministic mode, label-map augmentation,
all four models trained graphed and eager on 3 classes, train() / test_segmentation_model / predict_labels end to end."""
import json
import os

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def ref_loss(z, y, weight, ignore_index, w_ce, w_dice, smooth):
    """fp64: w_ce * F.cross_entropy + w_dice * (1 - mean over classes 1..K-1 of the soft Dice), ignored pixels out"""
    k = z.shape[1]
    yl = y.reshape(z.shape[0], *z.shape[2:]).long()
    ce = F.cross_entropy(z, yl, weight=None if weight is None else weight.double(), ignore_index=ignore_index)
    valid = (yl != ignore_index).unsqueeze(1).double()
    p = torch.softmax(z, 1) * valid
    t = F.one_hot(torch.where(yl == ignore_index, 0, yl), k).permute(0, 3, 1, 2).double() * valid
    dims = (0, 2, 3)
    dice = (2 * (p * t).sum(dims) + smooth) / (p.sum(dims) + t.sum(dims) + smooth)
    return w_ce * ce + w_dice * (1 - dice[1:].mean())


def make_case(n, k, h, w, label_dtype, ignore_index, seed, frac_ignored=0.1):
    g = torch.Generator(device="cuda").manual_seed(seed)
    z = torch.randn(n, k, h, w, device="cuda", generator=g) * 3
    y = torch.randint(0, k, (n, h, w), device="cuda", generator=g)
    y[torch.rand(n, h, w, device="cuda", generator=g) < frac_ignored] = ignore_index
    return z, y.to(label_dtype)


@pytest.mark.parametrize("shape", [(2, 37, 29), (4, 256, 256)], ids=["ragged", "4x256x256"])
@pytest.mark.parametrize("weighted", [False, True], ids=["unweighted", "weighted"])
@pytest.mark.parametrize("label_dtype", [torch.uint8, torch.int64], ids=["u8", "i64"])
@pytest.mark.parametrize("k", [2, 3, 5, 8])
def test_ce_dice_loss_and_gradient_match_fp64(k, label_dtype, weighted, shape):
    from b200seg import ops
    n, h, w = shape
    ii = 255 if label_dtype == torch.uint8 else -100
    z, y = make_case(n, k, h, w, label_dtype, ii, seed=k * 10 + h)
    weight = (0.5 + torch.rand(k, device="cuda", generator=torch.Generator(device="cuda").manual_seed(k))) \
        if weighted else None
    for w_ce, w_dice in ((0.5, 0.5), (1.0, 0.0)):
        zr = z.requires_grad_(True)
        loss, sums = ops.seg_loss_ce(zr, y, weight, ii, w_ce, w_dice, 1.0)
        loss.backward()
        dz = zr.grad.clone()
        zr.grad = None
        zd = z.detach().double().requires_grad_(True)
        ref = ref_loss(zd, y, weight, ii, w_ce, w_dice, 1.0)
        ref.backward()
        assert abs(float(loss) - float(ref)) <= 1e-6 * abs(float(ref)), (w_ce, w_dice, float(loss), float(ref))
        err = float((dz.double() - zd.grad).abs().max())
        assert err <= 2e-6 * float(zd.grad.abs().max()), (w_ce, w_dice, err, float(zd.grad.abs().max()))
        z = z.detach()


def test_ce_sums_layout_and_hard_iou_counts():
    from b200seg import kernels as K
    k = 4
    z, y = make_case(2, k, 40, 36, torch.int64, -100, seed=5)
    _, sums = K.ce_loss_fwd(z, y, None, -100)
    f = K.ce_sums_fields(sums, k)
    valid = y != -100
    pred = z.argmax(1)
    for c in range(k):
        t, p = (y == c) & valid, (pred == c) & valid
        assert float(f["t"][c]) == float(t.sum())
        assert float(f["inter"][c]) == float((t & p).sum())
        assert float(f["union"][c]) == float((t | p).sum())
    assert float(f["invalid"]) == 0.0
    assert abs(float(f["p"].sum()) - float(valid.sum())) < 1e-3


def test_invalid_label_gives_nan_and_is_counted():
    """torch asserts on the device for a label >= K; the fused loss reports NaN and counts the label, no fault"""
    from b200seg import kernels as K
    z, y = make_case(2, 3, 32, 32, torch.uint8, 255, seed=1, frac_ignored=0.0)
    y[1, 5, 7] = 3
    loss, sums = K.ce_loss_fwd(z, y, None, 255, 0.5, 0.5, 1.0)
    torch.cuda.synchronize()
    assert torch.isnan(loss).item()
    assert float(K.ce_sums_fields(sums, 3)["invalid"]) == 1.0


def test_all_pixels_ignored_gives_nan():
    from b200seg import kernels as K
    z, _ = make_case(2, 3, 32, 32, torch.int64, -100, seed=2)
    y = torch.full((2, 32, 32), -100, dtype=torch.int64, device="cuda")
    loss, _ = K.ce_loss_fwd(z, y, None, -100, 1.0, 0.0, 1.0)
    ref = F.cross_entropy(z.double(), y, ignore_index=-100)
    assert torch.isnan(loss).item() and torch.isnan(ref).item()


@pytest.mark.parametrize("shape", [(3, 37, 29), (2, 64, 64)], ids=["ragged", "aligned"])
@pytest.mark.parametrize("label_dtype", [torch.uint8, torch.int64], ids=["u8", "i64"])
@pytest.mark.parametrize("k", [2, 3, 8])
def test_counts_and_argmax_are_exact_with_ties(k, label_dtype, shape):
    """integer-valued logits in [-2, 2]: most pixels have tied maxima, and argmax must take the first one"""
    from b200seg import kernels as K
    n, h, w = shape
    ii = 255 if label_dtype == torch.uint8 else -100
    g = torch.Generator(device="cuda").manual_seed(k + h)
    z = torch.randint(-2, 3, (n, k, h, w), device="cuda", generator=g).float()
    y = torch.randint(0, k, (n, h, w), device="cuda", generator=g)
    y[torch.rand(n, h, w, device="cuda", generator=g) < 0.1] = ii
    y[0, 0, :3] = k + 1 if label_dtype == torch.uint8 else -7               # invalid labels: excluded
    y = y.to(label_dtype)
    pred = torch.argmax(z, 1)
    assert torch.equal(K.logits_to_labels(z), pred.to(torch.uint8))
    counts = K.seg_counts_mc(z, y, ii)
    yl = y.long()
    valid = (yl >= 0) & (yl < k) & (yl != ii)
    ref = torch.empty((n, k, 3), dtype=torch.int64, device="cuda")
    for c in range(k):
        t, p = (yl == c) & valid, (pred == c) & valid
        ref[:, c, 0] = (t & p).flatten(1).sum(1)
        ref[:, c, 1] = p.flatten(1).sum(1)
        ref[:, c, 2] = t.flatten(1).sum(1)
    assert torch.equal(counts, ref)


def test_deterministic_mode_is_bit_reproducible():
    from b200seg import kernels as K
    z, y = make_case(8, 3, 256, 256, torch.uint8, 255, seed=9)
    wt = torch.tensor([0.3, 1.0, 2.0], device="cuda")

    def run():
        loss, sums = K.ce_loss_fwd(z, y, wt, 255, 0.5, 0.5, 1.0)
        dz = K.ce_loss_bwd(z, y, wt, 255, sums, None, 0.5, 0.5, 1.0)
        return loss.clone(), sums.clone(), dz

    K.set_deterministic(True)
    try:
        a, b = run(), run()
    finally:
        K.set_deterministic(False)
    c = run()
    for u, v in zip(a, b):
        assert torch.equal(u, v)
    assert float(((a[1] - c[1]).abs() / c[1].abs().clamp_min(1e-300)).max()) <= 1e-12
    # the fp32 loss and dz come from sums that agree to ~1e-16: at most a few ulps apart, element by element
    for u, v in ((a[0], c[0]), (a[2], c[2])):
        big = torch.maximum(u.abs(), v.abs())
        ulp = torch.nextafter(big, torch.full_like(big, float("inf"))) - big
        assert bool(((u - v).abs() <= 4 * ulp).all()), float((u - v).abs().max())


def test_class_weight_on_another_device_is_rejected_before_any_launch():
    """nn.CrossEntropyLoss(weight=torch.tensor([...])) habit: a host weight must raise, not reach the kernel"""
    from b200seg import kernels as K
    from b200seg import ops
    z, y = make_case(2, 3, 16, 16, torch.int64, -100, seed=4)
    w_host = torch.tensor([0.5, 1.0, 2.0])
    with pytest.raises(ValueError):
        ops.seg_loss_ce(z, y, w_host, -100, 1.0, 0.0, 1.0)
    with pytest.raises(ValueError):
        K.ce_loss_bwd(z, y, w_host, -100, torch.zeros(K.ce_nsums(3), dtype=torch.float64, device="cuda"), None)
    with pytest.raises(ValueError):
        K.ce_loss_fwd(z, y, torch.ones(4, device="cuda"))


def test_augment_labels_matches_the_nearest_mask_path():
    """b2_seg_augment_labels: the label map equals the nearest-resize / nearest-warp / flip mask that b2_seg_augment
    writes (pinned against cv2 by tests/golden/augment.npz) times 255, and the image output is bit-equal"""
    from b200seg.data import GpuSegAugment
    g = torch.Generator().manual_seed(3)
    n, hs, ws = 6, 300, 280
    img = torch.randint(0, 256, (n, hs, ws, 3), dtype=torch.uint8, generator=g)
    masks = (torch.randint(0, 3, (n, hs, ws), dtype=torch.uint8, generator=g),
             torch.randint(0, 256, (n, hs, ws), dtype=torch.uint8, generator=g))
    for mask, border in ((masks[0], "constant"), (masks[1], "constant"), (masks[0], "reflect101")):
        aug_f = GpuSegAugment(size=256, train=True, seed=11, border=border)
        aug_l = GpuSegAugment(size=256, train=True, seed=11, labels=True, border=border)
        samples = aug_f.sample(n)
        samples[0] = {"flip": True}                                   # no warp, flip only
        samples[1] = {"angle": 10.0, "scale": 1.03, "dx": 0.04, "dy": -0.03, "flip": True}
        x_f, t_f = aug_f(img, mask, samples=samples)
        x_l, y_l = aug_l(img, mask, samples=samples)
        assert y_l.dtype == torch.uint8 and y_l.shape == (n, 256, 256)
        assert torch.equal(x_f, x_l)
        assert torch.equal(torch.round(t_f[:, 0] * 255).to(torch.uint8), y_l)
    with pytest.raises(ValueError):
        GpuSegAugment(labels=True, mask_nearest_resize=False)


MODELS = [("AttentionUNet", {"out_channel": 3}), ("R2U_Net", {"out_channels": 3, "t": 2}),
          ("R2AttU_Net", {"out_channels": 3, "t": 2}), ("ResNetUnet", {"n_classes": 3, "freeze": True}),
          ("ResNetUnet", {"n_classes": 3, "freeze": False})]
IDS = ["AttentionUNet", "R2U_Net", "R2AttU_Net", "ResNetUnet_frozen", "ResNetUnet_unfrozen"]


def _model(name, kw):
    from b200seg.models import segmentation_models as M
    torch.manual_seed(0)
    return getattr(M, name)(**kw).cuda().to(memory_format=torch.channels_last).train()


@pytest.mark.parametrize("name,kw", MODELS, ids=IDS)
def test_graphed_ce_dice_step_matches_eager_step(name, kw):
    from b200seg import kernels as K
    from b200seg.engine import GraphedTrainStep
    from b200seg.optim import FusedClipAdamW
    from b200seg.utils.synthetic import xray_batch_multiclass
    batches = [xray_batch_multiclass(4, 128, 128, seed=60 + i, device="cuda") for i in range(6)]

    def run(graph):
        model = _model(name, kw)
        opt = FusedClipAdamW([p for p in model.parameters() if p.requires_grad], lr=1e-3, weight_decay=5e-4,
                             max_norm=1.0)
        st = GraphedTrainStep(model, opt, graph=graph, warmup=3, wgrad_overlap=True, loss="ce",
                              loss_weights=(0.5, 0.5, 1.0))
        losses = [float(st(x, y)) for x, y in batches]
        torch.cuda.synchronize()
        assert st.capture_error is None, st.capture_error
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


# 30 AdamW steps (lr 1e-3) on one fixed 4 x 128^2 batch must bring the CE+Dice loss below this fraction of the first
# step's loss.  The first B200 run (NVIDIA B200, 1000 W power limit) measured last / first = 0.294 AttentionUNet,
# 0.378 R2U_Net(t=2), 0.187 R2AttU_Net(t=2), 0.407 ResNetUnet(freeze=True), 0.408 ResNetUnet(freeze=False); the limit
# is the worst of these times 1.5, rounded.  B200SEG_MC_LOSS_LOG=<file> appends the measured values.
_LOSS_DROP_LIMIT = 0.6


@pytest.mark.parametrize("name,kw", MODELS, ids=IDS)
def test_eager_loss_matches_fp64_and_training_lowers_it(name, kw):
    from b200seg import ops
    from b200seg.optim import FusedClipAdamW
    from b200seg.utils.synthetic import xray_batch_multiclass
    x, y = xray_batch_multiclass(4, 128, 128, seed=77, device="cuda")
    model = _model(name, kw)
    opt = FusedClipAdamW([p for p in model.parameters() if p.requires_grad], lr=1e-3, weight_decay=5e-4,
                             max_norm=1.0)
    losses = []
    for step in range(31):
        opt.zero_grad(set_to_none=True)
        logits = model(x)
        loss, _ = ops.seg_loss_ce(logits, y, None, -100, 0.5, 0.5, 1.0)
        if step == 0:
            ref = ref_loss(logits.detach().double(), y, None, -100, 0.5, 0.5, 1.0)
            assert logits.shape == (4, 3, 128, 128)
            assert abs(float(loss) - float(ref)) <= 1e-6 * abs(float(ref)), (float(loss), float(ref))
        losses.append(float(loss))
        if step < 30:
            loss.backward()
            opt.step()
    ratio = losses[-1] / losses[0]
    out = os.environ.get("B200SEG_MC_LOSS_LOG")
    if out:
        with open(out, "a") as f:
            f.write(json.dumps({"model": name, "kw": kw, "first": losses[0], "last": losses[-1], "ratio": ratio}) + "\n")
    assert ratio < _LOSS_DROP_LIMIT, (losses[0], losses[-1], ratio)


def test_train_ce_replays_a_graph_and_saves(tmp_path):
    from b200seg.utils.helpers import train
    from b200seg.utils.synthetic import xray_batch_multiclass
    from b200seg.models.segmentation_models import AttentionUNet
    x, y = xray_batch_multiclass(6, 64, 64, seed=5)
    train_dl = [(x[0:2], y[0:2]), (x[2:4], y[2:4])]
    val_dl = [(x[4:6], y[4:6])]
    torch.manual_seed(0)
    model = AttentionUNet(out_channel=3)
    logs = []
    best = train(model, train_dl, val_dl, torch.device("cuda"), epochs=3, lr=1e-3, name="mc", save_dir=str(tmp_path),
                 seg=True, log=logs.append, loss="ce+dice", class_weight=[0.5, 1.0, 2.0])
    st = train.last_stepper
    assert st.capture_error is None, st.capture_error
    assert st.replays > 0, (st.eager_steps, st.replays)
    assert (tmp_path / "mc_best_loss.pt").exists()
    assert best == best and best < float("inf")
    assert any("IoU" in line for line in logs)


class _Echo(torch.nn.Module):
    """returns its input: test_segmentation_model then scores exactly the logits the loader hands it"""

    def __init__(self):
        super().__init__()
        self.p = torch.nn.Parameter(torch.zeros(1))

    def forward(self, x):
        return x


def test_segmentation_model_per_class_metrics_match_fp64():
    from b200seg.utils.tester import METRIC_KEYS, test_segmentation_model
    k, eps = 3, 1e-7
    g = torch.Generator(device="cuda").manual_seed(4)
    batches = []
    for _ in range(2):
        z = torch.randn(3, k, 48, 40, device="cuda", generator=g) * 2
        y = torch.randint(0, k, (3, 48, 40), device="cuda", generator=g)
        y[0] = torch.where(y[0] == 2, 1, y[0])                  # class 2 absent from one sample's labels
        batches.append((z, y.to(torch.uint8)))
    got = test_segmentation_model(_Echo().cuda(), batches, "cuda", "echo", log=lambda *a: None)
    per = {key: [] for key in ("iou", "dice", "precision", "recall", "f1")}
    pix = []
    for z, y in batches:
        pred = z.double().argmax(1)
        yl = y.long()
        tp = torch.stack([((pred == c) & (yl == c)).flatten(1).sum(1) for c in range(k)], 1).double()
        npred = torch.stack([(pred == c).flatten(1).sum(1) for c in range(k)], 1).double()
        ntgt = torch.stack([(yl == c).flatten(1).sum(1) for c in range(k)], 1).double()
        prec = (tp + eps) / (npred + eps)
        rec = (tp + eps) / (ntgt + eps)
        per["iou"].append((tp + eps) / (npred + ntgt - tp + eps))
        per["dice"].append((2 * tp + eps) / (npred + ntgt + eps))
        per["precision"].append(prec)
        per["recall"].append(rec)
        per["f1"].append(2 * prec * rec / (prec + rec + eps))
        pix.append(tp.sum(1) / ntgt.sum(1))
    assert set(METRIC_KEYS) <= set(got)
    for key, v in per.items():
        m = torch.cat(v).mean(0) * 100                      # per-class mean over samples
        for c in range(k):
            assert abs(got[f"{key}_c{c}"] - float(m[c])) < 1e-9, (key, c)
        assert abs(got[key] - float(m[1:].mean())) < 1e-9, key
    assert abs(got["pixel_accuracy"] - float(torch.cat(pix).mean() * 100)) < 1e-9


def test_segmentation_model_rejects_a_loader_mixing_label_maps_and_float_masks():
    from b200seg.utils.tester import test_segmentation_model
    z = torch.randn(2, 3, 16, 16, device="cuda")
    y = torch.randint(0, 3, (2, 16, 16), device="cuda", dtype=torch.uint8)
    with pytest.raises(ValueError):
        test_segmentation_model(_Echo().cuda(), [(z, y), (z, y.float())], "cuda", "echo", log=lambda *a: None)


def test_predict_labels_is_the_argmax_of_the_logits():
    """bf16 (BatchNorm-folded eval path) and fp32 parity mode, 3 classes; the fp32 logits also match the fp64 oracle"""
    import b200seg
    from b200seg.models.segmentation_models import AttentionUNet
    from b200seg.utils.synthetic import fill_state_dict_, xray_batch
    from b200seg.utils.tester import predict_labels
    from oracle import unet_oracle as O
    model = AttentionUNet(out_channel=3)
    fill_state_dict_(model.state_dict(), seed=3)
    model = model.cuda().eval()
    x, _ = xray_batch(2, 64, 64, seed=8, device="cuda")
    sd = {k: (v.detach().double().cpu() if v.is_floating_point() else v.detach().cpu())
          for k, v in model.state_dict().items()}
    ref, _ = O.attention_unet_forward(sd, x.double().cpu(), training=False)
    for mode, tol in (("bf16", 1e-2), ("fp32", 1e-4)):
        with torch.no_grad(), b200seg.precision(mode):
            logits = model(x).float()
        err = float((logits.double().cpu() - ref).norm() / ref.norm())
        assert logits.shape == (2, 3, 64, 64) and err < tol, (mode, err)
        lab = predict_labels(model, x, precision=mode)
        assert lab.dtype.name == "uint8" and lab.shape == (2, 64, 64)
        assert (torch.from_numpy(lab) == torch.argmax(logits, 1).cpu().to(torch.uint8)).all(), mode
