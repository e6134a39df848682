"""GPU: gradient accumulation folded into kernels (DESIGN.md section 4) against autograd's own accumulation.

  * ops.maxpool2x2_pass — the skip tensor's decoder-side gradient is added inside the pool-backward kernel
    (b2_maxpool2x2_bwd_add): one rounding of the exact sum, exactly like ATen's add of the two bf16 gradients, so every
    gradient must be BIT-identical to the plain path;
  * AttentionGate.gate_pass — the UpConv output's concat-side gradient rides the W_g dgrad epilogue as its addend (fp32
    add before the single bf16 rounding, where ATen rounds the dgrad first): equal up to that rounding.

Both are compared on whole models in deterministic-reduction mode (otherwise train-mode runs differ by their atomics'
summation order)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


@pytest.fixture()
def deterministic():
    from b200seg import kernels as K
    K.set_deterministic(True)
    try:
        yield
    finally:
        K.set_deterministic(False)


def _grads(model, x, t):
    from b200seg import kernels as K, ops
    model.zero_grad(set_to_none=True)
    K.step_begin()
    logits = model(x)
    loss, _ = ops.seg_loss(logits, t, 1.0, 0.0, 1.0)
    loss.backward()
    torch.cuda.synchronize()
    return logits.detach().clone(), {k: p.grad.detach().clone() for k, p in model.named_parameters()}


def _rel(a, b):
    return float((a.double() - b.double()).norm() / (b.double().norm() + 1e-30))


@pytest.mark.parametrize("name,kw", [("AttentionUNet", {}), ("R2U_Net", {"t": 2}), ("R2AttU_Net", {"t": 1})])
def test_pool_pass_is_bit_identical_to_autograd_accumulation(deterministic, name, kw):
    from b200seg import ops, ops_gate
    from b200seg.models import segmentation_models as M
    from b200seg.utils.synthetic import xray_batch
    torch.manual_seed(0)
    model = getattr(M, name)(**kw).cuda().train()
    x, t = xray_batch(2, 64, 64, seed=3, device=torch.device("cuda"))
    gate_pass = ops_gate._GATE_PASS
    ops_gate._GATE_PASS = False            # isolate the pool pass-through
    try:
        assert ops._POOL_PASS
        state = {k: v.clone() for k, v in model.state_dict().items()}
        lo1, g1 = _grads(model, x, t)
        ops._POOL_PASS = False
        model.load_state_dict(state)
        lo0, g0 = _grads(model, x, t)
    finally:
        ops._POOL_PASS = True
        ops_gate._GATE_PASS = gate_pass
    assert torch.equal(lo1, lo0)
    bad = [k for k in g0 if not torch.equal(g0[k], g1[k])]
    assert not bad, f"{len(bad)} gradients differ, e.g. {bad[:4]}"


def test_gate_pass_matches_autograd_accumulation(deterministic):
    from b200seg import ops_gate
    from b200seg.models.segmentation_models import AttentionUNet
    from b200seg.utils.synthetic import xray_batch
    torch.manual_seed(0)
    model = AttentionUNet().cuda().eval()        # eval-mode BatchNorm: no chaotic amplification of the one rounding
    for p in model.parameters():
        p.requires_grad_(True)
    x, t = xray_batch(2, 64, 64, seed=4, device=torch.device("cuda"))
    assert ops_gate._GATE_PASS
    lo1, g1 = _grads(model, x, t)
    ops_gate._GATE_PASS = False
    try:
        lo0, g0 = _grads(model, x, t)
    finally:
        ops_gate._GATE_PASS = True
    assert torch.equal(lo1, lo0)
    num = sum(float((g1[k].double() - g0[k].double()).pow(2).sum()) for k in g0) ** 0.5
    den = sum(float(g0[k].double().pow(2).sum()) for k in g0) ** 0.5
    assert num / den < 2e-3, num / den
    worst = max(_rel(g1[k], g0[k]) for k in g0 if g0[k].numel() > 1000)
    assert worst < 2e-2, worst
