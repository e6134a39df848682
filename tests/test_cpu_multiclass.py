"""CPU checks of the multi-class layer: the sums layout the Python side reads matches the header's, the fake kernels of
the new ops propagate shapes, arguments are validated before anything reaches a device, and the synthetic 3-class
batch has the promised classes."""
import re
from pathlib import Path

import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def test_ce_sums_layout_matches_header():
    from b200seg import kernels as K
    text = (ROOT / "include" / "b200seg.h").read_text()
    macros = dict(re.findall(r"#define (B2_CE_\w+)(?:\(k\))?\s+\(?(.+?)\)?\s*$", text, flags=re.M))
    for k in range(2, K.MAX_CLASSES + 1):
        ev = {name: eval(expr, {"k": k}) for name, expr in macros.items()}
        assert ev["B2_CE_NSUMS"] == K.ce_nsums(k)
        f = K.ce_sums_fields(torch.arange(K.ce_nsums(k), dtype=torch.float64), k)
        assert int(f["loss"]) == ev["B2_CE_LOSS"] and int(f["wsum"]) == ev["B2_CE_WSUM"]
        assert int(f["invalid"]) == ev["B2_CE_INVALID"]
        for key, name in (("pt", "B2_CE_PT"), ("p", "B2_CE_P"), ("t", "B2_CE_T"), ("inter", "B2_CE_INTER"),
                          ("union", "B2_CE_UNION")):
            assert f[key].tolist() == list(range(ev[name], ev[name] + k)), (k, key)


def test_fake_kernels_of_the_multiclass_ops():
    import b200seg.ops as ops
    from torch._subclasses.fake_tensor import FakeTensorMode
    with FakeTensorMode():
        z = torch.empty(2, 5, 32, 32, device="cuda")
        y = torch.empty(2, 32, 32, dtype=torch.uint8, device="cuda")
        loss, sums = ops.seg_loss_ce(z, y, None, -100, 0.5, 0.5, 1.0)
        assert loss.shape == () and sums.shape == (28,) and sums.dtype == torch.float64
        dz = ops.seg_loss_ce_bwd(loss, z, y, None, -100, sums, 0.5, 0.5, 1.0)
        assert dz.shape == z.shape and dz.dtype == torch.float32


def test_arguments_are_validated_before_any_launch():
    from b200seg.data import GpuSegAugment
    from b200seg.engine import GraphedTrainStep
    from b200seg.utils.helpers import train
    with pytest.raises(ValueError):
        GpuSegAugment(labels=True, mask_nearest_resize=False)
    with pytest.raises(ValueError):
        GraphedTrainStep(None, None, loss="focal")
    with pytest.raises(ValueError):
        train(None, [], [], "cpu", 1, 1e-3, "m", "/nonexistent", seg=True, loss="dice")


def test_synthetic_multiclass_batch():
    from b200seg.utils.synthetic import xray_batch, xray_batch_multiclass
    x, y = xray_batch_multiclass(4, 96, 80, seed=3)
    x0, m0 = xray_batch(4, 96, 80, seed=3)
    assert torch.equal(x, x0)                                   # the same image as the binary batch
    assert y.dtype == torch.uint8 and y.shape == (4, 96, 80)
    assert set(torch.unique(y).tolist()) == {0, 1, 2}
    assert torch.equal(y > 0, m0[:, 0] > 0.5)                   # lesions lie inside the lungs
    assert all(int((y[i] == 2).sum()) > 0 for i in range(4))
    x1, y1 = xray_batch_multiclass(4, 96, 80, seed=3)
    assert torch.equal(y, y1)
