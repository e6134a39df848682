"""pytest configuration: registers the `gpu` marker and puts the package directory on sys.path.

`-m "not gpu"` tests run on the CPU-only build box; `-m gpu` tests are the parity tests proper and call the
sm_100a kernels through the C ABI (they never read /root/reference).
"""
import os
import sys
from pathlib import Path

import pytest

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "medical-image-segmentation-and-classification_b200"
for p in (str(ROOT), str(PKG)):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")
    # ResNetUnet asks torchvision for the ImageNet ResNet-50 checkpoint, a download: every such request fails at once, as
    # it does offline, so the tests use the model's seeded random-init fallback on every machine and none of them reaches
    # the network or depends on what the user's torch cache holds
    from torchvision.models import WeightsEnum

    def no_download(self, *args, **kwargs):
        raise RuntimeError(f"{self} is not fetched: the tests use random init")

    WeightsEnum.get_state_dict = no_download


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(autouse=True)
def _exact_fp32_reference():
    """torch/cuDNN fp32 references must not silently drop to TF32"""
    import torch

    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    yield
