import os, sys
from pathlib import Path
ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "medical-image-segmentation-and-classification_b200"))
import torch
from b200seg import kernels as K

def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)

def run(n, h, w, cin, cout, k):
    g = torch.Generator(device="cuda").manual_seed(1)
    x = nhwc(torch.randn(n, cin, h, w, device="cuda", generator=g))
    wt = torch.randn(cout, cin, k, k, device="cuda", generator=g) / (cin * k * k) ** 0.5
    wf, wd = K.pack_weights(wt)
    stats = torch.zeros(2, cout, dtype=torch.float64, device="cuda")
    y = K.conv_igemm(x, wf, cout, k, stats=stats)
    torch.cuda.synchronize()
    return y, stats

shape = tuple(int(v) for v in sys.argv[1].split(",")) if len(sys.argv) > 1 else (2, 64, 64, 128, 256, 3)
y0, s0 = run(*shape)
for env, val in (("B200SEG_PAIR", "1"), ("B200SEG_PAIR", "2")):
    os.environ[env] = val
    try:
        y1, s1 = run(*shape)
        print(env, val, "equal" if torch.equal(y0, y1) else f"DIFF max {float((y0.float()-y1.float()).abs().max())}",
              float((s0 - s1).abs().max()), flush=True)
    except Exception as e:
        print(env, val, "ERROR", str(e)[:300], flush=True)
    del os.environ[env]
