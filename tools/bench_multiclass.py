"""Cost of multi-class training on the B200: AttU_Net 256^2 graphed training steps with one output channel and BCE (the
binary default) against three output channels and CE + Dice, alternated in ONE process, plus the multi-class loss
kernels timed on their own with CUDA events.

    python tools/bench_multiclass.py [--batch 64] [--side 256] [--rounds 5] [--steps 20] [--out FILE]

Both steps run like bench.py's: deterministic-reduction mode, weight gradients on the side stream, FusedClipAdamW,
one CUDA graph per step.  Kernel rates are bytes the kernel must move (computed from the shapes) over its time; each
timed launch follows a 512 MiB READ that evicts the 126 MB L2 (clean lines: no write-back of the eviction falls into the
timed window), so the inputs come from HBM.  A plain device copy of the logits, timed the same way, is the reference
rate of a memory-bound kernel under these conditions.  Prints one JSON document.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "medical-image-segmentation-and-classification_b200"))

import torch  # noqa: E402

HBM_TBPS = 7.7          # HGX B200 data sheet, per GPU


def gpu_identity():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm,driver_version",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        info["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def make_stepper(k, batch, side):
    from b200seg.engine import GraphedTrainStep
    from b200seg.models.segmentation_models import AttentionUNet
    from b200seg.optim import FusedClipAdamW
    from b200seg.utils.synthetic import xray_batch, xray_batch_multiclass
    torch.manual_seed(0)
    model = AttentionUNet(out_channel=k).cuda().to(memory_format=torch.channels_last).train()
    opt = FusedClipAdamW(model.parameters(), lr=1e-6, weight_decay=5e-4, max_norm=1.0)
    if k == 1:
        x, t = xray_batch(batch, side, side, seed=100, device="cuda")
        st = GraphedTrainStep(model, opt, warmup=3, wgrad_overlap=True)
    else:
        x, t = xray_batch_multiclass(batch, side, side, seed=100, device="cuda")
        st = GraphedTrainStep(model, opt, warmup=3, wgrad_overlap=True, loss="ce", loss_weights=(0.5, 0.5, 1.0))
    for _ in range(5):                      # 3 eager steps, capture, one replay
        st(x, t)
    torch.cuda.synchronize()
    assert st.graph_for(x, t) is not None, st.capture_error
    return st, x, t


def time_steps(st, x, t, steps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(st.stream)
    for _ in range(steps):
        st(x, t)
    e1.record(st.stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def time_kernel(fn, reps, flush):
    """median / min ms of fn() over reps launches, each after an L2-evicting read"""
    fn()
    ts = []
    for _ in range(reps):
        flush.sum()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts), min(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--side", type=int, default=256)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--kernel-reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_multiclass.py measures the B200: no CUDA device")
    from b200seg import _lib
    from b200seg import kernels as K
    _lib.check(_lib.load().b2_arch_check(), "b2_arch_check")
    K.set_deterministic(True)
    B, S = args.batch, args.side
    res = {"gpu": gpu_identity(), "batch": B, "side": S, "rounds": args.rounds, "steps_per_round": args.steps}

    # -- steps, alternated ---------------------------------------------------------------------------------------
    arms = {"k1_bce": make_stepper(1, B, S), "k3_ce_dice": make_stepper(3, B, S)}
    per = {name: [] for name in arms}
    for _ in range(args.rounds):
        for name, (st, x, t) in arms.items():
            per[name].append(time_steps(st, x, t, args.steps))
    for name, v in per.items():
        res[name] = {"ms_per_step_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v),
                     "ms_rounds": v}
    res["step_delta_ms_median"] = res["k3_ce_dice"]["ms_per_step_median"] - res["k1_bce"]["ms_per_step_median"]
    del arms
    torch.cuda.empty_cache()

    # -- loss kernels in isolation (K = 3, uint8 labels, the step's shapes) ----------------------------------------
    k = 3
    g = torch.Generator(device="cuda").manual_seed(0)
    z = torch.randn(B, k, S, S, device="cuda", generator=g)
    y = torch.randint(0, k, (B, S, S), device="cuda", generator=g).to(torch.uint8)
    flush = torch.ones(128 << 20, dtype=torch.float32, device="cuda")      # 512 MiB
    zc = torch.empty_like(z)
    K.set_deterministic(False)
    zb, yb = z.numel() * 4, y.numel()
    loss, sums = K.ce_loss_fwd(z, y, None, -100, 0.5, 0.5, 1.0)
    acc = torch.zeros_like(sums)
    kernels = {
        "ce_loss_fwd": (lambda: _lib.call("b2_ce_loss_fwd", K._p(z), K._p(y), 1, B, k, S * S, None, -100, K._p(acc),
                                          K._stream()), zb + yb),
        "ce_loss_finalize": (lambda: _lib.call("b2_ce_loss_finalize", K._p(sums), k, 0.5, 0.5, 1.0, K._p(loss),
                                               K._stream()), 0),
        "ce_loss_bwd": (lambda: K.ce_loss_bwd(z, y, None, -100, sums, None, 0.5, 0.5, 1.0), 2 * zb + yb),
        "seg_counts_mc": (lambda: K.seg_counts_mc(z, y), zb + yb),
        "logits_to_labels": (lambda: K.logits_to_labels(z), zb + yb),
        "copy_baseline": (lambda: zc.copy_(z), 2 * zb),
    }
    res["kernels"] = {}
    for name, (fn, nbytes) in kernels.items():
        med, best = time_kernel(fn, args.kernel_reps, flush)
        gbs = nbytes / (med * 1e-3) / 1e9
        res["kernels"][name] = {"bytes": nbytes, "ms_median": med, "ms_min": best, "GB_per_s": gbs,
                                "fraction_of_7.7TBps": gbs / (HBM_TBPS * 1e3)}
    loss_ms = sum(res["kernels"][n]["ms_median"] for n in ("ce_loss_fwd", "ce_loss_finalize", "ce_loss_bwd"))
    res["loss_kernels_ms"] = loss_ms
    res["claim_step_delta_le_loss_kernels"] = res["step_delta_ms_median"] <= loss_ms
    res["claim_kernels_ge_70pct"] = all(v["fraction_of_7.7TBps"] >= 0.7 for n, v in res["kernels"].items()
                                        if n not in ("ce_loss_finalize", "copy_baseline"))
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
