#!/usr/bin/env python
"""det_cost.py — what the deterministic-reduction mode costs the flagship training step.

    python tools/det_cost.py --det 0|1 [--replays N] [--trace DIR]

Builds the bench.py workload (channels_last AttentionUNet, FusedClipAdamW, GraphedTrainStep with the weight-gradient
side stream, batch 64, 256x256, seed 0) with the library's deterministic mode on (--det 1) or off (--det 0), times
N graph replays with CUDA events and prints one JSON line with the GPU's name and power limit.  With --trace DIR a
second, separate pass runs torch.profiler (CUDA activities) over two replays and writes the per-kernel time and
count of one step to DIR/det<mode>_kernels.txt, memset nodes included.

Run one process per mode: set_deterministic(False) frees the workspace a graph captured in deterministic mode
points into, so the mode is never toggled inside a process.
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
PKG = ROOT / "medical-image-segmentation-and-classification_b200"
for _p in (str(ROOT), str(PKG)):
    if _p not in sys.path:
        sys.path.insert(0, _p)


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [s.strip() for s in out.splitlines()[0].split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:       # the timing does not depend on it; say that it is missing
        return {"gpu": f"unknown ({e})"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--det", type=int, choices=[0, 1], required=True)
    ap.add_argument("--replays", type=int, default=50)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--side", type=int, default=256)
    ap.add_argument("--trace", metavar="DIR", default=None)
    args = ap.parse_args()

    import torch
    from b200seg import _lib, kernels as K
    from b200seg.engine import GraphedTrainStep
    from b200seg.models.segmentation_models import AttentionUNet
    from b200seg.optim import FusedClipAdamW
    from b200seg.utils.synthetic import xray_batch

    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    _lib.check(_lib.load().b2_arch_check(), "b2_arch_check")
    K.set_wgrad_overlap(True)
    K.set_deterministic(bool(args.det))
    torch.manual_seed(0)
    model = AttentionUNet().to(dev, memory_format=torch.channels_last)
    model.train()
    opt = FusedClipAdamW([p for p in model.parameters() if p.requires_grad], lr=1e-6, weight_decay=5e-4, max_norm=1.0)
    x, t = xray_batch(args.batch, args.side, args.side, seed=100)
    x, t = x.to(dev), t.to(dev)
    stepper = GraphedTrainStep(model, opt, graph=True, warmup=3, wgrad_overlap=True)
    stepper.stream.wait_stream(torch.cuda.current_stream())
    torch.cuda.set_stream(stepper.stream)
    for _ in range(4):                    # 3 eager warm-up steps, then capture + one replay
        stepper(x, t)
    torch.cuda.synchronize()
    static = stepper.static_inputs(x.shape, t.shape)
    assert static is not None, f"graph capture failed: {stepper.capture_error}"
    xs, ts = static

    def replay():
        return stepper(xs, ts, inputs_are_static=True)

    for _ in range(5):
        replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.replays):
        loss = replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.replays
    line = {"det": args.det, "ms_per_step": round(ms, 4), "img_per_s": round(args.batch * 1000.0 / ms, 1),
            "replays": args.replays, "batch": args.batch, "side": args.side, "loss": float(loss),
            "launches_per_step": stepper.launches_per_replay.get((tuple(x.shape), tuple(t.shape))),
            "deterministic": K.deterministic_enabled(), **gpu_info()}

    if args.trace:
        from torch.profiler import ProfilerActivity, profile
        out = Path(args.trace)
        out.mkdir(parents=True, exist_ok=True)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(2):
                replay()
            torch.cuda.synchronize()
        rows = {}
        for ev in prof.events():
            if ev.device_type != torch.autograd.DeviceType.CUDA:
                continue
            r = rows.setdefault(ev.name, [0.0, 0])
            r[0] += ev.device_time_total / 2.0     # per step, microseconds
            r[1] += 1
        total = sum(v[0] for v in rows.values())
        lines = [f"det={args.det}  {line['gpu']}  power limit {line.get('power_limit')}  "
                 f"event-timed {ms:.3f} ms/step (untraced pass)",
                 f"per step (mean of 2 traced replays): device time summed over entries {total / 1e3:.3f} ms "
                 "(the two streams overlap, so this exceeds the step time)",
                 f"{'us/step':>10} {'n/step':>7}  name"]
        for name, (us, n) in sorted(rows.items(), key=lambda kv: -kv[1][0]):
            lines.append(f"{us:10.1f} {n / 2:7.1f}  {name[:140]}")
        (out / f"det{args.det}_kernels.txt").write_text("\n".join(lines) + "\n")
        fin = [v for k, v in rows.items() if "det_finish" in k]
        mem = [v for k, v in rows.items() if "memset" in k.lower()]
        line["trace"] = {"det_finish_us": round(sum(v[0] for v in fin), 1), "det_finish_n": sum(v[1] for v in fin) / 2,
                         "memset_us": round(sum(v[0] for v in mem), 1), "memset_n": sum(v[1] for v in mem) / 2,
                         "summed_device_ms": round(total / 1e3, 3)}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
