#!/usr/bin/env python
"""bench.py — AttU_Net 256x256 training throughput (images/s) on N B200s, one JSON line on rank 0.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--batch B] [--model NAME]
                    [--dump-outputs DIR]

A step = zero_grad -> forward -> BCEWithLogits -> backward -> (gradient all-reduce) -> clip_grad_norm_(1.0) ->
AdamW step, i.e. the body of the reference's train() hot loop (utils/helpers.py:317-337) on synthetic
chest-X-ray-shaped 3x256x256 inputs with binary masks and random-init weights (BASELINE.json configs[1]:
"AttU_Net training batch 64 bf16 ... on 1 B200"; per-GPU batch stays 64 as N grows => weak scaling).

value  : images/s with the batch resident in HBM when the timed region starts (CUDA events, max over ranks).
e2e    : same step through the public nn.Module API with the batch copied from pinned host memory and the loss
         read back to the host inside the timed region, every step.
roofline : tcgen05 implicit-GEMM convolution kernel (fprop + dgrad launches): algorithmic FLOPs of every launch
         / CUDA-event time of those launches, measured in an instrumented pass after the timed region, against
         the measured sustained bf16 peak in MEASURED_PEAKS.json.
cpu_baseline / --impl reference : the oracle port of the reference (oracle/unet_oracle.py, pinned to the real
         reference by tests/golden) timed on the host cores, batch 4 per step (BASELINE.json configs[0]).
reductions : every run of the B200 arm uses the library's deterministic-reduction mode (fixed-order sums instead of
         atomics), so that the same arguments compute the same bits.  With atomics the summation order varies, and
         AdamW turns the rounding noise of near-zero gradients (the conv biases ahead of BatchNorm) into steps of about
         lr that spread to every weight: two runs would train different models.
--dump-outputs DIR : after the timed steps, DIR/<name>.npy holds what the last of them computed (see output_arrays);
         the inputs depend on the arguments alone, so two builds can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
PKG = ROOT / "medical-image-segmentation-and-classification_b200"
for _p in (str(ROOT), str(PKG)):
    if _p not in sys.path:
        sys.path.insert(0, _p)

METRIC = "AttU_Net 256x256 train images/sec"     # other --model values report "<model> ... train images/sec"
TRAIN_GFLOP_PER_IMG = {"AttentionUNet": 398.32, "R2U_Net": 1697.66, "R2AttU_Net": 1704.13,
                       "ResNetUnet": 234.43}   # SURVEY.md §8(d); R2 figures are for the ctor default t=5


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="per-GPU batch")
    ap.add_argument("--global-batch", type=int, default=0,
                    help="fixed GLOBAL batch split over the ranks (strong scaling: BASELINE.json configs[2] R2AttU b32, "
                         "configs[3] ResNetUnet b128); overrides --batch")
    ap.add_argument("--model", default="AttentionUNet", choices=["AttentionUNet", "R2U_Net", "R2AttU_Net", "ResNetUnet"])
    ap.add_argument("--t", type=int, default=None, help="recurrence depth for the R2 models (reference default 5)")
    ap.add_argument("--side", type=int, default=256)
    ap.add_argument("--cpu-batch", type=int, default=4)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--optimizer", default="fused", choices=["fused", "torch"],
                    help="fused: b200seg FusedClipAdamW (clip + AdamW, 2 launches); torch: clip_grad_norm_ + AdamW(fused)")
    ap.add_argument("--wgrad-overlap", type=int, default=1,
                    help="1: weight-gradient kernels on a side stream, overlapping the memory-bound backward kernels")
    ap.add_argument("--graph", type=int, default=1,
                    help="capture the whole training step in a CUDA graph (single-GPU runs); 0 = eager launches")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and the model state of the last timed step as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the b200 path computed; it does not apply to --impl reference")
    return args


DUMP_BYTES = 64 << 20        # cap on what --dump-outputs writes
DUMP_SAMPLE = 16384          # elements kept of a larger tensor


def output_arrays(loss, model):
    """What a caller of the training step receives: the step's loss and the state the step leaves in the model (parameters
    and BatchNorm running statistics), as {name: float32 or float64 array}.  A tensor of more than DUMP_SAMPLE elements
    is cut to a fixed, seeded sample of its flattened values, the same positions on every run."""
    import numpy as np
    import torch
    out = {"loss": loss.detach().float().cpu().numpy()}
    for k, v in model.state_dict().items():
        v = v.detach()
        if v.numel() > DUMP_SAMPLE:
            idx = np.sort(np.random.default_rng(0).choice(v.numel(), DUMP_SAMPLE, replace=False))
            v = v.reshape(-1)[torch.from_numpy(idx).to(v.device)]
        wide = v.dtype == torch.float64 or not v.is_floating_point()       # num_batches_tracked counts, fp64 state
        out[k] = v.to(torch.float64 if wide else torch.float32).cpu().numpy()
    assert sum(a.nbytes for a in out.values()) <= DUMP_BYTES
    return out


TRAFFIC_FILE = "r02f_traffic.json"      # ncu DRAM counters of one step of the default workload (tools/profile_step.py)


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d.get("bf16_tflops_sustained", 1407.6), d.get("hbm_gbs", 6468.0), "measured (MEASURED_PEAKS.json, sustained)"
    return 1400.0, 6650.0, "fallback (B200_PROFILING.md)"


def measured_traffic():
    """mean DRAM bytes per launch of the tensor-core kernels, from the committed ncu capture of one training step of
    the default workload (tools/profile_step.py + tools/summarize_traffic.py); {} if the capture is absent"""
    p = ROOT / "profiles" / TRAFFIC_FILE
    if not p.exists():
        return {}
    d = json.loads(p.read_text())
    out = {}
    # fprop / dgrad launches are conv_igemm_kernel or, for the Cout = 64 3x3 layers on wide images, conv_c64_kernel
    for short, names in (("conv_igemm", ("b2::conv_igemm_kernel", "b2::conv_c64_kernel")),
                         ("conv_wgrad", ("b2::conv_wgrad_kernel",))):
        n = sum(d[k]["launches"] for k in names if k in d)
        if n:
            out[short] = sum(d[k]["read_GB"] + d[k]["write_GB"] for k in names if k in d) * 1e9 / n
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None

    def start(self):
        """Started BEFORE the warm-up: nvidia-smi takes a few hundred ms to come up, longer than a short timed region.
        Rows are stamped on arrival; stop() keeps those that fall between mark_begin() and mark_end()."""
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        t0 = self.t0 if self.t0 is not None else float("-inf")
        t1 = self.t1 if self.t1 is not None else float("inf")
        inside = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.05]
        window = "timed region"
        if not inside:       # a timed region shorter than one sampling period: the rows taken under load around it
            inside = [r for ts, r in self.rows if ts >= t0 - 1.0]
            window = "timed region +- 1 s (under load)"
        sm, mx, reasons = [], [], set()
        for r in inside:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 4), ("hw_thermal_slowdown", 5), ("sw_thermal_slowdown", 6),
                              ("sw_power_cap", 7)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "window": window, "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port of the reference on the host cores
# ----------------------------------------------------------------------------------------------------------
def cpu_reference_steps(model_name, kw, batch, side, steps, warmup, with_optimizer=True):
    import numpy as np
    import torch
    from oracle import unet_oracle as O           # the CPU arm is the one place bench.py may execute oracle/
    from oracle.synthetic import xray_batch
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    # weights: the reference's state_dict layout (recorded from the real modules in tests/golden/) + synthetic fill;
    # nothing of the CUDA package is imported on this arm
    lay = np.load(ROOT / "tests" / "golden" / f"{model_name}.npz", allow_pickle=True)
    sd = O.state_dict_from_layout(lay["keys"], lay["shapes"], lay["dtypes"], seed=0)
    frozen = ("encoder",) if model_name == "ResNetUnet" else ()      # reference default freeze=True
    params = {k: v.requires_grad_(True) for k, v in sd.items()
              if v.is_floating_point() and not k.endswith(("running_mean", "running_var"))
              and not k.startswith(frozen or ("\0",))}
    opt = torch.optim.AdamW(list(params.values()), lr=1e-6, weight_decay=5e-4)
    x, t = xray_batch(batch, side, side, seed=0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        opt.zero_grad(set_to_none=True)
        logits, newb = O.FORWARDS[model_name](sd, x, training=True, **kw)
        loss = O.bce_with_logits(logits, t)
        loss.backward()
        if with_optimizer:
            torch.nn.utils.clip_grad_norm_(list(params.values()), 1.0)
            opt.step()
        for k, v in newb.items():
            sd[k] = v.detach()
        float(loss)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    return times


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    kw = {"t": args.t} if (args.t is not None and args.model != "AttentionUNet") else {}
    steps, warmup = args.steps, max(args.warmup, 1)
    times = cpu_reference_steps(args.model, kw, args.cpu_batch, args.side, steps, warmup)
    total = sum(times)
    ips = args.cpu_batch * len(times) / total
    sample = (f"oracle port of the reference ({args.model} fwd+BCE+bwd+clip+AdamW, fp32, torch CPU), "
              f"batch {args.cpu_batch} per step x {len(times)} steps, {os.cpu_count()} threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": ips, "unit": "images/s", "n_gpus": args.gpus,
        "steps": len(times), "warmup": warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{args.model} {args.side}x{args.side} training step, bounded CPU sample "
                               f"(batch {args.cpu_batch}/step) of the batch-{args.batch} workload"},
        "cpu_baseline": {"value": ips, "unit": "images/s", "cores": os.cpu_count(), "kind": "port", "sample": sample},
        "e2e": {"value": ips, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------
# B200 arm
# ----------------------------------------------------------------------------------------------------------
def _tick(msg, t0=[None]):
    """wall-clock phase markers on stderr (B200SEG_BENCH_VERBOSE=1)"""
    if os.environ.get("B200SEG_BENCH_VERBOSE"):
        now = time.perf_counter()
        if t0[0] is None:
            t0[0] = now
        print(f"[bench +{now - t0[0]:7.2f}s] {msg}", file=sys.stderr, flush=True)


def run_b200(args):
    _tick("start")
    import torch
    import torch.distributed as dist

    from b200seg import _lib, kernels as K, ops
    from b200seg.models import segmentation_models as M
    from b200seg.ddp import GradReducer
    from b200seg.utils.synthetic import xray_batch
    from torchvision.models import WeightsEnum

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    saved_stdout = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner on stdout from native code: park fd 1 on stderr until the JSON line is due, so
        # that rank 0's stdout carries exactly ONE line
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group("nccl", device_id=dev)
    _lib.check(_lib.load().b2_arch_check(), "b2_arch_check")
    K.set_wgrad_overlap(bool(args.wgrad_overlap))
    K.set_deterministic(True)             # the same arguments compute the same bits (see "reductions" above)

    kw = {"t": args.t} if (args.t is not None and args.model != "AttentionUNet") else {}
    def no_download(self, *args, **kwargs):
        raise RuntimeError(f"{self} is not fetched: the benchmark uses random init")
    # ResNetUnet: every pretrained-weight request fails as it does offline, so the model takes its seeded random-init
    # fallback, never a downloaded or cached checkpoint, and the inputs depend on the arguments alone
    WeightsEnum.get_state_dict = no_download
    torch.manual_seed(0)
    model = getattr(M, args.model)(**kw).to(dev, memory_format=torch.channels_last)   # helpers.py:243
    model.train()
    use_graph = bool(args.graph)     # the bucketed NCCL all-reduces are captured in the graph as well
    trainable = [p for p in model.parameters() if p.requires_grad]
    if args.optimizer == "fused":     # clip_grad_norm_(1.0) + AdamW in two launches of libb200seg (helpers.py:251,333-335)
        from b200seg.optim import FusedClipAdamW
        opt = FusedClipAdamW(trainable, lr=1e-6, weight_decay=5e-4, max_norm=1.0)
    else:
        opt = torch.optim.AdamW(trainable, lr=1e-6, weight_decay=5e-4, fused=True, capturable=use_graph)
    reducer = GradReducer(model, bucket_mb=32) if world > 1 else None
    if args.global_batch:
        assert args.global_batch % world == 0, "--global-batch must be divisible by the number of ranks"
        args.batch = args.global_batch // world
    B, S = args.batch, args.side
    x_host, t_host = xray_batch(B, S, S, seed=100 + rank)
    x_host, t_host = x_host.pin_memory(), t_host.pin_memory()
    x_dev, t_dev = x_host.to(dev), t_host.to(dev)
    params = [p for p in model.parameters() if p.requires_grad]

    def step(x, t):      # the eager step, used by the instrumented roofline pass below
        opt.zero_grad(set_to_none=True)
        K.step_begin()
        logits = model(x)
        loss, _ = ops.seg_loss(logits, t, 1.0, 0.0, 1.0)
        loss.backward()
        if reducer is not None:
            reducer.finish()
        if args.optimizer != "fused":
            torch.nn.utils.clip_grad_norm_(params, 1.0)
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            out = fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms), out

    # The package's own fast step (b200seg.engine.GraphedTrainStep — the same object utils.helpers.train() drives):
    # the first calls run eagerly (warm-up), then the whole step — forward, loss, backward, bucketed NCCL all-reduces,
    # clip, AdamW, weight re-pack — is captured in ONE CUDA graph and every later call is a replay.
    from b200seg.engine import GraphedTrainStep, PinnedPrefetcher
    n_warm = max(args.warmup, 3)
    stepper = GraphedTrainStep(model, opt, reducer=reducer, graph=use_graph, warmup=n_warm,
                               wgrad_overlap=bool(args.wgrad_overlap),
                               clip_fn=None if args.optimizer == "fused"
                               else (lambda: torch.nn.utils.clip_grad_norm_(params, 1.0)))
    run_stream = stepper.stream           # everything below runs on the stepper's stream (no per-step stream hops)
    run_stream.wait_stream(torch.cuda.current_stream())
    torch.cuda.set_stream(run_stream)
    _tick("model built, warm-up begins")
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()                   # (comes up during the warm-up; only rows inside the timed region are used)
    for _ in range(n_warm):
        stepper(x_dev, t_dev)
    torch.cuda.synchronize()
    _tick("warm-up done")
    stepper(x_dev, t_dev)                 # captures (if enabled) and replays once
    torch.cuda.synchronize()
    graphed = stepper.graph_for(x_dev, t_dev) is not None
    if use_graph and not graphed:
        print(f"[bench] CUDA graph capture failed ({stepper.capture_error}); timing eager launches", file=sys.stderr)
    static = stepper.static_inputs(x_dev.shape, t_dev.shape)
    if static is not None:
        x_run, t_run = static             # batch resident in the graph's input buffers when the timed region starts
    else:
        x_run, t_run = x_dev, t_dev
    launches_per_step = stepper.launches_per_replay.get((tuple(x_dev.shape), tuple(t_dev.shape)))
    _tick("graph captured and replayed once" if graphed else "eager mode")

    def run_step():
        return stepper(x_run, t_run, inputs_are_static=graphed)

    l0 = _lib.launch_count
    sampler.mark_begin()
    ms, loss = timed(run_step, args.steps)
    sampler.mark_end()
    launches = (_lib.launch_count - l0) if not graphed else launches_per_step * args.steps
    time.sleep(0.06)                      # let the sampler deliver the last row of the region
    clocks = sampler.stop() if rank == 0 else None
    _tick("timed region done")
    if args.dump_outputs and rank == 0:   # now: the passes below train the model further
        import numpy as np
        out_dir = Path(args.dump_outputs)
        out_dir.mkdir(parents=True, exist_ok=True)
        for name, a in output_arrays(loss, model).items():
            np.save(out_dir / f"{name}.npy", a)

    # end-to-end through the package API: every step's batch starts in pinned HOST memory (as DataLoader(pin_memory=True)
    # delivers it), PinnedPrefetcher copies batch i+1 on its copy stream while step i computes, the stepper copies it
    # into the graph's inputs and replays, and the loss is read back to the host — every step moves one full batch
    # host -> device and 4 bytes device -> host inside the timed region.
    class _HostBatches:
        def __init__(self, n):
            self.n = n

        def __len__(self):
            return self.n

        def __iter__(self):
            for _ in range(self.n):
                yield x_host, t_host

    pre = PinnedPrefetcher(_HostBatches(args.steps + 1), dev)
    e2e_iter = iter(pre)

    def e2e_step():
        xb, tb = next(e2e_iter)
        return float(stepper(xb, tb))
    e2e_step()
    ms_e2e, _ = timed(e2e_step, args.steps)
    h2d_per_step = pre.h2d_bytes // (args.steps + 1)
    _tick("e2e done")
    # data-parallel sanity inside the measured run: after all those steps every replica must hold the same parameters
    replicas_in_sync = (reducer.param_checksum() == 0.0) if reducer is not None else None
    graph = stepper if graphed else None

    # instrumented pass for the roofline of the tensor-core kernels
    # (single stream: with the weight gradients on the side stream the per-launch event times would include the
    # kernels they overlap with)
    K.set_wgrad_overlap(False)
    K.PROFILE = []
    for _ in range(2):
        # the pass launches eagerly: park the GPU on a ~25 ms spin first so that the host has enqueued the step's
        # launches and events before the device reaches them — the event pairs then bracket kernel time, not launch
        # gaps (matters for the small-batch configs, whose kernels are shorter than a Python launch)
        torch.cuda._sleep(int(5e7))
        step(x_dev, t_dev)
    torch.cuda.synchronize()
    agg = {}
    if os.environ.get("B200SEG_BENCH_DUMP") and rank == 0:
        with open(os.environ["B200SEG_BENCH_DUMP"], "w") as f:
            for kind, flops, _alg, _nb, a, b in K.PROFILE[len(K.PROFILE) // 2:]:
                ms_ = a.elapsed_time(b)
                f.write(f"{kind} {flops / 1e9:10.2f} GF {ms_:8.4f} ms {flops / ms_ / 1e9:8.1f} TF/s\n")
    for kind, flops, alg, nb, a, b in K.PROFILE:
        f, fa, by, tms, n = agg.get(kind, (0.0, 0.0, 0.0, 0.0, 0))
        agg[kind] = (f + flops, fa + alg, by + nb, tms + a.elapsed_time(b), n + 1)
    K.PROFILE = None
    peak_tf, peak_hbm, peak_src = measured_peaks()

    def leave():
        """Multi-rank exit: NCCL communicator teardown can block while a captured graph still references NCCL work, so
        ranks rendezvous once more and leave without destroying the process group."""
        if world > 1:
            _tick("leaving")
            torch.cuda.synchronize()
            dist.barrier()
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)

    if rank != 0:
        leave()
        return
    imgs = B * world * args.steps
    value = imgs / (ms / 1e3)
    e2e = imgs / (ms_e2e / 1e3)
    f, fa, by_i, tms, n = agg.get("conv_igemm", (0.0, 0.0, 0.0, 1.0, 1))
    ach = f / (tms * 1e-3) / 1e12
    ach_alg = fa / (tms * 1e-3) / 1e12
    fw, fwa, by_w, tw, nw = agg.get("conv_wgrad", (0.0, 0.0, 0.0, 1.0, 1))
    traffic = measured_traffic()
    ach_w = fw / (tw * 1e-3) / 1e12
    ach_w_alg = fwa / (tw * 1e-3) / 1e12
    step_ms = ms / args.steps
    line = {
        "metric": METRIC if args.model == "AttentionUNet" else f"{args.model} {S}x{S} train images/sec",
        "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": step_ms, "higher_is_better": True,
        "scaling": "strong" if args.global_batch else "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"{args.model} {S}x{S} training step (fwd + BCEWithLogits + bwd + clip_grad_norm + "
                               f"AdamW), batch {B} per GPU, random init, synthetic X-ray-shaped inputs",
                   "per_gpu_batch": B, "global_batch": B * world, "parallelism": f"dp{world}",
                   "l2": "working set per step (>10 GB of activations) far exceeds the 126 MB L2",
                   "model_kwargs": kw, "cuda_graph": graph is not None, "optimizer": args.optimizer,
                   "wgrad_side_stream": bool(args.wgrad_overlap),
                   "deterministic_reductions": K.deterministic_enabled()},
        "e2e": {"value": e2e, "unit": "images/s", "h2d_bytes_per_step": int(h2d_per_step),
                "d2h_bytes_per_step": 4, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": launches,
        "replicas_in_sync": replicas_in_sync,
        "clocks": clocks,
        "roofline": {"kernel": "conv_igemm_kernel + conv_c64_kernel (tcgen05 implicit GEMM; every fprop + dgrad launch of the step)",
                     "bound": "tensor", "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf,
                     "achieved_algorithmic": ach_alg,
                     "note": "achieved = FLOPs the launches executed / their CUDA-event time; achieved_algorithmic "
                             "counts the folded UpConv launches at the reference's 3x3-on-the-fine-grid FLOPs (x2.25)",
                     "traffic": traffic.get("conv_igemm"), "traffic_unit": "bytes per launch (mean over the step's "
                     "launches; ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/" + TRAFFIC_FILE + ")",
                     "algorithmic_bytes_per_launch": by_i / max(n, 1),
                     "peak_source": peak_src, "launches_per_step": n // 2,
                     "ms_per_step_in_kernel": tms / 2, "share_of_step": (tms / 2) / step_ms},
        "roofline_wgrad": {"kernel": "conv_wgrad_kernel + wgrad_reduce_kernel", "bound": "tensor", "achieved": ach_w,
                           "achieved_algorithmic": ach_w_alg, "traffic": traffic.get("conv_wgrad"),
                           "algorithmic_bytes_per_launch": by_w / max(nw, 1),
                           "peak": peak_tf, "unit": "TFLOP/s", "frac": ach_w / peak_tf,
                           "launches_per_step": nw // 2, "ms_per_step_in_kernel": tw / 2,
                           "share_of_step": (tw / 2) / step_ms},
        "model_tflops": TRAIN_GFLOP_PER_IMG[args.model] * value / 1e3 if kw == {} else None,
    }
    if world == 1 and not args.no_cpu_baseline:
        times = cpu_reference_steps(args.model, kw, args.cpu_batch, S, 3, 1)
        best = min(times)
        line["cpu_baseline"] = {
            "value": args.cpu_batch / best, "unit": "images/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"oracle port of the reference, {args.model} batch {args.cpu_batch} fp32 train step "
                      f"(fwd+BCE+bwd+clip+AdamW), best of 3 after 1 warm-up, {os.cpu_count()} threads",
            "median_s_per_step": statistics.median(times)}
    if saved_stdout is not None:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
    print(json.dumps(line), flush=True)
    leave()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
