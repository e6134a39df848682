"""CPU: host-side logic added in round 2 that needs no GPU — the augmentation parameter packing (against OpenCV's own
matrix routines), the layout contract check behind the side-stream / gradient-slot paths, the precision switch, and the
header <-> ctypes agreement of the new argument structs."""
import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest
import torch

ROOT = Path(__file__).resolve().parent.parent


def test_affine_matrices_match_opencv():
    cv2 = pytest.importorskip("cv2")
    from b200seg.data import affine_matrix, invert_affine, pack_params
    for size, ang, sc, dx, dy in [(256, 11.0, 1.04, 0.03, -0.05), (64, -15.0, 0.95, -0.05, 0.02), (128, 0.0, 1.0, 0.0, 0.0)]:
        m = affine_matrix(size, ang, sc, dx, dy)
        ref = cv2.getRotationMatrix2D((size / 2 - 0.5, size / 2 - 0.5), ang, sc)
        ref[0, 2] += dx * size
        ref[1, 2] += dy * size
        assert np.allclose(m, ref, atol=1e-12)
        assert np.allclose(invert_affine(m), cv2.invertAffineTransform(ref), atol=1e-10)
    p = pack_params(64, [{"angle": 5.0, "scale": 1.0, "dx": 0.0, "dy": 0.0, "flip": True, "alpha": 1.1, "beta": -0.05},
                         {"flip": False}], border="reflect101")
    assert p.shape == (2, 12) and p.dtype == np.float32
    iv = p.view(np.int32)
    assert list(iv[0, 8:12]) == [1, 1, 1, 1] and list(iv[1, 8:12]) == [0, 0, 0, 1]
    assert np.allclose(p[1, 0:6], [1, 0, 0, 0, 1, 0]) and p[1, 6] == 1.0 and p[1, 7] == 0.0


def test_grad_is_stolen_layout_contract():
    from b200seg.kernels import grad_is_stolen
    w = torch.nn.Parameter(torch.randn(8, 4, 3, 3))
    assert not grad_is_stolen(w)                                   # contiguous 3x3: AccumulateGrad would clone
    w_cl = torch.nn.Parameter(torch.randn(8, 4, 3, 3).contiguous(memory_format=torch.channels_last))
    assert grad_is_stolen(w_cl)
    w_cl.grad = torch.zeros_like(w_cl)
    assert not grad_is_stolen(w_cl)                                # a gradient is already there: accumulation
    w11 = torch.nn.Parameter(torch.randn(8, 4, 1, 1))
    assert grad_is_stolen(w11)                                     # 1x1: both layouts coincide (size-1 dims are free)


def test_precision_switch_and_inference_only_guard():
    import b200seg
    from b200seg import ops_fp32
    assert b200seg.get_precision() == "bf16"
    with b200seg.precision("fp32"):
        assert b200seg.get_precision() == "fp32"
        m = torch.nn.Linear(2, 2).train()
        with pytest.raises(RuntimeError, match="inference path only"):
            ops_fp32.active(m)
        with torch.no_grad():
            assert ops_fp32.active(m.eval())
    assert b200seg.get_precision() == "bf16"
    with pytest.raises(ValueError):
        b200seg.set_precision("fp16")


def _struct_fields(name):
    text = (ROOT / "include" / "b200seg.h").read_text()
    body = re.search(r"typedef struct " + name + r" \{(.*?)\} " + name + ";", text, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    n = 0
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        names = decl.split(",")
        arr = re.search(r"\[(\d+)\]", names[0])
        n += int(arr.group(1)) if arr else len(names)
    return n


@pytest.mark.parametrize("cname,pyname", [("b2_conv_args", "ConvArgs"), ("b2_wgrad_args", "WgradArgs"),
                                          ("b2_gate_args", "GateArgs"), ("b2_f32_conv_args", "F32ConvArgs"),
                                          ("b2_bn_run_ref", "BnRunRef")])
def test_ctypes_structs_have_the_headers_field_count(cname, pyname):
    from b200seg import _lib
    assert len(getattr(_lib, pyname)._fields_) == _struct_fields(cname)
    if pyname == "BnRunRef":
        assert C.sizeof(_lib.BnRunRef) == 48          # 64 of them travel as one kernel parameter


def test_aug_params_size_matches_header():
    from b200seg.data import PARAM_FLOATS
    assert _struct_fields("b2_aug_params") == PARAM_FLOATS          # 6 + 2 floats + 4 ints, 4 bytes each
    assert C.sizeof(C.c_float) == 4


def _load_bench():
    import importlib.util
    import sys
    spec = importlib.util.spec_from_file_location("bench_mod", ROOT / "bench.py")
    argv, sys.argv = sys.argv, ["bench.py"]
    try:
        bench = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(bench)
    finally:
        sys.argv = argv
    return bench


def test_bench_clock_sampler_keeps_the_rows_of_the_timed_region():
    """bench.py's nvidia-smi sampler starts before the warm-up and stamps its rows; only those inside the timed region
    count (median clock, throttle reasons), with the rows around it as the fallback for a region shorter than one period."""
    bench = _load_bench()

    class _Proc:
        def terminate(self):
            pass

        def wait(self, timeout=None):
            return 0

    def row(mhz, cap):
        return ["0", str(mhz), "1965", "900.0", "Not Active", "Not Active", "Not Active", "Active" if cap else "Not Active"]

    s = bench.ClockSampler(0)
    s.proc = _Proc()
    s.rows = [(0.5, row(1965, False)), (1.1, row(1700, True)), (1.2, row(1650, True)), (1.3, row(1600, True)),
              (2.5, row(1965, False))]
    s.t0, s.t1 = 1.0, 1.35
    out = s.stop()
    assert out["samples"] == 3 and out["sm_mhz"] == 1650 and out["sm_max_mhz"] == 1965
    assert out["reasons"] == ["sw_power_cap"] and out["window"] == "timed region"
    s = bench.ClockSampler(0)
    s.proc = _Proc()
    s.rows = [(0.2, row(1900, False)), (1.5, row(1800, True))]
    s.t0, s.t1 = 1.0, 1.01                      # no row inside: the rows taken under load around it
    out = s.stop()
    assert out["samples"] == 2 and "under load" in out["window"]
    assert bench.ClockSampler(0).stop()["sm_mhz"] is None          # nvidia-smi unavailable


@pytest.mark.parametrize("name", ["AttentionUNet", "R2U_Net", "R2AttU_Net", "ResNetUnet"])
def test_bench_output_arrays_are_a_fixed_sample_within_budget(name):
    """bench.py --dump-outputs: the loss and every state_dict entry of the model, float32 / float64, large tensors cut
    to the same seeded positions on every run, the whole at most 64 MB"""
    import warnings
    from b200seg.models import segmentation_models as M
    bench = _load_bench()
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        torch.manual_seed(0)
        m = getattr(M, name)()
    sd = m.state_dict()
    out = bench.output_arrays(torch.tensor(0.25), m)
    assert list(out) == ["loss"] + list(sd) and float(out["loss"]) == 0.25
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(a.nbytes for a in out.values()) <= 64 << 20
    big = [k for k, v in sd.items() if v.numel() > bench.DUMP_SAMPLE]
    assert big
    for k in big:
        n = sd[k].numel()
        idx = np.sort(np.random.default_rng(0).choice(n, bench.DUMP_SAMPLE, replace=False))
        assert np.array_equal(out[k], sd[k].reshape(-1).numpy()[idx]), k
    again = bench.output_arrays(torch.tensor(0.25), m)
    assert all(np.array_equal(out[k], again[k]) for k in out)
    small = next(k for k, v in sd.items() if v.is_floating_point() and v.numel() <= bench.DUMP_SAMPLE)
    assert np.array_equal(out[small], sd[small].numpy())


def test_bench_rejects_zero_steps():
    import subprocess
    import sys
    r = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=300)
    assert r.returncode == 2 and "--steps" in r.stderr


def test_bench_reference_arm_contract():
    """`bench.py --impl reference` (the CPU arm the driver runs beside ours): rank 0 prints ONE JSON line with the base
    keys plus impl / cpu_baseline / e2e (zero copy bytes); every other rank exits 0 without work."""
    import json
    import os
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    cmd = [sys.executable, str(root / "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1", "--cpu-batch", "1",
           "--side", "64"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=dict(os.environ, RANK="0"))
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "images/s" and d["higher_is_better"] is True
    assert d["metric"] == "AttU_Net 256x256 train images/sec" and d["steps"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "workload" in d["config"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=300, env=dict(os.environ, RANK="1", WORLD_SIZE="2"))
    assert r.returncode == 0 and r.stdout.strip() == "", (r.stdout, r.stderr[-500:])


def test_nvtx_ranges_behind_env_flag():
    """B200SEG_NVTX=1 wraps every library call in an NVTX range named after the entry point (a no-op without a
    profiler) and leaves return-code checking and launch counting untouched."""
    import os
    import subprocess
    import sys
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    code = ("from b200seg import _lib\n"
            "assert _lib._NVTX\n"
            "n = _lib.launch_count\n"
            "_lib.call('b2_reload_env')\n"
            "assert _lib.launch_count == n + 1\n"
            "import torch\n"
            "if not torch.cuda.is_available():\n"
            "    try:\n"
            "        _lib.call('b2_arch_check')\n"
            "        raise SystemExit('no error raised')\n"
            "    except _lib.B2Error:\n"
            "        pass\n"
            "print('NVTX_OK')\n")
    env = dict(os.environ, B200SEG_NVTX="1",
               PYTHONPATH=str(root / "medical-image-segmentation-and-classification_b200") + os.pathsep + os.environ.get("PYTHONPATH", ""))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and "NVTX_OK" in r.stdout, (r.stdout, r.stderr[-1000:])
