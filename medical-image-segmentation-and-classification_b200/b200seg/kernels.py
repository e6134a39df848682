"""Tensor-level wrappers over the C ABI: take torch CUDA tensors, pass raw pointers + dims + the current stream.

Activations are NHWC bf16 tensors of shape [N, H, W, C]; the channel stride of the underlying buffer may exceed C
(channel-slice views are passed without a copy).  Every function here launches kernels of libb200seg.so and
nothing else — torch is used only to allocate outputs.
"""
from __future__ import annotations

import contextlib
import ctypes as C
import os

import torch

from . import _lib
from ._lib import ConvArgs, GateCoef, WgradArgs, call

BF16 = torch.bfloat16


# Optional per-launch timing hook used by bench.py's roofline pass: when set to a list, the tensor-core
# convolution wrappers append (kind, flops, start_event, end_event) recorded on the launching stream.
PROFILE = None


def _prof_begin():
    if PROFILE is None:
        return None
    ev = torch.cuda.Event(enable_timing=True)
    ev.record()
    return ev


def _prof_end(kind, flops, start, alg_scale=1.0, nbytes=0.0):
    """flops = executed by the launch; alg_scale * flops = the reference's algorithmic count for the same work
    (9/4 for the folded UpConv phases, which do 4 taps on the coarse grid instead of 9 on the fine one)"""
    if start is not None:
        end = torch.cuda.Event(enable_timing=True)
        end.record()
        PROFILE.append((kind, flops, flops * alg_scale, nbytes, start, end))


# ----------------------------------------------------------------------------------------------------------
# Weight-gradient overlap: dW is only needed after backward, so its kernels can run on a side stream while the main
# stream goes on with the memory-bound BatchNorm / gate / pooling backward of the next layers (they fit next to the
# persistent wgrad CTAs on an SM; the tensor-core kernels of the main stream do not, those simply take turns).
# Opt-in (set_wgrad_overlap / B200SEG_WGRAD_OVERLAP=1): the caller must not touch a weight gradient before
# loss.backward() has returned — true for utils.helpers.train() and bench.py (zero_grad(set_to_none=True),
# channels_last parameters, gradients read by GradReducer.finish() / the optimizer).  Weights shared between several
# autograd nodes (Recurrent_block) qualify too: their applications accumulate into one buffer inside the wgrad kernel
# (ops.conv_bn_act, share_index / share_count), so autograd never sums them on the main stream.
# ----------------------------------------------------------------------------------------------------------
_OVERLAP = {"enabled": os.environ.get("B200SEG_WGRAD_OVERLAP", "0") == "1", "side": {}, "refs": [], "pending": False,
            "task": -1}


def set_wgrad_overlap(flag: bool) -> None:
    _OVERLAP["enabled"] = bool(flag)


def wgrad_overlap_enabled() -> bool:
    return _OVERLAP["enabled"]


def _join_wgrad_stream():
    """End of backward (autograd engine callback): the calling stream waits for the side stream, references drop."""
    main = torch.cuda.current_stream()
    for side in _OVERLAP["side"].values():
        main.wait_stream(side)
    _OVERLAP["refs"].clear()
    _OVERLAP["pending"] = False


def wgrad_side_stream():
    """The side stream if weight gradients of the running backward pass are in flight on it, else None."""
    if not _OVERLAP["pending"]:
        return None
    return _OVERLAP["side"].get(torch.cuda.current_device())


def wgrad_side_streams():
    """every side stream created so far on the current device (for callers that must order work after them)"""
    side = _OVERLAP["side"].get(torch.cuda.current_device())
    return [side] if side is not None else []


def grad_is_stolen(weight) -> bool:
    """True when autograd's AccumulateGrad will adopt the [Cout, taps, Cin] weight-gradient buffer as `weight.grad`
    without touching it on the main stream: no gradient accumulated yet and the parameter's memory order is the
    buffer's (channels_last; size-1 dims are free).  Otherwise AccumulateGrad clones / adds on the main stream and a
    side-stream wgrad kernel would race it — callers then keep the weight gradient on the main stream."""
    if weight.grad is not None or weight.dim() != 4:
        return False
    cout, cin, kh, kw = weight.shape
    want = (kh * kw * cin, 1, kw * cin, cin)
    return all(d == 1 or s == w for d, s, w in zip(weight.shape, weight.stride(), want))


@contextlib.contextmanager
def wgrad_stream(*keep, allow=True):
    """Run the enclosed launches on the weight-gradient side stream (ordered after everything already queued on the
    current stream).  `keep`: tensors produced on the current stream that the side stream reads — references are
    held until the join so the caching allocator cannot hand their memory out again.  No-op unless enabled, inside a
    backward pass and `allow`."""
    if not (allow and _OVERLAP["enabled"] and torch.cuda.is_available()):
        yield
        return
    task = torch._C._current_graph_task_id()       # -1 outside backward
    if task < 0:
        yield                                       # not inside a backward pass: nothing to overlap with
        return
    if not _OVERLAP["pending"] or _OVERLAP["task"] != task:
        if _OVERLAP["pending"]:
            # a previous backward pass ended without its callback (an exception unwound it): join what it left behind
            _join_wgrad_stream()
        try:
            torch.autograd.Variable._execution_engine.queue_callback(_join_wgrad_stream)
        except RuntimeError:
            yield
            return
        _OVERLAP["pending"] = True
        _OVERLAP["task"] = task
    main = torch.cuda.current_stream()
    dev = torch.cuda.current_device()
    side = _OVERLAP["side"].get(dev)
    if side is None:
        side = _OVERLAP["side"][dev] = torch.cuda.Stream(device=dev)
    ev = torch.cuda.Event()
    ev.record(main)
    side.wait_event(ev)
    _OVERLAP["refs"].extend(t for t in keep if t is not None)
    with torch.cuda.stream(side):
        yield


# ----------------------------------------------------------------------------------------------------------
# Zeroed scratch for the small reduction buffers of a step (BatchNorm statistics, backward sums, loss sums): ~75
# torch.zeros fills per AttU_Net step become slices of one arena that step_begin() clears with a single memset.
# Opt-in: without step_begin() (or once the arena is exhausted) zeros_scratch() is torch.zeros.  Slices are only valid
# until the next step_begin(), so nothing that outlives a step (gradients) is ever taken from it.
# ----------------------------------------------------------------------------------------------------------
_ARENA = {"enabled": os.environ.get("B200SEG_ZERO_ARENA", "1") != "0", "bufs": {}, "bytes": 1 << 20}


def step_begin():
    """Start of a training step (train() / bench.py call it): clear what the previous step used of the arena."""
    if not _ARENA["enabled"] or not torch.cuda.is_available():
        return
    dev = torch.cuda.current_device()
    st = _ARENA["bufs"].get(dev)
    if st is None:
        st = _ARENA["bufs"][dev] = {"buf": torch.zeros(_ARENA["bytes"], dtype=torch.uint8, device=f"cuda:{dev}"),
                                    "off": 0, "high": 0, "armed": False}
    else:
        # the high-water mark of all earlier steps: a captured CUDA graph replays this one memset for every step
        st["high"] = max(st["high"], st["off"])
        if st["high"]:
            st["buf"][:st["high"]].zero_()
    st["off"] = 0
    st["armed"] = True
    _ZPOOL.pop(dev, None)


# Zero-filled op OUTPUTS that may outlive the step (bias gradients that autograd adopts as .grad, statistics a caller
# may keep): slices of a pool that is allocated FRESH once per step (one fill launch instead of ~50), never recycled —
# a slice keeps the pool's storage alive for as long as anyone holds it.  Main-stream tensors only, and at most ONE slice
# among the inputs and outputs of any custom op (torch.library rejects outputs that share a storage with each other
# or with an input).
_ZPOOL = {}
_ZPOOL_BYTES = 256 << 10


def zeros_out(shape, dtype, device):
    dev = device.index if device.index is not None else torch.cuda.current_device()
    st = _ARENA["bufs"].get(dev) if device.type == "cuda" else None
    if st is None or not st["armed"]:
        return torch.zeros(shape, dtype=dtype, device=device)
    n = 1
    for d in shape:
        n *= int(d)
    nbytes = n * torch.empty((), dtype=dtype).element_size()
    if nbytes > _ZPOOL_BYTES // 4:
        return torch.zeros(shape, dtype=dtype, device=device)
    pool = _ZPOOL.get(dev)
    off = 0 if pool is None else (pool["off"] + 255) & ~255
    if pool is None or off + nbytes > _ZPOOL_BYTES:
        pool = _ZPOOL[dev] = {"buf": torch.zeros(_ZPOOL_BYTES, dtype=torch.uint8, device=device), "off": 0}
        off = 0
    pool["off"] = off + nbytes
    return pool["buf"][off:off + nbytes].view(dtype).view(shape)


def zeros_scratch(shape, dtype, device):
    """Zero-filled reduction buffer that is dead by the end of the step."""
    st = _ARENA["bufs"].get(device.index if device.index is not None else torch.cuda.current_device()) \
        if device.type == "cuda" else None
    if st is None or not st["armed"]:
        return torch.zeros(shape, dtype=dtype, device=device)
    n = 1
    for d in shape:
        n *= int(d)
    nbytes = n * torch.empty((), dtype=dtype).element_size()
    off = (st["off"] + 15) & ~15
    if off + nbytes > st["buf"].numel():
        return torch.zeros(shape, dtype=dtype, device=device)
    st["off"] = off + nbytes
    return st["buf"][off:off + nbytes].view(dtype).view(shape)


# ----------------------------------------------------------------------------------------------------------
# Deterministic-reduction mode (b2_set_deterministic): per-block partials + fixed-order second stage instead of
# atomics, so that two runs on the same inputs are bit-identical (set_deterministic(True) or B200SEG_DETERMINISTIC=1).
# The workspace belongs to the launches of one compute stream at a time; the weight-gradient side stream only runs
# the (always deterministic) wgrad kernels and never touches it.
# ----------------------------------------------------------------------------------------------------------
_DET = {"want": os.environ.get("B200SEG_DETERMINISTIC", "0") == "1", "bufs": {}, "bytes": 64 << 20}


def set_deterministic(flag: bool) -> None:
    _DET["want"] = bool(flag)
    if torch.cuda.is_available():
        _sync_deterministic()


def deterministic_enabled() -> bool:
    return _DET["want"]


def _sync_deterministic():
    """register / drop the workspace of the current device so that the library state follows _DET['want']"""
    dev = torch.cuda.current_device()
    have = dev in _DET["bufs"]
    if _DET["want"] and not have:
        buf = torch.empty(_DET["bytes"], dtype=torch.uint8, device=f"cuda:{dev}")
        _lib.check(_lib.load().b2_set_deterministic(C.c_void_p(buf.data_ptr()), buf.numel()), "b2_set_deterministic")
        _DET["bufs"][dev] = buf
    elif not _DET["want"] and have:
        _lib.check(_lib.load().b2_set_deterministic(C.c_void_p(0), 0), "b2_set_deterministic")
        torch.cuda.synchronize(dev)          # no launch may still be writing partials when the buffer is freed
        del _DET["bufs"][dev]


def reload_switches():
    """the library caches the B200SEG_* environment switches: re-read them after changing os.environ"""
    _lib.check(_lib.load().b2_reload_env(), "b2_reload_env")


def _stream():
    if _DET["want"] != (torch.cuda.current_device() in _DET["bufs"]):
        _sync_deterministic()
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def _nhwc(t):
    """(N, H, W, C, ld) of an NHWC bf16 activation; rows must be dense apart from the channel stride."""
    assert t.dtype == BF16 and t.dim() == 4 and t.is_cuda, (t.dtype, t.shape, t.device)
    n, h, w, c = t.shape
    ld = t.stride(2)
    assert t.stride(3) == 1 and t.stride(1) == w * ld and t.stride(0) == h * w * ld, (t.shape, t.stride())
    return n, h, w, c, ld


def new_act(n, h, w, c, device):
    return torch.empty((n, h, w, c), dtype=BF16, device=device)


# ----------------------------------------------------------------------------------------------------------
# weights
# ----------------------------------------------------------------------------------------------------------
# Packed (bf16, MMA-layout) copies of the convolution weights are cached per parameter and kept fresh by the optimizer:
# FusedClipAdamW re-packs every registered weight in ONE multi-tensor launch right after its AdamW kernel
# (b2_pack_weights_multi), so the conv calls of a training step pack nothing.  Any other writer goes through torch
# (in-place ops bump Tensor._version) and simply invalidates the entry.
#
# Entries are keyed by (data_ptr, kind) and validated against a weak reference to the parameter object: a freed
# parameter whose address is reused by another tensor can never alias a stale entry (the old object is dead).
_PACKS = {"cache": {}, "serial": 0, "epoch": 0}


class _Pack:
    __slots__ = ("ref", "ptr", "version", "kind", "wf", "wd", "cout", "cin", "ksize", "strides", "code", "cols")


def invalidate_pack_cache():
    """drop every cached packed weight (they are rebuilt on next use)"""
    _PACKS["cache"].clear()
    _PACKS["serial"] += 1


def bump_param_epoch():
    """called by whoever updated parameters through raw pointers (FusedClipAdamW.step, a graph replay of it): derived
    caches that the optimizer does NOT refresh itself (BN-folded inference weights) become stale"""
    _PACKS["epoch"] += 1


def param_epoch() -> int:
    return _PACKS["epoch"]


def pack_serial() -> int:
    return _PACKS["serial"]


def _pack_valid(pk, weight):
    o = pk.ref()
    return (o is not None and pk.ptr == weight.data_ptr() and o.data_ptr() == pk.ptr
            and o._version == pk.version and weight._version == pk.version)


_PACK_KINDS = {"plain": 0, "upfold": 1, "stem": 2, "convT_f": 0, "convT_d": 0}


def packed(weight, kind="plain", want_dgrad=False):
    """Cached packed copies of a conv weight: (wf, wd) with wd None unless a dgrad layout was ever requested.
    kind: 'plain'   [Cout,Cin,k,k] -> wf [k*k,Cout,Cin], wd [k*k,Cin,Cout] (flipped taps)
          'upfold'  [Cout,Cin,3,3] -> wf [4,4,Cout,Cin], wd [4,4,Cin,Cout]           (UpConv folding)
          'stem'    [Cout,<=3,3,3] -> wf [1,Cout,32] im2col matrix                   (image stem as a GEMM)
          'convT_f' ConvTranspose weight [Cin,Cout,2,2] -> wf [4,Cout,Cin]           (forward: rows = Cout)
          'convT_d' ConvTranspose weight [Cin,Cout,2,2] -> wf [4,Cin,Cout]           (input gradient: rows = Cin)"""
    key = (weight.data_ptr(), kind)
    pk = _PACKS["cache"].get(key)
    if pk is not None and _pack_valid(pk, weight) and (pk.wd is not None or not want_dgrad):
        return pk.wf, pk.wd
    import weakref
    view = weight.permute(1, 0, 2, 3) if kind == "convT_f" else weight
    cout, cin, kh, kw = view.shape
    assert kh == kw and weight.dtype == torch.float32
    dev = weight.device
    reuse = pk is not None and pk.ref() is weight and pk.ptr == weight.data_ptr() and pk.strides == tuple(view.stride())
    wf = pk.wf if reuse else None
    wd = pk.wd if reuse else None
    need_wd = want_dgrad or wd is not None
    if kind == "upfold":
        wf = wf if wf is not None else torch.empty((4, 4, cout, cin), dtype=BF16, device=dev)
        if need_wd and wd is None:
            wd = torch.empty((4, 4, cin, cout), dtype=BF16, device=dev)
        sv = view.stride()
        call("b2_pack_weights_upfold", _p(view), cout, cin, sv[0], sv[1], sv[2], sv[3], _p(wf), _p(wd), _stream())
    elif kind == "stem":
        cols = stem_cols(weight)
        wf = wf if wf is not None else torch.empty((1, cout, cols), dtype=BF16, device=dev)
        wm = stem_weight_matrix(weight)
        sm = wm.stride()
        call("b2_pack_weights", _p(wm), cout, cols, 1, sm[0], sm[1], sm[2], sm[3], _p(wf), _p(None), _stream())
    else:
        taps = kh * kw
        wf = wf if wf is not None else torch.empty((taps, cout, cin), dtype=BF16, device=dev)
        if need_wd and wd is None:
            wd = torch.empty((taps, cin, cout), dtype=BF16, device=dev)
        sv = view.stride()
        call("b2_pack_weights", _p(view), cout, cin, kh, sv[0], sv[1], sv[2], sv[3], _p(wf), _p(wd), _stream())
    new = _Pack()
    new.ref, new.ptr, new.version, new.kind = weakref.ref(weight), weight.data_ptr(), weight._version, kind
    new.wf, new.wd, new.cout, new.cin, new.ksize = wf, wd, cout, cin, kh
    new.strides, new.code = tuple(view.stride()), _PACK_KINDS[kind]
    new.cols = stem_cols(weight) if kind == "stem" else 0
    cache = _PACKS["cache"]
    if len(cache) > 4096:
        for k in [k for k, v in cache.items() if v.ref() is None]:
            del cache[k]
    cache[key] = new
    if not (reuse and wd is pk.wd and wf is pk.wf):
        _PACKS["serial"] += 1          # new buffers: optimizers rebuild their re-pack tables
    return wf, wd


# ----------------------------------------------------------------------------------------------------------
# Gradient slots: a data-parallel reducer (ddp.GradReducer) registers, per conv weight, the slice of its flat bucket
# where that weight's gradient belongs.  The weight-gradient kernels then write straight into the bucket and autograd
# adopts a view of it as `weight.grad` — no pack copy before the all-reduce, no copy back after it.
# ----------------------------------------------------------------------------------------------------------
_GRAD_SLOTS = {}


def register_grad_slot(weight, flat_slice):
    """flat_slice: 1-D fp32 view (weight.numel() elements) of the bucket; memory order = [Cout][taps][Cin]"""
    import weakref
    assert flat_slice.dtype == torch.float32 and flat_slice.numel() == weight.numel() and flat_slice.is_contiguous()
    _GRAD_SLOTS[weight.data_ptr()] = (weakref.ref(weight), flat_slice)


def unregister_grad_slots(weights=None):
    if weights is None:
        _GRAD_SLOTS.clear()
        return
    for w in weights:
        _GRAD_SLOTS.pop(w.data_ptr(), None)


def grad_slot(weight, shape):
    """a FRESH tensor (so AccumulateGrad can adopt it) viewing the registered bucket slice as `shape`, or None"""
    hit = _GRAD_SLOTS.get(weight.data_ptr())
    if hit is None or hit[0]() is not weight or not grad_is_stolen(weight):
        return None
    return hit[1].view(shape)


def packs_of(params):
    """every live cached pack whose master is one of `params` (FusedClipAdamW builds its re-pack table from this)"""
    ptrs = {p.data_ptr(): p for p in params}
    out = []
    for (ptr, _kind), pk in _PACKS["cache"].items():
        p = ptrs.get(ptr)
        if p is not None and _pack_valid(pk, p):
            out.append(pk)
    return out


def pack_weights(weight, want_dgrad=True):
    """fp32 [Cout, Cin, k, k] parameter (any strides) -> (bf16 [k*k, Cout, Cin], bf16 [k*k, Cin, Cout] flipped)."""
    cout, cin, kh, kw = weight.shape
    assert kh == kw and weight.dtype == torch.float32
    taps = kh * kw
    wf = torch.empty((taps, cout, cin), dtype=BF16, device=weight.device)
    wd = torch.empty((taps, cin, cout), dtype=BF16, device=weight.device) if want_dgrad else None
    s = weight.stride()
    call("b2_pack_weights", _p(weight), cout, cin, kh, s[0], s[1], s[2], s[3], _p(wf), _p(wd), _stream())
    return wf, wd


def pack_weights_upfold(weight, want_dgrad=True):
    """UpConv folding: fp32 [Cout, Cin, 3, 3] -> bf16 [4 phases, 4 taps, Cout, Cin] (+ [4, 4 flipped, Cin, Cout])"""
    cout, cin, kh, kw = weight.shape
    assert kh == 3 and kw == 3 and weight.dtype == torch.float32
    wf = torch.empty((4, 4, cout, cin), dtype=BF16, device=weight.device)
    wd = torch.empty((4, 4, cin, cout), dtype=BF16, device=weight.device) if want_dgrad else None
    s = weight.stride()
    call("b2_pack_weights_upfold", _p(weight), cout, cin, s[0], s[1], s[2], s[3], _p(wf), _p(wd), _stream())
    return wf, wd


def pack_weights_folded(weight, bias, coef, upfold=False):
    """eval-mode BN folding: (bf16 packed W * scale[co], fp32 bias * scale + shift); coef = [mean, invstd, scale, shift]"""
    cout, cin, kh, kw = weight.shape
    shape = (4, 4, cout, cin) if upfold else (kh * kw, cout, cin)
    wf = torch.empty(shape, dtype=BF16, device=weight.device)
    bf = torch.empty((cout,), dtype=torch.float32, device=weight.device)
    s = weight.stride()
    call("b2_pack_weights_folded", _p(weight), cout, cin, kh, s[0], s[1], s[2], s[3], _p(coef[2]), _p(coef[3]),
         _p(bias), int(upfold), _p(wf), _p(bf), _stream())
    return wf, bf


def fold_upconv_wgrad(dweff, out=None):
    """fp32 [4 phases, Cout, 4 taps, Cin] -> fp32 [Cout, 9, Cin]"""
    _, cout, _, cin = dweff.shape
    dw = out if out is not None else torch.empty((cout, 9, cin), dtype=torch.float32, device=dweff.device)
    assert dw.is_contiguous() and dw.numel() == cout * 9 * cin
    call("b2_fold_upconv_wgrad", _p(dweff), cout, cin, _p(dw), _stream())
    return dw


# ----------------------------------------------------------------------------------------------------------
# tcgen05 convolutions
# ----------------------------------------------------------------------------------------------------------
def conv_igemm(x0, wpk, cout, ksize, x1=None, bias=None, addend=None, stats=None, relu=False, out=None,
               row_offset=0, dgrad=False, stride=1, out_mul=1, out_off=(0, 0), in_mul=1, in_off=(0, 0), pad=None,
               alg_scale=1.0, add_after_act=False, fold=0):
    """y = conv(x0 | x1; wpk) (+bias) (+addend) (relu); wpk is [taps, rows, ktot] bf16, rows [row_offset,
    row_offset+cout) are used.  `stats` (fp64 [2, cout]) accumulates sum / sumsq of the rounded output.
    stride=2 samples the input on a 2x finer grid (strided conv / ConvTranspose dgrad); out_mul=2 places the result
    at pixels (2h+off_h, 2w+off_w) of `out` (ConvTranspose pixel shuffle).
    fold: merged launches of the folded UpConv, wpk = its 16 packed taps [16, rows, ktot] — 1: x0 coarse -> y on the 2x
    grid (all four phases, one launch); 2: x0 = dz on the 2x grid -> coarse dx (16-tap K loop, one launch)."""
    n, hi, wi, c0, ld0 = _nhwc(x0)
    if fold:
        assert ksize == 2 and x1 is None and addend is None and stride == 1 and out_mul == 1 and in_mul == 1
        out_mul = 2 if fold == 1 else 1
        h, w = (hi, wi) if fold == 1 else (hi // 2, wi // 2)
    else:
        assert hi % (stride * in_mul) == 0 and wi % (stride * in_mul) == 0
        h, w = hi // (stride * in_mul), wi // (stride * in_mul)     # output grid (in_mul: x0 is read as a sub-lattice)
    c1, ld1 = 0, 0
    if x1 is not None:
        n1, h1, w1, c1, ld1 = _nhwc(x1)
        assert (n1, h1, w1) == (n, hi, wi)
    taps, rows, ktot = wpk.shape
    assert taps == (16 if fold else ksize * ksize) and wpk.dtype == BF16 and wpk.is_contiguous()
    assert ktot >= c0 + c1 and row_offset + cout <= rows
    y = out if out is not None else new_act(n, h * out_mul, w * out_mul, cout, x0.device)
    ny, hy, wy, cy, ldy = _nhwc(y)
    assert cy == cout and (ny, hy, wy) == (n, h * out_mul, w * out_mul)
    a = ConvArgs()
    a.n, a.h, a.w, a.ksize = n, h, w, ksize
    a.x0, a.c0, a.ldx0 = x0.data_ptr(), c0, ld0
    a.x1, a.c1, a.ldx1 = (x1.data_ptr() if x1 is not None else None), c1, ld1
    a.wpk = wpk.data_ptr() + row_offset * ktot * 2
    a.ktot = ktot
    a.w_tap_stride = rows * ktot
    a.cout = cout
    a.y, a.ldy = y.data_ptr(), ldy
    a.bias = bias.data_ptr() if bias is not None else None
    if addend is not None:
        _, _, _, ca, lda = _nhwc(addend)
        assert ca == cout
        a.addend, a.ldadd = addend.data_ptr(), lda
    if stats is not None:
        assert stats.dtype == torch.float64 and stats.numel() == 2 * cout
        a.stats = stats.data_ptr()
    a.relu = int(relu)
    a.stride, a.out_mul, a.out_off_h, a.out_off_w = stride, (1 if fold else out_mul), out_off[0], out_off[1]
    a.in_mul, a.in_off_h, a.in_off_w = in_mul, in_off[0], in_off[1]
    a.add_after_act = int(add_after_act)
    a.fold_mode = int(fold)
    if pad is not None:
        a.custom_pad, a.pad_h, a.pad_w = 1, pad[0], pad[1]
    t0 = _prof_begin()
    call("b2_conv_dgrad" if dgrad else "b2_conv_fprop", C.byref(a), _stream())
    # algorithmic DRAM bytes of the launch: every input element once, every output element once, the weights once
    _prof_end("conv_igemm", 2.0 * n * h * w * cout * (c0 + c1) * taps, t0, alg_scale,
              2.0 * (n * hi * wi * (c0 + c1) // (in_mul * in_mul) + n * h * w * cout * (4 if fold == 1 else 1)
                     + taps * cout * (c0 + c1)))
    return y


def conv_wgrad(dy, x0, ksize, x1=None, out=None, accumulate=False, x_stride=1, dy_mul=1, dy_off=(0, 0), pad=None,
               alg_scale=1.0, fold=False):
    """dW fp32 [Cout, k*k, C0+C1] = sum_p dY[p] (x) X[p+tap].  x_stride=2 (ksize 2): X lives on the 2x finer grid
    (weight gradient of ConvTranspose2d(k=2,s=2) with dy := its input, x := its output gradient).
    fold=True (ksize 2, dy_mul 2): all four phase gradients of a folded UpConv, [4, Cout, 4, Cin], in one launch;
    returns None when the library does not take the shape in that mode (the caller launches the phases)."""
    n, hd, wd_, cout, lddy = _nhwc(dy)
    assert hd % dy_mul == 0 and wd_ % dy_mul == 0
    h, w = hd // dy_mul, wd_ // dy_mul                          # dY is read as a sub-lattice when dy_mul > 1
    nx, hx, wx, c0, ld0 = _nhwc(x0)
    assert (nx, hx, wx) == (n, h * x_stride, w * x_stride)
    c1, ld1 = 0, 0
    if x1 is not None:
        _, _, _, c1, ld1 = _nhwc(x1)
    taps = 16 if fold else ksize * ksize
    dw = out if out is not None else torch.empty((cout, taps, c0 + c1), dtype=torch.float32, device=dy.device)
    assert dw.is_contiguous() and dw.numel() == cout * taps * (c0 + c1)
    a = WgradArgs()
    a.n, a.h, a.w, a.ksize = n, h, w, ksize
    a.dy, a.cout, a.lddy = dy.data_ptr(), cout, lddy
    a.x0, a.c0, a.ldx0 = x0.data_ptr(), c0, ld0
    a.x1, a.c1, a.ldx1 = (x1.data_ptr() if x1 is not None else None), c1, ld1
    a.dw = dw.data_ptr()
    a.accumulate = int(accumulate)
    a.x_stride = x_stride
    a.dy_mul, a.dy_off_h, a.dy_off_w = dy_mul, dy_off[0], dy_off[1]
    if pad is not None:
        a.custom_pad, a.pad_h, a.pad_w = 1, pad[0], pad[1]
    a.fold = int(fold)
    need = _lib.load().b2_conv_wgrad_workspace(C.byref(a))
    if need == -1 and fold:                 # B2_ERR_SHAPE
        return None
    if need < 0:
        _lib.check(int(need), "b2_conv_wgrad_workspace")
    ws = torch.empty(int(need), dtype=torch.uint8, device=dy.device)
    a.workspace, a.workspace_bytes = ws.data_ptr(), int(need)
    t0 = _prof_begin()
    call("b2_conv_wgrad", C.byref(a), _stream())
    _prof_end("conv_wgrad", 2.0 * n * h * w * cout * (c0 + c1) * taps, t0, alg_scale,
              2.0 * (n * h * w * cout * (4 if fold else 1) + n * hx * wx * (c0 + c1)) + 4.0 * taps * cout * (c0 + c1))
    return dw


# ----------------------------------------------------------------------------------------------------------
# small-channel convolutions
# ----------------------------------------------------------------------------------------------------------
def image_to_nhwc4(x):
    """NCHW fp32 image [N, C<=4, H, W] -> NHWC bf16 [N, H, W, 4] (zero padded channels)."""
    assert x.dtype == torch.float32 and x.dim() == 4 and x.is_contiguous() and x.shape[1] <= 4
    n, c, h, w = x.shape
    y = torch.empty((n, h, w, 4), dtype=BF16, device=x.device)
    call("b2_nchw_f32_to_nhwc_bf16", _p(x), n, c, h, w, _p(y), 4, _stream())
    return y


STEM_COLS = 32          # im2col columns of the 3x3 stem (27 used for a 3-channel image)


def stem_im2col3x3(x):
    """NCHW fp32 image [N, C<=3, H, W] -> NHWC bf16 [N, H, W, 32]: 3x3 neighbourhood, column = tap * C + c."""
    assert x.dtype == torch.float32 and x.dim() == 4 and x.is_contiguous() and x.shape[1] <= 3
    n, c, h, w = x.shape
    xc = torch.empty((n, h, w, STEM_COLS), dtype=BF16, device=x.device)
    call("b2_stem_im2col3x3", _p(x), n, c, h, w, _p(xc), _stream())
    return xc


def stem_cols(weight):
    """im2col columns of an image stem: 32 for the 3x3 stems, ks*ks*cin rounded up to 8 otherwise (7x7: 152)"""
    cout, cin, kh, kw = weight.shape
    return STEM_COLS if kh == 3 else (kh * kw * cin + 7) // 8 * 8


def stem_weight_matrix(weight):
    """fp32 [Cout, Cin<=3, k, k] -> fp32 [Cout, cols, 1, 1] with column = tap * Cin + c (the im2col order)."""
    cout, cin, kh, kw = weight.shape
    cols = stem_cols(weight)
    wm = torch.zeros((cout, cols), dtype=torch.float32, device=weight.device)
    wm[:, :kh * kw * cin] = weight.detach().permute(0, 2, 3, 1).reshape(cout, kh * kw * cin)
    return wm.view(cout, cols, 1, 1)


def stem_im2col(x, ksize, stride, pad, cols):
    """NCHW fp32 image -> NHWC bf16 [N, Ho, Wo, cols] im2col (column = tap * C + c) for any stem geometry"""
    assert x.dtype == torch.float32 and x.dim() == 4 and x.is_contiguous()
    n, c, h, w = x.shape
    ho, wo = (h + 2 * pad - ksize) // stride + 1, (w + 2 * pad - ksize) // stride + 1
    xc = torch.empty((n, ho, wo, cols), dtype=BF16, device=x.device)
    call("b2_stem_im2col", _p(x), n, c, h, w, ksize, stride, pad, cols, _p(xc), _stream())
    return xc


def maxpool3x3s2_bwd(dy, x):
    n, h, w, c, ld = _nhwc(x)
    lddy = _nhwc(dy)[4]
    dx = new_act(n, h, w, c, x.device)
    call("b2_maxpool3x3s2_bwd", _p(dy), lddy, _p(x), ld, n, h, w, c, _p(dx), c, _stream())
    return dx


def zero_insert2x(x):
    """y[2h, 2w] = x[h, w], zero elsewhere"""
    n, h, w, c, ld = _nhwc(x)
    y = new_act(n, 2 * h, 2 * w, c, x.device)
    call("b2_zero_insert2x", _p(x), ld, n, h, w, c, _p(y), c, _stream())
    return y


def relu_mask(dy, out):
    """g = out > 0 ? dy : 0"""
    n, h, w, c, lddy = _nhwc(dy)
    ldo = _nhwc(out)[4]
    g = new_act(n, h, w, c, dy.device)
    call("b2_relu_mask", _p(dy), lddy, _p(out), ldo, n * h * w, c, _p(g), c, _stream())
    return g


def stem_weight_grad(dwc, cin, taps=9):
    """[Cout, 1, cols] gradient of the im2col weight matrix -> [Cout, taps, Cin] (tap-major, as conv_wgrad returns)."""
    cout = dwc.shape[0]
    return dwc.reshape(cout, -1)[:, :taps * cin].reshape(cout, taps, cin).contiguous()


def pack_small_weight(weight):
    """fp32 [Cout, Cin<=4, k, k] -> fp32 [Cout, k*k, 4] (tiny; done with torch indexing on the host stream)."""
    cout, cin, kh, kw = weight.shape
    wk = torch.zeros((cout, kh * kw, 4), dtype=torch.float32, device=weight.device)
    wk[:, :, :cin] = weight.permute(0, 2, 3, 1).reshape(cout, kh * kw, cin)
    return wk


def conv_smallc_fprop(x4, wk, bias, ksize, relu=False):
    n, h, w, c4 = x4.shape
    assert c4 == 4 and x4.is_contiguous()
    cout = wk.shape[0]
    y = new_act(n, h, w, cout, x4.device)
    call("b2_conv_smallc_fprop", _p(x4), n, h, w, ksize, _p(wk), _p(bias), cout, _p(y), cout, int(relu), _stream())
    return y


def conv_smallc_wgrad(dy, x4, ksize):
    n, h, w, cout, lddy = _nhwc(dy)
    dw = torch.zeros((cout, ksize * ksize, 4), dtype=torch.float32, device=dy.device)
    call("b2_conv_smallc_wgrad", _p(dy), lddy, _p(x4), n, h, w, ksize, cout, _p(dw), _stream())
    return dw


def head_fwd(x, weight2d, bias):
    """x NHWC bf16 -> logits fp32 NCHW [N, Cout, H, W]; weight2d fp32 [Cout, Cin]."""
    n, h, w, cin, ld = _nhwc(x)
    cout = weight2d.shape[0]
    y = torch.empty((n, cout, h, w), dtype=torch.float32, device=x.device)
    call("b2_head_fwd", _p(x), ld, n * h * w, h * w, cin, _p(weight2d), _p(bias), cout, _p(y), _stream())
    return y


def head_bwd(dy, x, weight2d, need_dx=True):
    n, h, w, cin, ld = _nhwc(x)
    cout = weight2d.shape[0]
    assert dy.dtype == torch.float32 and dy.is_contiguous()
    dx = new_act(n, h, w, cin, x.device) if need_dx else None
    dw = torch.zeros((cout, cin), dtype=torch.float32, device=x.device)
    db = torch.zeros((cout,), dtype=torch.float32, device=x.device)
    call("b2_head_bwd", _p(dy), _p(x), ld, n * h * w, h * w, cin, _p(weight2d), cout, _p(dx), cin, _p(dw), _p(db),
         _stream())
    return dx, dw, db


# ----------------------------------------------------------------------------------------------------------
# batch norm
# ----------------------------------------------------------------------------------------------------------
def channel_stats(z, stats):
    n, h, w, c, ld = _nhwc(z)
    call("b2_channel_stats", _p(z), ld, n * h * w, c, _p(stats), _stream())


def channel_sum(dy):
    n, h, w, c, ld = _nhwc(dy)
    db = torch.empty((c,), dtype=torch.float32, device=dy.device)
    call("b2_channel_sum", _p(dy), ld, n * h * w, c, _p(db), _stream())
    return db


def bn_finalize(stats, count, gamma, beta, eps, momentum, running_mean, running_var, nbt):
    """-> coef fp32 [4, C] = (mean, invstd, scale, shift); updates running stats in place."""
    c = stats.numel() // 2
    coef = torch.empty((4, c), dtype=torch.float32, device=stats.device)
    call("b2_bn_finalize", _p(stats), c, int(count), _p(gamma), _p(beta), float(eps), float(momentum),
         _p(running_mean), _p(running_var), _p(nbt), _p(coef[0]), _p(coef[1]), _p(coef[2]), _p(coef[3]), _stream())
    return coef


def bn_eval_coeffs(gamma, beta, running_mean, running_var, eps):
    c = running_mean.numel()
    coef = torch.empty((4, c), dtype=torch.float32, device=running_mean.device)
    call("b2_bn_eval_coeffs", _p(gamma), _p(beta), _p(running_mean), _p(running_var), float(eps), c, _p(coef[0]),
         _p(coef[1]), _p(coef[2]), _p(coef[3]), _stream())
    return coef


def stem7x7_fprop(x4, wk):
    """ResNet stem: 7x7/s2/p3, <=4 -> 64, no bias.  x4 NHWC bf16 [N,H,W,4]; wk fp32 [64, 49, 4]."""
    n, h, w, c4 = x4.shape
    assert c4 == 4 and x4.is_contiguous()
    cout = wk.shape[0]
    y = new_act(n, h // 2, w // 2, cout, x4.device)
    call("b2_stem7x7_fprop", _p(x4), n, h, w, _p(wk), cout, _p(y), cout, _stream())
    return y


def maxpool3x3s2_fwd(x):
    n, h, w, c, ld = _nhwc(x)
    y = new_act(n, h // 2, w // 2, c, x.device)
    call("b2_maxpool3x3s2_fwd", _p(x), ld, n, h, w, c, _p(y), c, _stream())
    return y


def bn_apply(z, coef, relu=True, addend=None, want_sum=False, sum_only=False):
    """want_sum: also return y + addend; sum_only: return ONLY act(bn(z)) + addend (the x + x1 re-injection of
    Recurrent_block, R2U_Net.py:19); addend without either: y = act(bn(z) + addend) (ResNet residual)"""
    n, h, w, c, ld = _nhwc(z)
    y = None if sum_only else new_act(n, h, w, c, z.device)
    ysum = new_act(n, h, w, c, z.device) if (want_sum or sum_only) else None
    lda = _nhwc(addend)[4] if addend is not None else 0
    call("b2_bn_apply", _p(z), ld, n * h * w, c, _p(coef[2]), _p(coef[3]), int(relu), _p(y), c, _p(addend), lda,
         _p(ysum), c, _stream())
    if sum_only:
        return ysum
    return (y, ysum) if want_sum else y


# Deferred running-statistics updates: they are off the data path (nothing in the step reads running_mean / running_var)
# but each was a launch of its own on the step's critical stream — 34 per AttU_Net step, 70 per R2AttU_Net(t=2) step.
# Inside `deferred_running_updates()` (engine.GraphedTrainStep) they are queued and flushed as ONE launch per round;
# round k holds the k-th update of every BatchNorm of the step, so the t + 1 sequential updates of a Recurrent_block's
# shared BatchNorm (R2U_Net.py:15-20) keep their order.
_RUN = {"defer": False, "queue": []}


@contextlib.contextmanager
def deferred_running_updates():
    if os.environ.get("B200SEG_DEFER_RUNNING", "1") == "0":      # A/B switch: one launch per BatchNorm call
        yield
        return
    prev = _RUN["defer"]
    _RUN["defer"] = True
    try:
        yield
        flush_running_updates()
    finally:
        _RUN["defer"] = prev
        if not prev:
            _RUN["queue"].clear()


def flush_running_updates():
    q, _RUN["queue"] = _RUN["queue"], []
    if not q:
        return
    rounds, seen = [], {}
    for e in q:                                     # e = (stats, count, momentum, rm, rv, nbt)
        k = seen.get(e[3].data_ptr(), 0)
        seen[e[3].data_ptr()] = k + 1
        while len(rounds) <= k:
            rounds.append([])
        rounds[k].append(e)
    for rnd in rounds:
        refs = (_lib.BnRunRef * len(rnd))()
        max_c = 0
        for i, (stats, count, momentum, rm, rv, nbt) in enumerate(rnd):
            c = stats.numel() // 2
            max_c = max(max_c, c)
            refs[i].stats, refs[i].running_mean, refs[i].running_var = stats.data_ptr(), rm.data_ptr(), rv.data_ptr()
            refs[i].num_batches_tracked, refs[i].count, refs[i].c, refs[i].momentum = nbt.data_ptr(), count, c, momentum
        call("b2_bn_update_running_multi", refs, len(rnd), max_c, _stream())


def bn_update_running(stats, count, momentum, running_mean, running_var, nbt):
    """momentum update of the running statistics from epilogue-produced (sum, sumsq); no coefficient outputs"""
    if _RUN["defer"]:
        _RUN["queue"].append((stats, int(count), float(momentum), running_mean, running_var, nbt))
        return
    c = stats.numel() // 2
    z = C.c_void_p(0)
    call("b2_bn_finalize", _p(stats), c, int(count), z, z, 0.0, float(momentum), _p(running_mean), _p(running_var),
         _p(nbt), z, z, z, z, _stream())


def bn_bwd(dy, z, coef, gamma, relu=True, training=True, want_dbias=False):
    """-> (dz bf16, dgamma fp32, dbeta fp32[, dbias fp32])"""
    n, h, w, c, lddy = _nhwc(dy)
    ldz = _nhwc(z)[4]
    npix = n * h * w
    sums = zeros_scratch((2, c), torch.float64, z.device)
    call("b2_bn_bwd_reduce", _p(dy), lddy, _p(z), ldz, npix, c, _p(coef[2]), _p(coef[3]), _p(coef[0]), _p(coef[1]),
         int(relu), _p(sums), _stream())
    dz = new_act(n, h, w, c, z.device)
    dgamma = torch.empty((c,), dtype=torch.float32, device=z.device)
    dbeta = torch.empty((c,), dtype=torch.float32, device=z.device)
    dbias = zeros_out((c,), torch.float32, z.device) if want_dbias else None
    call("b2_bn_bwd_apply", _p(dy), lddy, _p(z), ldz, npix, c, _p(coef[2]), _p(coef[3]), _p(coef[0]), _p(coef[1]),
         _p(gamma), int(relu), int(training), _p(sums), _p(dz), c, _p(dgamma), _p(dbeta), _p(dbias), _stream())
    return (dz, dgamma, dbeta, dbias) if want_dbias else (dz, dgamma, dbeta)


# ----------------------------------------------------------------------------------------------------------
# pooling / upsampling / add
# ----------------------------------------------------------------------------------------------------------
def maxpool_fwd(x):
    n, h, w, c, ld = _nhwc(x)
    y = new_act(n, h // 2, w // 2, c, x.device)
    call("b2_maxpool2x2_fwd", _p(x), ld, n, h, w, c, _p(y), c, _stream())
    return y


def maxpool_bwd(dy, x, addend=None):
    n, h, w, c, ld = _nhwc(x)
    lddy = _nhwc(dy)[4]
    dx = new_act(n, h, w, c, x.device)
    if addend is not None:
        assert addend.shape == x.shape
        call("b2_maxpool2x2_bwd_add", _p(dy), lddy, _p(x), ld, n, h, w, c, _p(addend), _nhwc(addend)[4], _p(dx), c,
             _stream())
    else:
        call("b2_maxpool2x2_bwd", _p(dy), lddy, _p(x), ld, n, h, w, c, _p(dx), c, _stream())
    return dx


def upsample_fwd(x):
    n, h, w, c, ld = _nhwc(x)
    y = new_act(n, 2 * h, 2 * w, c, x.device)
    call("b2_upsample2x_fwd", _p(x), ld, n, h, w, c, _p(y), c, _stream())
    return y


def upsample_bwd(dy):
    n, h2, w2, c, lddy = _nhwc(dy)
    dx = new_act(n, h2 // 2, w2 // 2, c, dy.device)
    call("b2_upsample2x_bwd", _p(dy), lddy, n, h2 // 2, w2 // 2, c, _p(dx), c, _stream())
    return dx


def add(a, b):
    n, h, w, c, lda = _nhwc(a)
    ldb = _nhwc(b)[4]
    out = new_act(n, h, w, c, a.device)
    call("b2_add", _p(a), lda, _p(b), ldb, n * h * w, c, _p(out), c, _stream())
    return out


def to_nhwc_bf16(x):
    """NCHW fp32 [N, C, H, W] -> NHWC bf16 [N, H, W, C]"""
    assert x.dtype == torch.float32 and x.dim() == 4 and x.is_contiguous()
    n, c, h, w = x.shape
    y = new_act(n, h, w, c, x.device)
    call("b2_layout_nchw_to_nhwc", _p(x), n, c, h, w, _p(y), c, _stream())
    return y


def to_nchw_f32(x):
    """NHWC bf16 -> NCHW fp32"""
    n, h, w, c, ld = _nhwc(x)
    y = torch.empty((n, c, h, w), dtype=torch.float32, device=x.device)
    call("b2_layout_nhwc_to_nchw", _p(x), ld, n, c, h, w, _p(y), _stream())
    return y


# ----------------------------------------------------------------------------------------------------------
# attention gate (memory-bound part)
# ----------------------------------------------------------------------------------------------------------
def gate_psi_fwd(g1p, x1p, coef_g, coef_x, wpsi, bpsi):
    n, h, w, fint, ld = _nhwc(g1p)
    assert _nhwc(x1p)[4] == ld
    q = torch.empty((n, h, w), dtype=BF16, device=g1p.device)
    qstats = zeros_out((2,), torch.float64, g1p.device)    # an output of the gate op: not arena memory
    call("b2_gate_psi_fwd", _p(g1p), _p(x1p), ld, n * h * w, fint, _p(coef_g[2]), _p(coef_g[3]), _p(coef_x[2]),
         _p(coef_x[3]), _p(wpsi), _p(bpsi), _p(q), _p(qstats), _stream())
    return q, qstats


def gate_apply_fwd(x, q, coef1):
    n, h, w, c, ld = _nhwc(x)
    psi = torch.empty((n, h, w), dtype=BF16, device=x.device)
    out = new_act(n, h, w, c, x.device)
    call("b2_gate_apply_fwd", _p(x), ld, _p(q), n * h * w, c, _p(coef1[2]), _p(coef1[3]), _p(psi), _p(out), c,
         _stream())
    return out, psi


def gate_apply_bwd(dout, x, psi, q, coef1):
    n, h, w, c, ldx = _nhwc(x)
    lddo = _nhwc(dout)[4]
    dx = new_act(n, h, w, c, x.device)
    dsig = torch.empty((n, h, w), dtype=torch.float32, device=x.device)
    sums1 = zeros_scratch((2,), torch.float64, x.device)
    call("b2_gate_apply_bwd", _p(dout), lddo, _p(x), ldx, _p(psi), _p(q), n * h * w, c, _p(coef1[0]),
         _p(coef1[1]), _p(dx), c, _p(dsig), _p(sums1), _stream())
    return dx, dsig, sums1


def _gate_coef(coef_g, gamma_g, coef_x, gamma_x, coef1, gamma1, wpsi):
    k = GateCoef()
    k.scale_g, k.shift_g, k.mean_g, k.invstd_g = (coef_g[2].data_ptr(), coef_g[3].data_ptr(), coef_g[0].data_ptr(),
                                                  coef_g[1].data_ptr())
    k.gamma_g = gamma_g.data_ptr()
    k.scale_x, k.shift_x, k.mean_x, k.invstd_x = (coef_x[2].data_ptr(), coef_x[3].data_ptr(), coef_x[0].data_ptr(),
                                                  coef_x[1].data_ptr())
    k.gamma_x = gamma_x.data_ptr()
    k.gamma1, k.mean1, k.invstd1 = gamma1.data_ptr(), coef1[0].data_ptr(), coef1[1].data_ptr()
    k.wpsi = wpsi.data_ptr()
    return k


def gate_psi_bwd(dsig, sums1, q, g1p, x1p, coef_g, gamma_g, coef_x, gamma_x, coef1, gamma1, wpsi, training=True):
    """-> dg1p, dx1p (bf16), dgb fp32 [4, fint] (dgamma_g, dbeta_g, dgamma_x, dbeta_x), dbn1 fp32 [2],
    dwpsi fp32 [fint], dbpsi fp32 [1]"""
    n, h, w, fint, ld = _nhwc(g1p)
    npix = n * h * w
    dev = g1p.device
    k = _gate_coef(coef_g, gamma_g, coef_x, gamma_x, coef1, gamma1, wpsi)
    sums = zeros_scratch((4, fint), torch.float64, dev)
    dwpsi = torch.zeros((fint,), dtype=torch.float32, device=dev)   # (one pool slice per custom op at most: the outputs
    dbpsi = torch.zeros((1,), dtype=torch.float32, device=dev)      # of an op may not share a storage)
    call("b2_gate_psi_bwd_reduce", _p(dsig), _p(q), _p(g1p), _p(x1p), ld, npix, fint, C.byref(k), _p(sums1),
         int(training), _p(sums), _p(dwpsi), _p(dbpsi), _stream())
    dg1p = new_act(n, h, w, fint, dev)
    dx1p = new_act(n, h, w, fint, dev)
    dgb = torch.empty((4, fint), dtype=torch.float32, device=dev)
    dbn1 = torch.empty((2,), dtype=torch.float32, device=dev)
    dbias = zeros_out((2, fint), torch.float32, dev)     # bias grads of the W_g / W_x convs
    assert ld == fint
    call("b2_gate_psi_bwd_apply", _p(dsig), _p(q), _p(g1p), _p(x1p), ld, npix, fint, C.byref(k), _p(sums1),
         int(training), _p(sums), _p(dg1p), _p(dx1p), _p(dgb), _p(dbn1), _p(dbias), _stream())
    return dg1p, dx1p, dgb, dbn1, dwpsi, dbpsi, dbias


# ----------------------------------------------------------------------------------------------------------
# loss
# ----------------------------------------------------------------------------------------------------------
def loss_fwd(z, t, w_bce=1.0, w_dice=0.0, smooth=1.0):
    assert z.dtype == torch.float32 and t.dtype == torch.float32 and z.is_contiguous() and t.is_contiguous()
    assert z.numel() == t.numel()
    sums = zeros_out((6,), torch.float64, z.device)   # an output of seg_loss the caller may keep: not arena memory
    loss = torch.empty((), dtype=torch.float32, device=z.device)
    call("b2_loss_fwd", _p(z), _p(t), z.numel(), _p(sums), _stream())
    call("b2_loss_finalize", _p(sums), z.numel(), float(w_bce), float(w_dice), float(smooth), _p(loss), _stream())
    return loss, sums


def _thr_logit(threshold):
    import math
    if threshold <= 0.0:
        return -float("inf")
    if threshold >= 1.0:
        return float("inf")
    return math.log(threshold / (1.0 - threshold))


def seg_counts(z, t, threshold=0.5, probabilities=False):
    """[N, ...] fp32 logits (or probabilities) / targets -> int64 [N, 3] = (TP, #pred, #target) per sample
    (b2_seg_counts); pred = sigmoid(z) > threshold, evaluated as z > logit(threshold)."""
    assert z.dtype == torch.float32 and t.dtype == torch.float32 and z.is_contiguous() and t.is_contiguous()
    assert z.shape == t.shape and z.dim() >= 2
    n = z.shape[0]
    counts = torch.empty((n, 3), dtype=torch.int64, device=z.device)
    thr = float(threshold) if probabilities else _thr_logit(threshold)
    call("b2_seg_counts", _p(z), _p(t), n, z.numel() // n, thr, float(threshold), _p(counts), _stream())
    return counts


def logits_to_mask(z, threshold=0.5):
    """fp32 logits -> uint8 {0, 255} mask of the same shape (b2_logits_to_mask)."""
    assert z.dtype == torch.float32 and z.is_contiguous()
    mask = torch.empty(z.shape, dtype=torch.uint8, device=z.device)
    call("b2_logits_to_mask", _p(z), z.numel(), _thr_logit(threshold), _p(mask), _stream())
    return mask


def loss_bwd(z, t, sums, grad_out, w_bce=1.0, w_dice=0.0, smooth=1.0):
    dz = torch.empty_like(z)
    call("b2_loss_bwd", _p(z), _p(t), z.numel(), _p(sums), float(w_bce), float(w_dice), float(smooth),
         _p(grad_out), _p(dz), _stream())
    return dz


# ----------------------------------------------------------------------------------------------------------
# multi-class: softmax cross-entropy + soft Dice, per-class counts, argmax label map (csrc/loss_mc.cu)
# ----------------------------------------------------------------------------------------------------------
MAX_CLASSES = 8


def ce_nsums(k):
    """number of fp64 sums b2_ce_loss_fwd accumulates for k classes (B2_CE_NSUMS)"""
    return 3 + 5 * k


def ce_sums_fields(sums, k):
    """named views of the b2_ce_loss_fwd sums (layout: include/b200seg.h, B2_CE_*)"""
    return {"loss": sums[0], "wsum": sums[1], "pt": sums[2:2 + k], "p": sums[2 + k:2 + 2 * k],
            "t": sums[2 + 2 * k:2 + 3 * k], "inter": sums[2 + 3 * k:2 + 4 * k], "union": sums[2 + 4 * k:2 + 5 * k],
            "invalid": sums[2 + 5 * k]}


def _mc_args(z, labels):
    """(n, k, hw, label_bytes) of fp32 NCHW logits [N, K, H, W] and uint8 / int64 labels [N, H, W] or [N, 1, H, W]"""
    assert z.dtype == torch.float32 and z.is_contiguous() and z.dim() == 4 and z.is_cuda, (z.dtype, z.shape)
    n, k, h, w = z.shape
    if not 2 <= k <= MAX_CLASSES:
        raise ValueError(f"multi-class kernels take 2..{MAX_CLASSES} classes, the logits have {k} channels")
    if labels.dtype not in (torch.uint8, torch.int64):
        raise TypeError(f"labels must be uint8 or int64 class indices, got {labels.dtype}")
    if labels.numel() != n * h * w or labels.shape[0] != n or labels.shape[-2:] != (h, w):
        raise ValueError(f"labels {tuple(labels.shape)} do not match logits {tuple(z.shape)}")
    assert labels.is_contiguous() and labels.device == z.device
    return n, k, h * w, labels.element_size()


def _mc_weight(weight, z, k):
    """the class-weight vector the kernels read with device loads: fp32, contiguous, K entries, on the logits' device"""
    if weight is None:
        return
    if weight.device != z.device:
        raise ValueError(f"class weight is on {weight.device}, the logits on {z.device}")
    if weight.dtype != torch.float32 or not weight.is_contiguous() or weight.numel() != k:
        raise ValueError(f"class weight must be a contiguous fp32 vector of {k} entries, got {weight.dtype} "
                         f"{tuple(weight.shape)}")


def ce_loss_fwd(z, labels, weight=None, ignore_index=-100, w_ce=1.0, w_dice=0.0, smooth=1.0):
    """-> (loss fp32 scalar, sums fp64 [3 + 5K]); loss is NaN when a label is outside [0, K) and not ignore_index, or
    when no pixel is valid"""
    n, k, hw, lb = _mc_args(z, labels)
    _mc_weight(weight, z, k)
    sums = zeros_out((ce_nsums(k),), torch.float64, z.device)   # an output of seg_loss_ce: not arena memory
    loss = torch.empty((), dtype=torch.float32, device=z.device)
    call("b2_ce_loss_fwd", _p(z), _p(labels), lb, n, k, hw, _p(weight), int(ignore_index), _p(sums), _stream())
    call("b2_ce_loss_finalize", _p(sums), k, float(w_ce), float(w_dice), float(smooth), _p(loss), _stream())
    return loss, sums


def ce_loss_bwd(z, labels, weight, ignore_index, sums, grad_out, w_ce=1.0, w_dice=0.0, smooth=1.0):
    n, k, hw, lb = _mc_args(z, labels)
    _mc_weight(weight, z, k)
    assert sums.dtype == torch.float64 and sums.numel() == ce_nsums(k) and sums.device == z.device
    assert grad_out is None or (grad_out.dtype == torch.float32 and grad_out.device == z.device)
    dz = torch.empty_like(z)
    call("b2_ce_loss_bwd", _p(z), _p(labels), lb, n, k, hw, _p(weight), int(ignore_index), _p(sums), float(w_ce),
         float(w_dice), float(smooth), _p(grad_out), _p(dz), _stream())
    return dz


def seg_counts_mc(z, labels, ignore_index=-100):
    """fp32 logits [N, K, H, W] + labels -> int64 [N, K, 3] = (TP, #pred, #target) per sample and class, pred = argmax"""
    n, k, hw, lb = _mc_args(z, labels)
    counts = torch.empty((n, k, 3), dtype=torch.int64, device=z.device)
    call("b2_seg_counts_mc", _p(z), _p(labels), lb, n, k, hw, int(ignore_index), _p(counts), _stream())
    return counts


def logits_to_labels(z):
    """fp32 logits [N, K, H, W] -> uint8 label map [N, H, W] (argmax, first maximum on ties)"""
    assert z.dtype == torch.float32 and z.is_contiguous() and z.dim() == 4 and z.is_cuda
    n, k, h, w = z.shape
    if not 2 <= k <= MAX_CLASSES:
        raise ValueError(f"multi-class kernels take 2..{MAX_CLASSES} classes, the logits have {k} channels")
    out = torch.empty((n, h, w), dtype=torch.uint8, device=z.device)
    call("b2_logits_to_labels", _p(z), n, k, h * w, _p(out), _stream())
    return out
