"""The fast training step as a package component (what bench.py times and utils.helpers.train() runs):

  GraphedTrainStep   zero_grad -> forward -> loss -> backward -> (bucketed all-reduce) -> clip + AdamW, the body of the
                     reference's hot loop (utils/helpers.py:317-337), captured ONCE per batch shape in a CUDA graph and
                     replayed: ~600 kernel launches per AttU_Net step cost no Python / launch overhead any more.
  PinnedPrefetcher   the other half of the reference's loop, `x, y = x.to(device, non_blocking=True), ...`
                     (helpers.py:318): batches are staged in pinned host memory and copied on a copy stream into
                     double-buffered device slots while the previous step computes.

Both are plain PyTorch plumbing (streams, events, graphs); every kernel inside the step is libb200seg's.
"""
from __future__ import annotations

from typing import Callable, Dict, Optional, Tuple

import torch

from . import kernels as K
from . import ops


class GraphedTrainStep:
    """step(x, t) -> loss (a device scalar, valid until the next call).

    The first `warmup` calls for a batch shape run eagerly (they are real training steps: the caching allocator, the
    autograd stream bindings and the optimizer's pointer table settle); the next call captures the step into a CUDA
    graph with static input buffers and every later call of that shape is one graph replay.  At most `max_graphs`
    shapes are captured (a ragged last batch gets its own graph; further shapes stay eager); all graphs share one
    memory pool.  Everything runs on one private non-default stream — AccumulateGrad nodes bind to the stream of their
    first use, so the eager warm-up, the capture and the replays must not hop streams.

    `loss_weights` = (w_bce, w_dice, smooth) of b200seg::seg_loss (BCEWithLogits = (1, 0, 1), helpers.py:245;
    CombinedLoss = (0.5, 0.5, 1), clip_seg_finetuner.py:61-74).
    `loss="ce"`: multi-class training on K >= 2 logit channels and integer label maps (uint8 / int64 [N, H, W]) through
    b200seg::seg_loss_ce; `loss_weights` then means (w_ce, w_dice, smooth), `class_weight` (K floats) and
    `ignore_index` have nn.CrossEntropyLoss's meaning.
    """

    def __init__(self, model: torch.nn.Module, optimizer, reducer=None, loss_weights=(1.0, 0.0, 1.0), graph: bool = True,
                 warmup: int = 3, max_graphs: int = 2, wgrad_overlap: Optional[bool] = None,
                 clip_fn: Optional[Callable[[], None]] = None, loss: str = "bce", class_weight=None,
                 ignore_index: int = -100):
        if loss not in ("bce", "ce"):
            raise ValueError(f"loss must be 'bce' or 'ce', got {loss!r}")
        self.model, self.optimizer, self.reducer = model, optimizer, reducer
        self.loss_weights = tuple(float(v) for v in loss_weights)
        self.loss = loss
        self.ignore_index = int(ignore_index)
        self.use_graph = bool(graph)
        self.warmup = max(int(warmup), 1)
        self.max_graphs = int(max_graphs)
        self.wgrad_overlap = wgrad_overlap
        self.clip_fn = clip_fn                      # for non-fused optimizers: called between backward and step
        self.device = next(model.parameters()).device
        self.class_weight = None if class_weight is None else \
            torch.as_tensor(class_weight, dtype=torch.float32).to(self.device).contiguous()
        self.stream = torch.cuda.Stream(device=self.device)
        self._seen: Dict[Tuple, int] = {}
        self._graphs: Dict[Tuple, Tuple] = {}       # shape key -> (graph, x_static, t_static, loss_static, launches)
        self._pool = None
        self.replays = 0
        self.eager_steps = 0
        self.capture_error: Optional[str] = None

    # -- one eager step on the current stream --------------------------------------------------------------
    def _step(self, x, t):
        self.optimizer.zero_grad(set_to_none=True)
        K.step_begin()
        with K.deferred_running_updates():          # the BatchNorm running-statistics updates of the forward: one launch
            logits = self.model(x)
        if logits.dim() == 3:
            logits = logits.unsqueeze(1)            # helpers.py:323-324
        if self.loss == "ce":
            loss, _sums = ops.seg_loss_ce(logits, t, self.class_weight, self.ignore_index, *self.loss_weights)
        else:
            loss, _sums = ops.seg_loss(logits, t, *self.loss_weights)
        loss.backward()
        if self.reducer is not None:
            self.reducer.finish()
        if self.clip_fn is not None:
            self.clip_fn()
        self.optimizer.step()
        return loss

    def _sync_lr(self):
        sync = getattr(self.optimizer, "sync_lr", None)
        if sync is not None:
            sync()                                   # scheduler updates reach the device scalar the graph reads

    def graph_for(self, x, t):
        return self._graphs.get((tuple(x.shape), tuple(t.shape)))

    @property
    def launches_per_replay(self):
        return {k: v[4] for k, v in self._graphs.items()}

    def __call__(self, x: torch.Tensor, t: torch.Tensor, inputs_are_static: bool = False) -> torch.Tensor:
        """`inputs_are_static`: x / t ARE the graph's static buffers (see static_inputs) — skip the device copy."""
        key = (tuple(x.shape), tuple(t.shape))
        cur = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(cur)
        prev_overlap = K.wgrad_overlap_enabled()
        if self.wgrad_overlap is not None:
            K.set_wgrad_overlap(self.wgrad_overlap)
        try:
            with torch.cuda.stream(self.stream):
                entry = self._graphs.get(key)
                if entry is None and self.use_graph and self.capture_error is None \
                        and self._seen.get(key, 0) >= self.warmup and len(self._graphs) < self.max_graphs:
                    entry = self._capture(key, x, t)
                if entry is not None:
                    graph, xs, ts, loss_s, _n = entry
                    if not inputs_are_static:
                        xs.copy_(x, non_blocking=True)
                        ts.copy_(t, non_blocking=True)
                    self._sync_lr()
                    graph.replay()
                    K.bump_param_epoch()             # the replayed optimizer step rewrote the parameters
                    self.replays += 1
                    loss = loss_s
                else:
                    self._sync_lr()
                    loss = self._step(x, t)
                    self._seen[key] = self._seen.get(key, 0) + 1
                    self.eager_steps += 1
                    x.record_stream(self.stream)
                    t.record_stream(self.stream)
        finally:
            if self.wgrad_overlap is not None:
                K.set_wgrad_overlap(prev_overlap)
        cur.wait_stream(self.stream)
        return loss

    def _capture(self, key, x, t):
        from . import _lib
        xs, ts = torch.empty_like(x), torch.empty_like(t)
        xs.copy_(x)
        ts.copy_(t)
        self.optimizer.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()
        try:
            before = _lib.launch_count
            kwargs = {"pool": self._pool} if self._pool is not None else {}
            with torch.cuda.graph(graph, stream=self.stream, **kwargs):
                loss_s = self._step(xs, ts)
            launches = _lib.launch_count - before
        except Exception as e:      # keep training eagerly if capture is refused (e.g. an op that syncs)
            self.capture_error = f"{type(e).__name__}: {e}"
            torch.cuda.synchronize(self.device)
            return None
        if self._pool is None:
            self._pool = graph.pool()
        entry = (graph, xs, ts, loss_s, launches)
        self._graphs[key] = entry
        return entry

    def static_inputs(self, x_shape, t_shape):
        """the captured graph's input buffers for this shape (None before capture): a prefetcher may copy straight
        into them and call step(xs, ts, inputs_are_static=True)"""
        e = self._graphs.get((tuple(x_shape), tuple(t_shape)))
        return (e[1], e[2]) if e is not None else None


class PinnedPrefetcher:
    """Iterate a loader of (x, y) CPU batches as device batches: pinned staging + asynchronous H2D on a copy stream,
    two device slots per shape, the copy of batch i+1 overlapping the compute of batch i (SURVEY.md §8f N4; reference:
    DataLoader(pin_memory=True) + .to(device, non_blocking=True), utils/trainer.py:153-160, utils/helpers.py:318).

    Yields (x_dev, y_dev); the tensors stay valid until the SECOND next batch is requested."""

    def __init__(self, loader, device, depth: int = 2, device_transform=None):
        """device_transform(x_dev, y_dev) -> (x, y): applied on the consumer's stream when a batch is handed out, e.g.
        data.GpuSegAugment turning raw uint8 image / mask batches into normalised fp32 tensors on the device"""
        self.loader, self.device, self.depth = loader, torch.device(device), max(int(depth), 2)
        self.device_transform = device_transform
        self.copy_stream = torch.cuda.Stream(device=self.device)
        self._pinned: Dict[Tuple, list] = {}
        self._slots: Dict[Tuple, list] = {}
        self._turn: Dict[Tuple, int] = {}
        self._hold: Dict[Tuple, list] = {}
        self.h2d_bytes = 0

    def __len__(self):
        return len(self.loader)

    @property
    def dataset(self):
        return self.loader.dataset

    def _stage(self, x, y):
        key = (tuple(x.shape), x.dtype, tuple(y.shape), y.dtype)
        if key not in self._slots:
            self._pinned[key] = [(torch.empty(x.shape, dtype=x.dtype).pin_memory(),
                                  torch.empty(y.shape, dtype=y.dtype).pin_memory()) for _ in range(self.depth)]
            self._slots[key] = [(torch.empty(x.shape, dtype=x.dtype, device=self.device),
                                 torch.empty(y.shape, dtype=y.dtype, device=self.device), torch.cuda.Event(),
                                 torch.cuda.Event()) for _ in range(self.depth)]
            self._turn[key] = 0
            self._hold[key] = [None] * self.depth
        i = self._turn[key]
        self._turn[key] = (i + 1) % self.depth
        xd, yd, ready, consumed = self._slots[key][i]
        if x.is_pinned() and y.is_pinned():       # DataLoader(pin_memory=True): copy straight out of the batch
            px, py = x, y
            self._hold[key][i] = (x, y)           # keep the source alive until its H2D has run
        else:
            px, py = self._pinned[key][i]
            ready.synchronize()                   # the previous H2D out of this pinned pair has finished
            px.copy_(x)
            py.copy_(y)
        self.copy_stream.wait_event(consumed)     # the slot's previous consumer is done with it
        with torch.cuda.stream(self.copy_stream):
            xd.copy_(px, non_blocking=True)
            yd.copy_(py, non_blocking=True)
            ready.record(self.copy_stream)
        self.h2d_bytes += x.numel() * x.element_size() + y.numel() * y.element_size()
        return xd, yd, ready, consumed

    def __iter__(self):
        it = iter(self.loader)
        nxt = None
        try:
            x, y = next(it)
        except StopIteration:
            return
        if x.is_cuda:                             # already on the device: nothing to stage
            yield x, y
            yield from it
            return
        nxt = self._stage(x, y)
        while nxt is not None:
            xd, yd, ready, consumed = nxt
            try:
                x, y = next(it)
                following = self._stage(x, y)     # issue the next copy before handing out the current batch
            except StopIteration:
                following = None
            torch.cuda.current_stream(self.device).wait_event(ready)
            if self.device_transform is not None:
                yield self.device_transform(xd, yd)
            else:
                yield xd, yd
            consumed.record(torch.cuda.current_stream(self.device))
            nxt = following
