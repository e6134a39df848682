"""Mirror of the segmentation half of the reference's utils/helpers.py: get_seg_model / iou / train with the same
names, argument meaning, prints, checkpoint names and return value, driving the b200seg modules.

Differences from the reference, all forced by the B200 path and listed in DESIGN.md:
  * compute precision is bf16 inside the kernels, so the fp16 GradScaler of helpers.py:285 is not needed (bf16 has
    fp32's exponent range); the autocast context is not used either — the modules always run bf16;
  * the loss is the fused b200seg::seg_loss op (BCEWithLogits, helpers.py:245), which also yields the IoU counts,
    so validation does not launch per-sample reductions (iou() below is kept for API compatibility);
  * only `seg=True` is supported (the classification branch, helpers.py:257-283, is outside the hot path);
  * the training step (zero_grad .. optimizer.step, helpers.py:317-337) is captured once per batch shape in a CUDA graph
    and replayed (engine.GraphedTrainStep; B200SEG_TRAIN_GRAPH=0 launches eagerly), and CPU batches are staged through
    pinned memory and copied on a copy stream while the previous step computes (engine.PinnedPrefetcher);
  * B200SEG_TRAIN_LOG=<file> appends one JSON line per epoch (losses, IoU, images/s of the training loop, graph
    replays) next to the reference's per-epoch print (SURVEY.md §5, metrics / logging);
  * train(loss="ce" | "ce+dice") trains K >= 2 mutually exclusive classes on integer label maps with the fused
    b200seg::seg_loss_ce op (softmax cross-entropy, + soft Dice over the foreground classes for "ce+dice").
"""
from __future__ import annotations

import json
import os
import time

import torch

from .. import ops


def get_seg_model(name):
    """helpers.py:195-213 — same names, default constructors (=> t=5 for the R2 models, frozen ResNet encoder)."""
    from ..models.segmentation_models import AttentionUNet, R2AttU_Net, R2U_Net

    name_lower = name.lower()
    if name_lower == "resnetunet":
        from ..models.segmentation_models import ResnetUnet
        return ResnetUnet.ResNetUnet()
    elif name_lower == "attentionunet":
        return AttentionUNet()
    elif name_lower == "r2unet":
        return R2U_Net()
    elif name_lower == "r2attunet":
        return R2AttU_Net()
    raise ValueError(f"Unknown segmentation model: {name}")


def iou(pred, mask, t=0.5):
    """helpers.py:223-227 (host-syncing, per call) — kept for drop-in use; train() uses the fused counts."""
    p = (pred > t).float()
    inter = (p * mask).sum()
    union = ((p + mask) > 0).float().sum()
    return (inter / (union + 1e-7)).item()


def _dataset_len(dl, fallback):
    """len(dl.dataset) as the reference divides by (helpers.py:361,367); `fallback` for loaders without a dataset"""
    try:
        return len(dl.dataset)
    except (AttributeError, TypeError):
        return fallback


# multi-class loss modes -> (w_ce, w_dice, smooth) of b200seg::seg_loss_ce; "ce+dice" weighs like CombinedLoss
_CE_MODES = {"ce": (1.0, 0.0, 1.0), "ce+dice": (0.5, 0.5, 1.0)}


def train(model, train_dl, val_dl, device, epochs, lr, name, save_dir, seg=False, cls_head_name=None,
          reducer=None, log=print, loss="bce", class_weight=None, ignore_index=-100):
    """helpers.py:231-412, segmentation branch.  Returns the best validation loss.

    loss="bce" (default) is the reference's BCEWithLogits on one mask channel.  "ce" / "ce+dice" train the model's K >= 2
    output channels as mutually exclusive classes on integer label maps (uint8 / int64 [N, H, W]; `class_weight` and
    `ignore_index` as in nn.CrossEntropyLoss); the printed IoU is then the mean over the foreground classes 1..K-1 of
    inter / union per validation batch."""
    if not seg:
        raise NotImplementedError("b200seg.train covers the segmentation path only (seg=True)")
    if loss != "bce" and loss not in _CE_MODES:
        raise ValueError(f"loss must be 'bce', 'ce' or 'ce+dice', got {loss!r}")
    device = torch.device(device)
    model = model.to(device, memory_format=torch.channels_last)            # helpers.py:243
    from .. import kernels as K
    from ..optim import FusedClipAdamW
    # weight gradients on a side stream: safe here because gradients are only read after backward() (reducer.finish /
    # optimizer.step), parameters are channels_last and zero_grad(set_to_none=True) is used
    overlap_before = K.wgrad_overlap_enabled()
    K.set_wgrad_overlap(device.type == "cuda" and os.environ.get("B200SEG_WGRAD_OVERLAP", "1") != "0")
    optimizer = FusedClipAdamW(model.parameters(), lr=lr, weight_decay=5e-4, max_norm=1.0)   # helpers.py:251,333
    log(f"Training Segmentation model (all layers unfrozen) with LR: {lr}")
    scheduler = torch.optim.lr_scheduler.CosineAnnealingLR(optimizer, T_max=epochs)   # helpers.py:254
    best_score = float("inf")
    patience, patience_counter = 10, 0
    from ..engine import GraphedTrainStep, PinnedPrefetcher
    on_gpu = device.type == "cuda"
    graph = on_gpu and os.environ.get("B200SEG_TRAIN_GRAPH", "1") != "0"
    if loss == "bce":
        stepper = GraphedTrainStep(model, optimizer, reducer=reducer, loss_weights=(1.0, 0.0, 1.0),  # helpers.py:245
                                   graph=graph)
    else:
        stepper = GraphedTrainStep(model, optimizer, reducer=reducer, loss_weights=_CE_MODES[loss], graph=graph,
                                   loss="ce", class_weight=class_weight, ignore_index=ignore_index)
    train.last_stepper = stepper          # introspection for tests / tools: replays, eager steps, capture errors
    start_time = time.time()

    try:
        for epoch in range(1, epochs + 1):
            model.train()
            running = torch.zeros((), dtype=torch.float64, device=device)     # no per-step .item() (helpers.py:337)
            seen = 0
            t_epoch = time.time()
            batches = PinnedPrefetcher(train_dl, device) if on_gpu else train_dl
            for x, y in batches:
                if not x.is_cuda:
                    x, y = x.to(device, non_blocking=True), y.to(device, non_blocking=True)
                # zero_grad -> forward -> BCEWithLogits -> backward -> (all-reduce) -> clip_grad_norm_(1.0) + AdamW,
                # replayed from a CUDA graph after the first few (eager) steps of each batch shape
                step_loss = stepper(x.float(), y.float()) if loss == "bce" else stepper(x.float(), y)
                running += step_loss.detach().double() * x.size(0)
                seen += x.size(0)
            running_sum = float(running)              # the epoch's one host sync of the training loop
            train_s = time.time() - t_epoch

            model.eval()
            val_loss = torch.zeros((), dtype=torch.float64, device=device)
            val_iou = torch.zeros((), dtype=torch.float64, device=device)
            n_val, n_batches = 0, 0
            with torch.no_grad():
                for x, y in val_dl:
                    x, y = x.to(device), y.to(device)
                    out = model(x)
                    if out.dim() == 3:
                        out = out.unsqueeze(1)
                    if loss == "bce":
                        vloss, sums = ops.seg_loss(out, y, 1.0, 0.0, 1.0)
                        val_loss += vloss.double() * x.size(0)
                        val_iou += sums[4] / (sums[5] + 1e-7)                 # helpers.py:223-227 per batch
                    else:
                        vloss, sums = ops.seg_loss_ce(out, y, stepper.class_weight, ignore_index, *_CE_MODES[loss])
                        val_loss += vloss.double() * x.size(0)
                        f = K.ce_sums_fields(sums, out.shape[1])
                        val_iou += (f["inter"][1:] / (f["union"][1:] + 1e-7)).mean()   # foreground classes
                    n_val += x.size(0)
                    n_batches += 1
            if reducer is not None:
                # data parallel: every rank must take the SAME improved / patience / early-stop decision (BatchNorm
                # running statistics are per rank, so local validation losses differ) — decide on the global means
                import torch.distributed as dist
                tot = torch.stack([val_loss, val_iou, torch.tensor(float(n_val), dtype=torch.float64, device=device),
                                   torch.tensor(float(n_batches), dtype=torch.float64, device=device)])
                dist.all_reduce(tot, group=reducer.group)
                val_loss, val_iou, n_val, n_batches = tot[0], tot[1], float(tot[2]), float(tot[3])
                n_train = seen                                   # per-rank shard: samples this rank saw
            else:
                # the reference divides by len(dataset) / len(loader) (helpers.py:361-367) — differs from the number of
                # samples seen when the loader drops the last batch
                n_val, n_batches = _dataset_len(val_dl, n_val), max(n_batches, 1)
                n_train = _dataset_len(train_dl, seen)
            val_loss = float(val_loss) / max(n_val, 1)
            val_iou_f = float(val_iou) / max(n_batches, 1)
            log(f"[{name}] Ep{epoch}: TrainLoss {running_sum / max(n_train, 1):.3f} | ValLoss {val_loss:.3f} | "
                f"IoU {val_iou_f:.3f}")
            log_path = os.environ.get("B200SEG_TRAIN_LOG")
            if log_path and (reducer is None or reducer.rank == 0):
                rec = {"name": name, "epoch": epoch, "train_loss": running_sum / max(n_train, 1), "val_loss": val_loss,
                       "iou": val_iou_f, "images": seen, "train_s": train_s, "images_per_s": seen / max(train_s, 1e-9),
                       "lr": optimizer.param_groups[0]["lr"], "graph_replays": stepper.replays,
                       "eager_steps": stepper.eager_steps, "world_size": 1 if reducer is None else reducer.world}
                with open(log_path, "a") as f:
                    f.write(json.dumps(rec) + "\n")
            improved = val_loss < best_score
            scheduler.step()
            if improved:
                best_score = val_loss
                patience_counter = 0
                if reducer is None or reducer.rank == 0:      # one writer (rank 0's replica, its own BN statistics)
                    os.makedirs(save_dir, exist_ok=True)
                    torch.save(model.state_dict(), os.path.join(save_dir, f"{name}_best_loss.pt"))   # helpers.py:394-400
            else:
                patience_counter += 1
            if patience_counter >= patience:
                log(f"Early stopping at epoch {epoch}. Best score: {best_score:.2f}")
                break
    finally:
        K.set_wgrad_overlap(overlap_before)
    log(f"Training for {name} finished in {(time.time() - start_time) / 60:.2f} minutes.")
    return best_score
