"""Mirror of the segmentation half of the reference's utils/tester.py (metrics :92-193, test loop :249-312) on the
b200seg kernels: same function names, argument meaning, printed report and returned dict.

The reference evaluates every sample with ~10 tensor reductions and 8 `.item()` host syncs
(calculate_segmentation_metrics, tester.py:158-193).  Here one launch of b2_seg_counts per batch yields the three
integers per sample that all six metrics are functions of — TP, #pred, #target — and the metrics are evaluated from
them on the device in fp64 with the reference's 1e-7 guards; the test loop syncs with the host once, at the end.
Classification / CLIP / CLIPSeg testers are outside the hot path (SURVEY.md section 8) and are not mirrored.
"""
from __future__ import annotations

import torch

from .. import kernels as K

METRIC_KEYS = ("iou", "dice", "pixel_accuracy", "precision", "recall", "f1")


def segmentation_counts(logits, target, threshold=0.5, probabilities=False):
    """[N,1,H,W] (or [N,H,W]) logits and targets -> int64 [N,3] = (TP, #pred, #target), one kernel launch."""
    z = logits.detach().float().contiguous()
    t = target.detach().float().contiguous()
    if z.dim() == 1:
        z, t = z[None], t[None]
    return K.seg_counts(z, t, threshold, probabilities=probabilities)


def metrics_from_counts(counts, per_sample):
    """(TP, #pred, #target) per sample -> dict of fp64 [N] tensors in percent, tester.py:92-193 term by term."""
    c = counts.double()
    tp, npred, ntgt = c[:, 0], c[:, 1], c[:, 2]
    fp = npred - tp
    fn = ntgt - tp
    union = npred + ntgt - tp
    eps = 1e-7
    iou = (tp + eps) / (union + eps)                              # calculate_iou
    dice = (2.0 * tp + eps) / (npred + ntgt + eps)                # calculate_dice
    pix = (per_sample - fp - fn) / per_sample                     # calculate_pixel_accuracy: pred == target
    precision = (tp + eps) / (tp + fp + eps)
    recall = (tp + eps) / (tp + fn + eps)
    f1 = 2 * (precision * recall) / (precision + recall + eps)
    vals = (iou, dice, pix, precision, recall, f1)
    return {k: v * 100 for k, v in zip(METRIC_KEYS, vals)}


# per-class keys of the multi-class report: f"{key}_c{k}" for every class k
CLASS_METRIC_KEYS = ("iou", "dice", "precision", "recall", "f1")


def metrics_from_counts_mc(counts):
    """int64 [N, K, 3] = (TP, #pred, #target) per sample and class (kernels.seg_counts_mc) -> dict of fp64 tensors in
    percent: per-class [N, K] entries for CLASS_METRIC_KEYS and the per-sample pixel accuracy [N] = sum TP / #valid
    pixels; the reference's 1e-7 guards, so a class absent from both prediction and label scores 100"""
    c = counts.double()
    tp, npred, ntgt = c[..., 0], c[..., 1], c[..., 2]
    eps = 1e-7
    iou = (tp + eps) / (npred + ntgt - tp + eps)
    dice = (2.0 * tp + eps) / (npred + ntgt + eps)
    precision = (tp + eps) / (npred + eps)
    recall = (tp + eps) / (ntgt + eps)
    f1 = 2 * (precision * recall) / (precision + recall + eps)
    out = {k: v * 100 for k, v in zip(CLASS_METRIC_KEYS, (iou, dice, precision, recall, f1))}
    out["pixel_accuracy"] = tp.sum(1) / ntgt.sum(1).clamp_min(1) * 100
    return out


def _single(pred, target, threshold):
    p = pred.detach().float().reshape(1, -1).contiguous()
    t = target.detach().float().reshape(1, -1).contiguous()
    m = metrics_from_counts(K.seg_counts(p, t, threshold, probabilities=True), p.shape[1])
    return {k: float(v[0]) for k, v in m.items()}


def calculate_iou(pred, target, threshold=0.5):
    """tester.py:92-111 — pred holds probabilities (after sigmoid); returns a fraction, like the reference."""
    return _single(pred, target, threshold)["iou"] / 100


def calculate_dice(pred, target, threshold=0.5):
    """tester.py:114-134"""
    return _single(pred, target, threshold)["dice"] / 100


def calculate_pixel_accuracy(pred, target, threshold=0.5):
    """tester.py:137-155"""
    return _single(pred, target, threshold)["pixel_accuracy"] / 100


def calculate_segmentation_metrics(pred, target, threshold=0.5):
    """tester.py:158-193 — one sample, values in percent."""
    return _single(pred, target, threshold)


def test_segmentation_model(model, test_loader, device, model_name, log=print, ignore_index=-100):
    """tester.py:249-312: average of the per-sample metrics over the test set.

    Multi-class: when the masks are integer label maps and the model returns K >= 2 channels, pred = argmax and the
    metrics are counted per sample and class (kernels.seg_counts_mc; `ignore_index` pixels excluded).  The six keys are
    then the means over the foreground classes 1..K-1 (pixel accuracy: sum TP / valid pixels), and f"{key}_c{k}" holds
    each class's own average."""
    model.eval()
    device = torch.device(device)
    totals = None
    multiclass = None                                        # which counting the first batch selected
    num_samples = 0
    log(f"\n{'=' * 60}")
    log(f"Testing Segmentation Model: {model_name}")
    log(f"{'=' * 60}")
    with torch.no_grad():
        for images, masks in test_loader:
            images = images.to(device, non_blocking=True)
            masks = masks.to(device, non_blocking=True)
            outputs = model(images)
            if outputs.dim() == 3:
                outputs = outputs.unsqueeze(1)
            batch_mc = outputs.shape[1] >= 2 and not masks.is_floating_point()
            if multiclass is None:
                multiclass = batch_mc
            elif batch_mc != multiclass:
                raise ValueError("test loader mixes integer label maps and float masks")
            if batch_mc:
                z = outputs.detach().float().contiguous()
                m = metrics_from_counts_mc(K.seg_counts_mc(z, masks.contiguous(), ignore_index))
                batch = torch.cat([m["pixel_accuracy"].sum().view(1)] + [m[k].sum(0) for k in CLASS_METRIC_KEYS])
            else:
                counts = segmentation_counts(outputs, masks.reshape(outputs.shape), 0.5)
                m = metrics_from_counts(counts, outputs[0].numel())
                batch = torch.stack([m[k].sum() for k in METRIC_KEYS])
            if totals is None:
                totals = torch.zeros_like(batch)
            totals += batch
            num_samples += outputs.size(0)
    if totals is None:
        totals = torch.zeros(len(METRIC_KEYS), dtype=torch.float64, device=device)
    avg = (totals / max(num_samples, 1)).tolist()            # the only host sync
    if not multiclass:
        avg_metrics = dict(zip(METRIC_KEYS, avg))
    else:                                                    # [pixel accuracy, then K values per class metric]
        ncls = (len(avg) - 1) // len(CLASS_METRIC_KEYS)
        per_class = {key: avg[1 + i * ncls:1 + (i + 1) * ncls] for i, key in enumerate(CLASS_METRIC_KEYS)}
        avg_metrics = {key: sum(v[1:]) / (ncls - 1) for key, v in per_class.items()}
        avg_metrics["pixel_accuracy"] = avg[0]
        avg_metrics = {key: avg_metrics[key] for key in METRIC_KEYS}
        for key, v in per_class.items():
            avg_metrics.update({f"{key}_c{k}": v[k] for k in range(ncls)})
    log(f"\n{model_name} Test Results:")
    log(f"{'-' * 60}")
    log(f"IoU (Jaccard):     {avg_metrics['iou']:.2f}%")
    log(f"Dice Coefficient:  {avg_metrics['dice']:.2f}%")
    log(f"Pixel Accuracy:    {avg_metrics['pixel_accuracy']:.2f}%")
    log(f"Precision:         {avg_metrics['precision']:.2f}%")
    log(f"Recall:            {avg_metrics['recall']:.2f}%")
    log(f"F1 Score:          {avg_metrics['f1']:.2f}%")
    log(f"{'=' * 60}\n")
    return avg_metrics


test_segmentation_model.__test__ = False      # not a pytest test


def predict_mask(model, img_tensor, threshold=0.5, precision=None):
    """pipeline.py:340-357 (_predict_segmentation, U-Net branch): logits -> uint8 {0,255} mask on the host.
    `img_tensor`: [1,3,H,W] (or [N,3,H,W]) normalised image; returns a numpy array [H,W] (or [N,H,W]).
    precision="fp32": run the fp32 parity mode (ops_fp32.py) — the reference computes this path in fp32, and its masks
    are reproduced bit for bit only at that precision; None: whatever b200seg.get_precision() says (default bf16)."""
    import contextlib
    from .. import ops_fp32
    model.eval()
    dev = next(model.parameters()).device
    with torch.no_grad(), (ops_fp32.precision(precision) if precision else contextlib.nullcontext()):
        logits = model(img_tensor.to(dev)).float().contiguous()
        mask = K.logits_to_mask(logits, threshold)
    mask = mask.cpu()
    if mask.dim() == 4 and mask.shape[1] == 1:
        mask = mask[:, 0]
    if mask.shape[0] == 1:
        mask = mask[0]
    return mask.numpy()


def predict_labels(model, img_tensor, precision=None):
    """Multi-class counterpart of predict_mask: logits [N, K, H, W] (K >= 2) -> uint8 label map = argmax over the
    classes (first maximum on ties, as torch.argmax) on the host; [H, W] for one image, [N, H, W] otherwise.
    precision="fp32": the fp32 parity mode (ops_fp32.py); None: b200seg.get_precision()."""
    import contextlib
    from .. import ops_fp32
    model.eval()
    dev = next(model.parameters()).device
    with torch.no_grad(), (ops_fp32.precision(precision) if precision else contextlib.nullcontext()):
        logits = model(img_tensor.to(dev)).float().contiguous()
        labels = K.logits_to_labels(logits)
    labels = labels.cpu()
    if labels.shape[0] == 1:
        labels = labels[0]
    return labels.numpy()
