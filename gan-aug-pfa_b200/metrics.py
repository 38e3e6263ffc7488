"""Device-side evaluation metrics for the Siamese change-detection model (SURVEY.md §8f rank 3).

Mirrors ``calculate_metrics`` (evaluate.py:34-64) and the per-sample accumulation of ``evaluate_model``
(evaluate.py:129-210): the reference applies ``torch.sigmoid``, moves every prediction map to the CPU and thresholds it
there, one sample at a time.  Here one kernel (``gap_seg_confusion``) turns a batch of logits into per-sample
[TP, FP, FN, TN] counts on the GPU; only 4 integers per sample cross PCIe, and the ratios are formed from them with the
reference's formulas (fp32 arithmetic, ``smooth`` in the same places).

For the multi-class model (``SiameseUNet(n_channels, K)``, K = 2..16) ``gap_seg_confusion_ck`` forms a per-sample K x K
confusion matrix from the argmax over the class planes, and ``multiclass_metrics`` turns it into one-vs-rest
per-class ratios with the same formulas.
"""
from __future__ import annotations

from typing import Dict, List

import torch

from . import ops

METRIC_KEYS = ("accuracy", "precision", "recall", "f1", "iou")
MULTICLASS_KEYS = ("precision", "recall", "f1", "iou", "mean_iou", "accuracy")


def confusion_counts(logits: torch.Tensor, labels: torch.Tensor, out: torch.Tensor | None = None) -> torch.Tensor:
    """Per-sample int64 [n, 4] = [TP, FP, FN, TN] of ``sigmoid(logits) > 0.5`` against {0,1} ``labels`` (int64 [n,H,W]
    as the dataset yields them, or fp32).  ``out`` (zeroed by the caller) is accumulated into when given."""
    n = logits.shape[0]
    if out is None:
        out = torch.zeros(n, 4, device=logits.device, dtype=torch.int64)
    ops.seg_confusion(logits.contiguous(), labels.contiguous(), out)
    return out


def metrics_from_counts(tp, fp, fn, tn, smooth: float = 1e-6) -> Dict[str, float]:
    """The ratios of evaluate.py:47-64 from the four counts (fp32 arithmetic like the reference's tensors)."""
    f = torch.float32
    tp, fp, fn, tn = (torch.as_tensor(float(v), dtype=f) for v in (tp, fp, fn, tn))
    precision = (tp + smooth) / (tp + fp + smooth)
    recall = (tp + smooth) / (tp + fn + smooth)
    f1 = (2 * precision * recall + smooth) / (precision + recall + smooth)
    union = (tp + fp) + (tp + fn) - tp          # preds.sum() + targets.sum() - intersection
    iou = (tp + smooth) / (union + smooth)
    accuracy = (tp + tn + smooth) / (tp + tn + fp + fn + smooth)
    return {"accuracy": accuracy.item(), "precision": precision.item(), "recall": recall.item(), "f1": f1.item(),
            "iou": iou.item()}


def calculate_metrics(logits: torch.Tensor, targets: torch.Tensor, smooth: float = 1e-6) -> Dict[str, float]:
    """evaluate.py:34 for ONE sample or a whole flattened batch, from logits (the reference passes sigmoid(logits))."""
    c = confusion_counts(logits.reshape(1, -1), targets.reshape(1, -1)).cpu()[0]
    return metrics_from_counts(*c.tolist(), smooth=smooth)


def batch_metrics(logits: torch.Tensor, labels: torch.Tensor, smooth: float = 1e-6) -> List[Dict[str, float]]:
    """Per-sample metric dicts of a batch (the inner loop of evaluate.py:150-185) with one kernel and one small D2H."""
    c = confusion_counts(logits, labels).cpu()
    return [metrics_from_counts(*row.tolist(), smooth=smooth) for row in c]


def confusion_matrix(logits: torch.Tensor, labels: torch.Tensor, ignore_index: int = -100,
                     out: torch.Tensor | None = None) -> torch.Tensor:
    """Per-sample int64 [n, K, K] confusion matrices of ``logits.argmax(1)`` (fp32 class planes [n, K, h, w], ties to
    the lowest class) against int64 ``labels`` [n, h, w]: rows = label, columns = prediction.  Pixels labelled
    ``ignore_index`` or outside [0, K) are not counted.  ``out`` (zeroed by the caller) is accumulated into."""
    n, k = logits.shape[0], logits.shape[1]
    if out is None:
        out = torch.zeros(n, k, k, device=logits.device, dtype=torch.int64)
    ops.seg_confusion_ck(logits.contiguous(), labels.contiguous(), ignore_index, out)
    return out


def multiclass_metrics(counts, smooth: float = 1e-6) -> Dict[str, object]:
    """Per-class one-vs-rest precision / recall / F1 / IoU (lists of K floats) from a [K, K] confusion matrix (or a
    stack [n, K, K], which is summed first), with the formulas and ``smooth`` placement of ``metrics_from_counts``;
    plus ``mean_iou`` (the mean of the per-class IoU) and the overall pixel ``accuracy`` (trace / total, with smooth
    as in the binary accuracy)."""
    c = torch.as_tensor(counts).detach().cpu().to(torch.int64)
    if c.dim() == 3:
        c = c.sum(0)
    f = torch.float32
    tp = c.diagonal().to(f)
    fp = c.sum(0).to(f) - tp          # predicted as the class, labelled otherwise
    fn = c.sum(1).to(f) - tp          # labelled as the class, predicted otherwise
    precision = (tp + smooth) / (tp + fp + smooth)
    recall = (tp + smooth) / (tp + fn + smooth)
    f1 = (2 * precision * recall + smooth) / (precision + recall + smooth)
    union = (tp + fp) + (tp + fn) - tp
    iou = (tp + smooth) / (union + smooth)
    total = c.sum().to(f)
    accuracy = (tp.sum() + smooth) / (total + smooth)
    return {"precision": precision.tolist(), "recall": recall.tolist(), "f1": f1.tolist(), "iou": iou.tolist(),
            "mean_iou": float(iou.mean()), "accuracy": float(accuracy)}
