"""Change objects: connected-component labelling, minimum-area filtering and object-level scores of a change map, on
the device (csrc/objects.cu).

A change map (``SiameseEngine.predict_scene(...).pred`` or ``SiameseEngine.predict``) counts pixels; users count
objects: which buildings appeared, how many, how large, and without the single-pixel speckle a tiled network leaves
behind.  ``change_objects`` labels the objects of every non-zero class, drops those smaller than ``min_area``,
numbers the rest in raster order and lists them; with labels it also scores them against the reference objects of
the label map.  This is the post-processing the reference's README promises for evaluate.py.
"""
from __future__ import annotations

from typing import NamedTuple, Optional

import torch

from . import ops

MAX_CLASSES = ops.MAX_CLASSES


class ChangeObjects(NamedTuple):
    """change_objects' result; confusion and object_counts are None without labels.
    pred: uint8, the input's shape, with the objects below min_area set to 0.  ids: int32, same shape: 0 for background
    and dropped objects, else the object's id 1..n.  objects: int64 [n, 7], row id - 1 = (sample, class, area, y0, x0,
    y1, x1), inclusive box.  confusion: int64 [K, K] (rows = label) or, K = 1, [TP, FP, FN, TN] of pred.
    object_counts: int64 [max(K, 2), 4], per class (reference objects, detected ones, predicted objects, matched ones)."""
    pred: torch.Tensor
    ids: torch.Tensor
    objects: torch.Tensor
    confusion: Optional[torch.Tensor]
    object_counts: Optional[torch.Tensor]


def _is_int(v) -> bool:
    return isinstance(v, int) and not isinstance(v, bool)


def change_objects(pred: torch.Tensor, n_classes: int, labels: Optional[torch.Tensor] = None, min_area: int = 0,
                   connectivity: int = 8, min_overlap: float = 0.0, ignore_index: int = -100) -> ChangeObjects:
    """The objects of a class map, filtered by area, numbered and listed on the device.

    pred: uint8 [H, W] or [N, H, W] class map, on the host or a CUDA device (a host map is copied to the current
    device).  n_classes: the model's K in 1..16; K = 1 is the single-logit model's 0/1 map.  Class 0 is "no change".

    An object is a maximal `connectivity`-connected (4 or 8) set of pixels of one non-zero class inside one sample:
    scipy.ndimage.label with generate_binary_structure(2, 1) or (2, 2), run per class.  Objects of fewer than
    `min_area` pixels are set to 0 in the returned pred (the input is not modified).  The others get ids 1..n in raster
    order of their first pixel over (n, y, x); the numbering does not depend on scheduling.

    labels (int64, pred's shape): the reference.  Its objects are formed by the same rule; pixels labelled
    `ignore_index` or outside [0, K) ({0, 1} for K = 1) are background there and are not counted in the confusion,
    which is that of the filtered pred, with predict_scene's format.  A reference object of class c is detected when at
    least max(1, ceil(min_overlap * area)) of its pixels are predicted as c; a predicted object is matched when as many
    of its pixels are labelled c.  metrics.object_metrics turns object_counts into precision, recall and F1.

    The call synchronises with the host once, to size `objects`.  Scratch on the device: 4 bytes per pixel, 16 with
    labels (and 4 bytes per object).  Raises ValueError for bad arguments before any work is enqueued, and for a pred
    value >= max(K, 2) after the synchronisation."""
    if not isinstance(pred, torch.Tensor) or pred.dtype != torch.uint8 or pred.dim() not in (2, 3):
        raise ValueError(f"pred must be a uint8 [H, W] or [N, H, W] tensor, got {getattr(pred, 'dtype', type(pred))} "
                         f"{tuple(getattr(pred, 'shape', ()))}")
    if min(pred.shape) < 1:
        raise ValueError(f"pred is empty: {tuple(pred.shape)}")
    if not _is_int(n_classes) or not 1 <= n_classes <= MAX_CLASSES:
        raise ValueError(f"n_classes must be an int in 1..{MAX_CLASSES}, got {n_classes!r}")
    if labels is not None and (not isinstance(labels, torch.Tensor) or labels.dtype != torch.int64
                               or labels.shape != pred.shape):
        raise ValueError(f"labels must be an int64 tensor of pred's shape {tuple(pred.shape)}, got "
                         f"{getattr(labels, 'dtype', type(labels))} {tuple(getattr(labels, 'shape', ()))}")
    if not _is_int(min_area) or min_area < 0:
        raise ValueError(f"min_area must be an int >= 0, got {min_area!r}")
    if connectivity not in (4, 8) or isinstance(connectivity, bool):
        raise ValueError(f"connectivity must be 4 or 8, got {connectivity!r}")
    if isinstance(min_overlap, bool) or not isinstance(min_overlap, (int, float)) or not 0.0 <= min_overlap <= 1.0:
        raise ValueError(f"min_overlap must be a number in [0, 1], got {min_overlap!r}")
    if not _is_int(ignore_index):
        raise ValueError(f"ignore_index must be an int, got {ignore_index!r}")
    n, h, w = (1, *pred.shape) if pred.dim() == 2 else tuple(pred.shape)
    px = n * h * w
    if px >= 2 ** 31:
        raise ValueError(f"pred has {px} pixels; at most 2^31 - 1 are supported (int32 indices)")

    dev = pred.device if pred.is_cuda else torch.device("cuda", torch.cuda.current_device())
    k, kk = n_classes, max(n_classes, 2)
    with torch.cuda.device(dev):
        src = pred.to(dev).contiguous()
        parent = torch.empty(px, device=dev, dtype=torch.int32)
        ids = torch.empty(px, device=dev, dtype=torch.int32)         # the root areas until the objects are numbered
        info = torch.empty(2, device=dev, dtype=torch.int32)         # (object count, pred values >= max(K, 2))
        chunk = torch.empty(-(-px // ops.OBJECTS_CHUNK), device=dev, dtype=torch.int32)
        out = torch.empty(pred.shape, device=dev, dtype=torch.uint8)
        ops.objects_label(src, n, h, w, k, connectivity, parent, ids, info=info)
        ops.objects_number(src, parent, ids, min_area, chunk, info)
        lab = None
        if labels is not None:
            lab = {"lparent": torch.empty(px, device=dev, dtype=torch.int32),
                   "larea": torch.empty(px, device=dev, dtype=torch.int32),
                   "loverlap": torch.empty(px, device=dev, dtype=torch.int32),
                   "confusion": torch.empty((4,) if k == 1 else (k, k), device=dev, dtype=torch.int64),
                   "object_counts": torch.empty(kk, 4, device=dev, dtype=torch.int64)}
            # the label classes go to `out`, which the finish pass overwrites with the filtered pred
            ops.objects_label(labels.to(dev).contiguous(), n, h, w, k, connectivity, lab["lparent"], lab["larea"],
                              classes=out, ignore_index=ignore_index)
        count, bad = info.tolist()                                   # the one host synchronisation
        if bad:
            raise ValueError(f"pred has {bad} values >= {kk}, outside the classes of n_classes = {k}")
        objects = torch.empty(count, 7, device=dev, dtype=torch.int64)
        if lab is not None:
            lab["overlap"] = torch.empty(count, device=dev, dtype=torch.int32)
        ops.objects_finish(src, parent, ids, n, h, w, k, count, out, objects, min_overlap=float(min_overlap),
                           **(lab or {}))
    if lab is None:
        return ChangeObjects(out, ids.view(pred.shape), objects, None, None)
    return ChangeObjects(out, ids.view(pred.shape), objects, lab["confusion"], lab["object_counts"])
