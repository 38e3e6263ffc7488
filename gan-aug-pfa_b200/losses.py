"""Multi-class Dice losses for the drop-in ``SiameseUNet(n_channels, K)`` (K = 2..16): the K-class forms of the
reference's CombinedLoss (BCE + Dice, train.py:82-105) and FocalDiceLoss (train.py:108-128), as ``nn.Module`` criteria
for a train.py-style loop::

    criterion = SoftmaxFocalDiceLoss(beta=0.5, gamma=2.0).to(device)
    loss = criterion(outputs, labels)       # outputs [n, K, h, w] fp32, labels int64 [n, h, w]
    loss.backward()

The forward runs the fused loss-and-gradient kernels (gap_seg_softmax_dice) once and keeps the gradient; the backward
only scales it by grad_output.  The Dice term is 1 - the mean over classes 1..K-1 (class 0, "no change", is excluded
as in the reference's binary Dice) of (2 I_k + smooth) / (P_k + T_k + smooth), with I_k = sum p_k [y=k],
P_k = sum p_k, T_k = sum [y=k] over the counted pixels (label != ignore_index, 0 <= label < K) of the WHOLE batch, like
the reference's DiceLoss.  Under data parallelism each rank's Dice covers its own batch only.
"""
from __future__ import annotations

from typing import Optional, Sequence, Union

import torch
import torch.nn as nn

from . import ops


class _SoftmaxDiceFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logits, labels, crit):
        dev = logits.device
        weight = crit.weight
        if weight is not None and weight.device != dev:
            weight = weight.to(dev)
        if crit.bad_labels is None or crit.bad_labels.device != dev:
            crit.bad_labels = torch.zeros(1, device=dev, dtype=torch.int64)
        sums = torch.empty(ops.DICE_SUMS, device=dev, dtype=torch.float64)
        loss = torch.empty(1, device=dev, dtype=torch.float64)
        grad = torch.empty_like(logits) if ctx.needs_input_grad[0] else None
        ops.seg_softmax_dice_loss(logits, labels, crit.mode, crit.w_point, crit.gamma, crit.smooth, weight,
                                  crit.ignore_index, sums, crit.bad_labels, grad, 1.0, loss)
        ctx.grad = grad
        return loss.to(logits.dtype).reshape(())

    @staticmethod
    def backward(ctx, grad_output):
        return ctx.grad * grad_output, None, None


class _SoftmaxDice(nn.Module):
    mode = 0

    def __init__(self, w_point: float, gamma: float, smooth: float,
                 weight: Optional[Union[torch.Tensor, Sequence[float]]], ignore_index: int) -> None:
        super().__init__()
        name = type(self).__name__
        ops.check_dice_args(name, w_point, gamma, smooth)
        if weight is not None:
            weight = torch.as_tensor(weight, dtype=torch.float32).detach().reshape(-1).contiguous()
            if not 2 <= weight.numel() <= ops.MAX_CLASSES:
                raise ValueError(f"{name}: weight must have one entry per class (2..{ops.MAX_CLASSES}), got "
                                 f"{weight.numel()}")
        self.register_buffer("weight", weight)
        self.w_point, self.gamma, self.smooth = float(w_point), float(gamma), float(smooth)
        self.ignore_index = int(ignore_index)
        self.bad_labels: Optional[torch.Tensor] = None      # labels outside [0, K) that are not ignore_index (counted)

    def forward(self, logits: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        """logits: fp32 class planes [n, K, h, w] on the GPU; labels: int64 [n, h, w].  Returns the scalar loss."""
        name = type(self).__name__
        if not isinstance(logits, torch.Tensor) or logits.dim() != 4 or not 2 <= logits.shape[1] <= ops.MAX_CLASSES:
            raise ValueError(f"{name}: logits must be class planes [n, K, h, w] with K in 2..{ops.MAX_CLASSES}, got "
                             f"{tuple(logits.shape) if isinstance(logits, torch.Tensor) else type(logits).__name__}")
        if logits.dtype != torch.float32 or not isinstance(labels, torch.Tensor) or labels.dtype != torch.int64:
            raise ValueError(f"{name}: logits must be fp32 and labels int64")
        n, _, h, w = logits.shape
        if tuple(labels.shape) != (n, h, w):
            raise ValueError(f"{name}: labels must be [n={n}, h={h}, w={w}], got {tuple(labels.shape)}")
        if self.weight is not None and self.weight.numel() != logits.shape[1]:
            raise ValueError(f"{name}: weight has {self.weight.numel()} entries; the logits have {logits.shape[1]} "
                             "classes")
        if not (logits.is_cuda and labels.is_cuda):
            raise ValueError(f"{name} needs CUDA tensors (there is no CPU path)")
        return _SoftmaxDiceFn.apply(logits.contiguous(), labels.contiguous(), self)


class CEDiceLoss(_SoftmaxDice):
    """alpha * nn.CrossEntropyLoss(weight, ignore_index) + (1 - alpha) * Dice over K = 2..16 classes: CombinedLoss
    (train.py:82-105) for softmax outputs.  At K = 2 it equals alpha * F.cross_entropy + (1 - alpha) * the reference's
    DiceLoss on the logit difference z1 - z0."""
    mode = 0

    def __init__(self, alpha: float = 0.5, smooth: float = 1.0,
                 weight: Optional[Union[torch.Tensor, Sequence[float]]] = None, ignore_index: int = -100) -> None:
        super().__init__(alpha, 0.0, smooth, weight, ignore_index)
        self.alpha = float(alpha)


class SoftmaxFocalDiceLoss(_SoftmaxDice):
    """beta * Focal + (1 - beta) * Dice over K = 2..16 classes: FocalDiceLoss (train.py:108-128) for softmax outputs,
    Focal = mean over the counted pixels of a[y] (1 - p_y)^gamma (-log p_y) with a = weight (None: all 1).  At K = 2
    with weight = [1 - focal_alpha, focal_alpha] it equals the reference's FocalDiceLoss on z1 - z0."""
    mode = 1

    def __init__(self, beta: float = 0.5, gamma: float = 2.0, smooth: float = 1.0,
                 weight: Optional[Union[torch.Tensor, Sequence[float]]] = None, ignore_index: int = -100) -> None:
        super().__init__(beta, gamma, smooth, weight, ignore_index)
        self.beta = float(beta)
