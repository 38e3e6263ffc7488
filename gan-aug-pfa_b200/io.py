"""Host -> device input pipeline for the step loops (SURVEY.md §8(f) rank 2): replaces the reference's per-batch
`.to(DEVICE)` (train_gan.py:53-54, train.py:137-139) by a double-buffered prefetch on a copy stream.

Batches are tuples of PINNED host tensors — raw uint8 [n, h, w, C] images (normalised on the device by the first
kernels, dataset.py:28-29,155-159) or the fp32 NCHW tensors the reference's DataLoader yields.  While iteration i
computes, batch i+1 is copied into the other staging slot; the consumer calls `release()` once it has enqueued the
work that reads the current slot, which lets the copy stream refill it two iterations later."""
from __future__ import annotations

from typing import Iterable, Iterator, List, Optional, Sequence, Tuple

import torch

from . import ops


def load_pair_u8(a_u8: torch.Tensor, b_u8: torch.Tensor, size: Tuple[int, int],
                 label: Optional[torch.Tensor] = None):
    """The tensor half of BaseChangeDetectionDataset.__getitem__ (dataset.py:191, transform list at 185-191) on the
    device, for raw uint8 [n, h, w, C] image batches (C = 1..4) of any size: ToTensor -> JointResize(size, BILINEAR;
    labels NEAREST) -> JointNormalize.  Returns fp32 NCHW [n, C, H, W] tensors in [-1, 1] — what the reference's DataLoader
    yields and `train_step` / the drop-in modules accept — and the resized int64 label map if one was given."""
    H, W = size
    outs = []
    for x in (a_u8, b_u8):
        f = torch.empty(x.shape[0], x.shape[-1], H, W, device=x.device)
        ops.resize_u8_to_nhwc_bf16(x.contiguous(), None, f)
        outs.append(f)
    if label is not None:
        lab = torch.empty(label.shape[0], H, W, device=label.device, dtype=torch.int64)
        ops.resize_nearest_i64(label.contiguous(), lab)
        outs.append(lab)
    return tuple(outs)


class PairPrefetcher:
    """for a, b in PairPrefetcher(device, batches): step(a, b); prefetcher.release()"""

    def __init__(self, device, batches: Iterable[Sequence[torch.Tensor]], slots: int = 2) -> None:
        self.dev = torch.device(device)
        if self.dev.type != "cuda":
            raise ValueError("PairPrefetcher stages batches in CUDA memory")
        self.batches = batches
        self.slots = slots
        self.copy_stream = torch.cuda.Stream(self.dev)
        self._stage: List[Tuple[torch.Tensor, ...]] = []
        self._copied = [torch.cuda.Event() for _ in range(slots)]
        self._used = [torch.cuda.Event() for _ in range(slots)]
        self._used_valid = [False] * slots
        self._cur = -1
        self.h2d_bytes = 0

    def preallocate(self, example: Sequence[torch.Tensor]) -> "PairPrefetcher":
        """Create the device staging buffers for batches shaped like `example` up front (a cudaMalloc inside the loop
        would synchronise the device)."""
        while len(self._stage) < self.slots:
            self._stage.append(tuple(torch.empty(t.shape, dtype=t.dtype, device=self.dev) for t in example))
        return self

    def _issue(self, k: int, batch: Sequence[torch.Tensor]) -> None:
        for t in batch:
            if not t.is_pinned():
                raise ValueError("PairPrefetcher needs pinned host tensors (tensor.pin_memory())")
        if len(self._stage) <= k:
            self._stage.append(tuple(torch.empty(t.shape, dtype=t.dtype, device=self.dev) for t in batch))
        elif any(s.shape != t.shape or s.dtype != t.dtype for s, t in zip(self._stage[k], batch)):
            self._stage[k] = tuple(torch.empty(t.shape, dtype=t.dtype, device=self.dev) for t in batch)
        with torch.cuda.stream(self.copy_stream):
            if self._used_valid[k]:
                self.copy_stream.wait_event(self._used[k])       # the consumer of this slot's previous batch is done
            for dst, src in zip(self._stage[k], batch):
                dst.copy_(src, non_blocking=True)
                self.h2d_bytes += src.numel() * src.element_size()
            self._copied[k].record(self.copy_stream)

    def __iter__(self) -> Iterator[Tuple[torch.Tensor, ...]]:
        it = iter(self.batches)
        self.copy_stream.wait_stream(torch.cuda.current_stream(self.dev))
        nxt = next(it, None)
        i = 0
        if nxt is not None:
            self._issue(0, nxt)
        while nxt is not None:
            k = i % self.slots
            ahead = next(it, None)
            if ahead is not None:
                self._issue((i + 1) % self.slots, ahead)
            torch.cuda.current_stream(self.dev).wait_event(self._copied[k])
            self._cur = k
            yield self._stage[k]
            if self._cur == k:
                self.release()          # a consumer that did not: everything enqueued so far counts as the reader
            nxt = ahead
            i += 1

    def release(self) -> None:
        """Call after enqueueing the work that reads the batch just yielded."""
        k = self._cur
        if k >= 0:
            self._used[k].record(torch.cuda.current_stream(self.dev))
            self._used_valid[k] = True
            self._cur = -1
