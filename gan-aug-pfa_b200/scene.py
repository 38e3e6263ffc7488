"""The tile grid and blending window of sliding-window scene inference, shared by SiameseEngine.predict_scene and
GeneratorEngine.translate_scene (csrc/scene.cu derives the same origins and window on the device)."""
from __future__ import annotations

from typing import List, Tuple

import torch


def scene_axis(length: int, tile: int, overlap: int, align: int = 16) -> Tuple[List[int], int]:
    """The tile origins along one scene axis of `length` pixels and the tile extent E.  length <= tile: one tile at 0
    with E = length rounded up to `align` (a multiple of 16 that divides `tile`), whose reads past the scene clamp to
    its last row / column.  Otherwise E = tile, step S = tile - overlap and n = ceil((length - tile) / S) + 1 tiles at
    min(i*S, length - tile): the last one is snapped to the edge."""
    if length <= tile:
        return [0], -(-length // align) * align
    step = tile - overlap
    n = -(-(length - tile) // step) + 1
    return [min(i * step, length - tile) for i in range(n)], tile


def scene_window(extent: int) -> torch.Tensor:
    """The 1-D blending window of a tile axis, fp64 [extent]: g(t) = exp(-(t + 0.5 - E/2)^2 / (2 sigma^2)), sigma = E/8
    (nnU-Net's choice); a tile's weight is g_y(ty) * g_x(tx).  Its smallest value is about exp(-8), so every covered
    pixel has a positive weight sum, and with overlap 0 it cancels (plain stitching)."""
    t = torch.arange(extent, dtype=torch.float64)
    sigma = extent / 8
    return torch.exp(-(t + 0.5 - extent / 2) ** 2 / (2 * sigma ** 2))


def _scene_grid(h: int, w: int, tile: int, overlap: int, align: int = 16):
    """((len, ext, step, n) of the y axis, same of the x axis): the grid in the form the scene kernels take."""
    out = []
    for length in (h, w):
        origins, ext = scene_axis(length, tile, overlap, align)
        out.append((length, ext, tile - overlap if len(origins) > 1 else ext, len(origins)))
    return tuple(out)
