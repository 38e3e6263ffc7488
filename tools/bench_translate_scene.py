"""Sliding-window image translation of a whole scene (GeneratorEngine.translate_scene) on the GPU, in one process:

1. an 8192 x 8192 seeded uint8 RGB scene (already on the device) through a 3 -> 3 BatchNorm num_downs = 7 generator
   whose running statistics come from a few training steps, at tile 256 / overlap 0 and 64 with batch 32, 64, 128,
   and tile 512 / overlap 64 / batch 16: the whole call (CUDA events, one warm-up call, median of --calls) and scene
   Mpx/s;
2. the eval forward alone, run as many times as the call has tile batches (on the staged input);
3. one instrumented call with CUDA events around every gather, blend and finalize launch: their summed times, the
   bytes each must move (gather: the tile pixels read and the 4-slot bf16 batch written; blend: the 16-byte tile
   outputs of every real tile read, the accumulators read where an earlier batch started them and written where the
   batch covers; finalize: the accumulators read and the uint8 image written) and their fraction of the 6527 GB/s HBM
   roof the other benches use;
4. the device name and enforced power limit, read from NVML in the same run.

    python tools/bench_translate_scene.py [--calls 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from gan_aug_pfa_b200 import ops  # noqa: E402
from gan_aug_pfa_b200.pix2pix import Pix2PixTrainer  # noqa: E402
from gan_aug_pfa_b200.scene import _scene_grid, scene_axis  # noqa: E402

ROOF_GBS = 6527.0
SIZE = 8192
C = 3
CONFIGS = ((256, 32, 0), (256, 64, 0), (256, 128, 0), (256, 32, 64), (256, 64, 64), (256, 128, 64),
           (512, 16, 64))                                                  # (tile, batch, overlap)


def device_info() -> dict:
    import pynvml as nv
    nv.nvmlInit()
    h = nv.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
    name = nv.nvmlDeviceGetName(h)
    return {"device": name.decode() if isinstance(name, bytes) else name,
            "power_limit_w": nv.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0}


def _cells(origins, ext, length):
    """Compressed coordinates of one axis: cell boundaries and, per tile, its [first, last) cell range."""
    b = sorted({0, length, *origins, *(min(o + ext, length) for o in origins)})
    return np.diff(b), [(b.index(o), b.index(min(o + ext, length))) for o in origins]


def blend_bytes(h: int, w: int, tile: int, overlap: int, batch: int, align: int) -> int:
    """Bytes the image blend must move over a whole call: the 16-byte 4-slot output of every real tile pixel, plus per
    batch the accumulators ((C + 1) * 4 B per pixel) written where the batch covers and read where an earlier batch
    started them."""
    oy, ey = scene_axis(h, tile, overlap, align)
    ox, ex = scene_axis(w, tile, overlap, align)
    dy, ry = _cells(oy, ey, h)
    dx, rx = _cells(ox, ex, w)
    area = np.outer(dy, dx).astype(np.int64)
    tiles = [(a, b) for a in ry for b in rx]
    first = np.full(area.shape, len(tiles))
    for t in reversed(range(len(tiles))):
        (y0, y1), (x0, x1) = tiles[t]
        first[y0:y1, x0:x1] = t
    total = len(tiles) * ey * ex * 16
    for t0 in range(0, len(tiles), batch):
        touched = np.zeros(area.shape, dtype=bool)
        for (y0, y1), (x0, x1) in tiles[t0:t0 + batch]:
            touched[y0:y1, x0:x1] = True
        total += int(area[touched].sum()) * (C + 1) * 4
        total += int(area[touched & (first < t0)].sum()) * (C + 1) * 4
    return total


def timed_call(eng, img, tile, overlap, batch) -> dict:
    """translate_scene's loop with CUDA events around each scene kernel (the same launches as the call)."""
    h, w = img.shape[:2]
    align = 1 << eng.L
    grid = _scene_grid(h, w, tile, overlap, align)
    (_, ey, _, ny), (_, ex, _, nx) = grid
    acc = torch.empty(C, h, w, device=img.device)
    wsum = torch.empty(h, w, device=img.device)
    image = torch.empty(h, w, C, device=img.device, dtype=torch.uint8)
    ev = {"gather": [], "blend": [], "finalize": []}

    def rec(name, fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        ev[name].append((e0, e1))

    eng.training = False
    eng._alloc(batch, ey, ex)
    for t0 in range(0, ny * nx, batch):
        rec("gather", lambda: ops.scene_gather_one(img, grid, t0, eng.x_nhwc))
        eng.forward(None, x_ready=True)
        rec("blend", lambda: ops.scene_blend_image(eng.fake_f32, grid, t0, acc, wsum))
    rec("finalize", lambda: ops.scene_finalize_image(acc, wsum, image, False))
    torch.cuda.synchronize()
    return {name: sum(a.elapsed_time(b) for a, b in pairs) for name, pairs in ev.items()}


def forward_only_ms(eng, n_batches: int) -> float:
    eng.training = False
    eng.forward(None, x_ready=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_batches):
        eng.forward(None, x_ready=True)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def trained_generator(dev):
    """A 3 -> 3 BatchNorm generator after a few training steps (non-trivial running statistics)."""
    torch.manual_seed(0)
    tr = Pix2PixTrainer(dev)
    g = torch.Generator().manual_seed(1)
    for _ in range(3):
        a = (torch.rand(4, 3, 256, 256, generator=g) * 2 - 1).to(dev)
        b = (torch.rand(4, 3, 256, 256, generator=g) * 2 - 1).to(dev)
        tr.train_step(a, b)
    torch.cuda.synchronize()
    return tr.G


def run(calls: int) -> list:
    dev = torch.device("cuda:0")
    eng = trained_generator(dev)
    g = torch.Generator(device=dev).manual_seed(0)
    img = torch.randint(0, 256, (SIZE, SIZE, C), device=dev, generator=g, dtype=torch.uint8)
    align = 1 << eng.L
    rows = []
    for tile, batch, overlap in CONFIGS:
        grid = _scene_grid(SIZE, SIZE, tile, overlap, align)
        (_, ey, _, ny), (_, ex, _, nx) = grid
        n_tiles = ny * nx
        n_batches = -(-n_tiles // batch)
        eng.translate_scene(img, tile=tile, overlap=overlap, batch=batch)          # warm-up
        torch.cuda.synchronize()
        times = []
        for _ in range(calls):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            eng.translate_scene(img, tile=tile, overlap=overlap, batch=batch)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        call_ms = statistics.median(times)
        fwd_ms = forward_only_ms(eng, n_batches)
        parts = timed_call(eng, img, tile, overlap, batch)
        px = SIZE * SIZE
        nbytes = {
            "gather": n_batches * batch * ey * ex * 4 * 2 + n_tiles * ey * ex * C,
            "blend": blend_bytes(SIZE, SIZE, tile, overlap, batch, align),
            "finalize": px * ((C + 1) * 4 + C),
        }
        row = {"tile": tile, "batch": batch, "overlap": overlap, "tiles": n_tiles, "batches": n_batches,
               "call_ms_median": round(call_ms, 2), "call_ms": [round(t, 2) for t in times],
               "scene_mpx_s": round(px / 1e6 / (call_ms / 1e3), 1), "forward_ms": round(fwd_ms, 2),
               "call_over_forward": round(call_ms / fwd_ms, 3)}
        for name, ms in parts.items():
            gbs = nbytes[name] / (ms * 1e-3) / 1e9
            row[name] = {"ms": round(ms, 3), "MB": round(nbytes[name] / 1e6, 1), "GB/s": round(gbs, 1),
                         "frac_roof": round(gbs / ROOF_GBS, 3)}
        row["blend_us_per_batch"] = round(parts["blend"] * 1e3 / n_batches, 1)
        row["scene_kernels_frac_of_call"] = round(sum(parts.values()) / call_ms, 4)
        rows.append(row)
        print(json.dumps(row), flush=True)
    return rows


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_translate_scene needs a CUDA device")
    res = {"info": device_info(), "roof_GBs": ROOF_GBS, "scene": [SIZE, SIZE, C], "rows": run(a.calls)}
    print(json.dumps(res["info"]))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
