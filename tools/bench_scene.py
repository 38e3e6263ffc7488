"""Sliding-window scene inference (SiameseEngine.predict_scene) on the GPU, in one process:

1. an 8192 x 8192 seeded uint8 RGB pair (already on the device), K = 1, 2, 7, at tile 512 / batch 4 and tile 256 /
   batch 16, overlap 0 and 64: the whole call (CUDA events, one warm-up call, median of --calls) and scene Mpx/s;
2. the eval forward alone, run as many times as the call has tile batches (on the staged inputs);
3. one instrumented call with CUDA events around every gather, blend and finalize launch: their summed times, the
   bytes each must move (gather: the tile pixels of both scenes read and the two 4-slot bf16 batches written; blend:
   the batch logits read, the accumulators read where an earlier batch started them and written where the batch
   covers; finalize: the accumulators read and the uint8 map written) and their fraction of the 6527 GB/s HBM roof
   the other benches use;
4. the device name and enforced power limit, read from NVML in the same run.

    python tools/bench_scene.py [--calls 5] [--out FILE]
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

from gan_aug_pfa_b200 import ops, spec  # noqa: E402
from gan_aug_pfa_b200.siamese import SiameseEngine, _scene_grid, scene_axis  # noqa: E402

ROOF_GBS = 6527.0
SIZE = 8192
CONFIGS = ((512, 4, 0), (512, 4, 64), (256, 16, 0), (256, 16, 64))       # (tile, batch, overlap)


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


def blend_bytes(h: int, w: int, tile: int, overlap: int, batch: int, k: int) -> int:
    """Bytes the blend must move over a whole call: logits of every real tile, plus per batch the accumulators
    ((K + 1) * 4 B per pixel) written where the batch covers and read where an earlier batch started them."""
    oy, ey = scene_axis(h, tile, overlap)
    ox, ex = scene_axis(w, tile, overlap)
    dy, ry = _cells(oy, ey, h)
    dx, rx = _cells(ox, ex, w)
    area = np.outer(dy, dx).astype(np.int64)
    tiles = [(a, b) for a in ry for b in rx]
    first = np.full(area.shape, len(tiles))
    for t in reversed(range(len(tiles))):
        (y0, y1), (x0, x1) = tiles[t]
        first[y0:y1, x0:x1] = t
    total = len(tiles) * k * ey * ex * 4
    for t0 in range(0, len(tiles), batch):
        touched = np.zeros(area.shape, dtype=bool)
        for (y0, y1), (x0, x1) in tiles[t0:t0 + batch]:
            touched[y0:y1, x0:x1] = True
        total += int(area[touched].sum()) * (k + 1) * 4
        total += int(area[touched & (first < t0)].sum()) * (k + 1) * 4
    return total


def timed_call(eng, img1, img2, tile, overlap, batch) -> dict:
    """predict_scene's loop with CUDA events around each scene kernel (the same launches as the call)."""
    h, w = img1.shape[:2]
    k = eng.n_classes
    grid = _scene_grid(h, w, tile, overlap)
    (_, ey, _, ny), (_, ex, _, nx) = grid
    acc = torch.empty(k, h, w, device=img1.device)
    wsum = torch.empty(h, w, device=img1.device)
    pred = torch.empty(h, w, device=img1.device, dtype=torch.uint8)
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
        rec("gather", lambda: ops.scene_gather(img1, img2, grid, t0, eng.x_in[0], eng.x_in[1]))
        eng._forward_from((None, None))
        rec("blend", lambda: ops.scene_blend(eng.logits, grid, t0, acc, wsum))
    rec("finalize", lambda: ops.scene_finalize(acc, wsum, pred, False))
    torch.cuda.synchronize()
    eng._tape = []
    return {name: sum(a.elapsed_time(b) for a, b in pairs) for name, pairs in ev.items()}


def forward_only_ms(eng, n_batches: int) -> float:
    eng.training = False
    eng._forward_from((None, None))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n_batches):
        eng._forward_from((None, None))
    e1.record()
    torch.cuda.synchronize()
    eng._tape = []
    return e0.elapsed_time(e1)


def run(calls: int) -> list:
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(0)
    img1 = torch.randint(0, 256, (SIZE, SIZE, 3), device=dev, generator=g, dtype=torch.uint8)
    img2 = torch.randint(0, 256, (SIZE, SIZE, 3), device=dev, generator=g, dtype=torch.uint8)
    rows = []
    for k in (1, 2, 7):
        torch.manual_seed(0)
        eng = SiameseEngine(dev, 3, k)
        eng.load_state_dict(spec.SiameseSpec(3, k).default_state_dict())
        for tile, batch, overlap in CONFIGS:
            grid = _scene_grid(SIZE, SIZE, tile, overlap)
            (_, ey, _, ny), (_, ex, _, nx) = grid
            n_tiles = ny * nx
            n_batches = -(-n_tiles // batch)
            eng.predict_scene(img1, img2, tile=tile, overlap=overlap, batch=batch)        # warm-up
            torch.cuda.synchronize()
            times = []
            for _ in range(calls):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                eng.predict_scene(img1, img2, tile=tile, overlap=overlap, batch=batch)
                e1.record()
                torch.cuda.synchronize()
                times.append(e0.elapsed_time(e1))
            call_ms = statistics.median(times)
            fwd_ms = forward_only_ms(eng, n_batches)
            parts = timed_call(eng, img1, img2, tile, overlap, batch)
            px = SIZE * SIZE
            nbytes = {
                "gather": n_batches * batch * ey * ex * 4 * 2 * 2 + n_tiles * ey * ex * 3 * 2,
                "blend": blend_bytes(SIZE, SIZE, tile, overlap, batch, k),
                "finalize": px * ((k + 1) * 4 + 1),
            }
            row = {"k": k, "tile": tile, "batch": batch, "overlap": overlap, "tiles": n_tiles, "batches": n_batches,
                   "call_ms_median": round(call_ms, 2), "call_ms": [round(t, 2) for t in times],
                   "scene_mpx_s": round(px / 1e6 / (call_ms / 1e3), 1), "forward_ms": round(fwd_ms, 2)}
            for name, ms in parts.items():
                gbs = nbytes[name] / (ms * 1e-3) / 1e9
                row[name] = {"ms": round(ms, 3), "MB": round(nbytes[name] / 1e6, 1), "GB/s": round(gbs, 1),
                             "frac_roof": round(gbs / ROOF_GBS, 3)}
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
        raise SystemExit("bench_scene needs a CUDA device")
    res = {"info": device_info(), "roof_GBs": ROOF_GBS, "scene": [SIZE, SIZE, 3], "rows": run(a.calls)}
    print(json.dumps(res["info"]))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
