"""Multi-class Dice losses on the GPU, in one process:

1. gap_seg_softmax_dice (kind="ce_dice" = mode 0, kind="softmax_focal_dice" = mode 1: zero the sums, stats pass,
   gradient pass) beside gap_seg_ce_loss at batch 4 @512^2 (1,048,576 pixels) for K = 2, 7, 16, CUDA events over
   --iters back-to-back launches after warm-up.  Bytes are what the two passes must move: (8K + 16) B per pixel (the
   planes and labels read by each pass) plus 4K B per pixel for the gradient; gap_seg_ce_loss moves 16 B per pixel of
   labels (two passes) plus 8K B of planes.  The roof is the 6527 GB/s HBM figure DESIGN.md uses.  The planes
   (8-64 MB) fit in the 126 MB L2, so the second pass may read them from there: the fraction of roof is of the bytes,
   not a claim that all of them came from HBM;
2. SiameseEngine.train_step at batch 4 @512^2 with kind "ce", "ce_dice" and "softmax_focal_dice" at K = 2 and 7,
   interleaved in --blocks blocks of --steps steps (median block);
3. the device name and enforced power limit, read from NVML in the same run.

    python tools/bench_siamese_losses.py [--iters 50] [--steps 10] [--blocks 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from gan_aug_pfa_b200 import ops, spec  # noqa: E402
from gan_aug_pfa_b200.siamese import SiameseEngine  # noqa: E402

ROOF_GBS = 6527.0
N, H, W = 4, 512, 512
KW = {"ce": {}, "ce_dice": dict(alpha=0.5, smooth=1.0), "softmax_focal_dice": dict(beta=0.5, gamma=2.0, smooth=1.0)}


def device_info() -> dict:
    import pynvml as nv
    nv.nvmlInit()
    h = nv.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
    name = nv.nvmlDeviceGetName(h)
    return {"device": name.decode() if isinstance(name, bytes) else name,
            "power_limit_w": nv.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0}


def time_us(fn, iters: int) -> float:
    for _ in range(3):
        fn()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) * 1000.0 / iters


def row(name: str, k: int, us: float, nbytes: int, ce_us: float) -> dict:
    gbs = nbytes / us / 1e3
    return {"kernel": name, "k": k, "us": round(us, 2), "MB": round(nbytes / 1e6, 1), "GB/s": round(gbs, 1),
            "frac_roof": round(gbs / ROOF_GBS, 3), "vs_seg_ce_loss": round(us / ce_us, 3)}


def kernel_rows(iters: int) -> list:
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(0)
    pix = N * H * W
    rows = []
    for k in (2, 7, 16):
        logits = torch.randn(N, k, H, W, device=dev, generator=g) * 3
        lab = torch.randint(0, k, (N, H, W), device=dev, generator=g)
        cw = torch.rand(k, device=dev, generator=g) + 0.5
        grad = torch.empty_like(logits)
        bad = torch.zeros(1, device=dev, dtype=torch.int64)
        loss = torch.zeros(1, device=dev, dtype=torch.float64)
        ce_sums = torch.zeros(2, device=dev, dtype=torch.float64)
        sums = torch.zeros(ops.DICE_SUMS, device=dev, dtype=torch.float64)
        ce_us = time_us(lambda: ops.seg_ce_loss(logits, lab, cw, -100, ce_sums, bad, grad, 1.0, loss), iters)
        rows.append(row("seg_ce_loss", k, ce_us, pix * (16 + 8 * k), ce_us))
        for mode, name in ((0, "seg_softmax_dice[ce_dice]"), (1, "seg_softmax_dice[softmax_focal_dice]")):
            us = time_us(lambda: ops.seg_softmax_dice_loss(logits, lab, mode, 0.5, 2.0, 1.0, cw, -100, sums, bad, grad,
                                                           1.0, loss), iters)
            rows.append(row(name, k, us, pix * (8 * k + 16 + 4 * k), ce_us))
    return rows


def step_rows(steps: int, blocks: int) -> list:
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(1)
    x1 = torch.rand(N, 3, H, W, device=dev, generator=g) * 2 - 1
    x2 = torch.rand(N, 3, H, W, device=dev, generator=g) * 2 - 1
    runs = {}
    for k in (2, 7):
        lab = torch.randint(1, k, (N, H, W), device=dev, generator=g) * (torch.rand(N, H, W, device=dev, generator=g) < 0.1)
        for kind in KW:
            torch.manual_seed(0)
            e = SiameseEngine(dev, 3, k)
            e.load_state_dict(spec.SiameseSpec(3, k).default_state_dict())
            runs[(k, kind)] = (e, lab)
    times = {key: [] for key in runs}
    for (k, kind), (e, lab) in runs.items():                  # warm-up
        for _ in range(3):
            e.train_step(x1, x2, lab, kind=kind, **KW[kind])
    torch.cuda.synchronize()
    for _ in range(blocks):
        for (k, kind), (e, lab) in runs.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                loss = e.train_step(x1, x2, lab, kind=kind, **KW[kind])
            torch.cuda.synchronize()
            times[(k, kind)].append((time.perf_counter() - t0) * 1e3 / steps)
            assert torch.isfinite(loss).all()
    out = []
    for (k, kind), t in times.items():
        base = statistics.median(times[(k, "ce")])
        out.append({"k": k, "kind": kind, "ms_per_step_median": round(statistics.median(t), 3),
                    "blocks_ms": [round(v, 3) for v in t], "vs_ce": round(statistics.median(t) / base, 4)})
    return out


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_siamese_losses needs a CUDA device")
    res = {"info": device_info(), "roof_GBs": ROOF_GBS, "kernels": kernel_rows(a.iters),
           "train_step_b4_512": step_rows(a.steps, a.blocks)}
    for r in res["kernels"]:
        print(json.dumps(r))
    for r in res["train_step_b4_512"]:
        print(json.dumps(r))
    print(json.dumps(res["info"]))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
