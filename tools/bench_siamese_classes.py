"""Multi-class Siamese head on the GPU, in one process:

1. the conv_last head at batch 4 @512^2 (1,048,576 pixels; the 64-channel bf16 input is 134 MB): forward, input
   gradient and weight gradient for K = 1 (the single-class conv1x1_cout1 kernels) and K = 2, 7, 16
   (gap_conv1x1_ck_*), CUDA events over --iters back-to-back launches after warm-up;
2. gap_seg_ce_loss (loss + gradient) and gap_seg_confusion_ck on the same planes and int64 labels;
   bytes are the tensors each kernel must read and write, the roof is the 6527 GB/s HBM figure DESIGN.md uses;
3. SiameseEngine.train_step at batch 4 @512^2 for K = 1 (CombinedLoss), 2 and 7 (cross-entropy), interleaved in
   --blocks blocks of --steps steps (median block);
4. the device name and enforced power limit, read from NVML.

    python tools/bench_siamese_classes.py [--iters 50] [--steps 10] [--blocks 5] [--out FILE]
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

from gan_aug_pfa_b200 import ops  # noqa: E402
from gan_aug_pfa_b200.siamese import SiameseEngine  # noqa: E402

ROOF_GBS = 6527.0
N, H, W = 4, 512, 512


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


def row(name: str, k: int, us: float, nbytes: int) -> dict:
    gbs = nbytes / us / 1e3
    return {"kernel": name, "k": k, "us": round(us, 2), "MB": round(nbytes / 1e6, 1), "GB/s": round(gbs, 1),
            "frac_roof": round(gbs / ROOF_GBS, 3)}


def kernel_rows(iters: int) -> list:
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(0)
    pix = N * H * W
    x = torch.randn(N, H, W, 64, device=dev, generator=g).to(torch.bfloat16)
    gx = torch.empty_like(x)
    xb = x.numel() * 2
    rows = []
    for k in (1, 2, 7, 16):
        w = torch.randn(k, 64, device=dev, generator=g) / 8
        b = torch.randn(k, device=dev, generator=g)
        dw, db = torch.zeros_like(w), torch.zeros_like(b)
        planes = torch.empty(N, k, H, W, device=dev)
        dl = torch.randn(N, k, H, W, device=dev, generator=g) * 1e-3
        pb = planes.numel() * 4
        if k == 1:
            fwd = lambda: ops.conv1x1_cout1_fwd(x, w.view(-1), b, planes.view(-1))       # noqa: E731
            dgr = lambda: ops.conv1x1_cout1_dgrad(dl.view(-1), w.view(-1), gx)           # noqa: E731
            wgr = lambda: ops.conv1x1_cout1_wgrad(dl.view(-1), x, dw.view(-1), db)       # noqa: E731
            tag = "conv1x1_cout1"
        else:
            pred = torch.empty(N, H, W, device=dev, dtype=torch.uint8)
            fwd = lambda: ops.conv1x1_ck_fwd(x, w, b, planes)                            # noqa: E731
            rows.append(row("conv1x1_ck_fwd+pred", k, time_us(lambda: ops.conv1x1_ck_fwd(x, w, b, planes, pred), iters),
                            xb + pb + pix))
            dgr = lambda: ops.conv1x1_ck_dgrad(dl, w, gx)                                # noqa: E731
            wgr = lambda: ops.conv1x1_ck_wgrad(dl, x, dw, db)                            # noqa: E731
            tag = "conv1x1_ck"
        rows.append(row(tag + "_fwd", k, time_us(fwd, iters), xb + pb))
        rows.append(row(tag + "_dgrad", k, time_us(dgr, iters), xb + pb))
        rows.append(row(tag + "_wgrad", k, time_us(wgr, iters), xb + pb))
        if k > 1:
            lab = torch.randint(0, k, (N, H, W), device=dev, generator=g)
            cw = torch.rand(k, device=dev, generator=g) + 0.5
            sums = torch.zeros(2, device=dev, dtype=torch.float64)
            bad = torch.zeros(1, device=dev, dtype=torch.int64)
            loss = torch.zeros(1, device=dev, dtype=torch.float64)
            grad = torch.empty_like(dl)
            # label pre-pass (8 B/pixel) + planes and labels read once + gradient planes written
            rows.append(row("seg_ce_loss", k, time_us(lambda: ops.seg_ce_loss(dl, lab, cw, -100, sums, bad, grad, 1.0,
                                                                              loss), iters), 2 * lab.numel() * 8 + 2 * pb))
            counts = torch.zeros(N, k, k, device=dev, dtype=torch.int64)
            rows.append(row("seg_confusion_ck", k, time_us(lambda: ops.seg_confusion_ck(dl, lab, -100, counts), iters),
                            pb + lab.numel() * 8))
    return rows


def step_rows(steps: int, blocks: int) -> list:
    dev = torch.device("cuda:0")
    g = torch.Generator(device=dev).manual_seed(1)
    x1 = torch.rand(N, 3, H, W, device=dev, generator=g) * 2 - 1
    x2 = torch.rand(N, 3, H, W, device=dev, generator=g) * 2 - 1
    engines = {}
    for k in (1, 2, 7):
        torch.manual_seed(0)
        e = SiameseEngine(dev, 3, k)
        from gan_aug_pfa_b200 import spec
        e.load_state_dict(spec.SiameseSpec(3, k).default_state_dict())
        lab = (torch.rand(N, H, W, device=dev, generator=g) < 0.1).long() if k == 1 else \
            torch.randint(0, k, (N, H, W), device=dev, generator=g)
        engines[k] = (e, lab)
    times = {k: [] for k in engines}
    for k, (e, lab) in engines.items():                  # warm-up
        for _ in range(3):
            e.train_step(x1, x2, lab)
    torch.cuda.synchronize()
    for _ in range(blocks):
        for k, (e, lab) in engines.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(steps):
                loss = e.train_step(x1, x2, lab)
            torch.cuda.synchronize()
            times[k].append((time.perf_counter() - t0) * 1e3 / steps)
            assert torch.isfinite(loss).all()
    base = statistics.median(times[1])
    return [{"k": k, "ms_per_step_median": round(statistics.median(t), 3), "blocks_ms": [round(v, 3) for v in t],
             "vs_k1": round(statistics.median(t) / base, 4)} for k, t in times.items()]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_siamese_classes needs a CUDA device")
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
