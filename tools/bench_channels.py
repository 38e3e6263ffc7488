"""Image channel counts on the GPU, in one process:

1. thin_convT_fwd (the generator's last ConvTranspose2d: [64,128,128,128] bf16 input, 268 MB, + bias + Tanh into the
   fp32 and bf16 4-slot outputs; and the discriminator's input gradient: [64,128,128,64] input into the fp32 output) at
   CO = 1..4 output channels, against CO = 3 (the existing entry point) on the same tensors;
2. gen_out_bwd (L1 + Tanh backward, fp32 real_B) at C = 1..4 on [64,256,256] images;
   both with CUDA events over --iters back-to-back launches after warm-up.  Bytes are the tensors each kernel must read
   and write; the roof is the 6527 GB/s HBM figure DESIGN.md uses.  Every working set exceeds the 126 MB L2;
3. Pix2PixTrainer.train_step_graphed at batch 64, 256x256 for input_nc -> output_nc = 3 -> 3, 1 -> 3 and 4 -> 4,
   interleaved in blocks;
4. the device name and enforced power limit, read from NVML.

    python tools/bench_channels.py [--iters 50] [--steps 60] [--blocks 6] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import sys
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from gan_aug_pfa_b200 import ops  # noqa: E402
from gan_aug_pfa_b200.pix2pix import Pix2PixTrainer  # noqa: E402

ROOF_GBS = 6527.0
CONFIGS = [(3, 3), (1, 3), (4, 4)]


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


def convT_rows(iters: int) -> list:
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(0)
    rows = []
    for what, cw, act, with_bf in (("generator_out", 128, ops.ACT_TANH, True), ("disc_input_grad", 64, ops.ACT_NONE, False)):
        n, ih, iw = 64, 128, 128
        wide = torch.randn(n, ih, iw, cw, generator=g, device=dev).to(torch.bfloat16)
        o32 = torch.zeros(n, 2 * ih, 2 * iw, 4, device=dev)
        obf = torch.zeros(n, 2 * ih, 2 * iw, 4, device=dev, dtype=torch.bfloat16) if with_bf else None
        bias = torch.zeros(4, device=dev) if act == ops.ACT_TANH else None
        t = {}
        for co in (1, 2, 3, 4):
            wcol = (torch.randn(16 * co, cw, generator=g, device=dev) / 32).to(torch.bfloat16)
            t[co] = time_us(lambda: ops.thin_convT_fwd(wide, wcol, bias, act, obf, o32, co=co), iters)
        nbytes = wide.numel() * 2 + o32.numel() * 4 + (obf.numel() * 2 if with_bf else 0)
        for co in (1, 2, 3, 4):
            rows.append({"kernel": "thin_convT_fwd", "use": what, "cw": cw, "co": co, "us": round(t[co], 2),
                         "GB/s": round(nbytes / t[co] / 1e3, 1), "roof_frac": round(nbytes / t[co] / 1e3 / ROOF_GBS, 3),
                         "over_co3": round(t[co] / t[3], 4)})
    return rows


def gen_out_rows(iters: int) -> list:
    dev = "cuda"
    g = torch.Generator(device=dev).manual_seed(1)
    n, h, w = 64, 256, 256
    fake = torch.tanh(torch.randn(n, h, w, 4, generator=g, device=dev))
    dd = torch.randn(n, h, w, 4, generator=g, device=dev) * 1e-3
    dpre = torch.zeros(n, h, w, 4, device=dev, dtype=torch.bfloat16)
    loss = torch.zeros(1, device=dev, dtype=torch.float64)
    rows, t = [], {}
    for c in (1, 2, 3, 4):
        real = torch.rand(n, c, h, w, generator=g, device=dev) * 2 - 1
        t[c] = time_us(lambda: ops.gen_out_bwd(fake, real, dd, 1e-6, dpre, loss), iters)
        nbytes = n * h * w * (16 + 16 + 4 * c + 8)
        rows.append({"kernel": "gen_out_bwd", "c": c, "us": round(t[c], 2), "GB/s": round(nbytes / t[c] / 1e3, 1),
                     "roof_frac": round(nbytes / t[c] / 1e3 / ROOF_GBS, 3)})
    for r in rows:
        r["over_c3"] = round(t[r["c"]] / t[3], 4)
    return rows


def steps(n_steps: int, blocks: int) -> list:
    dev = torch.device("cuda")
    trainers, data = {}, {}
    for ic, oc in CONFIGS:
        g = torch.Generator().manual_seed(0)
        data[(ic, oc)] = ((torch.rand(64, ic, 256, 256, generator=g) * 2 - 1).to(dev),
                          (torch.rand(64, oc, 256, 256, generator=g) * 2 - 1).to(dev))
        torch.manual_seed(0)
        trainers[(ic, oc)] = Pix2PixTrainer(dev, input_nc=ic, output_nc=oc)
        for _ in range(5):
            trainers[(ic, oc)].train_step_graphed(*data[(ic, oc)])
    torch.cuda.synchronize()
    per = max(1, n_steps // blocks)
    times = {k: [] for k in trainers}
    for _ in range(blocks):
        for key, tr in trainers.items():
            A, B = data[key]
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(per):
                tr.train_step_graphed(A, B)
            e1.record()
            torch.cuda.synchronize()
            times[key].append(e0.elapsed_time(e1) / per)
    out = []
    med = {k: sorted(t)[len(t) // 2] for k, t in times.items()}
    for (ic, oc), t in times.items():
        out.append({"step": "train_step_graphed", "input_nc": ic, "output_nc": oc, "batch": 64, "size": 256,
                    "steps": per * blocks, "ms_per_step_median_block": round(med[(ic, oc)], 3),
                    "ms_blocks": [round(x, 3) for x in t], "over_3to3": round(med[(ic, oc)] / med[(3, 3)], 4)})
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=50, help="timed launches per kernel (>= 20)")
    ap.add_argument("--steps", type=int, default=60, help="timed training steps per configuration (>= 50)")
    ap.add_argument("--blocks", type=int, default=6, help="interleaved blocks the steps are split into")
    ap.add_argument("--out", type=Path, default=None, help="also write all results as JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_channels needs a CUDA device (the gap_* kernels have no CPU path)")
    res = {"env": device_info(), "kernels": [], "steps": []}
    print(json.dumps(res["env"]), flush=True)
    for r in convT_rows(a.iters) + gen_out_rows(a.iters):
        res["kernels"].append(r)
        print(json.dumps(r), flush=True)
    for r in steps(a.steps, a.blocks):
        res["steps"].append(r)
        print(json.dumps(r), flush=True)
    if a.out is not None:
        a.out.parent.mkdir(parents=True, exist_ok=True)
        a.out.write_text(json.dumps(res, indent=1))


if __name__ == "__main__":
    main()
