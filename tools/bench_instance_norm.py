"""InstanceNorm2d against BatchNorm2d on the GPU, in one process:

1. every gap_in_* kernel against its BatchNorm counterpart on the same tensors (CUDA events over --iters launches after
   warm-up): in_stats + in_act vs bn_act (whose statistics come from the conv epilogue), in_bwd_reduce vs
   bn_bwd_reduce, in_bwd_apply vs bn_bwd_apply.  The generator's pattern: two activated outputs (LeakyReLU, ReLU skip)
   forward, a second gradient source (the skip) backward.  Bytes are the tensors each kernel must read and write; the
   roof is the 6527 GB/s HBM figure DESIGN.md uses.  The [64,128,128,64] tensor (134 MB) exceeds the 126 MB L2; the
   two 63-67 MB tensors do not, but each kernel's working set (3-4 such tensors) does;
2. Pix2PixTrainer(norm=...).train_step_graphed at batch 64, 256x256, norm="batch" and "instance" interleaved in blocks;
3. the device name and enforced power limit, read from NVML.

    python tools/bench_instance_norm.py [--iters 50] [--steps 50] [--out FILE]
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
SHAPES = [(64, 128, 128, 64), (64, 64, 64, 128), (64, 31, 31, 512)]


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


def kernels(shape, iters: int) -> list:
    n, h, w, c = shape
    dev = "cuda"
    bf = dict(device=dev, dtype=torch.bfloat16)
    g = torch.Generator(device=dev).manual_seed(0)
    y, g1, g2 = (torch.randn(n, h, w, c, generator=g, device=dev).to(torch.bfloat16) for _ in range(3))
    o1, o2, dy = (torch.empty(n, h, w, c, **bf) for _ in range(3))
    size = y.numel() * 2
    # BatchNorm per-channel state
    bsc, bsh, bmu, biv = torch.ones(c, device=dev), torch.zeros(c, device=dev), torch.zeros(c, device=dev), torch.ones(c, device=dev)
    bsums = torch.zeros(2 * c, device=dev, dtype=torch.float64)
    # InstanceNorm per-(image, channel) state, from real statistics
    isums = torch.zeros(2 * n * c, device=dev, dtype=torch.float64)
    isc, ish, imu, iiv = (torch.empty(n, c, device=dev) for _ in range(4))
    dbias = torch.zeros(c, device=dev)
    count = n * h * w

    def in_stats():
        ops.in_stats(y, isums)

    def in_finalize():
        ops.bn_finalize(isums, h * w, None, None, 1e-5, 0.0, 1, None, None, None, isc, ish, imu, iiv)

    in_stats()
    in_finalize()
    rows = []

    def row(name, bn_name, t_in, t_bn, nbytes, bn_bytes):
        rows.append({"shape": list(shape), "kernel": name, "us": round(t_in, 2), "GB/s": round(nbytes / t_in / 1e3, 1),
                     "roof_frac": round(nbytes / t_in / 1e3 / ROOF_GBS, 3), "bn_kernel": bn_name, "bn_us": round(t_bn, 2),
                     "bn_GB/s": round(bn_bytes / t_bn / 1e3, 1), "in_over_bn": round(t_in / t_bn, 3)})

    t_bn_act = time_us(lambda: ops.bn_act(y, bsc, bsh, o1, ops.ACT_LRELU, o2, ops.ACT_RELU), iters)
    t_stats = time_us(lambda: (in_stats(), in_finalize()), iters)
    t_act = time_us(lambda: ops.in_act(y, isc, ish, o1, ops.ACT_LRELU, o2, ops.ACT_RELU), iters)
    row("in_stats+bn_finalize", "(conv epilogue)", t_stats, t_bn_act, size, 3 * size)
    row("in_act", "bn_act", t_act, t_bn_act, 3 * size, 3 * size)
    row("in_stats+in_act", "bn_act", t_stats + t_act, t_bn_act, 4 * size, 3 * size)
    t_bred = time_us(lambda: ops.bn_bwd_reduce(y, g1, g2, 0.2, bsc, bsh, bmu, biv, bsums), iters)
    t_ired = time_us(lambda: ops.in_bwd_reduce(y, g1, g2, 0.2, isc, ish, isums), iters)
    row("in_bwd_reduce", "bn_bwd_reduce", t_ired, t_bred, 3 * size, 3 * size)
    bsums.zero_()
    isums.zero_()
    ops.in_bwd_reduce(y, g1, g2, 0.2, isc, ish, isums)
    t_bapp = time_us(lambda: ops.bn_bwd_apply(y, g1, g2, 0.2, bsc, bsh, bmu, biv, bsums, count, dy), iters)
    t_iapp = time_us(lambda: ops.in_bwd_apply(y, g1, g2, 0.2, isc, ish, isums, dy, dbias), iters)
    row("in_bwd_apply(+dbias)", "bn_bwd_apply", t_iapp, t_bapp, 4 * size, 4 * size)
    return rows


def steps(n_steps: int, blocks: int) -> list:
    dev = torch.device("cuda")
    g = torch.Generator().manual_seed(0)
    A = (torch.rand(64, 3, 256, 256, generator=g) * 2 - 1).to(dev)
    B = (torch.rand(64, 3, 256, 256, generator=g) * 2 - 1).to(dev)
    trainers = {}
    for norm in ("batch", "instance"):
        torch.manual_seed(0)
        trainers[norm] = Pix2PixTrainer(dev, norm=norm)
        for _ in range(5):
            trainers[norm].train_step_graphed(A, B)
    torch.cuda.synchronize()
    per = max(1, n_steps // blocks)
    times = {k: [] for k in trainers}
    for _ in range(blocks):
        for norm, tr in trainers.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(per):
                tr.train_step_graphed(A, B)
            e1.record()
            torch.cuda.synchronize()
            times[norm].append(e0.elapsed_time(e1) / per)
    out = []
    for norm, t in times.items():
        ms = sorted(t)[len(t) // 2]
        out.append({"step": "train_step_graphed", "norm": norm, "batch": 64, "size": 256, "steps": per * blocks,
                    "ms_per_step_median_block": round(ms, 3), "ms_blocks": [round(x, 3) for x in t],
                    "images_per_s": round(64 / ms * 1e3, 1)})
    out.append({"step": "instance_over_batch", "ratio": round(out[1]["ms_per_step_median_block"]
                                                              / out[0]["ms_per_step_median_block"], 4)})
    return out


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--iters", type=int, default=50, help="timed launches per kernel (>= 20)")
    ap.add_argument("--steps", type=int, default=50, help="timed training steps per norm (>= 50)")
    ap.add_argument("--blocks", type=int, default=5, help="interleaved blocks the steps are split into")
    ap.add_argument("--out", type=Path, default=None, help="also write all results as JSON here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_instance_norm needs a CUDA device (the gap_* kernels have no CPU path)")
    res = {"env": device_info(), "kernels": [], "steps": []}
    print(json.dumps(res["env"]), flush=True)
    for shape in SHAPES:
        for r in kernels(shape, a.iters):
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
