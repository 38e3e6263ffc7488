#!/usr/bin/env python
"""Benchmark of the Pix2Pix G+D training iteration (BASELINE.json metric: "Pix2Pix G+D train
images/sec at 256^2").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

ours:       one process per GPU (torchrun for N > 1), batch 64 per GPU, 256x256 synthetic RGB pairs,
            bf16 tensor-core kernels from libgap_b200.so; prints ONE JSON line on rank 0.
reference:  the reference's own CPU implementation of the path — its unmodified models.py + train_gan.train_gan_one_epoch,
            byte-compiled into oracle/_ref by oracle/stage_ref.py — timed on this box's host cores with every host
            thread, same config (batch 64 per step), metric and unit.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

BATCH_PER_GPU = 64
HW = 256
GFLOP_PER_IMG = 86.789062656     # SURVEY.md §8(d): 3*G + 8*D - 2*D.0 - G.0, convolutions only
METRIC = "pix2pix_gd_train_images_per_sec_256"
UNIT = "images/s"


def _peaks() -> dict:
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        d["_source"] = "measured"
        return d
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "_source": "fallback"}


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons while the timed region runs, every 25 ms (the profiling recipe polls
    every 200 ms).  Polling every 4 ms, as this did at first, cost the timed region 3-4 %: the device-resident loop
    measured 7.70 / 8.07 / 7.89 ms per iteration on three boxes where the end-to-end loop right after it, which does
    strictly more work but ran without the sampler, took 7.57 / 7.65 / 7.59 ms (NVML queries take the driver's per-GPU
    lock, which the launching thread needs ~170 times per iteration; an in-process sampler thread, which used to run
    beside the child, also takes the GIL from it)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    _CHILD = r'''
import sys, time
import pynvml as nv
nv.nvmlInit()
uuid, idx = sys.argv[1], int(sys.argv[2])
try:
    h = nv.nvmlDeviceGetHandleByUUID(uuid.encode())
except Exception:
    h = nv.nvmlDeviceGetHandleByIndex(idx)
mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
while True:
    try:
        rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
    except Exception:
        rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
    print(time.time(), nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM), mx, nv.nvmlDeviceGetPowerUsage(h) / 1000.0, rs,
          flush=True)
    time.sleep(0.025)
'''

    def __init__(self, index: int) -> None:
        """Starts an NVML sampler in a child process right away (it needs ~1 s to come up and, unlike a thread, does not
        compete with the launching thread for the GIL); `with sampler:` marks the window whose samples are kept."""
        self.index = index
        self.rows: list[list[str]] = []
        self._stop = threading.Event()
        self._t = None
        self._t0 = self._t1 = 0.0
        self._child = None
        try:
            uuid = "GPU-" + str(torch.cuda.get_device_properties(index).uuid)
            self._child = subprocess.Popen([sys.executable, "-c", self._CHILD, uuid, str(index)], stdout=subprocess.PIPE,
                                           stderr=subprocess.DEVNULL, text=True)
            import atexit
            atexit.register(self._kill_child)      # never leave the sampler behind, whatever happens to the run
        except Exception:
            self._child = None

    def _kill_child(self) -> None:
        c = self._child
        if c is not None and c.poll() is None:
            try:
                c.kill()
            except Exception:
                pass

    def _run_nvml(self) -> bool:
        """In-process NVML sampling every 25 ms (the same counters nvidia-smi prints; one nvidia-smi invocation takes
        longer than a whole default timed region).  Returns False when NVML is unavailable."""
        try:
            import pynvml as nv
            nv.nvmlInit()
            try:        # NVML ignores CUDA_VISIBLE_DEVICES: find the device torch calls `index` by its UUID
                h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + str(torch.cuda.get_device_properties(self.index).uuid)).encode())
            except Exception:
                h = nv.nvmlDeviceGetHandleByIndex(self.index)
            mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
        except Exception:
            return False
        bits = ((0x8, 3), (0x40, 4), (0x20, 5), (0x4, 6))      # hw_slowdown, hw_thermal, sw_thermal, sw_power_cap
        while not self._stop.is_set():
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                row = [str(sm), str(mx), str(nv.nvmlDeviceGetPowerUsage(h) / 1000.0), "", "", "", ""]
                for mask, col in bits:
                    row[col] = "Active" if rs & mask else "Not Active"
                self.rows.append(row)
            except Exception:
                pass
            self._stop.wait(0.025)
        return True

    def _run(self) -> None:
        if self._run_nvml():
            return
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5)
                if out.returncode == 0 and out.stdout.strip():
                    self.rows.append([c.strip() for c in out.stdout.strip().splitlines()[0].split(",")])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._t0 = time.time()
        # the in-process thread is only the fallback for a child that could not be started: a second Python thread
        # contends with the launching thread for the GIL inside the timed region
        if self._child is None or self._child.poll() is not None:
            self._child = None
            self._t = threading.Thread(target=self._run, daemon=True)
            self._t.start()
        return self

    def __exit__(self, *a):
        self._t1 = time.time()
        self._stop.set()
        if self._t is not None:
            self._t.join(timeout=6)
        if self._child is not None:
            try:
                self._child.terminate()
                out, _ = self._child.communicate(timeout=5)
            except Exception:
                out = ""
            rows = []
            for slack in (0.0, 0.03):       # a window shorter than the sampling period: take the samples next to it
                for line in out.splitlines():
                    f = line.split()
                    if len(f) != 5:
                        continue
                    try:
                        ts, sm, mx, pw, rs = float(f[0]), f[1], f[2], f[3], int(f[4])
                    except ValueError:
                        continue
                    if self._t0 - slack <= ts <= self._t1 + slack:
                        act = lambda m: "Active" if rs & m else "Not Active"
                        rows.append([sm, mx, pw, act(0x8), act(0x40), act(0x20), act(0x4)])
                if rows:
                    break
            if len(rows) > len(self.rows):      # the child saw more of the window than the in-process thread
                self.rows = rows

    def summary(self) -> dict:
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        mx = max((float(r[1]) for r in self.rows if r[1].replace(".", "").isdigit()), default=None)
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        pw = sorted(float(r[2]) for r in self.rows if r[2].replace(".", "").isdigit())
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": reasons,
                "samples": len(self.rows), "power_w": pw[len(pw) // 2] if pw else None}


def _host_threads() -> int:
    """Host threads this process may use (torchrun exports OMP_NUM_THREADS=1, which must not throttle the CPU arm)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def _gan_config(world: int) -> dict:
    """The workload description shared by both arms (the driver compares these)."""
    return {"workload": "pix2pix_gan_train_b64_256x256", "batch_per_gpu": BATCH_PER_GPU, "image": f"{HW}x{HW}x3",
            "parallelism": f"dp{world}", "algorithmic_gflop_per_image": GFLOP_PER_IMG,
            "l2": "no flush needed: the per-step working set (several GB of activations) >> 126 MB L2, and two input "
                  "batches alternate"}


class ReferenceGanLoop:
    """The reference's OWN iteration: `train_gan.train_gan_one_epoch` (train_gan.py:46-75) over its own
    `models.UNetGenerator` / `NLayerDiscriminator` with `optim.Adam(1e-4, (0.5, 0.999))` (train_gan.py:138-141), loaded
    from oracle/_ref (the unmodified reference, byte-compiled by oracle/stage_ref.py).  mode "fp32" = the reference as
    it is; "bf16_cl" = the same loop under torch.autocast(bfloat16) with channels_last modules and inputs (the best
    the existing library kernels offer).  `models` swaps in another implementation of the models.py surface (the
    drop-in modules).  Falls back to the oracle port (kind "port") when oracle/_ref is not staged."""

    def __init__(self, device, batch: int, mode: str = "fp32", models=None, tag: str = "ref") -> None:
        from oracle import ref_loader
        self.dev = torch.device(device)
        self.mode = mode
        self.batch = batch
        g = torch.Generator().manual_seed(1234)
        self.batches = []
        for _ in range(2):
            a = (torch.rand(batch, 3, HW, HW, generator=g) * 2 - 1).to(self.dev)
            b = (torch.rand(batch, 3, HW, HW, generator=g) * 2 - 1).to(self.dev)
            if mode == "bf16_cl":
                a, b = a.contiguous(memory_format=torch.channels_last), b.contiguous(memory_format=torch.channels_last)
            self.batches.append({"image1": a, "image2": b})
        torch.manual_seed(0)
        if ref_loader.available():
            self.kind = "reference"
            ns = ref_loader.load(models=models, tag=tag)
            ns.train_gan.DEVICE = self.dev          # configuration constant of the script (train_gan.py:25)
            self.ns = ns
            self.gen = ns.train_gan.UNetGenerator(input_nc=3, output_nc=3).to(self.dev)
            self.disc = ns.train_gan.NLayerDiscriminator(input_nc=6).to(self.dev)
            if mode == "bf16_cl":
                self.gen = self.gen.to(memory_format=torch.channels_last)
                self.disc = self.disc.to(memory_format=torch.channels_last)
            self.opt_g = torch.optim.Adam(self.gen.parameters(), lr=1e-4, betas=(0.5, 0.999))
            self.opt_d = torch.optim.Adam(self.disc.parameters(), lr=1e-4, betas=(0.5, 0.999))
        else:
            if models is not None or mode != "fp32":
                raise FileNotFoundError("oracle/_ref is not staged")
            from oracle import pix2pix_oracle as O
            from gan_aug_pfa_b200 import spec as MI
            self.kind = "port"
            self.O = O
            sd_g, sd_d = MI.default_state_dicts()
            self.sd = tuple({k: v.to(self.dev) for k, v in sd.items()} for sd in (sd_g, sd_d))
            self.opt = (O.AdamState(self.sd[0], O.param_names(self.sd[0]), 1e-4, (0.5, 0.999)),
                        O.AdamState(self.sd[1], O.param_names(self.sd[1]), 1e-4, (0.5, 0.999)))

    def step(self, i: int):
        batch = self.batches[i % 2]
        if self.kind == "port":
            return self.O.gan_train_step(self.sd[0], self.sd[1], self.opt[0], self.opt[1], batch["image1"], batch["image2"])[:2]
        if self.mode == "bf16_cl":
            with torch.autocast(self.dev.type, dtype=torch.bfloat16):
                return self.ns.train_gan.train_gan_one_epoch(self.gen, self.disc, [batch], self.opt_g, self.opt_d)
        return self.ns.train_gan.train_gan_one_epoch(self.gen, self.disc, [batch], self.opt_g, self.opt_d)


def _time_cpu_loop(loop: ReferenceGanLoop, steps: int, warmup: int, budget_s: float):
    """Runs `warmup` untimed and up to `steps` timed iterations; stops early when the projected total exceeds
    `budget_s` (each iteration is a full batch of the workload: ~7 TFLOP of fp32 on the host cores).  Returns
    (images/s, seconds per step, steps executed)."""
    t_w = time.perf_counter()
    for i in range(warmup):
        loop.step(i)
    per = (time.perf_counter() - t_w) / max(1, warmup)
    n_run = steps if warmup == 0 else max(1, min(steps, int(budget_s / max(per, 1e-9))))
    t0 = time.perf_counter()
    done = 0
    for i in range(n_run):
        loop.step(i)
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    el = time.perf_counter() - t0
    return done * loop.batch / el, el / done, done


def _cpu_baseline(budget_s: float = 25.0) -> dict:
    """The CPU arm on a bounded sample: the unmodified reference loop (oracle/_ref) at the workload's own batch (64),
    fp32, every host thread: one untimed iteration, then as many timed ones as fit in ~25 s."""
    threads = _host_threads()
    torch.set_num_threads(threads)
    loop = ReferenceGanLoop("cpu", BATCH_PER_GPU, "fp32", tag="cpubase")
    val, per, done = _time_cpu_loop(loop, steps=8, warmup=1, budget_s=budget_s)
    return {"value": val, "unit": UNIT, "cores": threads, "kind": loop.kind,
            "sample": f"{done} iteration(s) of train_gan_one_epoch at batch {BATCH_PER_GPU}, 256x256, fp32 after 1 warm-up "
                      f"({per:.1f} s each) on {threads} host threads"}


def run_reference(args) -> None:
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref: its unmodified models.py +
    train_gan.train_gan_one_epoch) on this box's host cores, same config / metric / unit as our arm.  Each step is one
    full batch-64 iteration; when K of them would not fit in ~4 minutes, fewer are executed and `steps_executed` says
    how many (the rate is per executed step)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = _host_threads()
    torch.set_num_threads(threads)
    loop = ReferenceGanLoop("cpu", BATCH_PER_GPU, "fp32", tag="cpuarm")
    val, per, done = _time_cpu_loop(loop, steps=args.steps, warmup=max(1, min(args.warmup, 1)), budget_s=200.0)
    sample = (f"{done} of {args.steps} steps executed, each one train_gan_one_epoch iteration at batch {BATCH_PER_GPU}, "
              f"256x256, fp32, {threads} host threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "steps_executed": done, "warmup": args.warmup, "ms_per_step": 1e3 * per, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _gan_config(args.gpus),
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": loop.kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def _gpu_loop_rate(loop: ReferenceGanLoop, steps: int, warmup: int) -> float:
    for i in range(warmup):
        loop.step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        loop.step(i)
    e1.record()
    torch.cuda.synchronize()
    return steps * loop.batch / (e0.elapsed_time(e1) * 1e-3)


def _library_baseline(dev) -> dict:
    """SURVEY.md §8(d) / BASELINE.md §2: the existing Blackwell library kernels on this very GPU — the unmodified
    reference loop with DEVICE=cuda (torch eager -> cuDNN 9 / ATen), batch 64, (a) as it is (fp32 tensors; torch's
    default lets cuDNN use TF32 for convolutions) and (b) under bf16 autocast with channels_last."""
    out = {"unit": UNIT, "batch": BATCH_PER_GPU,
           "what": "oracle/_ref train_gan_one_epoch + reference models on cuda via torch eager (cuDNN), "
                   "cudnn.benchmark on, 3 warm-up + 5 timed iterations, CUDA events"}
    prev = torch.backends.cudnn.benchmark
    torch.backends.cudnn.benchmark = True
    try:
        for mode in ("fp32", "bf16_cl"):
            key = "fp32" if mode == "fp32" else "bf16_autocast_channels_last"
            try:
                loop = ReferenceGanLoop(dev, BATCH_PER_GPU, mode, tag="lib_" + mode)
                out[key] = _gpu_loop_rate(loop, steps=5, warmup=3)
                del loop
            except Exception as e:      # a missing staged reference must not kill the bench line
                out[key] = None
                out[key + "_error"] = f"{type(e).__name__}: {e}"[:200]
            torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.benchmark = prev
    return out


def _dropin_leg(dev) -> dict:
    """The path the unchanged scripts take: the reference's real train_gan_one_epoch (oracle/_ref) driving the drop-in
    gan_aug_pfa_b200.models modules through torch autograd and torch.optim.Adam, batch 64."""
    from gan_aug_pfa_b200 import models as M
    try:
        loop = ReferenceGanLoop(dev, BATCH_PER_GPU, "fp32", models=M, tag="dropin")
        val = _gpu_loop_rate(loop, steps=5, warmup=3)
        del loop
        torch.cuda.empty_cache()
        return {"value": val, "unit": UNIT, "what": "oracle/_ref train_gan.train_gan_one_epoch on the drop-in modules "
                "(torch autograd + torch.optim.Adam around the native engine; the reference's second generator forward "
                "and its discarded D weight gradients are executed, 105.2 GFLOP/image)"}
    except Exception as e:
        return {"value": None, "error": f"{type(e).__name__}: {e}"[:200]}


def _roofline_dict(ach_tf: float, peaks: dict, **extra) -> dict:
    """Tensor-bound roofline entry.  `frac` is quoted against the BURST peak (MEASURED_PEAKS.json bf16_tflops): the
    timed regions here last a fraction of a second at ~1.75-1.8 GHz, the conditions the burst figure was measured
    under; `frac_sustained` divides by the seconds-long sustained figure (median 1357 MHz) for comparison."""
    burst = peaks["bf16_tflops"]
    sus = peaks.get("bf16_tflops_sustained", burst)
    d = {"bound": "tensor", "achieved": ach_tf, "peak": burst, "unit": "TFLOP/s", "frac": ach_tf / burst,
         "peak_sustained": sus, "frac_sustained": ach_tf / sus,
         "peak_source": f"{peaks['_source']} MEASURED_PEAKS.json: bf16_tflops (burst) for frac, bf16_tflops_sustained for "
                        "frac_sustained"}
    d.update(extra)
    return d


def _setup_dist():
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device: the gap_* kernels have no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not dist.is_initialized():
        dist.init_process_group("nccl", device_id=dev)
    return dist, world, rank, local, dev


def _barrier(dist, world):
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


def _max_over_ranks(dist, world, dev, *vals):
    if world > 1:
        t = torch.tensor(list(vals), device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(v) for v in t.tolist()]
    return list(vals)


DUMP_PARAM_SAMPLE = 1 << 19     # state_dict / gradient entries per network that --dump-outputs keeps


def dump_outputs(out_dir: str, tr, losses: torch.Tensor) -> None:
    """--dump-outputs: what one training step `tr` just ran hands its caller, as .npy files in `out_dir` (58 MB in
    all): the step's [loss_d, loss_g] (fp64), the generator's output images of the step (fp32 NCHW, the whole batch)
    and, for each network, one fixed seeded sample of its state_dict after the step's Adam update (floating-point
    entries flattened in key order, fp32) and of the step's parameter gradients (parameters in key order, fp32: a first
    Adam step moves every weight by about lr * sign(gradient), so the weights alone hardly show gradient magnitudes).
    Two builds run with the same arguments can be compared file by file."""
    import numpy as np
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    np.save(out / "losses.npy", losses.detach().cpu().double().numpy())
    np.save(out / "fake_B.npy", tr.G.output_nchw().cpu().numpy())
    for name, net in (("G", tr.G), ("D", tr.D)):
        flat = torch.cat([v.detach().reshape(-1).float() for v in net.state_dict().values() if v.is_floating_point()])
        idx = torch.randint(flat.numel(), (DUMP_PARAM_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
        np.save(out / f"{name}_state_sample.npy", flat[idx.to(flat.device)].cpu().numpy())
        flat = torch.cat([net.grad(k).reshape(-1) for k in net.key_order if k in net.views])
        idx = torch.randint(flat.numel(), (DUMP_PARAM_SAMPLE,), generator=torch.Generator().manual_seed(1)).sort().values
        np.save(out / f"{name}_grad_sample.npy", flat[idx.to(flat.device)].cpu().numpy())


def run_ours(args) -> None:
    from gan_aug_pfa_b200 import _lib, checkpoint, ops, parallel
    from gan_aug_pfa_b200.io import PairPrefetcher
    from gan_aug_pfa_b200.pix2pix import Pix2PixTrainer

    dist, world, rank, local, dev = _setup_dist()
    clock_sampler = ClockSampler(local)       # the child process needs a moment to come up: start it before the warm-up
    torch.manual_seed(0)
    tr = Pix2PixTrainer(dev, world=world)     # world > 1: bucketed NCCL all-reduce overlapped with the backward pass;
    #                                           replicas are broadcast from rank 0 at construction
    start = checkpoint.trainer_state(tr) if args.dump_outputs else None     # the seeded initial state
    N = BATCH_PER_GPU
    gen = torch.Generator().manual_seed(1234 + rank)
    n_batches = 2
    if args.inputs == "u8":     # raw uint8 images; ToTensor + JointNormalize run on the device (SURVEY 8f-2)
        host = [(torch.randint(0, 256, (N, HW, HW, 3), generator=gen, dtype=torch.uint8).pin_memory(),
                 torch.randint(0, 256, (N, HW, HW, 3), generator=gen, dtype=torch.uint8).pin_memory())
                for _ in range(n_batches)]
    else:                       # fp32 NCHW in [-1, 1]: what the reference's DataLoader hands to train_gan.py:53-54
        host = [(torch.rand(N, 3, HW, HW, generator=gen).mul_(2).sub_(1).pin_memory(),
                 torch.rand(N, 3, HW, HW, generator=gen).mul_(2).sub_(1).pin_memory()) for _ in range(n_batches)]
    devb = [(a.to(dev), b.to(dev)) for a, b in host]

    # Single GPU: the iteration's launches can be replayed from one CUDA graph (same kernels, no launch gaps) or
    # launched eagerly (three streams; the host enqueues a step faster than the GPU runs it).  Which is faster depends
    # on the host: calibrate both during warm-up (untimed, interleaved so clock drift cancels) and keep the faster.
    step_fn, use_graph = tr.train_step, False
    for i in range(args.warmup):
        step_fn(*devb[i % n_batches])
    if world == 1 and args.step_mode != "eager":
        use_graph = True
        if args.step_mode == "auto":
            def block(fn, n=5):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                a.record()
                for i in range(n):
                    fn(*devb[i % n_batches])
                b.record()
                torch.cuda.synchronize()
                return a.elapsed_time(b)
            block(tr.train_step_graphed, 3)                      # capture + first replays
            t_e = t_g = 0.0
            for r in range(4):                                   # ABBA order: clock drift cancels
                if r % 2 == 0:
                    t_e += block(tr.train_step)
                    t_g += block(tr.train_step_graphed)
                else:
                    t_g += block(tr.train_step_graphed)
                    t_e += block(tr.train_step)
            use_graph = t_g < t_e
        if use_graph:
            step_fn = tr.train_step_graphed
            for i in range(3):
                step_fn(*devb[i % n_batches])
    # ---- device-resident timing
    _barrier(dist, world)
    _lib.LAUNCHES = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with clock_sampler as clocks:
        _barrier(dist, world)
        e0.record()
        for i in range(args.steps):
            losses = step_fn(*devb[i % n_batches])
        e1.record()
        _barrier(dist, world)
    launches = _lib.LAUNCHES
    if use_graph:
        # graph replays do not pass through the Python launchers: count the launches of one eager iteration
        _lib.LAUNCHES = 0
        tr.train_step(*devb[0])
        launches = _lib.LAUNCHES * args.steps
    (ms,) = _max_over_ranks(dist, world, dev, e0.elapsed_time(e1))
    value = world * N * args.steps / (ms * 1e-3)
    loss_host = losses.cpu().tolist()
    if args.dump_outputs:
        # The timed steps train from the weights the warm-up and calibration steps left, and the step's fp32 atomic
        # reductions do not add up in the same order on every run, so those weights (and what is computed from them)
        # drift apart from run to run.  The step that is written out is therefore the timed step function once more,
        # on the last timed step's batch, from the seeded initial state: restored in place (captured graphs stay
        # valid), these inputs are the same on every run.
        checkpoint.load_trainer_state(tr, start, restore_rng=False)
        out = step_fn(*devb[(args.steps - 1) % n_batches])
        if rank == 0:
            dump_outputs(args.dump_outputs, tr, out)

    # ---- end to end through the public API: pinned host batches -> PairPrefetcher (H2D on a copy stream into two
    # staging buffers while the previous iteration computes) -> train_step -> the step's losses copied back to pinned
    # host memory EVERY step; the host waits for step i-1's losses while step i is already enqueued (a one-step lag:
    # the reference's `.item()` per step, train_gan.py:72-74, without draining the GPU between iterations).
    pre = PairPrefetcher(dev, [host[i % n_batches] for i in range(args.steps)]).preallocate(host[0])
    loss_pinned = [torch.empty(2, dtype=torch.float64).pin_memory() for _ in range(2)]
    ev_loss = [torch.cuda.Event(), torch.cuda.Event()]
    cur = torch.cuda.current_stream()
    seen = []
    zero_copy = not use_graph        # eager: the step's last kernel stores the losses straight into pinned host memory
    _barrier(dist, world)
    e0.record()
    for i, (a, b) in enumerate(pre):
        if zero_copy:
            step_fn(a, b, loss_host=loss_pinned[i % 2])
        else:
            out = step_fn(a, b)
        pre.release()                                    # the staging buffers of this batch may be refilled
        if not zero_copy:
            loss_pinned[i % 2].copy_(out, non_blocking=True)
        ev_loss[i % 2].record(cur)
        if i >= 1:
            ev_loss[(i - 1) % 2].synchronize()
            seen.append(loss_pinned[(i - 1) % 2].tolist())
    ev_loss[(args.steps - 1) % 2].synchronize()
    seen.append(loss_pinned[(args.steps - 1) % 2].tolist())
    e1.record()
    _barrier(dist, world)
    (ms_e2e,) = _max_over_ranks(dist, world, dev, e0.elapsed_time(e1))
    e2e_value = world * N * args.steps / (ms_e2e * 1e-3)
    assert len(seen) == args.steps

    # ---- per-kernel roofline: time every GEMM launch of a few steps with CUDA events
    # (side streams serialised for these steps: with the generator forward / the wgrads overlapping other kernels a
    # launch's event-to-event time would include the work it shares the GPU with)
    prof_steps = min(2, args.steps)
    saved = (tr.overlap_g_fwd, tr.G.overlap_wgrad, tr.D.overlap_wgrad)
    tr.overlap_g_fwd = tr.G.overlap_wgrad = tr.D.overlap_wgrad = False
    tr.train_step(*devb[0])
    ops.PROFILE = []
    for i in range(prof_steps):
        tr.train_step(*devb[i % n_batches])
    torch.cuda.synchronize()
    prof = ops.PROFILE
    ops.PROFILE = None
    tr.overlap_g_fwd, tr.G.overlap_wgrad, tr.D.overlap_wgrad = saved
    agg: dict = {}
    for name, flops, ev0, ev1 in prof:
        d = agg.setdefault(name, [0.0, 0.0, 0])
        d[0] += flops
        d[1] += ev0.elapsed_time(ev1) * 1e-3
        d[2] += 1
    peaks = _peaks()
    kern = {k: {"tflops": v[0] / v[1] / 1e12 if v[1] > 0 else 0.0, "seconds_per_step": v[1] / prof_steps,
                "launches_per_step": v[2] // prof_steps} for k, v in agg.items()}
    dom = max(agg.items(), key=lambda kv: kv[1][1])[0] if agg else None
    roofline = None
    if dom is not None:
        traffic = None
        for tname in ("r2_roofline_traffic.json", "r1_roofline_traffic.json"):
            tpath = ROOT / "profiles" / tname
            if tpath.exists():
                traffic = json.loads(tpath.read_text()).get(dom, {}).get("dram_bytes_per_launch")
                break
        step_tf = (value / world) * GFLOP_PER_IMG * 1e9 / 1e12
        roofline = _roofline_dict(
            kern[dom]["tflops"], peaks, kernel=dom, traffic=traffic,
            traffic_source=f"ncu dram__bytes_read+write per launch, averaged over the step's launches (profiles/{tname})"
            if traffic else None,
            algorithmic_flop_per_launch=agg[dom][0] / max(1, agg[dom][2]), per_kernel=kern,
            step_tflops=step_tf, step_frac_of_peak=step_tf / peaks["bf16_tflops"],
            step_frac_of_sustained=step_tf / peaks.get("bf16_tflops_sustained", peaks["bf16_tflops"]))

    # ---- data-parallel correctness signal + the other BASELINE configs, every rank takes part
    replica_diff = parallel.replica_param_max_abs_diff([tr.G, tr.D]) if world > 1 else None
    del tr, devb, pre
    torch.cuda.empty_cache()
    secondary = {}
    if args.secondary:
        for wl in ("gen_infer", "siamese_train"):
            secondary[wl] = measure_secondary(wl, steps=max(3, min(args.steps, 8)), warmup=3, dist=dist, world=world,
                                              rank=rank, dev=dev)
            torch.cuda.empty_cache()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": _gan_config(world), "cuda_graph": use_graph,
            "clocks": clocks.summary(),
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": sum(t.numel() * t.element_size() for t in host[0]),
                    "d2h_bytes_per_step": 16, "ms_per_step": ms_e2e / args.steps, "inputs": args.inputs,
                    "how": "PairPrefetcher (pinned host -> device staging on a copy stream) + train_step + the step's two "
                           "losses written to pinned host memory every step (by the last kernel itself when eager, by a "
                           "D2H copy after a graph replay), read by the host with a one-step lag"},
            "gpu_launches": launches,
            "roofline": roofline,
            "final_losses": {"loss_d": loss_host[0], "loss_g": loss_host[1]},
        }
        if replica_diff is not None:
            line["replica_param_max_abs_diff"] = replica_diff
        if secondary:
            line["secondary"] = secondary
        if world == 1 and args.baselines:
            line["dropin"] = _dropin_leg(dev)
            line["library_baseline"] = _library_baseline(dev)
            line["cpu_baseline"] = _cpu_baseline()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def measure_secondary(workload: str, steps: int, warmup: int, dist, world: int, rank: int, dev) -> dict:
    """BASELINE.json configs 4 and 5 with the same timing rules as the main leg: generator inference (batch 256, eval
    BatchNorm; independent replicas, no collective) and the Siamese U-Net training step at 512x512 (batch 4 per GPU,
    CombinedLoss; data parallel with the gradient all-reduce overlapped with the backward pass when world > 1)."""
    from gan_aug_pfa_b200 import _lib
    torch.manual_seed(0)
    gen = torch.Generator().manual_seed(1234 + rank)
    if workload == "gen_infer":
        from gan_aug_pfa_b200.pix2pix import GeneratorEngine
        N = 256
        eng = GeneratorEngine(dev)
        eng.training = True
        warm = (torch.rand(8, 3, HW, HW, generator=gen) * 2 - 1).to(dev)
        for _ in range(2):
            eng.forward(warm)                      # non-trivial running statistics, as after training
        eng.training = False
        # device-resident leg: fp32 NCHW inputs (the models.py contract).  End-to-end leg: what generate_synthetic_data.py's
        # loop moves — uint8 HWC images in (normalised on the device) and uint8 HWC images out (written by the last layer's
        # epilogue), pinned host buffers, H2D / D2H on copy streams overlapped with the previous / next batch's compute.
        host = [(torch.rand(N, 3, HW, HW, generator=gen) * 2 - 1).pin_memory() for _ in range(2)]
        devb = [h.to(dev) for h in host]
        host_u8 = [torch.randint(0, 256, (N, HW, HW, 3), generator=gen, dtype=torch.uint8).pin_memory() for _ in range(2)]
        in_u8 = [torch.empty(N, HW, HW, 3, device=dev, dtype=torch.uint8) for _ in range(2)]
        out_u8 = [torch.empty(N, HW, HW, 3, device=dev, dtype=torch.uint8) for _ in range(2)]
        out_host = [torch.empty(N, HW, HW, 3, dtype=torch.uint8).pin_memory() for _ in range(2)]
        cur = torch.cuda.current_stream()
        h2d_s, d2h_s = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
        ev_in = [torch.cuda.Event(), torch.cuda.Event()]
        ev_done = [torch.cuda.Event(), torch.cuda.Event()]
        ev_out = [torch.cuda.Event(), torch.cuda.Event()]
        state = {"i": 0}

        def step(i, e2e=False):
            if not e2e:
                eng.forward(devb[i % 2])
                return
            k = i % 2
            if state["i"] == 0:                         # first e2e call: start the input pipeline
                h2d_s.wait_stream(cur)
                d2h_s.wait_stream(cur)
                with torch.cuda.stream(h2d_s):
                    in_u8[k].copy_(host_u8[k], non_blocking=True)
                    ev_in[k].record(h2d_s)
            state["i"] += 1
            with torch.cuda.stream(h2d_s):              # prefetch the next batch while this one computes
                h2d_s.wait_event(ev_done[1 - k])        # (its buffer was consumed by the previous forward)
                in_u8[1 - k].copy_(host_u8[1 - k], non_blocking=True)
                ev_in[1 - k].record(h2d_s)
            cur.wait_event(ev_in[k])
            cur.wait_event(ev_out[k])                   # the D2H of two batches ago has drained out_u8[k]
            eng.forward(in_u8[k], out_u8=out_u8[k])
            ev_done[k].record(cur)
            with torch.cuda.stream(d2h_s):
                d2h_s.wait_event(ev_done[k])
                out_host[k].copy_(out_u8[k], non_blocking=True)
                ev_out[k].record(d2h_s)
            if i == steps - 1:
                d2h_s.synchronize()                     # every image of the timed region has reached the host
                cur.wait_stream(d2h_s)
        units, metric, unit = N, "generator_inference_images_per_sec_256", "images/s"
        gflop = 12.046041088
        h2d, d2h = N * 3 * HW * HW, N * 3 * HW * HW          # uint8 images both ways
        cfg = {"workload": "generator_inference_b256_256x256", "batch_per_gpu": N, "bn": "eval (running statistics)",
               "parallelism": f"replicas x{world}"}
        extra = {}
    else:
        from gan_aug_pfa_b200 import models as M
        from gan_aug_pfa_b200 import parallel
        from gan_aug_pfa_b200.siamese import SiameseEngine
        N, S = 4, 512
        eng = SiameseEngine(dev)
        torch.manual_seed(0)
        eng.load_state_dict({k: v.detach() for k, v in M.SiameseUNet(3, 1).state_dict().items()})
        if world > 1:
            parallel.broadcast_replica_state([eng])
            eng.reducer = parallel.TailReducer(eng.store.g)
        host = [((torch.rand(N, 3, S, S, generator=gen) * 2 - 1).pin_memory(),
                 (torch.rand(N, 3, S, S, generator=gen) * 2 - 1).pin_memory(),
                 (torch.rand(N, S, S, generator=gen) < 0.05).long().pin_memory()) for _ in range(2)]
        devb = [tuple(t.to(dev) for t in b) for b in host]
        stage = tuple(torch.empty_like(t) for t in devb[0])
        loss_host = torch.empty(1, dtype=torch.float64).pin_memory()

        def step(i, e2e=False):
            b = devb[i % 2]
            if e2e:
                for dst, src in zip(stage, host[i % 2]):
                    dst.copy_(src, non_blocking=True)
                b = stage
            loss = eng.train_step(*b, kind="combined", grad_scale=1.0 / world)
            if e2e:
                loss_host.copy_(loss, non_blocking=True)
                torch.cuda.current_stream().synchronize()
        units, metric, unit = N, "siamese_train_pairs_per_sec_512", "pairs/s"
        gflop = 2207.23
        h2d, d2h = 2 * N * 3 * S * S * 4 + N * S * S * 8, 8
        cfg = {"workload": "siamese_unet_train_b4_512x512_combined_loss", "batch_per_gpu": N, "loss": "CombinedLoss(0.5, 1:9)",
               "optimizer": "AdamW(1.0152e-4, wd 1.118e-5)",
               "parallelism": f"dp{world}" + (" (NCCL gradient all-reduce overlapped with the backward pass)" if world > 1 else "")}
        extra = {}

    for i in range(warmup):
        step(i)
    _barrier(dist, world)
    _lib.LAUNCHES = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    _barrier(dist, world)
    e0.record()
    for i in range(steps):
        step(i)
    e1.record()
    _barrier(dist, world)
    launches = _lib.LAUNCHES
    ms = e0.elapsed_time(e1)
    _barrier(dist, world)
    e0.record()
    for i in range(steps):
        step(i, e2e=True)
    e1.record()
    _barrier(dist, world)
    ms_e2e = e0.elapsed_time(e1)
    ms, ms_e2e = _max_over_ranks(dist, world, dev, ms, ms_e2e)
    if workload == "siamese_train":
        # the criterion train.py's main() actually builds (train.py:294, Optuna's constants): same step, other loss kernel
        fd = dict(kind="focal_dice", focal_alpha=0.6030489822904476, gamma=1.7930869982898021, beta=0.6699803915247974,
                  smooth=1.956571276926647e-06, grad_scale=1.0 / world)
        n_fd = max(2, min(steps, 5))
        for i in range(2):
            eng.train_step(*devb[i % 2], **fd)
        _barrier(dist, world)
        e0.record()
        for i in range(n_fd):
            eng.train_step(*devb[i % 2], **fd)
        e1.record()
        _barrier(dist, world)
        (ms_fd,) = _max_over_ranks(dist, world, dev, e0.elapsed_time(e1))
        extra["focal_dice_loss"] = {"value": world * units * n_fd / (ms_fd * 1e-3), "unit": unit, "steps": n_fd,
                                    "loss": "FocalDiceLoss(train.py:294 constants)"}
    if workload == "siamese_train" and world > 1:
        from gan_aug_pfa_b200 import parallel
        extra["replica_param_max_abs_diff"] = parallel.replica_param_max_abs_diff([eng])
    value = world * units * steps / (ms * 1e-3)
    peaks = _peaks()
    tf = (value / world) * gflop * 1e9 / 1e12
    out = {"metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": steps, "warmup": warmup,
           "ms_per_step": ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "bf16", "data": "synthetic", "config": cfg,
           "e2e": {"value": world * units * steps / (ms_e2e * 1e-3), "unit": unit, "h2d_bytes_per_step": h2d,
                   "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / steps},
           "gpu_launches": launches,
           "roofline": _roofline_dict(tf, peaks, traffic=None,
                                      note="whole-step algorithmic conv FLOP/s (SURVEY.md §8d) per GPU")}
    out.update(extra)
    return out


def run_secondary(args) -> None:
    dist, world, rank, local, dev = _setup_dist()
    clock_sampler = ClockSampler(local)
    with clock_sampler as clocks:
        out = measure_secondary(args.workload, args.steps, args.warmup, dist, world, rank, dev)
    out["clocks"] = clocks.summary()
    if rank == 0:
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pix2pix_train", choices=["pix2pix_train", "gen_infer", "siamese_train"],
                    help="pix2pix_train = the BASELINE.json metric (default; its JSON line also carries quick `secondary` "
                         "legs for the other two); gen_infer = generate_synthetic_data.py's generator forward at batch 256 "
                         "(config 4); siamese_train = train.py's step at 512x512, batch 4 per GPU (config 5, CombinedLoss)")
    ap.add_argument("--step-mode", default="auto", choices=["auto", "graph", "eager"],
                    help="single-GPU pix2pix_train: CUDA-graph replay, eager launches, or (default) whichever measures "
                         "faster in an untimed calibration after the warm-up")
    ap.add_argument("--inputs", default="u8", choices=["f32", "u8"],
                    help="pix2pix_train: host batches as raw uint8 HWC images normalised on the device (default: what an "
                         "image pipeline holds before dataset.py's ToTensor / JointNormalize) or as fp32 NCHW in [-1,1] "
                         "(the reference DataLoader's output, 4x the H2D bytes)")
    ap.add_argument("--no-secondary", dest="secondary", action="store_false",
                    help="skip the quick generator-inference / Siamese legs appended to the pix2pix_train line")
    ap.add_argument("--no-baselines", dest="baselines", action="store_false",
                    help="skip the drop-in, cuDNN library and CPU baseline legs (single GPU only)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="pix2pix_train: after the timed steps, run the timed step once more from the seeded initial "
                         "weights on the last timed batch and write what it computed (losses, generated images, a "
                         "seeded sample of the updated weights and of the step's gradients) as .npy files into DIR; the "
                         "legs after the timed window then continue from that restored-and-stepped state")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "pix2pix_train"):
        ap.error("--dump-outputs needs --impl ours --workload pix2pix_train")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "pix2pix_train":
        run_ours(args)
    else:
        run_secondary(args)


if __name__ == "__main__":
    main()
