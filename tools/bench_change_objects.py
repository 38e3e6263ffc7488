"""Change objects (objects.change_objects) on the GPU, in one process:

1. 8192 x 8192 seeded random maps (K = 2) at change densities 0.3 and 0.6, with and without labels of the same kind:
   the whole call (CUDA events, one warm-up call, median of --calls).  Each map is 67 MB, and with the int32 parents
   and ids the working set exceeds the 126 MB L2, so no pass is served from the previous one's cache;
2. the pred of a real 8192 x 8192 SiameseEngine.predict_scene call (K = 2, seeded weights, seeded uint8 pair on the
   device, tile 256 / overlap 64 / batch 8, the defaults), the time of that call, and change_objects on its map with
   min_area 16, as a share of the predict_scene call;
3. the bytes the passes must stream, from the shapes (the byte model is `streamed_bytes`; union-find chains and the
   scattered atomics are not counted), and their fraction of the 6527 GB/s HBM roof the other benches use;
4. scipy.ndimage.label on the host for the same maps (one call per change class), for reference;
5. the device name and enforced power limit, read from NVML in the same run.

    python tools/bench_change_objects.py [--calls 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
import time
from pathlib import Path

import torch
from scipy import ndimage

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

from gan_aug_pfa_b200 import models as M  # noqa: E402
from gan_aug_pfa_b200.objects import change_objects  # noqa: E402
from gan_aug_pfa_b200.siamese import SiameseEngine  # noqa: E402

ROOF_GBS = 6527.0
SIZE = 8192
K = 2


def device_info() -> dict:
    import pynvml as nv
    nv.nvmlInit()
    h = nv.nvmlDeviceGetHandleByIndex(torch.cuda.current_device())
    name = nv.nvmlDeviceGetName(h)
    return {"device": name.decode() if isinstance(name, bytes) else name,
            "power_limit_w": nv.nvmlDeviceGetEnforcedPowerLimit(h) / 1000.0}


def streamed_bytes(px: int, labels: bool) -> int:
    """Bytes per call that the passes stream, per pixel:
    pred: area clear 4; local: pred 1 + parent 4; flatten: pred 1 + parent 4; count and number: pred 1 + parent 4
    each; apply: parent 4 + ids 4 + pred 1 + filtered pred 1; table: ids 4 + parent 4 -> 42 B.
    labels: area and overlap clears 4 + 4; local: labels 8 + classes 1 + parent 4; flatten: classes 1 + parent 4;
    apply: label parent 4 + classes 1; table: label parent 4 -> 35 B more."""
    return px * (42 + (35 if labels else 0))


def time_calls(fn, calls: int) -> float:
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(calls):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return statistics.median(ts)


def scipy_ms(pred_cpu: torch.Tensor) -> float:
    p = pred_cpu.numpy()
    t = time.perf_counter()
    for c in range(1, K):
        ndimage.label(p == c, structure=ndimage.generate_binary_structure(2, 2))
    return (time.perf_counter() - t) * 1e3


def row(name: str, pred: torch.Tensor, labels, calls: int, **kw) -> dict:
    ms = time_calls(lambda: change_objects(pred, K, labels=labels, **kw), calls)
    r = change_objects(pred, K, labels=labels, **kw)
    b = streamed_bytes(pred.numel(), labels is not None)
    out = {"map": name, "labels": labels is not None, **kw, "objects": int(r.objects.shape[0]), "ms": round(ms, 3),
           "streamed_GB": round(b / 1e9, 3), "roof_fraction": round(b / 1e9 / (ms / 1e3) / ROOF_GBS, 3)}
    print(json.dumps(out), flush=True)
    return out


def main(calls: int) -> dict:
    dev = torch.device("cuda:0")
    res = {"info": device_info(), "rows": []}
    g = torch.Generator().manual_seed(0)
    for density in (0.3, 0.6):
        pred = (torch.rand(SIZE, SIZE, generator=g) < density).to(torch.uint8)
        lab = (torch.rand(SIZE, SIZE, generator=g) < density).long()
        pd, ld = pred.to(dev), lab.to(dev)
        for labels in (None, ld):
            res["rows"].append(row(f"random {density}", pd, labels, calls))
        res["rows"][-1]["scipy_ms"] = round(scipy_ms(pred), 1)
        del pd, ld
    torch.manual_seed(0)
    sd = {k: v.detach().clone() for k, v in M.SiameseUNet(3, K).state_dict().items()}
    eng = SiameseEngine(dev, 3, K)
    eng.load_state_dict(sd)
    u1, u2 = (torch.randint(0, 256, (SIZE, SIZE, 3), generator=g, dtype=torch.uint8).to(dev) for _ in range(2))
    lab = (torch.rand(SIZE, SIZE, generator=g) < 0.1).long().to(dev)
    box = {}
    scene_ms = time_calls(lambda: box.update(r=eng.predict_scene(u1, u2, labels=lab)), max(1, calls // 2))
    pred = box["r"].pred
    for labels in (None, lab):
        r = row("predict_scene pred", pred, labels, calls, min_area=16)
        r["predict_scene_ms"] = round(scene_ms, 1)
        r["share_of_predict_scene"] = round(r["ms"] / scene_ms, 4)
        res["rows"].append(r)
    res["rows"][-1]["scipy_ms"] = round(scipy_ms(pred.cpu()), 1)
    res["rows"][-1]["change_fraction"] = round(float(pred.float().mean()), 4)
    return res


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--calls", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = main(a.calls)
    print(json.dumps(res["info"]))
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(json.dumps(res, indent=1))
