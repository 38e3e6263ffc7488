"""Generate the golden fixtures under tests/golden/ from the UNMODIFIED reference at /root/reference.

Run in the build container (the reference tree is not available on the GPU box):
    python tests/golden/make_golden.py

Fixtures (all small; tensors are stored only for the reduced-size configurations):
  gan_small.pt      UNetGenerator(3,3,num_downs=5,ngf=8) / NLayerDiscriminator(6,ndf=8) at 32x32, batch 2:
                    sha256 of the seeded state_dicts, inputs, train-mode forward outputs, BatchNorm buffers
                    after the forward, parameter gradients of the reference D loss and G loss (the larger
                    generator gradients as a fixed seeded sample, see gan_small_fixture).
  gan_full.json     default-size models (ngf=64, 256x256, batch 1): sha256 of the seeded state_dicts,
                    output checksums, and the (loss_d, loss_g) sequence of three iterations of the
                    reference's own train_gan_one_epoch.
  siamese_small.pt  SiameseUNet(3,1) at 32x32, batch 2: outputs, CombinedLoss / FocalDiceLoss values,
                    a 2-step train_one_epoch loss sequence with AdamW.
  losses.pt         loss values / gradients of DiceLoss, FocalLoss, CombinedLoss, FocalDiceLoss on fixed logits.
"""
import hashlib
import importlib.util
import json
import os
import sys
import types
from pathlib import Path

import torch

REF = Path("/root/reference")
OUT = Path(__file__).resolve().parent


def _load(name, stubs=()):
    for s in stubs:
        sys.modules.setdefault(s, types.ModuleType(s))
    spec = importlib.util.spec_from_file_location(name, REF / f"{name}.py")
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def sd_hash(sd):
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(str(tuple(v.shape)).encode())
        h.update(str(v.dtype).encode())
        h.update(v.detach().contiguous().numpy().tobytes())
    return h.hexdigest()


GRAD_SAMPLE = 8192      # gan_small.pt keeps this many entries of each larger gradient tensor


def gan_small_fixture(full: dict) -> dict:
    """What gan_small.pt stores of `full`, kept under 1 MB: the seeded initial state_dicts as sha256 (spec.py reproduces
    them bit for bit), and of each generator gradient with more than GRAD_SAMPLE entries a fixed seeded sample of its
    flattened entries ("grads_g_sample": name -> {"idx": int32, "val": fp32}) instead of the whole tensor."""
    out = {k: v for k, v in full.items() if k not in ("sd_g", "sd_d", "grads_g")}
    out["sd_g_sha256"], out["sd_d_sha256"] = sd_hash(full["sd_g"]), sd_hash(full["sd_d"])
    out["grads_g"], out["grads_g_sample"] = {}, {}
    for n, g in full["grads_g"].items():
        if g.numel() <= GRAD_SAMPLE:
            out["grads_g"][n] = g
        else:
            idx = torch.randperm(g.numel(), generator=torch.Generator().manual_seed(0))[:GRAD_SAMPLE].sort().values
            out["grads_g_sample"][n] = {"idx": idx.to(torch.int32), "val": g.reshape(-1)[idx].clone()}
    return out


def main():
    sys.path.insert(0, str(REF))
    real_makedirs = os.makedirs
    os.makedirs = lambda *a, **k: None          # train_gan.py creates /Users/mac/... at import
    models = _load("models")
    _load("dataset")
    train_gan = _load("train_gan")
    train = _load("train", stubs=("optuna",))
    os.makedirs = real_makedirs
    torch.set_num_threads(8)

    # ---------------- gan_small
    torch.manual_seed(0)
    G = models.UNetGenerator(3, 3, num_downs=5, ngf=8)
    D = models.NLayerDiscriminator(6, ndf=8)
    sd_g0 = {k: v.clone() for k, v in G.state_dict().items()}
    sd_d0 = {k: v.clone() for k, v in D.state_dict().items()}
    gen = torch.Generator().manual_seed(1234)
    A = torch.rand(2, 3, 32, 32, generator=gen) * 2 - 1
    B = torch.rand(2, 3, 32, 32, generator=gen) * 2 - 1
    G.train(); D.train()
    fake = G(A)
    pred_real = D(torch.cat((A, B), 1))
    pred_fake = D(torch.cat((A, fake.detach()), 1))
    bce = torch.nn.BCEWithLogitsLoss()
    loss_d = 0.5 * (bce(pred_real, torch.ones_like(pred_real)) + bce(pred_fake, torch.zeros_like(pred_fake)))
    gd = torch.autograd.grad(loss_d, list(D.parameters()))
    pred_g = D(torch.cat((A, fake), 1))
    loss_g = bce(pred_g, torch.ones_like(pred_g)) + torch.nn.L1Loss()(fake, B) * 100.0
    gg = torch.autograd.grad(loss_g, list(G.parameters()))
    torch.save(gan_small_fixture({
        "sd_g": sd_g0, "sd_d": sd_d0, "A": A, "B": B, "fake": fake.detach(), "pred_real": pred_real.detach(),
        "pred_fake": pred_fake.detach(), "loss_d": float(loss_d), "loss_g": float(loss_g),
        "buffers_g": {k: v.clone() for k, v in G.state_dict().items() if "running" in k or "num_batches" in k},
        "buffers_d": {k: v.clone() for k, v in D.state_dict().items() if "running" in k or "num_batches" in k},
        "grads_d": {n: g for (n, _), g in zip(D.named_parameters(), gd)},
        "grads_g": {n: g for (n, _), g in zip(G.named_parameters(), gg)},
    }), OUT / "gan_small.pt")

    # ---------------- gan_full: the reference's own loop, default sizes
    torch.manual_seed(0)
    G = models.UNetGenerator(3, 3)
    D = models.NLayerDiscriminator(6)
    full = {"sd_g_sha256": sd_hash(G.state_dict()), "sd_d_sha256": sd_hash(D.state_dict()),
            "n_params_g": sum(p.numel() for p in G.parameters()), "n_params_d": sum(p.numel() for p in D.parameters()),
            "keys_g": list(G.state_dict().keys()), "keys_d": list(D.state_dict().keys())}
    opt_g = torch.optim.Adam(G.parameters(), lr=1e-4, betas=(0.5, 0.999))
    opt_d = torch.optim.Adam(D.parameters(), lr=1e-4, betas=(0.5, 0.999))
    gen = torch.Generator().manual_seed(1234)
    batches = [{"image1": torch.rand(1, 3, 256, 256, generator=gen) * 2 - 1,
                "image2": torch.rand(1, 3, 256, 256, generator=gen) * 2 - 1} for _ in range(3)]
    G.eval()
    with torch.no_grad():
        out_eval = G(batches[0]["image1"])
    full["eval_out_sum"] = float(out_eval.double().sum())
    full["eval_out_abs_sum"] = float(out_eval.double().abs().sum())
    train_gan.tqdm = lambda it, **k: _NoBar(it)
    seq = []
    for b in batches:
        ld, lg = train_gan.train_gan_one_epoch(G, D, [b], opt_g, opt_d)
        seq.append([ld, lg])
    full["loss_sequence"] = seq
    full["nbt_g_after"] = int(next(v for k, v in G.state_dict().items() if k.endswith("num_batches_tracked")))
    full["nbt_d_after"] = int(next(v for k, v in D.state_dict().items() if k.endswith("num_batches_tracked")))
    (OUT / "gan_full.json").write_text(json.dumps(full, indent=1))

    # ---------------- siamese_small
    torch.manual_seed(0)
    S = models.SiameseUNet(3, 1)
    sd_s0 = None  # 41M parameters: not stored; the seeded construction is reproduced by the test
    gen = torch.Generator().manual_seed(77)
    x1 = torch.rand(2, 3, 32, 32, generator=gen) * 2 - 1
    x2 = torch.rand(2, 3, 32, 32, generator=gen) * 2 - 1
    lab = (torch.rand(2, 32, 32, generator=gen) < 0.05).long()
    S.train()
    out = S(x1, x2)
    crit_c = train.CombinedLoss()
    crit_f = train.FocalDiceLoss(beta=0.6701, focal_gamma=1.7929, focal_alpha=0.6032, dice_smooth=1.96e-6)
    sia = {"x1": x1, "x2": x2, "label": lab, "out": out.detach(), "sd_sha256": None,
           "combined": float(crit_c(out, lab)), "focal_dice": float(crit_f(out, lab))}
    torch.manual_seed(0)
    S = models.SiameseUNet(3, 1)
    sia["sd_sha256"] = sd_hash(S.state_dict())
    sia["keys"] = list(S.state_dict().keys())
    opt = torch.optim.AdamW(S.parameters(), lr=1.0152e-4, weight_decay=1.118e-5)
    train.tqdm = lambda it, **k: _NoBar(it)
    batch = {"image1": x1, "image2": x2, "label": lab}
    sia["loss_sequence"] = [train.train_one_epoch(S, [batch], opt, crit_c, torch.device("cpu")) for _ in range(2)]
    torch.save(sia, OUT / "siamese_small.pt")

    # ---------------- losses
    gen = torch.Generator().manual_seed(5)
    logits = torch.randn(3, 1, 16, 16, generator=gen) * 3
    labels = (torch.rand(3, 16, 16, generator=gen) < 0.2).long()
    res = {"logits": logits, "labels": labels}
    for name, crit in (("dice", train.DiceLoss()), ("focal", train.FocalLoss(gamma=1.7929, alpha=0.6032)),
                       ("combined", train.CombinedLoss()), ("focal_dice", crit_f)):
        lg = logits.clone().requires_grad_(True)
        tgt = labels.float().unsqueeze(1) if name == "dice" else labels
        val = crit(lg, tgt)
        (g,) = torch.autograd.grad(val, lg)
        res[name] = float(val)
        res[name + "_grad"] = g
    x = torch.randn(4, 1, 30, 30, generator=gen)
    res["bce_x"] = x
    res["bce_ones"] = float(torch.nn.BCEWithLogitsLoss()(x, torch.ones_like(x)))
    res["bce_zeros"] = float(torch.nn.BCEWithLogitsLoss()(x, torch.zeros_like(x)))
    torch.save(res, OUT / "losses.pt")
    print("wrote", [p.name for p in OUT.iterdir()])


class _NoBar:
    def __init__(self, it):
        self.it = it

    def __iter__(self):
        return iter(self.it)

    def set_postfix(self, **k):
        pass


if __name__ == "__main__":
    main()
