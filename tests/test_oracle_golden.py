"""The CPU oracle against golden vectors produced by the reference (tests/golden/make_golden.py) and
against definition-level numpy convolutions.  Needs only the vectors under tests/golden."""
import hashlib
import json

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from gan_aug_pfa_b200 import spec
from oracle import pix2pix_oracle as O


def test_direct_numpy_conv_pins_library_semantics():
    g = torch.Generator().manual_seed(3)
    x = torch.randn(2, 3, 9, 8, generator=g)
    w = torch.randn(5, 3, 4, 4, generator=g)
    b = torch.randn(5, generator=g)
    for stride, pad in ((2, 1), (1, 1)):
        ref = F.conv2d(x, w, b, stride=stride, padding=pad).numpy()
        got = O.conv2d_direct_np(x.numpy(), w.numpy(), b.numpy(), stride, pad)
        np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-5)
    wt = torch.randn(3, 4, 4, 4, generator=g)
    bt = torch.randn(4, generator=g)
    ref = F.conv_transpose2d(x, wt, bt, stride=2, padding=1).numpy()
    got = O.conv_transpose2d_direct_np(x.numpy(), wt.numpy(), bt.numpy(), 2, 1)
    np.testing.assert_allclose(got, ref, rtol=1e-5, atol=1e-5)
    # empty batch edge case
    assert O.conv2d_direct_np(np.zeros((0, 3, 8, 8)), w.numpy(), None, 2, 1).shape == (0, 5, 4, 4)


def _sd_hash(sd):
    h = hashlib.sha256()
    for k, v in sd.items():
        h.update(k.encode())
        h.update(str(tuple(v.shape)).encode())
        h.update(str(v.dtype).encode())
        h.update(v.detach().contiguous().numpy().tobytes())
    return h.hexdigest()


def test_gan_small_forward_grads_buffers(golden_dir):
    gold = torch.load(golden_dir / "gan_small.pt")
    # the reference's seeded weights (make_golden.py: manual_seed(0), G then D), stored as their sha256
    torch.manual_seed(0)
    sd_g0, sd_d0 = spec.default_state_dicts(num_downs=5, ngf=8, ndf=8)
    assert _sd_hash(sd_g0) == gold["sd_g_sha256"] and _sd_hash(sd_d0) == gold["sd_d_sha256"]
    sd_g = O.clone_state_dict(sd_g0)
    sd_d = O.clone_state_dict(sd_d0)
    A, B = gold["A"], gold["B"]
    for sd in (sd_g, sd_d):
        for k in O.param_names(sd):
            sd[k].requires_grad_(True)
    nb_g, nb_d = {}, {}
    fake = O.unet_generator_forward(sd_g, A, True, nb_g)
    assert torch.allclose(fake, gold["fake"], atol=1e-6)
    pr = O.discriminator_forward(sd_d, torch.cat((A, B), 1), True, nb_d)
    pf = O.discriminator_forward(sd_d, torch.cat((A, fake.detach()), 1), True, nb_d)
    assert torch.allclose(pr, gold["pred_real"], atol=1e-6)
    assert torch.allclose(pf, gold["pred_fake"], atol=1e-6)
    loss_d = 0.5 * (O.bce_with_logits(pr, torch.ones_like(pr)) + O.bce_with_logits(pf, torch.zeros_like(pf)))
    assert abs(float(loss_d) - gold["loss_d"]) < 1e-6
    names_d = O.param_names(sd_d)
    gd = torch.autograd.grad(loss_d, [sd_d[k] for k in names_d])
    for k, g in zip(names_d, gd):
        assert torch.allclose(g, gold["grads_d"][k], rtol=1e-4, atol=1e-7), k
    pg = O.discriminator_forward(sd_d, torch.cat((A, fake), 1), True, nb_d)
    loss_g = O.bce_with_logits(pg, torch.ones_like(pg)) + O.l1_mean(fake, B) * 100.0
    assert abs(float(loss_g) - gold["loss_g"]) < 1e-4
    names_g = O.param_names(sd_g)
    gg = torch.autograd.grad(loss_g, [sd_g[k] for k in names_g])
    assert set(gold["grads_g"]) | set(gold["grads_g_sample"]) == set(names_g)
    for k, g in zip(names_g, gg):
        if k in gold["grads_g_sample"]:      # larger tensors: the reference's values at a fixed seeded sample
            smp = gold["grads_g_sample"][k]
            assert torch.allclose(g.reshape(-1)[smp["idx"].long()], smp["val"], rtol=1e-3, atol=1e-6), k
        else:
            assert torch.allclose(g, gold["grads_g"][k], rtol=1e-3, atol=1e-6), k
    for k, v in gold["buffers_g"].items():
        assert torch.allclose(nb_g[k].float(), v.float(), atol=1e-6), k
    for k, v in gold["buffers_d"].items():
        assert torch.allclose(nb_d[k].float(), v.float(), atol=1e-6), k


def test_gan_full_three_step_loss_sequence(golden_dir):
    """The oracle's gan_train_step reproduces three iterations of the reference's own
    train_gan_one_epoch at the default sizes (batch 1, 256x256)."""
    gold = json.loads((golden_dir / "gan_full.json").read_text())
    torch.manual_seed(0)
    sd_g, sd_d = spec.default_state_dicts()
    gen = torch.Generator().manual_seed(1234)
    batches = [(torch.rand(1, 3, 256, 256, generator=gen) * 2 - 1, torch.rand(1, 3, 256, 256, generator=gen) * 2 - 1)
               for _ in range(3)]
    with torch.no_grad():
        out = O.unet_generator_forward(sd_g, batches[0][0], False, None)
    assert abs(float(out.double().sum()) - gold["eval_out_sum"]) < 1e-2
    assert abs(float(out.double().abs().sum()) - gold["eval_out_abs_sum"]) / gold["eval_out_abs_sum"] < 1e-5
    og = O.AdamState(sd_g, O.param_names(sd_g), 1e-4, (0.5, 0.999))
    od = O.AdamState(sd_d, O.param_names(sd_d), 1e-4, (0.5, 0.999))
    for (A, B), (ld_ref, lg_ref) in zip(batches, gold["loss_sequence"]):
        ld, lg, _ = O.gan_train_step(sd_g, sd_d, og, od, A, B)
        assert abs(ld - ld_ref) < 2e-4 * max(1.0, abs(ld_ref)), (ld, ld_ref)
        assert abs(lg - lg_ref) < 2e-4 * max(1.0, abs(lg_ref)), (lg, lg_ref)
    nbt_g = next(v for k, v in sd_g.items() if k.endswith("num_batches_tracked"))
    nbt_d = next(v for k, v in sd_d.items() if k.endswith("num_batches_tracked"))
    assert int(nbt_g) == gold["nbt_g_after"] == 6 and int(nbt_d) == gold["nbt_d_after"] == 9


def test_losses_against_reference_values(golden_dir):
    gold = torch.load(golden_dir / "losses.pt")
    logits, labels = gold["logits"], gold["labels"]
    tf = labels.float().unsqueeze(1)
    cases = {
        "dice": lambda lg: O.dice_loss(lg, tf),
        "focal": lambda lg: O.focal_loss(lg, tf, gamma=1.7929, alpha=0.6032),
        "combined": lambda lg: O.combined_loss(lg, labels),
        "focal_dice": lambda lg: O.focal_dice_loss(lg, labels, 0.6701, 1.7929, 0.6032, 1.96e-6),
    }
    for name, fn in cases.items():
        lg = logits.clone().requires_grad_(True)
        val = fn(lg)
        (g,) = torch.autograd.grad(val, lg)
        assert abs(float(val) - gold[name]) < 1e-6, name
        assert torch.allclose(g, gold[name + "_grad"], rtol=1e-4, atol=1e-8), name
    x = gold["bce_x"]
    assert abs(float(O.bce_with_logits(x, torch.ones_like(x))) - gold["bce_ones"]) < 1e-6
    assert abs(float(O.bce_with_logits(x, torch.zeros_like(x))) - gold["bce_zeros"]) < 1e-6
    with pytest.raises(ValueError):
        O.combined_loss(logits, labels[:, :8])          # shape mismatch is an error in the reference too


def test_siamese_small(golden_dir):
    gold = torch.load(golden_dir / "siamese_small.pt")
    torch.manual_seed(0)
    sd = spec.SiameseSpec().default_state_dict()
    x1, x2, lab = gold["x1"], gold["x2"], gold["label"]
    with torch.no_grad():
        out = O.siamese_forward(O.clone_state_dict(sd), x1, x2, True, {})
    assert torch.allclose(out, gold["out"], atol=2e-5)
    assert abs(float(O.combined_loss(out, lab)) - gold["combined"]) < 1e-5
    assert abs(float(O.focal_dice_loss(out, lab, 0.6701, 1.7929, 0.6032, 1.96e-6)) - gold["focal_dice"]) < 1e-5
    opt = O.AdamState(sd, O.param_names(sd), 1.0152e-4, (0.9, 0.999), 1e-8, 1.118e-5, decoupled=True)
    seq = [O.siamese_train_step(sd, opt, x1, x2, lab, O.combined_loss) for _ in range(2)]
    for a, b in zip(seq, gold["loss_sequence"]):
        assert abs(a - b) < 2e-4 * max(1.0, abs(b)), (seq, gold["loss_sequence"])


def test_adam_matches_torch_optim():
    g = torch.Generator().manual_seed(0)
    p0 = torch.randn(257, generator=g)
    for decoupled, wd in ((False, 0.0), (True, 1.118e-5)):
        p_ref = p0.clone().requires_grad_(True)
        opt = (torch.optim.AdamW if decoupled else torch.optim.Adam)([p_ref], lr=1e-3, betas=(0.5, 0.999),
                                                                    weight_decay=wd)
        p = p0.clone()
        m, v = torch.zeros_like(p), torch.zeros_like(p)
        for step in range(1, 4):
            grad = torch.randn(257, generator=g)
            p_ref.grad = grad.clone()
            opt.step()
            O.adam_update(p, grad, m, v, step, 1e-3, 0.5, 0.999, 1e-8, wd, decoupled)
        assert torch.allclose(p, p_ref.detach(), atol=1e-7)
