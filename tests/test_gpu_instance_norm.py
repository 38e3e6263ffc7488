"""InstanceNorm2d on the device (pix2pix's `--norm instance`): known-answer tests of the gap_in_* kernels against torch
fp32 on the CPU, and the InstanceNorm networks (engines, stand-alone blocks, drop-in modules, CUDA graphs, checkpoints)
against the CPU oracle with nn.InstanceNorm2d layers (tests/in_oracle.py).

Tolerances: statistics rel <= 1e-5; bf16 outputs and input gradients rel-L2 <= 4e-3; the other limits are those of
test_gpu_engine.py / test_gpu_models_dropin.py.  A conv bias that feeds an affine-free InstanceNorm cancels
(IN(y + b) = IN(y)): its gradient is zero up to rounding, so it is bounded by 1e-3 * sum|dy| per channel instead of
compared by cosine."""
import functools
import io

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from gan_aug_pfa_b200 import checkpoint, ops  # noqa: E402
from gan_aug_pfa_b200 import models as M  # noqa: E402
from gan_aug_pfa_b200.pix2pix import Pix2PixTrainer  # noqa: E402
from in_oracle import IN_EPS, instance_norm  # noqa: E402
from oracle import pix2pix_oracle as O  # noqa: E402

DEV = torch.device("cuda:0")
ACTS = {ops.ACT_NONE: (1.0, lambda v: v), ops.ACT_LRELU: (0.2, lambda v: F.leaky_relu(v, 0.2)),
        ops.ACT_RELU: (0.0, F.relu)}


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(a @ b / (a.norm() * b.norm()).clamp_min(1e-30))


def _slot(n, h, w, c, pad, fill=float("nan")):
    """A [n, h, w, c] channel slot at offset 8 of a wider NaN-filled buffer (pixel stride c + pad)."""
    buf = torch.full((n, h, w, c + pad), fill, device=DEV, dtype=torch.bfloat16)
    return buf, buf[..., 8:8 + c]


def _guards_nan(buf, c):
    return bool(torch.isnan(buf[..., :8]).all()) and bool(torch.isnan(buf[..., 8 + c:]).all())


def _stats(y, n, c):
    hw = y.shape[1] * y.shape[2]
    sums = torch.zeros(2 * n * c, device=DEV, dtype=torch.float64)
    sc, sh, mu, iv = (torch.empty(n, c, device=DEV) for _ in range(4))
    ops.in_stats(y, sums)
    ops.bn_finalize(sums, hw, None, None, IN_EPS, 0.0, 1, None, None, None, sc, sh, mu, iv)
    return sums, sc, sh, mu, iv


# (n, h, w, c, pixel-stride padding, act1, act2 or None, second gradient source)
KAT = [
    (1, 2, 2, 64, 0, ops.ACT_LRELU, ops.ACT_RELU, True),
    (3, 4, 4, 512, 16, ops.ACT_RELU, None, False),
    (64, 2, 2, 512, 0, ops.ACT_NONE, None, False),
    (3, 31, 31, 512, 0, ops.ACT_LRELU, None, False),
    (64, 31, 31, 64, 8, ops.ACT_LRELU, None, False),
    (1, 64, 64, 64, 16, ops.ACT_NONE, ops.ACT_LRELU, True),
    (3, 64, 64, 512, 0, ops.ACT_LRELU, ops.ACT_RELU, True),
    (1, 128, 128, 512, 0, ops.ACT_RELU, None, False),
    (64, 128, 128, 64, 0, ops.ACT_LRELU, ops.ACT_RELU, True),
]


@pytest.mark.parametrize("n,h,w,c,pad,act1,act2,g2", KAT)
def test_in_kernels_known_answer(n, h, w, c, pad, act1, act2, g2):
    gen = torch.Generator().manual_seed(n * 7 + h + c)
    hw = h * w
    # per-channel offsets and scales so that the statistics are not trivially (0, 1)
    y_cpu = (torch.randn(n, h, w, c, generator=gen) * (0.5 + torch.rand(c, generator=gen)) + torch.randn(c, generator=gen))
    y_cpu = y_cpu.to(torch.bfloat16)
    ybuf, y = _slot(n, h, w, c, pad + 16)
    y.copy_(y_cpu.to(DEV))
    sums, sc, sh, mu, iv = _stats(y, n, c)
    yd = y_cpu.double().reshape(n, hw, c)
    mref = yd.mean(1)
    ivref = 1.0 / torch.sqrt(yd.var(1, unbiased=False) + IN_EPS)
    assert rel(mu.cpu(), mref) <= 1e-5 and rel(iv.cpu(), ivref) <= 1e-5
    assert float(sums.abs().max()) == 0.0                       # re-zeroed by finalize
    # forward: torch fp32 F.instance_norm on the same bf16 values
    yf = y_cpu.float().permute(0, 3, 1, 2).contiguous().requires_grad_(True)
    xhat = F.instance_norm(yf, eps=IN_EPS)
    o1buf, o1 = _slot(n, h, w, c, pad + 16)
    o2buf, o2 = _slot(n, h, w, c, 16) if act2 is not None else (None, None)
    ops.in_act(y, sc, sh, o1, act1, o2, act2 if act2 is not None else ops.ACT_NONE)
    r1 = ACTS[act1][1](xhat)
    assert rel(o1.cpu().float(), r1.detach().permute(0, 2, 3, 1)) <= 4e-3 and _guards_nan(o1buf, c)
    if o2 is not None:
        assert rel(o2.cpu().float(), ACTS[act2][1](xhat).detach().permute(0, 2, 3, 1)) <= 4e-3 and _guards_nan(o2buf, c)
    # backward: d = act1'(xhat)*g1 (+ relu'(xhat)*g2), then the InstanceNorm backward; torch autograd as reference
    slope = ACTS[act1][0]
    g1_cpu = torch.randn(n, h, w, c, generator=gen).to(torch.bfloat16)
    g2_cpu = torch.randn(n, h, w, c, generator=gen).to(torch.bfloat16) if g2 else None
    g1buf, g1 = _slot(n, h, w, c, 8)
    g1.copy_(g1_cpu.to(DEV))
    g2d = None
    if g2:
        _, g2d = _slot(n, h, w, c, 24)
        g2d.copy_(g2_cpu.to(DEV))
    loss = (r1 * g1_cpu.float().permute(0, 3, 1, 2)).sum()
    if g2:
        loss = loss + (F.relu(xhat) * g2_cpu.float().permute(0, 3, 1, 2)).sum()
    dy_ref = torch.autograd.grad(loss, yf)[0].permute(0, 2, 3, 1)
    dybuf, dy = _slot(n, h, w, c, pad + 16)
    dbias = torch.zeros(c, device=DEV)
    ops.in_bwd_reduce(y, g1, g2d, slope, sc, sh, sums)
    ops.in_bwd_apply(y, g1, g2d, slope, sc, sh, sums, dy, dbias)
    ops.bn_param_grads(sums, None, None)
    assert rel(dy.cpu().float(), dy_ref) <= 4e-3 and _guards_nan(dybuf, c)
    assert float(sums.abs().max()) == 0.0
    col = dy_ref.double().sum((0, 1, 2))
    bound = 1e-3 * dy_ref.double().abs().sum((0, 1, 2))
    assert bool(((dbias.cpu().double() - col).abs() <= bound).all())


def test_in_forward_graph_replays_give_the_same_result():
    n, h, w, c = 4, 16, 16, 128
    gen = torch.Generator().manual_seed(2)
    y = (torch.randn(n, h, w, c, generator=gen) * 3 + 1).to(torch.bfloat16).to(DEV)
    sums = torch.zeros(2 * n * c, device=DEV, dtype=torch.float64)
    sc, sh, mu, iv = (torch.empty(n, c, device=DEV) for _ in range(4))
    out = torch.empty_like(y)

    def fwd():
        ops.in_stats(y, sums)
        ops.bn_finalize(sums, h * w, None, None, IN_EPS, 0.0, 1, None, None, None, sc, sh, mu, iv)
        ops.in_act(y, sc, sh, out, ops.ACT_LRELU)

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fwd()
    torch.cuda.current_stream().wait_stream(side)
    eager = out.clone()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        fwd()
    res = []
    for _ in range(2):
        out.zero_()
        graph.replay()
        torch.cuda.synchronize()
        res.append(out.clone())
    # the fp64 atomics may add up in another order: the statistics agree to the last bits, the bf16 outputs almost always
    assert rel(res[0].float(), eager.float()) < 1e-3 and rel(res[1].float(), eager.float()) < 1e-3
    assert float(sums.abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------------------------
# networks
# ------------------------------------------------------------------------------------------------------------------
def _cpu_sd(net):
    return {k: v.detach().cpu().clone().contiguous() for k, v in net.state_dict().items()}


def _images(n, hw, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, 3, hw, hw, generator=g) * 2 - 1, torch.rand(n, 3, hw, hw, generator=g) * 2 - 1


def _in_fed_biases(G):
    """state_dict key of every generator conv bias that feeds an InstanceNorm -> the engine's gradient buffer at the norm
    input (dyu for up convs, dyd for down convs)."""
    out = {}
    for j in range(1, G.L):
        out[G.k_up[j] + ".bias"] = lambda j=j: G.dyu[j]
        if G.dbn[j] is not None:
            out[G.k_down[j] + ".bias"] = lambda j=j: G.dyd[j]
    return out


def _check_grads(engine_grad, ref_grads, yardstick, in_fed, what):
    """cosine >= 0.97 per tensor, or the torch-bf16 yardstick rule; biases in front of an InstanceNorm are bounded."""
    bad = []
    for k, r in ref_grads.items():
        gk = engine_grad(k).detach().cpu()
        if k in in_fed:
            dy = in_fed[k]().float().cpu()
            bound = 1e-3 * dy.abs().sum(dim=tuple(range(dy.dim() - 1)))
            assert bool((gk.abs() <= bound).all()), f"{what} {k}: {gk.abs().max()} vs {bound.min()}"
            continue
        if cos(gk, r) < 0.97:
            bad.append(k)
    if bad:
        ys = yardstick()
        for k in bad:
            c, cy = cos(engine_grad(k).detach().cpu(), ref_grads[k]), cos(ys[k], ref_grads[k])
            assert 1 - c <= max(0.03, 2.25 * (1 - cy)), f"{what} {k}: cos {c:.4f}, torch-bf16 yardstick {cy:.4f}"


def _oracle_step(sd_g, sd_d, A, B, autocast=False):
    """One oracle iteration (lr 1e-4, betas (0.5, 0.999) as the trainer's defaults) from copies of the given weights;
    autocast: under CPU bf16 autocast (the torch-bf16 yardstick)."""
    sd_g = {k: v.clone() for k, v in sd_g.items()}
    sd_d = {k: v.clone() for k, v in sd_d.items()}
    og = O.AdamState(sd_g, O.param_names(sd_g), 1e-4, (0.5, 0.999))
    od = O.AdamState(sd_d, O.param_names(sd_d), 1e-4, (0.5, 0.999))
    with instance_norm(), torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
        return O.gan_train_step(sd_g, sd_d, og, od, A, B, return_grads=True)


def _step_parity(tr, A, B):
    sd_g, sd_d = _cpu_sd(tr.G), _cpu_sd(tr.D)
    ld, lg, aux = _oracle_step(sd_g, sd_d, A, B)
    yardstick = functools.lru_cache(None)(lambda: _oracle_step(sd_g, sd_d, A, B, autocast=True)[2])
    losses = tr.train_step(A.to(DEV), B.to(DEV)).cpu()
    assert abs(float(losses[0]) - ld) < 2e-3 * max(1.0, abs(ld)), (float(losses[0]), ld)
    assert abs(float(losses[1]) - lg) < 2e-3 * max(1.0, abs(lg)), (float(losses[1]), lg)
    torch.cuda.synchronize()
    _check_grads(tr.D.grad, aux["grads_d"], lambda: yardstick()["grads_d"], {}, "D")
    _check_grads(tr.G.grad, aux["grads_g"], lambda: yardstick()["grads_g"], _in_fed_biases(tr.G), "G")


def test_engines_match_the_oracle_batch2():
    torch.manual_seed(0)
    tr = Pix2PixTrainer(DEV, norm="instance")
    assert not tr.G.bns and not tr.D.bns and not tr.D.fuse_head
    A, B = _images(2, 256, 11)
    sd_g, sd_d = _cpu_sd(tr.G), _cpu_sd(tr.D)
    with instance_norm():
        for training in (True, False):
            tr.G.training = tr.D.training = training
            tr.G.forward(A.to(DEV))
            fake = tr.G.output_nchw().cpu()
            ref = O.unet_generator_forward(sd_g, A, training, None)
            assert rel(fake, ref) <= 2e-2, training
            xa = torch.zeros(2, 256, 256, 4, device=DEV, dtype=torch.bfloat16)
            xb = torch.zeros_like(xa)
            ops.nchw_to_nhwc_bf16(A.to(DEV), xa)
            ops.nchw_to_nhwc_bf16(B.to(DEV), xb)
            logits = tr.D.forward(xa, xb).cpu().permute(0, 3, 1, 2)
            lref = O.discriminator_forward(sd_d, torch.cat([A, B], 1), training, None)
            assert rel(logits, lref) <= 2e-2, training
    _step_parity(tr, A, B)


def test_full_batch64_step_matches_the_oracle():
    torch.manual_seed(0)
    tr = Pix2PixTrainer(DEV, norm="instance")
    A, B = _images(64, 256, 64)
    _step_parity(tr, A, B)


def _block_parity(blk, x, prefix_grads_in_fed):
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in blk.state_dict().items()}
    xg = x.to(DEV).requires_grad_(True)
    out = blk(xg)
    w = torch.randn(out.shape, generator=torch.Generator().manual_seed(3))
    (out * w.to(DEV)).sum().backward()
    xr = x.clone().requires_grad_(True)
    with instance_norm():
        ref = O._unet_block(sd, "model", xr, True, None, False)
    gref = torch.autograd.grad((ref * w).sum(), [xr] + [sd[k] for k, _ in blk.named_parameters()])
    assert rel(out.detach().cpu(), ref.detach()) <= 2e-2
    assert cos(xg.grad.cpu(), gref[0]) >= 0.97
    eng = blk._engine_obj
    for (k, p), r in zip(blk.named_parameters(), gref[1:]):
        if k in prefix_grads_in_fed:
            dy = prefix_grads_in_fed[k](eng).float().cpu()
            assert bool((p.grad.abs().cpu() <= 1e-3 * dy.abs().sum((0, 1, 2))).all()), k
        else:
            assert cos(p.grad.cpu(), r) >= 0.97, k


def test_standalone_blocks_match_the_oracle():
    torch.manual_seed(0)
    inner = M.UnetSkipConnectionBlock(512, 512, innermost=True, norm_layer=nn.InstanceNorm2d).to(DEV)
    x = torch.randn(2, 512, 8, 8, generator=torch.Generator().manual_seed(1))
    _block_parity(inner, x, {"model.3.bias": lambda e: e.dyu[1]})
    torch.manual_seed(1)
    inner = M.UnetSkipConnectionBlock(512, 512, innermost=True, norm_layer=nn.InstanceNorm2d)
    outer = M.UnetSkipConnectionBlock(256, 512, submodule=inner, norm_layer=nn.InstanceNorm2d).to(DEV)
    x = torch.randn(2, 256, 16, 16, generator=torch.Generator().manual_seed(2))
    _block_parity(outer, x, {"model.1.bias": lambda e: e.dyd[1], "model.5.bias": lambda e: e.dyu[1],
                             "model.3.model.3.bias": lambda e: e.dyu[2]})


def test_reference_loop_runs_on_instance_norm_modules():
    norm = functools.partial(nn.InstanceNorm2d, affine=False, track_running_stats=False)
    torch.manual_seed(0)
    gen = M.UNetGenerator(input_nc=3, output_nc=3, norm_layer=nn.InstanceNorm2d).to(DEV)
    disc = M.NLayerDiscriminator(input_nc=6, norm_layer=norm).to(DEV)
    sd_g = {k: v.detach().cpu().clone() for k, v in gen.state_dict().items()}
    sd_d = {k: v.detach().cpu().clone() for k, v in disc.state_dict().items()}
    opt_g = torch.optim.Adam(gen.parameters(), lr=1e-4, betas=(0.5, 0.999))
    opt_d = torch.optim.Adam(disc.parameters(), lr=1e-4, betas=(0.5, 0.999))
    og = O.AdamState(sd_g, O.param_names(sd_g), 1e-4, (0.5, 0.999))
    od = O.AdamState(sd_d, O.param_names(sd_d), 1e-4, (0.5, 0.999))
    # the same run under CPU bf16 autocast: how far bf16 rounding alone carries the weights in two steps
    sd_gy, sd_dy = {k: v.clone() for k, v in sd_g.items()}, {k: v.clone() for k, v in sd_d.items()}
    ogy = O.AdamState(sd_gy, O.param_names(sd_gy), 1e-4, (0.5, 0.999))
    ody = O.AdamState(sd_dy, O.param_names(sd_dy), 1e-4, (0.5, 0.999))
    loss_GAN, loss_L1 = nn.BCEWithLogitsLoss(), nn.L1Loss()
    g = torch.Generator().manual_seed(1234)
    for _ in range(2):
        A = torch.rand(2, 3, 256, 256, generator=g) * 2 - 1
        B = torch.rand(2, 3, 256, 256, generator=g) * 2 - 1
        with instance_norm():
            ld_ref, lg_ref, _ = O.gan_train_step(sd_g, sd_d, og, od, A, B)
            with torch.autocast("cpu", dtype=torch.bfloat16):
                O.gan_train_step(sd_gy, sd_dy, ogy, ody, A, B)
        real_A, real_B = A.to(DEV), B.to(DEV)
        opt_d.zero_grad()
        fake_B = gen(real_A).detach()
        pred_real = disc(torch.cat((real_A, real_B), 1))
        loss_d_real = loss_GAN(pred_real, torch.ones_like(pred_real))
        pred_fake = disc(torch.cat((real_A, fake_B), 1))
        loss_d_fake = loss_GAN(pred_fake, torch.zeros_like(pred_fake))
        loss_d = (loss_d_real + loss_d_fake) * 0.5
        loss_d.backward()
        opt_d.step()
        opt_g.zero_grad()
        fake_B_for_g = gen(real_A)
        pred_fake_for_g = disc(torch.cat((real_A, fake_B_for_g), 1))
        loss_g = loss_GAN(pred_fake_for_g, torch.ones_like(pred_fake_for_g)) + loss_L1(fake_B_for_g, real_B) * 100.0
        loss_g.backward()
        opt_g.step()
        assert abs(loss_d.item() - ld_ref) < 3e-3 * max(1, abs(ld_ref)), (loss_d.item(), ld_ref)
        assert abs(loss_g.item() - lg_ref) < 3e-3 * max(1, abs(lg_ref)), (loss_g.item(), lg_ref)
    gen.eval()
    with torch.no_grad(), instance_norm():
        out = gen(A.to(DEV))
        ref = O.unet_generator_forward(sd_g, A, False, None)
        ref_y = O.unet_generator_forward(sd_gy, A, False, None)
    # Unlike BatchNorm (0.15 % after two steps), per-image statistics over the 4x4 bottleneck maps amplify the rounding
    # of the first Adam steps: torch's own bf16 run lands 13 % away from the fp32 one.  Same rule as for gradients.
    r, ry = rel(out.cpu(), ref), rel(ref_y, ref)
    assert r <= max(5e-2, 2.25 * ry), (r, ry)
    gen2 = M.UNetGenerator(3, 3, norm_layer=nn.InstanceNorm2d).to(DEV)
    gen2.load_state_dict(gen.state_dict())
    gen2.eval()
    with torch.no_grad():
        assert torch.equal(gen2(A.to(DEV)), out)


def test_graphed_train_step_matches_eager():
    batches = [_images(2, 64, 20 + i) for i in range(3)]
    res = []
    for graphed in (False, True):
        torch.manual_seed(0)
        tr = Pix2PixTrainer(DEV, num_downs=5, norm="instance")
        fn = tr.train_step_graphed if graphed else tr.train_step
        res.append(torch.stack([fn(a.to(DEV), b.to(DEV)).cpu().clone() for a, b in batches]))
    assert torch.allclose(res[0], res[1], rtol=2e-3, atol=2e-4), (res[0], res[1])


def test_checkpoint_resume_and_norm_mismatch():
    data = [_images(2, 64, 40 + i) for i in range(4)]
    torch.manual_seed(0)
    a = Pix2PixTrainer(DEV, num_downs=5, norm="instance")
    for x, y in data[:2]:
        a.train_step(x.to(DEV), y.to(DEV))
    buf = io.BytesIO()
    checkpoint.save(buf, checkpoint.trainer_state(a))
    want = [a.train_step(x.to(DEV), y.to(DEV)).cpu() for x, y in data[2:]]
    torch.manual_seed(123)
    b = Pix2PixTrainer(DEV, num_downs=5, norm="instance")
    buf.seek(0)
    state = checkpoint.load(buf)
    assert state["norm"] == "instance"
    checkpoint.load_trainer_state(b, state)
    got = [b.train_step(x.to(DEV), y.to(DEV)).cpu() for x, y in data[2:]]
    for w, g in zip(want, got):
        assert torch.allclose(w, g, rtol=2e-3, atol=2e-4), (want, got)
    bn_state = checkpoint.trainer_state(Pix2PixTrainer(DEV, num_downs=5))
    with pytest.raises(ValueError, match="norm"):
        checkpoint.load_trainer_state(b, bn_state)
    with pytest.raises(ValueError, match="norm"):
        checkpoint.load_trainer_state(Pix2PixTrainer(DEV, num_downs=5), state)
