"""1-4-channel images on the GPU: known-answer tests of the channel-count kernels against fp32 torch on the CPU (outputs
inside NaN guard bands, pad slots zero), bit-identity of the C = 3 entry points with the existing ones, and the engines,
the drop-in modules, checkpoints and the Siamese U-Net against the CPU oracle for other channel counts.

Tolerances are those of test_gpu_thin_layers.py (kernels: bf16 outputs rel-L2 <= 4e-3, fp32 outputs and weight
gradients <= 1e-4 / 2e-4) and test_gpu_engine.py (steps: losses within 2e-3 relative; gradient cosine >= 0.97 per
tensor, or within the torch-bf16 yardstick rule of test_gpu_batch64.py, 1 - cos <= max(0.03, 2.25 (1 - yardstick cos)),
with the yardstick measured here by running the oracle under CPU bf16 autocast on the same fixture)."""
import ctypes
import functools

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F
import torch.optim as optim

pytestmark = pytest.mark.gpu

from gan_aug_pfa_b200 import _lib, checkpoint, ops  # noqa: E402
from gan_aug_pfa_b200 import models as M  # noqa: E402
from gan_aug_pfa_b200.pix2pix import Pix2PixTrainer  # noqa: E402
from in_oracle import instance_norm  # noqa: E402
from oracle import pix2pix_oracle as O  # noqa: E402

DEV = torch.device("cuda:0")
NAN = float("nan")


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous()


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


def cos(a, b):
    a, b = a.double().flatten(), b.double().flatten()
    return float(a @ b / (a.norm() * b.norm()).clamp_min(1e-30))


def _slots(x):
    """NCHW with 1..4 channels -> NHWC bf16 [n, h, w, 4], slots >= C zero."""
    n, c, h, w = x.shape
    out = torch.zeros(n, h, w, 4, dtype=torch.bfloat16)
    out[..., :c] = nhwc(x).to(torch.bfloat16)
    return out


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


# ------------------------------------------------------------------------------------------------------------------
# kernels
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("co", [1, 2, 3, 4])
@pytest.mark.parametrize("n,ih,iw,cw,bias,act", [
    (2, 16, 32, 128, True, "tanh"),      # generator last layer
    (3, 10, 18, 64, False, "none"),      # discriminator input gradient; partial tiles
    (1, 4, 4, 128, True, "none"),        # input smaller than one halo tile
])
def test_thin_convT_fwd_known_answer(co, n, ih, iw, cw, bias, act):
    g = torch.Generator().manual_seed(ih + cw + co)
    x = torch.randn(n, cw, ih, iw, generator=g).to(torch.bfloat16).float()
    wt = (torch.randn(cw, co, 4, 4, generator=g) / (4 * cw) ** 0.5).to(torch.bfloat16).float()
    b = torch.randn(co, generator=g) if bias else None
    ref = F.conv_transpose2d(x, wt, b, stride=2, padding=1)
    if act == "tanh":
        ref = torch.tanh(ref)
    w2 = wt.permute(2, 3, 1, 0).reshape(16 * co, cw).to(torch.bfloat16).contiguous()      # [(kh*4+kw)*co + c][ci]
    H, W = 2 * ih, 2 * iw
    g32 = torch.full((n + 2, H, W, 8), NAN, device=DEV)            # guard images and guard slots 4..7
    gbf = torch.full((n + 2, H, W, 8), NAN, device=DEV, dtype=torch.bfloat16)
    gu8 = torch.full((n + 2, H, W, co), 77, device=DEV, dtype=torch.uint8)
    o32, obf, ou8 = g32[1:-1, ..., :4], gbf[1:-1, ..., :4], gu8[1:-1]
    ops.thin_convT_fwd(nhwc(x).to(torch.bfloat16).to(DEV), w2.to(DEV), b.to(DEV) if bias else None,
                       ops.ACT_TANH if act == "tanh" else ops.ACT_NONE, obf, o32, ou8, co=co)
    torch.cuda.synchronize()
    assert rel(o32.cpu()[..., :co], nhwc(ref)) < 1e-4
    assert rel(obf.cpu().float()[..., :co], nhwc(ref)) < 4e-3
    assert float(o32.cpu()[..., co:].abs().max() if co < 4 else 0.0) == 0.0
    assert float(obf.cpu().float()[..., co:].abs().max() if co < 4 else 0.0) == 0.0
    for gt in (g32, gbf):
        assert torch.isnan(gt[0].float()).all() and torch.isnan(gt[-1].float()).all()
        assert torch.isnan(gt[..., 4:].float()).all()
    want = ((o32.cpu()[..., :co] * 0.5 + 0.5) * 255).clamp(0, 255).to(torch.uint8)    # same fp32 values, same truncation
    assert torch.equal(ou8.cpu(), want)
    assert bool((gu8[0] == 77).all()) and bool((gu8[-1] == 77).all())


def _convT_c(co, wide, wcol, bias, act, obf, o32, ou8):
    n, ih, iw, cw = wide.shape
    h = _lib.lib()
    args = (_ptr(wcol), _ptr(bias), act, _ptr(obf), 0 if obf is None else obf.stride(2), _ptr(o32),
            0 if o32 is None else o32.stride(2), _ptr(ou8), ops._stream())
    if co is None:
        _lib.check(h.gap_thin_convT_fwd(_ptr(wide), cw, n, ih, iw, cw, *args))
    else:
        _lib.check(h.gap_thin_convT_fwd_c(_ptr(wide), cw, n, ih, iw, cw, co, *args))


def test_c3_entry_points_are_bit_identical_to_the_existing_ones():
    g = torch.Generator().manual_seed(5)
    # thin_convT_fwd: all three outputs
    n, ih, iw, cw = 4, 64, 64, 128
    wide = torch.randn(n, ih, iw, cw, generator=g).to(torch.bfloat16).to(DEV)
    wcol = (torch.randn(48, cw, generator=g) / 16).to(torch.bfloat16).to(DEV)
    b = torch.randn(3, generator=g).to(DEV)
    res = []
    for co in (None, 3):
        o32 = torch.full((n, 2 * ih, 2 * iw, 4), NAN, device=DEV)
        obf = torch.full((n, 2 * ih, 2 * iw, 4), NAN, device=DEV, dtype=torch.bfloat16)
        ou8 = torch.zeros(n, 2 * ih, 2 * iw, 3, device=DEV, dtype=torch.uint8)
        _convT_c(co, wide, wcol, b, ops.ACT_TANH, obf, o32, ou8)
        res.append((o32, obf, ou8))
    for a, c in zip(*res):
        assert torch.equal(a, c)
    # the uint8 converter and the resize
    img = torch.randint(0, 256, (2, 70, 90, 3), generator=g, dtype=torch.uint8).to(DEV)
    h = _lib.lib()
    outs = []
    for new in (False, True):
        o = torch.full((2, 70, 90, 4), NAN, device=DEV, dtype=torch.bfloat16)
        r = torch.full((2, 64, 64, 4), NAN, device=DEV, dtype=torch.bfloat16)
        f = torch.full((2, 3, 64, 64), NAN, device=DEV)
        if new:
            _lib.check(h.gap_u8_hwc_to_nhwc_bf16_c(_ptr(img), 3, _ptr(o), 4, 2 * 70 * 90, ops._stream()))
            _lib.check(h.gap_resize_u8_to_nhwc_bf16_c(_ptr(img), 3, 2, 70, 90, 64, 64, _ptr(r), 4, _ptr(f), ops._stream()))
        else:
            _lib.check(h.gap_u8_hwc_to_nhwc_bf16(_ptr(img), _ptr(o), 4, 2 * 70 * 90, ops._stream()))
            _lib.check(h.gap_resize_u8_to_nhwc_bf16(_ptr(img), 2, 70, 90, 64, 64, _ptr(r), 4, _ptr(f), ops._stream()))
        outs.append((o, r, f))
    for a, c in zip(*outs):
        assert torch.equal(a, c)
    # Siamese im2col
    x = _slots(torch.randn(2, 3, 24, 40, generator=g)).to(DEV)
    cols = []
    for new in (False, True):
        col = torch.full((2, 24, 40, 64), NAN, device=DEV, dtype=torch.bfloat16)
        if new:
            _lib.check(h.gap_im2col_k3s1p1_c(_ptr(x), 4, 3, _ptr(col), 2, 24, 40, ops._stream()))
        else:
            _lib.check(h.gap_im2col_k3s1p1_c3(_ptr(x), 4, _ptr(col), 2, 24, 40, ops._stream()))
        cols.append(col)
    assert torch.equal(cols[0], cols[1])


@pytest.mark.parametrize("w", [256, 64])          # 256: the tcgen05 row kernels; 64: the warp-MMA kernels
@pytest.mark.parametrize("c0,c1", [(1, 0), (4, 0), (1, 3), (2, 2), (4, 4), (3, 3)])
def test_thin_conv_fwd_and_wgrad_per_source_channels(c0, c1, w):
    n, h, cw = 2, 16, 64
    g = torch.Generator().manual_seed(10 * c0 + c1 + w)
    cs = [c for c in (c0, c1) if c]
    xs = [torch.randn(n, c, h, w, generator=g).to(torch.bfloat16).float() for c in cs]
    c = c0 + c1
    wt = (torch.randn(cw, c, 4, 4, generator=g) / (16 * c) ** 0.5).to(torch.bfloat16).float()
    b = torch.randn(cw, generator=g)
    srcs = [_slots(x).to(DEV) for x in xs]
    s1 = srcs[1] if c1 else None
    # forward: the packed weights hold each source's channels in its 4 slots, zero in the rest
    pk = torch.zeros(cw, 16, 4 * len(cs), dtype=torch.bfloat16)
    pk[:, :, :c0] = wt[:, :c0].permute(0, 2, 3, 1).reshape(cw, 16, c0).to(torch.bfloat16)
    if c1:
        pk[:, :, 4:4 + c1] = wt[:, c0:].permute(0, 2, 3, 1).reshape(cw, 16, c1).to(torch.bfloat16)
    ref = F.conv2d(torch.cat(xs, 1), wt, b, stride=2, padding=1)
    guard = torch.full((n + 2, h // 2, w // 2, 2 * cw), NAN, device=DEV, dtype=torch.bfloat16)
    out = guard[1:-1][..., :cw]
    ops.thin_conv_fwd(srcs[0], s1, pk.reshape(cw, -1).contiguous().to(DEV), b.to(DEV), out, ops.ACT_LRELU)
    assert rel(out.cpu().float(), nhwc(F.leaky_relu(ref, 0.2))) < 4e-3
    assert torch.isnan(guard[1:-1][..., cw:].float()).all()
    assert torch.isnan(guard[0].float()).all() and torch.isnan(guard[-1].float()).all()
    # weight / bias gradient into the master layout [cw][(kh*4+kw)*c + ch]
    dy = torch.randn(n, cw, h // 2, w // 2, generator=g).to(torch.bfloat16).float()
    wr = torch.zeros(cw, c, 4, 4, requires_grad=True)
    br = torch.zeros(cw, requires_grad=True)
    F.conv2d(torch.cat(xs, 1), wr, br, stride=2, padding=1).backward(dy)
    krow = 64 if not c1 else 128
    dw = torch.zeros(cw, krow, device=DEV)
    db = torch.zeros(cw, device=DEV)
    dyd = nhwc(dy).to(torch.bfloat16).to(DEV)
    ops.thin_conv_wgrad(dyd, srcs[0], s1, dw.view(-1), krow, db, c0=c0, c1=c1)
    want = wr.grad.permute(0, 2, 3, 1).reshape(cw, 16 * c)
    assert rel(dw.cpu()[:, :16 * c], want) < 2e-4
    assert float(dw.cpu()[:, 16 * c:].abs().max() if 16 * c < krow else 0.0) == 0.0
    assert rel(db.cpu(), br.grad) < 2e-4
    if (c0, c1) in ((3, 0), (3, 3)):
        # the channel-count entry point against two runs of the existing one (fp32 atomics: run-to-run differences)
        olds = []
        for _ in range(2):
            d = torch.zeros(cw, krow, device=DEV)
            _lib.check(_lib.lib().gap_thin_conv_wgrad(_ptr(dyd), cw, _ptr(srcs[0]), 4, _ptr(s1), 4 if c1 else 0, n, h, w,
                                                      cw, _ptr(d), krow, None, ops._stream()))
            olds.append(d)
        new = torch.zeros(cw, krow, device=DEV)
        _lib.check(_lib.lib().gap_thin_conv_wgrad_c(_ptr(dyd), cw, _ptr(srcs[0]), 4, c0, _ptr(s1), 4 if c1 else 0, c1, n, h,
                                                    w, cw, _ptr(new), krow, None, ops._stream()))
        spread = float((olds[0] - olds[1]).abs().max())
        assert float((new - olds[0]).abs().max()) <= max(2 * spread, 1e-6 * float(olds[0].abs().max()))


@pytest.mark.parametrize("c", [1, 2, 3, 4])
@pytest.mark.parametrize("u8", [False, True])
@pytest.mark.parametrize("vec", [True, False])     # the four-pixel kernel and the general per-pixel kernel
def test_gen_out_bwd_per_channel_count(c, u8, vec):
    n, h, w = 2, 32, 48
    g = torch.Generator().manual_seed(c + 10 * u8)
    fake = torch.zeros(n, h, w, 4)
    fake[..., :c] = torch.tanh(torch.randn(n, h, w, c, generator=g))
    dd = torch.zeros(n, h, w, 4)
    dd[..., :c] = torch.randn(n, h, w, c, generator=g) * 1e-3
    if u8:
        real_u8 = torch.randint(0, 256, (n, h, w, c), generator=g, dtype=torch.uint8)
        real = (real_u8.float() / 255.0) * 2 - 1
        real_dev = real_u8.to(DEV)
    else:
        real = torch.rand(n, h, w, c, generator=g) * 2 - 1
        real_dev = real.permute(0, 3, 1, 2).contiguous().to(DEV)
    scale = 100.0 / (n * c * h * w)
    d = fake[..., :c] - real
    ref = (dd[..., :c] + scale * torch.sign(d)) * (1 - fake[..., :c] ** 2)
    dpre = torch.full((n, h, w, 4), NAN, device=DEV, dtype=torch.bfloat16)
    loss = torch.zeros(1, device=DEV, dtype=torch.float64)
    if not vec:
        _lib.debug_set("gen_out_c3", 0)
        dpre[..., c:] = 0                          # the general kernel writes only the C channels
    try:
        ops.gen_out_bwd(fake.to(DEV), real_dev, dd.to(DEV), scale, dpre, loss)
        torch.cuda.synchronize()
    finally:
        _lib.debug_set("gen_out_c3", 1)
    assert rel(dpre.cpu().float()[..., :c], ref) < 4e-3
    assert float(dpre.cpu().float()[..., c:].abs().max() if c < 4 else 0.0) == 0.0
    assert abs(float(loss) - float(d.abs().double().sum())) < 1e-5 * float(d.abs().double().sum())


@pytest.mark.parametrize("c", [1, 2, 3, 4])
def test_converters_resize_and_im2col_per_channel_count(c):
    g = torch.Generator().manual_seed(30 + c)
    img = torch.randint(0, 256, (2, 20, 28, c), generator=g, dtype=torch.uint8)
    out = torch.full((2, 20, 28, 4), NAN, device=DEV, dtype=torch.bfloat16)
    ops.u8_hwc_to_nhwc_bf16(img.to(DEV), out)
    assert rel(out.cpu().float()[..., :c], (img.float() / 255 - 0.5) / 0.5) < 4e-3
    assert float(out.cpu().float()[..., c:].abs().max() if c < 4 else 0.0) == 0.0
    # fp32 NCHW -> 4-slot NHWC
    x = torch.randn(2, c, 20, 28, generator=g)
    xs = torch.full((2, 20, 28, 4), NAN, device=DEV, dtype=torch.bfloat16)
    ops.nchw_to_nhwc_bf16(x.to(DEV), xs)
    assert torch.equal(xs.cpu()[..., :c], nhwc(x).to(torch.bfloat16))
    assert float(xs.cpu().float()[..., c:].abs().max() if c < 4 else 0.0) == 0.0
    # antialiased resize (dataset.py's JointResize + Normalize) in both output forms
    big = torch.randint(0, 256, (2, 300, 420, c), generator=g, dtype=torch.uint8)
    ref = F.interpolate(big.permute(0, 3, 1, 2).float() / 255.0, size=(128, 128), mode="bilinear", align_corners=False,
                        antialias=True) * 2.0 - 1.0
    r = torch.full((2, 128, 128, 4), NAN, device=DEV, dtype=torch.bfloat16)
    f = torch.full((2, c, 128, 128), NAN, device=DEV)
    ops.resize_u8_to_nhwc_bf16(big.to(DEV), r, f)
    assert rel(r.cpu().float()[..., :c], nhwc(ref)) < 4e-3
    assert float(r.cpu().float()[..., c:].abs().max() if c < 4 else 0.0) == 0.0
    assert float((f.cpu() - ref).abs().max()) < 2e-6
    # Siamese first-layer im2col: col[pix][(kh*3+kw)*c + ch], zero padded to 64
    xb = x.to(torch.bfloat16).float()
    col = torch.full((2, 20, 28, 64), NAN, device=DEV, dtype=torch.bfloat16)
    ops.im2col_k3s1p1(_slots(xb).to(DEV), col, c)
    un = F.unfold(xb, 3, padding=1).view(2, c, 9, 20, 28).permute(0, 3, 4, 2, 1).reshape(2, 20, 28, 9 * c)
    assert torch.equal(col.cpu().float()[..., :9 * c], un)
    assert float(col.cpu().float()[..., 9 * c:].abs().max()) == 0.0


# ------------------------------------------------------------------------------------------------------------------
# engines
# ------------------------------------------------------------------------------------------------------------------
def _cpu_sd(net):
    return {k: v.detach().cpu().clone().contiguous() for k, v in net.state_dict().items()}


def _images(n, hw, ic, oc, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.rand(n, ic, hw, hw, generator=g) * 2 - 1, torch.rand(n, oc, hw, hw, generator=g) * 2 - 1


def _oracle_step(sd_g, sd_d, A, B, norm, autocast=False):
    sd_g = {k: v.clone() for k, v in sd_g.items()}
    sd_d = {k: v.clone() for k, v in sd_d.items()}
    og = O.AdamState(sd_g, O.param_names(sd_g), 1e-4, (0.5, 0.999))
    od = O.AdamState(sd_d, O.param_names(sd_d), 1e-4, (0.5, 0.999))
    with torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
        if norm == "instance":
            with instance_norm():
                return O.gan_train_step(sd_g, sd_d, og, od, A, B, return_grads=True)
        return O.gan_train_step(sd_g, sd_d, og, od, A, B, return_grads=True)


def _step_parity(tr, A, B, yard_cos=None):
    """yard_cos: {"grads_d": {key: cos}, "grads_g": ...} of a torch-bf16 yardstick measured elsewhere; by default it is
    measured on this fixture, and only when some tensor is below 0.97."""
    sd_g, sd_d = _cpu_sd(tr.G), _cpu_sd(tr.D)
    ld, lg, aux = _oracle_step(sd_g, sd_d, A, B, tr.norm)
    ys = functools.lru_cache(None)(lambda: _oracle_step(sd_g, sd_d, A, B, tr.norm, autocast=True)[2])
    losses = tr.train_step(A.to(DEV), B.to(DEV)).cpu()
    assert abs(float(losses[0]) - ld) < 2e-3 * max(1.0, abs(ld)), (float(losses[0]), ld)
    assert abs(float(losses[1]) - lg) < 2e-3 * max(1.0, abs(lg)), (float(losses[1]), lg)
    assert rel(tr.G.output_nchw().cpu(), aux["fake_B"]) < 2e-2
    torch.cuda.synchronize()
    inst = tr.norm == "instance"
    for net, key in ((tr.D, "grads_d"), (tr.G, "grads_g")):
        for k, r in aux[key].items():
            if inst and net is tr.G and k.endswith(".bias") and k not in ("model.model.0.bias", "model.model.3.bias"):
                continue        # biases in front of an InstanceNorm: analytically zero gradients (pure rounding noise)
            c = cos(net.grad(k).cpu(), r)
            if c < 0.97:
                cy = yard_cos[key][k] if yard_cos is not None else cos(ys()[key][k], r)
                assert 1 - c <= max(0.03, 2.25 * (1 - cy)), f"{k}: cos {c:.4f}, torch-bf16 yardstick {cy:.4f}"
    # the image-side layers see the least accumulated bf16 noise: tight check there
    assert rel(tr.G.grad("model.model.3.weight").cpu(), aux["grads_g"]["model.model.3.weight"]) < 2e-2
    assert rel(tr.G.grad("model.model.0.weight").cpu(), aux["grads_g"]["model.model.0.weight"]) < 2e-2 or \
        cos(tr.G.grad("model.model.0.weight").cpu(), aux["grads_g"]["model.model.0.weight"]) >= 0.97
    assert rel(tr.D.grad("model.0.weight").cpu(), aux["grads_d"]["model.0.weight"]) < 2e-2 or \
        cos(tr.D.grad("model.0.weight").cpu(), aux["grads_d"]["model.0.weight"]) >= 0.97
    return aux


@pytest.mark.parametrize("ic,oc", [(1, 3), (4, 4), (2, 1)])
def test_training_step_matches_the_oracle_batch2(ic, oc):
    torch.manual_seed(0)
    tr = Pix2PixTrainer(DEV, input_nc=ic, output_nc=oc)
    assert tr.D.split == (ic, oc)
    A, B = _images(2, 256, ic, oc, 1234)
    _step_parity(tr, A, B)
    fake = tr.G.fake_f32.cpu()
    assert float(fake[..., oc:].abs().max() if oc < 4 else 0.0) == 0.0 and fake.shape[-1] == 4


def test_training_step_matches_the_oracle_instance_norm_1_to_3():
    torch.manual_seed(0)
    tr = Pix2PixTrainer(DEV, input_nc=1, output_nc=3, norm="instance")
    A, B = _images(2, 256, 1, 3, 77)
    _step_parity(tr, A, B)


def test_training_step_matches_the_oracle_batch64_1_to_3(golden_dir):
    """The torch-bf16 yardstick of the batch-64 3 -> 3 step (tests/golden/gan_yardstick_b64.json: same networks past
    the image-side layers, same batch and size) bounds the tensors below 0.97; a CPU bf16-autocast oracle run at batch
    64 would take minutes."""
    import json
    yard = json.loads((golden_dir / "gan_yardstick_b64.json").read_text())
    torch.manual_seed(0)
    tr = Pix2PixTrainer(DEV, input_nc=1, output_nc=3)
    A, B = _images(64, 256, 1, 3, 4321)
    _step_parity(tr, A, B, yard_cos={"grads_d": yard["cos_d"], "grads_g": yard["cos_g"]})


def test_graphed_train_step_matches_eager_1_to_3():
    res = []
    for graphed in (False, True):
        torch.manual_seed(0)
        tr = Pix2PixTrainer(DEV, input_nc=1, output_nc=3)
        step = tr.train_step_graphed if graphed else tr.train_step
        out = []
        for s in range(3):
            A, B = _images(2, 256, 1, 3, 50 + s)
            out.append(step(A.to(DEV), B.to(DEV)).cpu())
        res.append(torch.stack(out))
    assert tr._graph is not None
    assert torch.allclose(res[0], res[1], rtol=2e-3, atol=2e-4), (res[0], res[1])


@pytest.mark.parametrize("ic,oc", [(1, 3), (4, 2)])
def test_uint8_inputs_match_the_fp32_path(ic, oc):
    g = torch.Generator().manual_seed(9)
    a8 = torch.randint(0, 256, (2, 256, 256, ic), generator=g, dtype=torch.uint8)
    b8 = torch.randint(0, 256, (2, 256, 256, oc), generator=g, dtype=torch.uint8)
    res = []
    for u8 in (False, True):
        torch.manual_seed(0)
        tr = Pix2PixTrainer(DEV, input_nc=ic, output_nc=oc)
        if u8:
            losses = tr.train_step(a8.to(DEV), b8.to(DEV))
        else:
            A = ((a8.permute(0, 3, 1, 2).float() / 255.0) * 2 - 1).contiguous()
            B = ((b8.permute(0, 3, 1, 2).float() / 255.0) * 2 - 1).contiguous()
            losses = tr.train_step(A.to(DEV), B.to(DEV))
        torch.cuda.synchronize()
        res.append((losses.cpu(), tr.G.output_nchw().cpu(), tr.G.store.g.cpu(), tr.D.store.g.cpu()))
    (l0, f0, gg0, gd0), (l1, f1, gg1, gd1) = res
    # (the input kernel normalises x*(2/255) - 1 in fp32, which can round some bf16 inputs differently)
    assert torch.allclose(l0, l1, rtol=1e-3, atol=1e-5), (l0, l1)
    assert rel(f1, f0) < 2e-3, rel(f1, f0)
    # the step's gradients (not the updated weights: Adam's first step moves every weight by +-lr whatever the size of its
    # gradient, so noise-level gradients of either run flip weights by 2*lr)
    assert cos(gg1, gg0) >= 0.999 and cos(gd1, gd0) >= 0.999, (cos(gg1, gg0), cos(gd1, gd0))
    # the generator's uint8 image output writes output_nc bytes per pixel
    out_u8 = torch.zeros(2, 256, 256, oc, device=DEV, dtype=torch.uint8)
    tr.G.training = False
    tr.G.forward(a8.to(DEV), out_u8=out_u8)
    want = ((tr.G.fake_f32[..., :oc] * 0.5 + 0.5) * 255).clamp(0, 255).to(torch.uint8)
    assert int((out_u8.int() - want.int()).abs().max()) <= 1      # the kernel contracts v*0.5+0.5 into one fma


def test_reference_loop_on_dropin_modules_1_to_3_and_state_dicts():
    """The reference's loop body (train_gan.py:53-71) on UNetGenerator(1, 3) + NLayerDiscriminator(4): module calls,
    torch losses, loss.backward(), optim.Adam -- against the oracle; then a state_dict round trip."""
    torch.manual_seed(0)
    gen = M.UNetGenerator(1, 3).to(DEV)
    disc = M.NLayerDiscriminator(4).to(DEV)
    sd_g, sd_d = _cpu_sd(gen), _cpu_sd(disc)
    opt_g = optim.Adam(gen.parameters(), lr=1e-4, betas=(0.5, 0.999))
    opt_d = optim.Adam(disc.parameters(), lr=1e-4, betas=(0.5, 0.999))
    og = O.AdamState(sd_g, O.param_names(sd_g), 1e-4, (0.5, 0.999))
    od = O.AdamState(sd_d, O.param_names(sd_d), 1e-4, (0.5, 0.999))
    loss_GAN, loss_L1 = nn.BCEWithLogitsLoss(), nn.L1Loss()
    gen.train()
    disc.train()
    for s in range(2):
        A, B = _images(2, 256, 1, 3, 600 + s)
        ld_ref, lg_ref, _ = O.gan_train_step(sd_g, sd_d, og, od, A, B)
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
        fake_B = gen(real_A)
        pred_fake = disc(torch.cat((real_A, fake_B), 1))
        loss_g = loss_GAN(pred_fake, torch.ones_like(pred_fake)) + loss_L1(fake_B, real_B) * 100.0
        loss_g.backward()
        opt_g.step()
        assert fake_B.shape == (2, 3, 256, 256)
        assert abs(loss_d.item() - ld_ref) < 3e-3 * max(1, abs(ld_ref)), (loss_d.item(), ld_ref)
        assert abs(loss_g.item() - lg_ref) < 3e-3 * max(1, abs(lg_ref)), (loss_g.item(), lg_ref)
    # the discriminator's input gradient reaches both halves of cat(A, B) (split 2 | 2 for input_nc = 4); train mode,
    # the mode the engines' backward passes implement
    x = torch.cat(_images(2, 64, 2, 2, 3), 1).to(DEV).requires_grad_(True)
    sd_now = _cpu_sd(disc)
    w = torch.randn(2, 1, 6, 6, generator=torch.Generator().manual_seed(8))
    (disc(x) * w.to(DEV)).sum().backward()
    xr = x.detach().cpu().requires_grad_(True)
    (O.discriminator_forward(sd_now, xr, True, {}) * w).sum().backward()
    assert cos(x.grad.cpu()[:, :2], xr.grad[:, :2]) >= 0.97 and cos(x.grad.cpu()[:, 2:], xr.grad[:, 2:]) >= 0.97
    # state_dict round trip into fresh modules
    gen.eval()
    A, _ = _images(2, 256, 1, 3, 99)
    with torch.no_grad():
        out = gen(A.to(DEV))
    gen2 = M.UNetGenerator(1, 3).to(DEV)
    gen2.load_state_dict(gen.state_dict())
    gen2.eval()
    with torch.no_grad():
        assert torch.equal(gen2(A.to(DEV)), out)
    with pytest.raises(RuntimeError):
        M.UNetGenerator(3, 3).load_state_dict(gen.state_dict())


def test_checkpoint_round_trip_and_channel_mismatch(tmp_path):
    torch.manual_seed(0)
    tr = Pix2PixTrainer(DEV, input_nc=1, output_nc=2)
    A, B = _images(2, 256, 1, 2, 5)
    tr.train_step(A.to(DEV), B.to(DEV))
    path = tmp_path / "ck.pt"
    checkpoint.save(path, checkpoint.trainer_state(tr))
    state = checkpoint.load(path)
    assert state["channels"] == {"input_nc": 1, "output_nc": 2}
    torch.manual_seed(1)
    tr2 = Pix2PixTrainer(DEV, input_nc=1, output_nc=2)
    checkpoint.load_trainer_state(tr2, state)
    for net, net2 in ((tr.G, tr2.G), (tr.D, tr2.D)):
        assert torch.equal(net.store.p, net2.store.p) and torch.equal(net.store.m, net2.store.m)
    A, B = _images(2, 256, 1, 2, 6)
    l1, l2 = tr.train_step(A.to(DEV), B.to(DEV)).cpu(), tr2.train_step(A.to(DEV), B.to(DEV)).cpu()
    assert torch.allclose(l1, l2, rtol=2e-3, atol=2e-4), (l1, l2)
    for ic, oc in ((3, 3), (1, 3), (2, 2)):
        with pytest.raises(ValueError, match="input_nc=1, output_nc=2"):
            checkpoint.load_trainer_state(Pix2PixTrainer(DEV, input_nc=ic, output_nc=oc), state)


# ------------------------------------------------------------------------------------------------------------------
# Siamese U-Net
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n_channels", [1, 4])
def test_siamese_forward_and_gradients_match_the_oracle(n_channels):
    """Batch 4, 128x128.  The golden yardstick files are for 3-channel fixtures, so the bf16 yardstick is measured here:
    the oracle under CPU bf16 autocast on the same fixture.  Logits within max(0.15, 1.5 x yardstick) rel-L2 (the bound
    of test_gpu_siamese.py), whole-gradient cosine within the yardstick rule."""
    torch.manual_seed(0)
    net = M.SiameseUNet(n_channels, 1).to(DEV)
    sd = _cpu_sd(net)
    g = torch.Generator().manual_seed(17 + n_channels)
    x1 = torch.rand(4, n_channels, 128, 128, generator=g) * 2 - 1
    x2 = torch.rand(4, n_channels, 128, 128, generator=g) * 2 - 1
    lab = (torch.rand(4, 1, 128, 128, generator=g) < 0.1).long()
    net.train()
    out = net(x1.to(DEV), x2.to(DEV))
    loss = O.combined_loss(out, lab.to(DEV))
    loss.backward()
    names = O.param_names(sd)
    mine = torch.cat([dict(net.named_parameters())[k].grad.detach().cpu().flatten() for k in names])

    def oracle(autocast):
        s = {k: v.clone().requires_grad_(k in names) for k, v in sd.items()}
        with torch.autocast("cpu", dtype=torch.bfloat16, enabled=autocast):
            o = O.siamese_forward(s, x1, x2, True, {})
            lo = O.combined_loss(o.float(), lab)
        gr = torch.autograd.grad(lo, [s[k] for k in names])
        return o.detach().float(), float(lo.detach()), torch.cat([q.float().flatten() for q in gr])

    ref_o, ref_l, ref_g = oracle(False)
    yd_o, yd_l, yd_g = oracle(True)
    assert out.shape == (4, 1, 128, 128)
    assert rel(out.detach().cpu(), ref_o) <= max(0.15, 1.5 * rel(yd_o, ref_o))
    assert abs(float(loss) - ref_l) <= max(3e-2 * abs(ref_l), 1.5 * abs(yd_l - ref_l))
    assert 1 - cos(mine, ref_g) <= max(0.05, 2.25 * (1 - cos(yd_g, ref_g)))
    with pytest.raises(ValueError, match="n_channels"):
        net(torch.zeros(1, 3, 32, 32, device=DEV), torch.zeros(1, 3, 32, 32, device=DEV))


# ------------------------------------------------------------------------------------------------------------------
# two GPUs
# ------------------------------------------------------------------------------------------------------------------
def _dp_shard(rank, n=2, hw=64):
    g = torch.Generator().manual_seed(4321 + rank)
    return torch.rand(n, 1, hw, hw, generator=g) * 2 - 1, torch.rand(n, 3, hw, hw, generator=g) * 2 - 1


def _dp_worker(rank, world, port, q):
    import os
    import tempfile
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from gan_aug_pfa_b200 import parallel
        torch.manual_seed(rank)                       # different seeds: only the broadcast makes the replicas equal
        tr = Pix2PixTrainer(dev, num_downs=5, world=world, bucket_elems=1 << 18, input_nc=1, output_nc=3)
        sd_d0 = _cpu_sd(tr.D)
        A, B = _dp_shard(rank)
        losses = tr.train_step(A.to(dev), B.to(dev)).cpu()
        out = {"losses": losses, "sd_d0": sd_d0,
               "g_d": {k: tr.D.grad(k).cpu().clone() / world for k in O.param_names(sd_d0)},
               "diff": parallel.replica_param_max_abs_diff([tr.G, tr.D])}
        path = os.path.join(tempfile.gettempdir(), f"gap_dp2_channels_rank{rank}_{port}.pt")
        torch.save(out, path)
        q.put((rank, path))
    finally:
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_rank_step_with_one_channel_inputs():
    """Pix2PixTrainer(world=2, input_nc=1): bit-identical replicas after the step, each rank's discriminator loss on its
    shard against the oracle (the D losses precede any all-reduce), and the all-reduced discriminator gradient against
    the shard average of the oracle's (bf16 tolerances of test_gpu_dp2.py)."""
    import os
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_dp_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in range(world)])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    dumps = [torch.load(path) for _, path in res]
    for _, path in res:
        os.remove(path)
    sd_d0 = dumps[0]["sd_d0"]
    for k, v in dumps[1]["sd_d0"].items():
        assert torch.equal(v, sd_d0[k]), k            # rank 1 starts from rank 0's weights
    names = O.param_names(sd_d0)
    torch.manual_seed(0)
    sd_g0 = M.UNetGenerator(1, 3, num_downs=5).state_dict()
    grads = []
    for rank, d in enumerate(dumps):
        assert d["diff"] == 0.0, f"replicas diverged by {d['diff']}"
        A, B = _dp_shard(rank)
        sg, sdd = O.clone_state_dict(sd_g0), O.clone_state_dict(sd_d0)
        og = O.AdamState(sg, O.param_names(sg), 1e-4, (0.5, 0.999))
        od = O.AdamState(sdd, names, 1e-4, (0.5, 0.999))
        ld, _, aux = O.gan_train_step(sg, sdd, og, od, A, B, return_grads=True)
        assert abs(float(d["losses"][0]) - ld) < 2e-3 * max(1.0, abs(ld)), (rank, d["losses"], ld)
        grads.append(aux["grads_d"])
    avg = {k: sum(g[k] for g in grads) / world for k in names}
    for d in dumps:
        whole = cos(torch.cat([d["g_d"][k].flatten() for k in names]), torch.cat([avg[k].flatten() for k in names]))
        assert whole > 0.97, whole
        assert min(cos(d["g_d"][k], avg[k]) for k in names) > 0.9
