"""The generator's sliding-window scene inference (GeneratorEngine.translate_scene) on the GPU: the one-image gather
bit for bit against the existing converters, image blend + finalize on synthetic tile outputs against the fp64
reference of tests/translate_ref.py, single-tile equivalence with the eval forward and its out_u8 image, end-to-end
runs against per-tile eval-forward outputs blended in fp64, determinism, side effects, a trainer, the drop-in module
and a 4096 x 4096 scene."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from gan_aug_pfa_b200 import models as M  # noqa: E402
from gan_aug_pfa_b200 import ops  # noqa: E402
from gan_aug_pfa_b200.pix2pix import GeneratorEngine, Pix2PixTrainer  # noqa: E402
from gan_aug_pfa_b200.scene import _scene_grid  # noqa: E402
from translate_ref import blend_image_ref, cut_tiles, near_integer, tile_origins, u8_ref  # noqa: E402

DEV = torch.device("cuda:0")
NAN = float("nan")
G = 68          # guard elements on either side of every kernel output (bf16 / fp32 outputs stay 8 / 16-byte aligned)


def _guarded(numel, dtype, fill, guard=G):
    buf = torch.full((numel + 2 * guard,), fill, device=DEV, dtype=dtype)
    return buf, buf[guard:guard + numel]


def _guards_intact(buf, fill, guard=G):
    a, b = buf[:guard], buf[-guard:]
    if isinstance(fill, float) and fill != fill:
        return bool(torch.isnan(a).all() and torch.isnan(b).all())
    return bool((a == fill).all() and (b == fill).all())


# ------------------------------------------------------------------------------------------------
# gather
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [1, 2, 3, 4])
@pytest.mark.parametrize("u8", [True, False])
@pytest.mark.parametrize("h,w", [(37, 150), (130, 45)])
def test_gather_one_is_bit_identical_to_the_converters(c, u8, h, w):
    tile, overlap, align, batch = 64, 16, 32, 3
    g = torch.Generator().manual_seed(c * 10 + h)
    if u8:
        s = torch.randint(0, 256, (h, w, c), generator=g, dtype=torch.uint8)
        chw = s.permute(2, 0, 1)
    else:
        s = torch.randn(c, h, w, generator=g) * 1.5
        chw = s
    origins, (ey, ex) = tile_origins(h, w, tile, overlap, align)
    grid = _scene_grid(h, w, tile, overlap, align)
    n_t = len(origins)
    crops = cut_tiles(chw, tile, overlap, align)                     # [n_t, c, ey, ex]
    ref = torch.zeros(n_t, ey, ex, 4, device=DEV, dtype=torch.bfloat16)
    for t in range(n_t):
        if u8:
            ops.u8_hwc_to_nhwc_bf16(crops[t].permute(1, 2, 0).contiguous()[None].to(DEV), ref[t:t + 1])
        else:
            ops.nchw_to_nhwc_bf16(crops[t][None].contiguous().to(DEV), ref[t:t + 1])
    d = s.to(DEV)
    numel = batch * ey * ex * 4
    for t0 in range(0, n_t, batch):
        b, o = _guarded(numel, torch.bfloat16, NAN)
        ops.scene_gather_one(d, grid, t0, o.view(batch, ey, ex, 4))
        assert _guards_intact(b, NAN)
        o = o.view(batch, ey, ex, 4)
        nv = min(batch, n_t - t0)
        assert torch.equal(o[:nv].view(torch.int16), ref[t0:t0 + nv].view(torch.int16))
        assert (o[..., c:].view(torch.int16) == 0).all()                 # slots >= C
        assert (o[nv:].view(torch.int16) == 0).all()                     # padding tiles of the last batch
    if h < tile:
        assert ey == 64 and origins[0][0] == 0                            # one row of tiles, rows past h repeat


# ------------------------------------------------------------------------------------------------
# image blend + finalize on synthetic tile outputs
# ------------------------------------------------------------------------------------------------
def _run_blend(v, h, w, tile, overlap, align, batch):
    """blend every batch of v [n_t, C, ey, ex] into NaN-guarded accumulators; the unused slots of the 4-slot tile
    outputs and the padding tiles of the last batch hold NaN (never read)."""
    n_t, c, ey, ex = v.shape
    grid = _scene_grid(h, w, tile, overlap, align)
    ab, acc = _guarded(c * h * w, torch.float32, NAN)
    wb, ws = _guarded(h * w, torch.float32, NAN)
    vd = v.to(DEV).permute(0, 2, 3, 1)
    for t0 in range(0, n_t, batch):
        fake = torch.full((batch, ey, ex, 4), NAN, device=DEV)
        nv = min(batch, n_t - t0)
        fake[:nv, ..., :c] = vd[t0:t0 + nv]
        ops.scene_blend_image(fake, grid, t0, acc.view(c, h, w), ws.view(h, w))
    assert _guards_intact(ab, NAN) and _guards_intact(wb, NAN)
    return ab, acc.view(c, h, w), ws.view(h, w)


@pytest.mark.parametrize("c", [1, 2, 3, 4])
@pytest.mark.parametrize("overlap", [0, 24])
@pytest.mark.parametrize("h,w,img_guard", [(150, 232, 64), (149, 231, 68)])    # vector and scalar finalize paths
def test_image_blend_and_finalize_match_the_fp64_reference(c, overlap, h, w, img_guard):
    tile, align, batch = 64, 32, 5
    origins, (ey, ex) = tile_origins(h, w, tile, overlap, align)
    g = torch.Generator().manual_seed(c * 7 + overlap + h)
    v = torch.tanh(torch.randn(len(origins), c, ey, ex, generator=g) * 2)
    v[torch.rand(v.shape, generator=g) < 0.01] = 1.0
    v[torch.rand(v.shape, generator=g) < 0.01] = -1.0
    want = blend_image_ref(v, h, w, tile, overlap, align)
    ab, acc, ws = _run_blend(v, h, w, tile, overlap, align, batch)
    assert torch.isfinite(ws).all() and (ws > 0).all()
    ib, img = _guarded(h * w * c, torch.uint8, 0xEE, img_guard)
    before = acc.clone()
    ops.scene_finalize_image(acc, ws, img.view(h, w, c), False)            # without values: acc is left as it was
    assert torch.equal(acc, before)
    first = img.clone()
    ops.scene_finalize_image(acc, ws, img.view(h, w, c), True)
    assert _guards_intact(ib, 0xEE, img_guard) and _guards_intact(ab, NAN)
    assert torch.equal(img, first)
    err = float((acc.cpu().double() - want).abs().max())
    assert err < 1e-5, err
    got = img.view(h, w, c).cpu()
    ref = u8_ref(want).permute(1, 2, 0)
    ok = ~near_integer(want, 1e-3).permute(1, 2, 0)
    assert torch.equal(got[ok], ref[ok])
    assert int((got.int() - ref.int()).abs().max()) <= 1
    assert int(ok.sum()) > 0.98 * got.numel()


def test_image_blend_is_deterministic_and_independent_of_the_batch():
    c, h, w, tile, overlap, align = 3, 150, 230, 64, 24, 32
    origins, (ey, ex) = tile_origins(h, w, tile, overlap, align)
    v = torch.rand(len(origins), c, ey, ex, generator=torch.Generator().manual_seed(2)) * 2 - 1
    _, a5, w5 = _run_blend(v, h, w, tile, overlap, align, 5)
    _, b5, v5 = _run_blend(v, h, w, tile, overlap, align, 5)
    _, a1, w1 = _run_blend(v, h, w, tile, overlap, align, 1)
    _, a24, w24 = _run_blend(v, h, w, tile, overlap, align, 24)
    for a, ww in ((b5, v5), (a1, w1), (a24, w24)):
        assert torch.equal(a, a5) and torch.equal(ww, w5)          # bit for bit: the same per-pixel summation order


# ------------------------------------------------------------------------------------------------
# the network
# ------------------------------------------------------------------------------------------------
def _engine(ic=3, oc=3, norm="batch", num_downs=7, use_dropout=False, seed=0):
    """An engine with the reference's seeded init and non-trivial BatchNorm running statistics."""
    torch.manual_seed(seed)
    eng = GeneratorEngine(DEV, ic, oc, num_downs, use_dropout=use_dropout, norm=norm, dropout_seed=5)
    g = torch.Generator(device=DEV).manual_seed(seed + 1)
    for bn in eng.bns.values():
        bn.running_mean.copy_(torch.randn(bn.c, device=DEV, generator=g) * 0.2)
        bn.running_var.copy_(torch.rand(bn.c, device=DEV, generator=g) + 0.5)
        bn.nbt.fill_(7)
    return eng


def _scene(c, h, w, seed):
    """A normalised fp32 [C, H, W] scene on the device: smooth structure plus noise."""
    g = torch.Generator().manual_seed(seed)
    base = torch.nn.functional.interpolate(torch.rand(1, c, h // 8 + 2, w // 8 + 2, generator=g), size=(h, w),
                                           mode="bilinear", align_corners=False)[0]
    return (base * 2 - 1 + 0.1 * torch.randn(c, h, w, generator=g)).clamp(-1, 1).to(DEV)


def _tile_outputs(eng, x, tile, overlap, batch):
    """Per-tile outputs of the existing eval forward on torch-cut crops, run in batches of `batch` (zero-padded, as
    translate_scene runs them): [n_tiles, output_nc, ey, ex] fp32."""
    align = 1 << eng.L
    crops = cut_tiles(x, tile, overlap, align)
    out = []
    was = eng.training
    eng.training = False
    try:
        for t0 in range(0, crops.shape[0], batch):
            chunk = torch.zeros(batch, *crops.shape[1:], device=DEV)
            nv = min(batch, crops.shape[0] - t0)
            chunk[:nv] = crops[t0:t0 + nv]
            out.append(eng.forward(chunk.contiguous())[:nv, ..., :eng.output_nc].permute(0, 3, 1, 2).clone())
    finally:
        eng.training = was
    return torch.cat(out)


def test_a_one_tile_scene_gives_the_eval_forward():
    eng = _engine()
    x = _scene(3, 128, 256, 4)
    eng.training = False
    u8 = torch.empty(1, 128, 256, 3, device=DEV, dtype=torch.uint8)
    fake = eng.forward(x[None].contiguous(), out_u8=u8)[0, ..., :3].permute(2, 0, 1).clone()
    res = eng.translate_scene(x, tile=256, batch=1, return_float=True)
    assert res.image.shape == (128, 256, 3) and res.image.dtype == torch.uint8
    assert res.values.shape == (3, 128, 256) and res.values.dtype == torch.float32
    assert float((res.values - fake).abs().max()) < 1e-6
    ok = ~near_integer(fake.cpu(), 1e-3).permute(1, 2, 0)
    assert torch.equal(res.image.cpu()[ok], u8[0].cpu()[ok])
    plain = eng.translate_scene(x, tile=256, batch=1)
    assert plain.values is None and torch.equal(plain.image, res.image)


@pytest.mark.parametrize("ic,oc,norm", [(3, 3, "batch"), (1, 3, "batch"), (4, 4, "batch"), (3, 3, "instance")])
@pytest.mark.parametrize("h,w", [(300, 420), (7, 333)])
def test_end_to_end_against_per_tile_outputs_blended_in_fp64(ic, oc, norm, h, w):
    tile, overlap, batch = 128, 32, 4
    eng = _engine(ic, oc, norm)
    x = _scene(ic, h, w, 20 + ic + oc + h)
    want = blend_image_ref(_tile_outputs(eng, x, tile, overlap, batch), h, w, tile, overlap, 128)
    res = eng.translate_scene(x, tile=tile, overlap=overlap, batch=batch, return_float=True)
    assert res.values.shape == (oc, h, w) and res.image.shape == (h, w, oc)
    err = float((res.values.cpu().double() - want).abs().max())
    assert err < 1e-5, err
    ok = ~near_integer(want, 1e-3).permute(1, 2, 0)
    assert torch.equal(res.image.cpu()[ok], u8_ref(want).permute(1, 2, 0)[ok])


def test_uint8_scene_from_the_host_matches_its_normalised_form():
    h, w, tile, overlap = 300, 420, 128, 32
    eng = _engine()
    u = torch.randint(0, 256, (h, w, 3), generator=torch.Generator().manual_seed(77), dtype=torch.uint8)
    out = torch.zeros(1, h, w, 4, device=DEV, dtype=torch.bfloat16)
    ops.u8_hwc_to_nhwc_bf16(u[None].to(DEV), out)
    f = out[0, ..., :3].permute(2, 0, 1).float().contiguous()      # bf16 values are exact in fp32
    res = eng.translate_scene(u, tile=tile, overlap=overlap, batch=4, return_float=True)
    same = eng.translate_scene(f, tile=tile, overlap=overlap, batch=4, return_float=True)
    assert torch.equal(res.values, same.values) and torch.equal(res.image, same.image)
    dev_u8 = eng.translate_scene(u.to(DEV), tile=tile, overlap=overlap, batch=4, return_float=True)
    assert torch.equal(dev_u8.values, res.values) and torch.equal(dev_u8.image, res.image)


def _state(eng):
    bufs = [t.clone() for bn in eng.bns.values() for t in (bn.running_mean, bn.running_var, bn.nbt)]
    return eng.store.p.clone(), eng.store.g.clone(), bufs


def test_determinism_batch_independence_and_no_side_effects():
    h, w = 300, 420
    eng = _engine(use_dropout=True)
    eng.store.g.copy_(torch.randn(eng.store.g.shape, device=DEV, generator=torch.Generator(device=DEV).manual_seed(3)))
    x = _scene(3, h, w, 3)
    eng.training = True
    calls = eng.dropout_calls
    p0, g0, b0 = _state(eng)
    kw = dict(tile=128, overlap=32, return_float=True)
    r1 = eng.translate_scene(x, batch=4, **kw)
    r2 = eng.translate_scene(x, batch=4, **kw)
    assert torch.equal(r1.image, r2.image) and torch.equal(r1.values, r2.values)
    r3 = eng.translate_scene(x, batch=1, **kw)
    want = r1.values.double().cpu()
    assert float((r3.values.double().cpu() - want).abs().max()) < 1e-5
    ok = ~near_integer(want, 1e-3).permute(1, 2, 0)
    assert torch.equal(r3.image.cpu()[ok], r1.image.cpu()[ok])
    assert eng.training is True and eng.dropout_calls == calls
    p1, g1, b1 = _state(eng)
    assert torch.equal(p0, p1) and torch.equal(g0, g1)
    assert all(torch.equal(a, b) for a, b in zip(b0, b1))
    # device inputs: no host synchronisation anywhere in the call
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        r4 = eng.translate_scene(x, batch=4, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.equal(r4.values, r1.values) and torch.equal(r4.image, r1.image)


def test_training_after_a_scene_matches_a_trainer_that_never_translated():
    gen = torch.Generator().manual_seed(9)
    batches = [(torch.rand(2, 3, 64, 64, generator=gen) * 2 - 1, torch.rand(2, 3, 64, 64, generator=gen) * 2 - 1)
               for _ in range(4)]
    scene = torch.randint(0, 256, (150, 100, 3), generator=gen, dtype=torch.uint8)
    res, states = [], []
    for translate in (False, True):
        torch.manual_seed(0)
        tr = Pix2PixTrainer(DEV, num_downs=5)
        seq = [tr.train_step(batches[0][0].to(DEV), batches[0][1].to(DEV)).cpu().clone()]
        if translate:
            out = tr.G.translate_scene(scene, tile=64, overlap=16, batch=3)
            assert out.image.shape == (150, 100, 3)
        for a, b in batches[1:]:
            seq.append(tr.train_step_graphed(a.to(DEV), b.to(DEV)).cpu().clone())
        res.append(torch.stack(seq))
        states.append((tr.G.store.p.clone(), tr.G.dropout_calls, [t.clone() for bn in tr.G.bns.values()
                                                                  for t in (bn.running_mean, bn.nbt)]))
    assert torch.allclose(res[0], res[1], rtol=2e-3, atol=2e-4), (res[0], res[1])
    assert states[0][1] == states[1][1]
    assert all(int(a) == int(b) for a, b in zip(states[0][2][1::2], states[1][2][1::2]))     # num_batches_tracked
    assert float((states[0][0] - states[1][0]).abs().max()) < 1e-3


def test_dropin_module_matches_the_engine_in_train_and_eval_mode():
    h, w = 200, 260
    torch.manual_seed(3)
    m = M.UNetGenerator(3, 3)
    sd = {k: v.detach().clone() for k, v in m.state_dict().items()}
    eng = GeneratorEngine(DEV, init=False)
    eng.load_state_dict(sd)
    m = m.to(DEV)
    x = _scene(3, h, w, 11)
    kw = dict(tile=128, overlap=32, batch=4, return_float=True)
    want = eng.translate_scene(x, **kw)
    nbt = [b.clone() for n, b in m.named_buffers() if n.endswith("num_batches_tracked")]
    m.train()
    a = m.translate_scene(x, **kw)
    assert m.training and m._engine_obj.training
    m.eval()
    b = m.translate_scene(x, **kw)
    assert not m.training
    for r in (a, b):
        assert torch.equal(r.image, want.image) and torch.equal(r.values, want.values)
        assert not r.values.requires_grad
    assert all(torch.equal(x_, y_) for x_, y_ in zip(nbt, [b_ for n, b_ in m.named_buffers()
                                                          if n.endswith("num_batches_tracked")]))


def test_a_4096_scene_at_tile_256():
    h = w = 4096
    eng = _engine()
    u = torch.randint(0, 256, (h, w, 3), generator=torch.Generator().manual_seed(8), dtype=torch.uint8).to(DEV)
    res = eng.translate_scene(u, tile=256, overlap=64, batch=64, return_float=True)
    assert res.image.shape == (h, w, 3) and res.image.dtype == torch.uint8
    assert res.values.shape == (3, h, w)
    assert bool(torch.isfinite(res.values).all())
    assert float(res.values.abs().max()) <= 1 + 1e-6           # a convex blend of Tanh outputs (fp32 division)
    other = eng.translate_scene(u, tile=256, overlap=64, batch=16, return_float=True)
    assert float((other.values - res.values).abs().max()) < 1e-5
