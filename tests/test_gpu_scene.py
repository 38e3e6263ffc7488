"""Sliding-window scene inference (SiameseEngine.predict_scene) on the GPU: the gather kernel bit for bit against the
existing converters, blend + finalize on synthetic logits against the fp64 reference of tests/scene_ref.py, single-tile
equivalence with predict() / forward(), end-to-end runs against per-tile logits of the eval forward blended in fp64,
determinism, side effects, the drop-in module and a 2048 x 2048 scene."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from gan_aug_pfa_b200 import models as M  # noqa: E402
from gan_aug_pfa_b200 import ops  # noqa: E402
from gan_aug_pfa_b200.siamese import SiameseEngine, _scene_grid  # noqa: E402
from scene_ref import blend_ref, cut_tiles, near_tie, pred_ref, tile_origins  # noqa: E402

DEV = torch.device("cuda:0")
NAN = float("nan")
G = 68          # guard elements on either side of every kernel output (a multiple of 4: the gather writes
#                one 8-byte store per 4-slot bf16 pixel and needs 8-byte aligned outputs)


def _guarded(numel, dtype, fill):
    buf = torch.full((numel + 2 * G,), fill, device=DEV, dtype=dtype)
    return buf, buf[G:G + numel]


def _guards_intact(buf, fill):
    a, b = buf[:G], buf[-G:]
    if isinstance(fill, float) and fill != fill:
        return bool(torch.isnan(a).all() and torch.isnan(b).all())
    return bool((a == fill).all() and (b == fill).all())


# ------------------------------------------------------------------------------------------------
# gather
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [1, 2, 3, 4])
@pytest.mark.parametrize("u8", [True, False])
@pytest.mark.parametrize("h,w", [(37, 70), (20, 45)])
def test_gather_is_bit_identical_to_the_converters(c, u8, h, w):
    tile, overlap, batch = 32, 8, 4
    g = torch.Generator().manual_seed(c * 10 + h)
    if u8:
        s1, s2 = (torch.randint(0, 256, (h, w, c), generator=g, dtype=torch.uint8) for _ in range(2))
        chw = [s.permute(2, 0, 1) for s in (s1, s2)]
    else:
        s1, s2 = (torch.randn(c, h, w, generator=g) * 1.5 for _ in range(2))
        chw = [s1, s2]
    origins, (ey, ex) = tile_origins(h, w, tile, overlap)
    grid = _scene_grid(h, w, tile, overlap)
    n_t = len(origins)
    ref = []
    for s in chw:
        crops = cut_tiles(s, tile, overlap)                       # [n_t, c, ey, ex]
        out = torch.zeros(n_t, ey, ex, 4, device=DEV, dtype=torch.bfloat16)
        for t in range(n_t):
            if u8:
                ops.u8_hwc_to_nhwc_bf16(crops[t].permute(1, 2, 0).contiguous()[None].to(DEV), out[t:t + 1])
            else:
                ops.nchw_to_nhwc_bf16(crops[t][None].contiguous().to(DEV), out[t:t + 1])
        ref.append(out)
    d1, d2 = s1.to(DEV), s2.to(DEV)
    numel = batch * ey * ex * 4
    for t0 in range(0, n_t, batch):
        b1, o1 = _guarded(numel, torch.bfloat16, NAN)
        b2, o2 = _guarded(numel, torch.bfloat16, NAN)
        ops.scene_gather(d1, d2, grid, t0, o1.view(batch, ey, ex, 4), o2.view(batch, ey, ex, 4))
        assert _guards_intact(b1, NAN) and _guards_intact(b2, NAN)
        for o, r in ((o1, ref[0]), (o2, ref[1])):
            o = o.view(batch, ey, ex, 4)
            nv = min(batch, n_t - t0)
            assert torch.equal(o[:nv].view(torch.int16), r[t0:t0 + nv].view(torch.int16))
            assert (o[:, ..., c:].view(torch.int16) == 0).all()         # slots >= C
            assert (o[nv:].view(torch.int16) == 0).all()                 # padding tiles of the last batch
    if h < tile:
        assert ey == 32 and ex == 32 and origins[0][0] == 0          # one row of tiles, rows past 20 repeat row 19


# ------------------------------------------------------------------------------------------------
# blend + finalize on synthetic logits
# ------------------------------------------------------------------------------------------------
def _synthetic(k, h, w, tile, overlap, seed):
    origins, (ey, ex) = tile_origins(h, w, tile, overlap)
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(len(origins), k, ey, ex, generator=g) * 3
    big = torch.rand(z.shape, generator=g)
    z[big < 0.02] = 30.0
    z[big > 0.98] = -30.0
    lab = torch.randint(0, max(k, 2), (h, w), generator=g)
    r = torch.rand(h, w, generator=g)
    lab[r < 0.05] = -100
    lab[(r >= 0.05) & (r < 0.08)] = -1
    lab[(r >= 0.08) & (r < 0.11)] = max(k, 2)
    return z, lab


def _run_blend(z, h, w, tile, overlap, batch):
    """blend every batch into NaN-guarded accumulators (padding tiles of the last batch hold NaN: never read)."""
    n_t, k, ey, ex = z.shape
    grid = _scene_grid(h, w, tile, overlap)
    ab, acc = _guarded(k * h * w, torch.float32, NAN)
    wb, ws = _guarded(h * w, torch.float32, NAN)
    zd = z.to(DEV)
    for t0 in range(0, n_t, batch):
        lg = torch.full((batch, k, ey, ex), NAN, device=DEV)
        nv = min(batch, n_t - t0)
        lg[:nv] = zd[t0:t0 + nv]
        ops.scene_blend(lg[:, 0].contiguous() if k == 1 else lg, grid, t0, acc.view(k, h, w), ws.view(h, w))
    assert _guards_intact(ab, NAN) and _guards_intact(wb, NAN)
    return ab, acc.view(k, h, w), ws.view(h, w)


@pytest.mark.parametrize("k", [1, 2, 7, 16])
def test_blend_and_finalize_match_the_fp64_reference(k):
    h, w, tile, overlap, batch = 150, 230, 64, 24, 5
    z, lab = _synthetic(k, h, w, tile, overlap, 40 + k)
    want = blend_ref(z, h, w, tile, overlap)
    ab, acc, ws = _run_blend(z, h, w, tile, overlap, batch)
    assert torch.isfinite(ws).all() and (ws > 0).all()
    pb, pred = _guarded(h * w, torch.uint8, 0xEE)
    counts = torch.zeros((4,) if k == 1 else (k, k), device=DEV, dtype=torch.int64)
    ops.scene_finalize(acc, ws, pred.view(h, w), True, lab.to(DEV), -100, counts)
    assert _guards_intact(pb, 0xEE) and _guards_intact(ab, NAN)
    probs = acc.cpu().double()
    err = float((probs - want).abs().max())
    assert err < 2e-6, err
    got = pred.view(h, w).cpu()
    ok = ~near_tie(want, 1e-6)
    assert torch.equal(got[ok], pred_ref(want)[ok])
    # the exact comparison covers nearly every pixel (the +-30 logits make some exact ties: about 1 % at K = 16)
    assert int(ok.sum()) > 0.97 * h * w
    # confusion = bincount of (label, returned pred) over the counted labels
    lab_v, pr = lab.reshape(-1), got.reshape(-1).long()
    if k == 1:
        keep = (lab_v == 0) | (lab_v == 1)
        l, p = lab_v[keep], pr[keep]
        ref = torch.stack([((l == 1) & (p == 1)).sum(), ((l == 0) & (p == 1)).sum(), ((l == 1) & (p == 0)).sum(),
                           ((l == 0) & (p == 0)).sum()])
    else:
        keep = (lab_v >= 0) & (lab_v < k)
        ref = torch.bincount(lab_v[keep] * k + pr[keep], minlength=k * k).view(k, k)
    assert torch.equal(counts.cpu(), ref)
    # without probs the accumulators are left as they were; without labels nothing is counted
    _, acc2, ws2 = _run_blend(z, h, w, tile, overlap, batch)
    before = acc2.clone()
    pred2 = torch.empty(h, w, device=DEV, dtype=torch.uint8)
    ops.scene_finalize(acc2, ws2, pred2, False)
    assert torch.equal(acc2, before) and torch.equal(pred2.cpu(), got)


def test_blend_is_deterministic_and_independent_of_the_batch():
    k, h, w, tile, overlap = 7, 150, 230, 64, 24
    z, _ = _synthetic(k, h, w, tile, overlap, 9)
    _, a5, w5 = _run_blend(z, h, w, tile, overlap, 5)
    _, b5, v5 = _run_blend(z, h, w, tile, overlap, 5)
    _, a1, w1 = _run_blend(z, h, w, tile, overlap, 1)
    _, a24, w24 = _run_blend(z, h, w, tile, overlap, 24)
    for a, ww in ((b5, v5), (a1, w1), (a24, w24)):
        assert torch.equal(a, a5) and torch.equal(ww, w5)          # bit for bit: the same per-pixel summation order


# ------------------------------------------------------------------------------------------------
# the network
# ------------------------------------------------------------------------------------------------
def _engine(k, seed=0):
    torch.manual_seed(seed)
    sd = {kk: v.detach().clone() for kk, v in M.SiameseUNet(3, k).state_dict().items()}
    eng = SiameseEngine(DEV, 3, k)
    eng.load_state_dict(sd)
    return eng, sd


def _scene(h, w, seed, u8=False):
    g = torch.Generator().manual_seed(seed)
    if u8:
        return [torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8) for _ in range(2)]
    # smooth structure plus noise, so that the two images differ in places
    base = torch.nn.functional.interpolate(torch.rand(1, 3, h // 8 + 2, w // 8 + 2, generator=g), size=(h, w),
                                           mode="bilinear", align_corners=False)[0]
    x1 = (base * 2 - 1 + 0.1 * torch.randn(3, h, w, generator=g)).clamp(-1, 1)
    x2 = x1.clone()
    x2[:, h // 3:h // 2, w // 4:w // 2] = torch.rand(3, h // 2 - h // 3, w // 2 - w // 4, generator=g) * 2 - 1
    return [x1.to(DEV), x2.to(DEV)]


def _tile_logits(eng, x1, x2, tile, overlap):
    """Per-tile logits of the existing eval forward on torch-cut crops: [n_tiles, K, ey, ex]."""
    c1, c2 = cut_tiles(x1, tile, overlap), cut_tiles(x2, tile, overlap)
    was = eng.training
    eng.training = False
    try:
        z = eng.forward(c1.contiguous(), c2.contiguous()).clone()
    finally:
        eng.training = was
        eng._tape = []
    return z.unsqueeze(1) if z.dim() == 3 else z


@pytest.mark.parametrize("k", [1, 2, 7])
def test_a_one_tile_scene_gives_predict(k):
    eng, _ = _engine(k)
    x1, x2 = _scene(128, 192, 5 + k)
    eng.training = False
    logits = eng.forward(x1[None], x2[None]).clone()
    if k == 1:
        want = (torch.sigmoid(logits[0]) > 0.5).to(torch.uint8)
        tie = logits[0].abs() < 1e-6
    else:
        want = eng.predict(x1[None], x2[None])[0]
        top = logits[0].topk(2, dim=0).values
        tie = (top[0] - top[1]) < 1e-5
    res = eng.predict_scene(x1, x2, tile=256)
    assert res.pred.shape == (128, 192) and res.pred.dtype == torch.uint8
    assert res.probs is None and res.confusion is None
    assert torch.equal(res.pred[~tie], want[~tie])


@pytest.mark.parametrize("k", [1, 2, 7])
@pytest.mark.parametrize("h,w", [(300, 420), (7, 333)])
def test_end_to_end_against_per_tile_logits_blended_in_fp64(k, h, w):
    tile, overlap = 128, 32
    eng, _ = _engine(k)
    x1, x2 = _scene(h, w, 20 + k + h)
    want = blend_ref(_tile_logits(eng, x1, x2, tile, overlap), h, w, tile, overlap)
    res = eng.predict_scene(x1, x2, tile=tile, overlap=overlap, batch=4, return_probs=True)
    assert res.probs.shape == (k, h, w) and res.probs.dtype == torch.float32
    err = float((res.probs.cpu().double() - want).abs().max())
    assert err < 1e-5, err
    ok = ~near_tie(want, 1e-5)
    assert torch.equal(res.pred.cpu()[ok], pred_ref(want)[ok])


def test_uint8_scene_from_the_host_matches_its_normalised_form():
    k, h, w, tile, overlap = 2, 300, 420, 128, 32
    eng, _ = _engine(k)
    u1, u2 = _scene(h, w, 77, u8=True)
    # the fp32 form of what the device normalisation produces (bf16 values are exact in fp32)
    f = []
    for u in (u1, u2):
        out = torch.zeros(1, h, w, 4, device=DEV, dtype=torch.bfloat16)
        ops.u8_hwc_to_nhwc_bf16(u[None].to(DEV), out)
        f.append(out[0, ..., :3].permute(2, 0, 1).float().contiguous())
    want = blend_ref(_tile_logits(eng, f[0], f[1], tile, overlap), h, w, tile, overlap)
    res = eng.predict_scene(u1, u2, tile=tile, overlap=overlap, batch=4, return_probs=True)
    assert float((res.probs.cpu().double() - want).abs().max()) < 1e-5
    same = eng.predict_scene(f[0], f[1], tile=tile, overlap=overlap, batch=4, return_probs=True)
    assert torch.equal(res.probs, same.probs) and torch.equal(res.pred, same.pred)


def _state(eng):
    bufs = [t.clone() for bn in eng.bns.values() for t in (bn.running_mean, bn.running_var, bn.nbt)]
    return eng.store.p.clone(), eng.store.g.clone(), bufs


def test_determinism_batch_independence_and_no_side_effects():
    k, h, w = 2, 300, 420
    eng, _ = _engine(k)
    x1, x2 = _scene(h, w, 3)
    lab = (torch.rand(h, w, generator=torch.Generator().manual_seed(1)) < 0.3).long().to(DEV)
    eng.training = True
    p0, g0, b0 = _state(eng)
    kw = dict(tile=128, overlap=32, return_probs=True, labels=lab)
    r1 = eng.predict_scene(x1, x2, batch=4, **kw)
    r2 = eng.predict_scene(x1, x2, batch=4, **kw)
    assert torch.equal(r1.pred, r2.pred) and torch.equal(r1.probs, r2.probs) and torch.equal(r1.confusion, r2.confusion)
    r3 = eng.predict_scene(x1, x2, batch=1, **kw)
    want = r1.probs.double().cpu()
    assert float((r3.probs.double().cpu() - want).abs().max()) < 1e-5
    ok = ~near_tie(want, 1e-5)
    assert torch.equal(r3.pred.cpu()[ok], r1.pred.cpu()[ok])
    assert eng.training is True and eng._tape == []
    p1, g1, b1 = _state(eng)
    assert torch.equal(p0, p1) and torch.equal(g0, g1)
    assert all(torch.equal(a, b) for a, b in zip(b0, b1))
    assert int(r1.confusion.sum()) == h * w
    # device inputs: no host synchronisation anywhere in the call
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        r4 = eng.predict_scene(x1, x2, batch=4, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.equal(r4.probs, r1.probs)


def test_dropin_module_matches_the_engine_in_train_and_eval_mode():
    k, h, w = 7, 200, 260
    eng, sd = _engine(k, seed=3)
    m = M.SiameseUNet(3, k)
    m.load_state_dict(sd)
    m = m.to(DEV)
    x1, x2 = _scene(h, w, 11)
    kw = dict(tile=128, overlap=32, batch=4, return_probs=True)
    want = eng.predict_scene(x1, x2, **kw)
    nbt = [b.clone() for n, b in m.named_buffers() if n.endswith("num_batches_tracked")]
    m.train()
    a = m.predict_scene(x1, x2, **kw)
    assert m.training and m._engine_obj.training
    m.eval()
    b = m.predict_scene(x1, x2, **kw)
    for r in (a, b):
        assert torch.equal(r.pred, want.pred) and torch.equal(r.probs, want.probs)
    assert all(torch.equal(x, y) for x, y in zip(nbt, [b_ for n, b_ in m.named_buffers()
                                                        if n.endswith("num_batches_tracked")]))


def test_a_2048_scene_at_tile_512_with_labels():
    k, h, w = 2, 2048, 2048
    eng, _ = _engine(k)
    g = torch.Generator().manual_seed(8)
    u1, u2 = (torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8) for _ in range(2))
    lab = (torch.rand(h, w, generator=g) < 0.02).long()
    lab[torch.rand(h, w, generator=g) < 0.01] = -100
    res = eng.predict_scene(u1.to(DEV), u2.to(DEV), tile=512, overlap=64, batch=4, return_probs=True,
                            labels=lab.to(DEV))
    assert not torch.isnan(res.probs).any()
    assert int(res.confusion.sum()) == int((lab != -100).sum())
    assert torch.equal(res.pred.long(), res.probs.argmax(0))
