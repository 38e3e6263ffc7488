"""Test-time augmentation and checkpoint ensembles over whole scenes (siamese.predict_scene_ensemble) on the GPU: the
transformed gather bit for bit against the existing converters, the multi-pass blend against the fp64 reference of
tests/tta_ref.py, end-to-end runs against per-pass per-tile logits of the eval forward, equivariance on symmetric
grids, ensembles of two networks, side effects and the drop-in module."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from gan_aug_pfa_b200 import models as M  # noqa: E402
from gan_aug_pfa_b200 import ops  # noqa: E402
from gan_aug_pfa_b200.siamese import TTA_TRANSFORMS, SiameseEngine, _scene_grid, predict_scene_ensemble  # noqa: E402
from scene_ref import cut_tiles, near_tie, pred_ref, tile_origins  # noqa: E402
from tta_ref import blend_passes_ref, f, passes  # noqa: E402

DEV = torch.device("cuda:0")
NAN = float("nan")
G = 68          # guard elements on either side of every kernel output (a multiple of 4: 8-byte aligned gather stores)


def _guarded(numel, dtype, fill):
    buf = torch.full((numel + 2 * G,), fill, device=DEV, dtype=dtype)
    return buf, buf[G:G + numel]


def _guards_intact(buf):
    return bool(torch.isnan(buf[:G].float()).all() and torch.isnan(buf[-G:].float()).all())


# ------------------------------------------------------------------------------------------------
# gather
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c", [1, 2, 3, 4])
@pytest.mark.parametrize("u8", [True, False])
@pytest.mark.parametrize("h,w,tile", [(37, 150, 64), (100, 130, 32)])      # ey = 48 != ex = 64; square 32 x 32
def test_transformed_gather_is_bit_identical_to_the_converters(c, u8, h, w, tile):
    overlap, batch = 16, 3
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
    d1, d2 = s1.to(DEV), s2.to(DEV)
    for d in range(8):
        oy, ox = (ex, ey) if d & 4 else (ey, ex)
        ref = []
        for s in chw:
            crops = f(cut_tiles(s, tile, overlap), d)                       # [n_t, c, oy, ox]
            out = torch.zeros(n_t, oy, ox, 4, device=DEV, dtype=torch.bfloat16)
            for t in range(n_t):
                if u8:
                    ops.u8_hwc_to_nhwc_bf16(crops[t].permute(1, 2, 0).contiguous()[None].to(DEV), out[t:t + 1])
                else:
                    ops.nchw_to_nhwc_bf16(crops[t][None].contiguous().to(DEV), out[t:t + 1])
            ref.append(out)
        numel = batch * oy * ox * 4
        for t0 in range(0, n_t, batch):
            b1, o1 = _guarded(numel, torch.bfloat16, NAN)
            b2, o2 = _guarded(numel, torch.bfloat16, NAN)
            ops.scene_gather(d1, d2, grid, t0, o1.view(batch, oy, ox, 4), o2.view(batch, oy, ox, 4), d)
            assert _guards_intact(b1) and _guards_intact(b2)
            nv = min(batch, n_t - t0)
            for o, r in ((o1, ref[0]), (o2, ref[1])):
                o = o.view(batch, oy, ox, 4)
                assert torch.equal(o[:nv].view(torch.int16), r[t0:t0 + nv].view(torch.int16)), d
                assert (o[:, ..., c:].view(torch.int16) == 0).all()
                assert (o[nv:].view(torch.int16) == 0).all()                # padding tiles of the last batch


# ------------------------------------------------------------------------------------------------
# multi-pass blend on synthetic logits
# ------------------------------------------------------------------------------------------------
def _synthetic_passes(k, h, w, tile, overlap, ds, seed):
    origins, (ey, ex) = tile_origins(h, w, tile, overlap)
    g = torch.Generator().manual_seed(seed)
    out = []
    for d in ds:
        oy, ox = (ex, ey) if d & 4 else (ey, ex)
        z = torch.randn(len(origins), k, oy, ox, generator=g) * 3
        big = torch.rand(z.shape, generator=g)
        z[big < 0.02] = 30.0
        z[big > 0.98] = -30.0
        out.append((d, z))
    return out


def _run_passes(per_pass, h, w, tile, overlap, batch):
    """blend every pass into NaN-guarded accumulators (padding tiles of the last batch hold NaN: never read)."""
    k = per_pass[0][1].shape[1]
    grid = _scene_grid(h, w, tile, overlap)
    ab, acc = _guarded(k * h * w, torch.float32, NAN)
    wb, ws = _guarded(h * w, torch.float32, NAN)
    for i, (d, z) in enumerate(per_pass):
        n_t, _, oy, ox = z.shape
        zd = z.to(DEV)
        for t0 in range(0, n_t, batch):
            lg = torch.full((batch, k, oy, ox), NAN, device=DEV)
            nv = min(batch, n_t - t0)
            lg[:nv] = zd[t0:t0 + nv]
            ops.scene_blend(lg[:, 0].contiguous() if k == 1 else lg, grid, t0, acc.view(k, h, w), ws.view(h, w),
                            d=d, first_pass=i == 0)
    assert _guards_intact(ab) and _guards_intact(wb)
    return acc.view(k, h, w), ws.view(h, w)


@pytest.mark.parametrize("k", [1, 2, 7, 16])
@pytest.mark.parametrize("h,w", [(150, 230), (40, 230)])           # square 64 x 64 tiles; ey = 48 != ex = 64
def test_multi_pass_blend_matches_the_fp64_reference(k, h, w):
    tile, overlap, batch = 64, 24, 5
    per_pass = _synthetic_passes(k, h, w, tile, overlap, [5, 0, 3, 4, 7, 1, 6, 2, 4], 40 + k + h)
    want = blend_passes_ref(per_pass, h, w, tile, overlap)
    acc, ws = _run_passes(per_pass, h, w, tile, overlap, batch)
    assert torch.isfinite(ws).all() and (ws > 0).all()
    pred = torch.empty(h, w, device=DEV, dtype=torch.uint8)
    ops.scene_finalize(acc, ws, pred, True)
    err = float((acc.cpu().double() - want).abs().max())
    assert err < 1e-5, err
    ok = ~near_tie(want, 1e-5)
    assert torch.equal(pred.cpu()[ok], pred_ref(want)[ok])


def test_multi_pass_blend_is_deterministic_and_independent_of_the_batch():
    k, h, w, tile, overlap = 7, 40, 230, 64, 24
    per_pass = _synthetic_passes(k, h, w, tile, overlap, range(8), 9)
    a5, w5 = _run_passes(per_pass, h, w, tile, overlap, 5)
    for batch in (5, 1, 24):
        a, ww = _run_passes(per_pass, h, w, tile, overlap, batch)
        assert torch.equal(a, a5) and torch.equal(ww, w5)


def test_a_later_pass_never_restarts_a_pixel():
    """first_pass=False adds onto what the accumulators hold, even at a pixel's first covering tile."""
    k, h, w, tile, overlap = 2, 150, 230, 64, 24
    (d0, z), = _synthetic_passes(k, h, w, tile, overlap, [6], 3)
    grid = _scene_grid(h, w, tile, overlap)
    acc = torch.full((k, h, w), 2.0, device=DEV)
    ws = torch.full((h, w), 3.0, device=DEV)
    zd = z.to(DEV)
    for t0 in range(0, z.shape[0], 4):
        lg = torch.zeros(4, k, *z.shape[-2:], device=DEV)
        lg[:min(4, z.shape[0] - t0)] = zd[t0:t0 + 4]
        ops.scene_blend(lg, grid, t0, acc, ws, d=d0, first_pass=False)
    one = _run_passes([(d0, z)], h, w, tile, overlap, 4)
    assert float((acc - 2.0 - one[0]).abs().max()) < 1e-5 and float((ws - 3.0 - one[1]).abs().max()) < 1e-5


# ------------------------------------------------------------------------------------------------
# the network
# ------------------------------------------------------------------------------------------------
def _engine(k, seed=0, c=3):
    torch.manual_seed(seed)
    sd = {kk: v.detach().clone() for kk, v in M.SiameseUNet(c, k).state_dict().items()}
    eng = SiameseEngine(DEV, c, k)
    eng.load_state_dict(sd)
    return eng, sd


def _scene(h, w, seed):
    g = torch.Generator().manual_seed(seed)
    base = torch.nn.functional.interpolate(torch.rand(1, 3, h // 8 + 2, w // 8 + 2, generator=g), size=(h, w),
                                           mode="bilinear", align_corners=False)[0]
    x1 = (base * 2 - 1 + 0.1 * torch.randn(3, h, w, generator=g)).clamp(-1, 1)
    x2 = x1.clone()
    x2[:, h // 3:h // 2, w // 4:w // 2] = torch.rand(3, h // 2 - h // 3, w // 2 - w // 4, generator=g) * 2 - 1
    return [x1.to(DEV), x2.to(DEV)]


def _pass_logits(eng, x1, x2, tile, overlap, d):
    """Logits of the existing eval forward on torch-transformed crops f_d(tile): [n_tiles, K, oy, ox]."""
    c1, c2 = f(cut_tiles(x1, tile, overlap), d), f(cut_tiles(x2, tile, overlap), d)
    was = eng.training
    eng.training = False
    try:
        z = eng.forward(c1.contiguous(), c2.contiguous()).clone()
    finally:
        eng.training = was
        eng._tape = []
    return z.unsqueeze(1) if z.dim() == 3 else z


@pytest.mark.parametrize("k", [1, 2, 7])
@pytest.mark.parametrize("h,w", [(300, 420), (7, 333)])
@pytest.mark.parametrize("tta", ["flips", "d4"])
def test_tta_end_to_end_against_per_pass_tile_logits_blended_in_fp64(k, h, w, tta):
    tile, overlap = 128, 32
    eng, _ = _engine(k)
    x1, x2 = _scene(h, w, 20 + k + h)
    want = blend_passes_ref([(d, _pass_logits(eng, x1, x2, tile, overlap, d)) for _, d in passes(1, tta)],
                            h, w, tile, overlap)
    res = eng.predict_scene(x1, x2, tile=tile, overlap=overlap, batch=4, return_probs=True, tta=tta)
    assert res.probs.shape == (k, h, w) and res.probs.dtype == torch.float32
    err = float((res.probs.cpu().double() - want).abs().max())
    assert err < 1e-5, err
    ok = ~near_tie(want, 1e-5)
    assert torch.equal(res.pred.cpu()[ok], pred_ref(want)[ok])
    if tta == "d4" and h == 7:
        assert eng._n == (4, 128, 16)              # re-sized at the transposed passes: [batch, ex, ey]


@pytest.mark.parametrize("tta,h,w", [("flips", 160, 208), ("d4", 160, 160)])
def test_tta_is_equivariant_on_a_symmetric_grid(tta, h, w):
    tile, overlap = 64, 16                         # 160 = 64 + 2 * 48, 208 = 64 + 3 * 48
    eng, _ = _engine(2, seed=4)
    x1, x2 = _scene(h, w, 31)
    kw = dict(tile=tile, overlap=overlap, batch=4, return_probs=True, tta=tta)
    base = eng.predict_scene(x1, x2, **kw).probs
    for g in TTA_TRANSFORMS[tta]:
        got = eng.predict_scene(f(x1, g).contiguous(), f(x2, g).contiguous(), **kw).probs
        err = float((got - f(base, g)).abs().max())
        assert err < 1e-5, (g, err)


# ------------------------------------------------------------------------------------------------
# ensembles
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("tta", [None, "d4"])
def test_a_one_member_ensemble_is_predict_scene(tta):
    k, h, w = 2, 300, 420
    eng, _ = _engine(k)
    x1, x2 = _scene(h, w, 3)
    lab = (torch.rand(h, w, generator=torch.Generator().manual_seed(1)) < 0.3).long().to(DEV)
    kw = dict(tile=128, overlap=32, batch=4, return_probs=True, labels=lab, tta=tta)
    a = eng.predict_scene(x1, x2, **kw)
    b = predict_scene_ensemble([eng], x1, x2, **kw)
    assert torch.equal(a.pred, b.pred) and torch.equal(a.probs, b.probs) and torch.equal(a.confusion, b.confusion)


@pytest.mark.parametrize("tta", [None, "flips"])
def test_two_members_average_their_probabilities(tta):
    k, h, w = 7, 200, 260
    ea, _ = _engine(k, seed=1)
    eb, _ = _engine(k, seed=2)
    x1, x2 = _scene(h, w, 8)
    kw = dict(tile=128, overlap=32, batch=4, return_probs=True, tta=tta)
    pa = ea.predict_scene(x1, x2, **kw).probs.double()
    pb = eb.predict_scene(x1, x2, **kw).probs.double()
    assert float((pa - pb).abs().max()) > 1e-2                 # the members differ
    lab = torch.randint(-1, k + 1, (h, w), generator=torch.Generator().manual_seed(2)).to(DEV)
    res = predict_scene_ensemble([ea, eb], x1, x2, labels=lab, **kw)
    want = (pa + pb) / 2
    assert float((res.probs.double() - want).abs().max()) < 1e-5
    ok = ~near_tie(want.cpu(), 1e-5)
    assert torch.equal(res.pred.cpu()[ok], pred_ref(want.cpu())[ok])
    assert int(res.confusion.sum()) == int(((lab >= 0) & (lab < k)).sum())


# ------------------------------------------------------------------------------------------------
# hygiene
# ------------------------------------------------------------------------------------------------
def _state(eng):
    bufs = [t.clone() for bn in eng.bns.values() for t in (bn.running_mean, bn.running_var, bn.nbt)]
    return eng.store.p.clone(), eng.store.g.clone(), bufs


def test_no_side_effects_and_no_host_synchronisation():
    k, h, w = 2, 7, 333                            # ey != ex: the d4 passes re-size the buffers
    ea, _ = _engine(k, seed=1)
    eb, _ = _engine(k, seed=2)
    x1, x2 = _scene(h, w, 3)
    lab = (torch.rand(h, w, generator=torch.Generator().manual_seed(1)) < 0.3).long().to(DEV)
    ea.training, eb.training = True, False
    before = [_state(e) for e in (ea, eb)]
    kw = dict(tile=128, overlap=32, batch=4, return_probs=True, labels=lab, tta="d4")
    r1 = predict_scene_ensemble([ea, eb], x1, x2, **kw)
    assert ea.training is True and eb.training is False and ea._tape == [] and eb._tape == []
    for e, (p0, g0, b0) in zip((ea, eb), before):
        p1, g1, b1 = _state(e)
        assert torch.equal(p0, p1) and torch.equal(g0, g1)
        assert all(torch.equal(a, b) for a, b in zip(b0, b1))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        r2 = predict_scene_ensemble([ea, eb], x1, x2, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert torch.equal(r1.probs, r2.probs) and torch.equal(r1.confusion, r2.confusion)
    r3 = predict_scene_ensemble([ea, eb], x1, x2, **{**kw, "batch": 1})
    assert torch.equal(r1.probs, r3.probs)                      # bit for bit: the per-pixel order is fixed


def test_value_errors_come_before_any_work():
    ea, _ = _engine(2, seed=1)
    eb, _ = _engine(7, seed=2)
    x1, x2 = _scene(64, 64, 3)
    cases = [([], x2, {}), ([ea, eb], x2, {}), ([ea], x2, {"tta": "d8"}), ([ea], x2, {"tile": 40}),
             ([ea], x2, {"batch": 0}), ([ea], x2, {"labels": torch.zeros(3, 3, dtype=torch.int64)}),
             ([ea], x2[:, :32].contiguous(), {})]
    for engines, y2, kw in cases:
        with pytest.raises(ValueError):
            predict_scene_ensemble(engines, x1, y2, **kw)
        assert ea._n is None and eb._n is None                  # no buffers, so no pass ever started


def test_dropin_modules_match_the_engines_in_train_and_eval_mode():
    k, h, w = 7, 200, 260
    ea, sda = _engine(k, seed=3)
    eb, sdb = _engine(k, seed=5)
    ma, mb = M.SiameseUNet(3, k), M.SiameseUNet(3, k)
    ma.load_state_dict(sda)
    mb.load_state_dict(sdb)
    ma, mb = ma.to(DEV), mb.to(DEV)
    x1, x2 = _scene(h, w, 11)
    kw = dict(tile=128, overlap=32, batch=4, return_probs=True, tta="d4")
    one = ea.predict_scene(x1, x2, **kw)
    both = predict_scene_ensemble([ea, eb], x1, x2, **kw)
    for mode in (True, False):
        ma.train(mode)
        mb.train(mode)
        a = ma.predict_scene(x1, x2, **kw)
        b = M.predict_scene_ensemble([ma, mb], x1, x2, **kw)
        assert ma.training is mode and ma._engine_obj.training is mode and mb._engine_obj.training is mode
        assert torch.equal(a.pred, one.pred) and torch.equal(a.probs, one.probs)
        assert torch.equal(b.pred, both.pred) and torch.equal(b.probs, both.probs)
    with pytest.raises(ValueError):
        M.predict_scene_ensemble([ea], x1, x2)
    with pytest.raises(ValueError):
        M.predict_scene_ensemble(ma, x1, x2)
