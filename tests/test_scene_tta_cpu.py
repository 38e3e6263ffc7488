"""Test-time augmentation and checkpoint ensembles over whole scenes, without a GPU: the dihedral tile transforms,
the fp64 multi-pass reference blend the GPU tests use against an independent per-pixel loop, the D4 equivariance of
the "d4" average on a symmetric grid, and the argument checks of predict_scene_ensemble and of the new entry points."""
import ctypes
import itertools

import pytest
import torch

from gan_aug_pfa_b200 import siamese
from gan_aug_pfa_b200.siamese import scene_window
from scene_ref import cut_tiles, tile_origins
from tta_ref import blend_passes_ref, f, f_inv, passes


@pytest.mark.parametrize("d", range(8))
@pytest.mark.parametrize("shape", [(3, 16, 16), (2, 16, 48), (1, 48, 32)])
def test_inverse_undoes_each_transform(d, shape):
    x = torch.arange(torch.Size(shape).numel(), dtype=torch.float64).view(shape)
    y = f(x, d)
    assert y.shape[-2:] == ((shape[2], shape[1]) if d & 4 else shape[1:])
    assert torch.equal(f_inv(y, d), x)


def test_the_eight_transforms_are_distinct_and_closed_under_composition():
    x = torch.arange(64, dtype=torch.float64).view(8, 8)
    imgs = [f(x, d) for d in range(8)]
    assert all(not torch.equal(a, b) for a, b in itertools.combinations(imgs, 2))
    for a, b in itertools.product(range(8), repeat=2):
        y = f(f(x, a), b)
        assert sum(torch.equal(y, im) for im in imgs) == 1
    # the rotations by 90 and 270 degrees are the transposed members with one flip
    rot = {tuple(torch.rot90(x, k, (0, 1)).flatten().tolist()) for k in (1, 3)}
    assert rot == {tuple(f(x, 5).flatten().tolist()), tuple(f(x, 6).flatten().tolist())}
    # "flips" never transposes: it never changes a tile's shape
    assert all(d < 4 for d in siamese.TTA_TRANSFORMS["flips"])


def test_passes_run_member_by_member_in_ascending_d():
    assert passes(2, "flips") == [(0, 0), (0, 1), (0, 2), (0, 3), (1, 0), (1, 1), (1, 2), (1, 3)]
    assert passes(1, None) == [(0, 0)]
    assert [d for _, d in passes(1, "d4")] == list(range(8))


@pytest.mark.parametrize("k", [1, 3])
@pytest.mark.parametrize("h,w,tile,overlap", [(37, 53, 16, 4), (12, 41, 16, 6)])
def test_multi_pass_reference_matches_a_per_pixel_loop(k, h, w, tile, overlap):
    origins, (ey, ex) = tile_origins(h, w, tile, overlap)
    g = torch.Generator().manual_seed(k + h)
    per_pass = []
    for d in (0, 3, 4, 6, 1):                               # any order of transforms, repeats allowed
        oy, ox = (ex, ey) if d & 4 else (ey, ex)
        per_pass.append((d, torch.randn(len(origins), k, oy, ox, generator=g, dtype=torch.float64) * 2))
    got = blend_passes_ref(per_pass, h, w, tile, overlap)
    gy, gx = scene_window(ey), scene_window(ex)
    want = torch.zeros(k, h, w, dtype=torch.float64)
    for y in range(h):
        for x in range(w):
            acc = torch.zeros(k, dtype=torch.float64)
            ws = 0.0
            for d, z in per_pass:
                for t, (y0, x0) in enumerate(origins):
                    if not (y0 <= y < y0 + ey and x0 <= x < x0 + ex):
                        continue
                    ty, tx = y - y0, x - x0
                    # position of (ty, tx) in f_d(tile)
                    i, j = (tx, ty) if d & 4 else (ty, tx)
                    oy, ox = z.shape[-2:]
                    if d & 2:
                        i = oy - 1 - i
                    if d & 1:
                        j = ox - 1 - j
                    v = z[t, :, i, j]
                    p = torch.sigmoid(v) if k == 1 else torch.softmax(v, 0)
                    wt = float(gy[ty] * gx[tx])
                    acc += wt * p
                    ws += wt
            want[:, y, x] = acc / ws
    assert float((got - want).abs().max()) < 1e-12


def _toy_net(crops):
    """A position-dependent stand-in for the network: [n, C, a, b] -> [n, 2, a, b] logits that mix the pixel values with
    the row and column index, so that a single pass is not equivariant."""
    n, _, a, b = crops.shape
    r = torch.arange(a, dtype=torch.float64)[:, None] / a
    c = torch.arange(b, dtype=torch.float64)[None, :] / b
    z0 = crops[:, 0] * 1.5 - crops[:, 1] + 2.0 * r - 0.7 * c * c
    z1 = crops[:, 1] * crops[:, 0] + 1.3 * r * c - 0.4 * r
    return torch.stack([z0, z1], 1)


def _toy_scene_probs(scene, tile, overlap, tta):
    _, h, w = scene.shape
    tiles = cut_tiles(scene, tile, overlap)
    per_pass = [(d, _toy_net(f(tiles, d))) for _, d in passes(1, tta)]
    return blend_passes_ref(per_pass, h, w, tile, overlap)


@pytest.mark.parametrize("tta,h,w", [("d4", 64 + 2 * 48, 64 + 2 * 48), ("flips", 64 + 2 * 48, 64 + 3 * 48)])
def test_the_tta_average_is_equivariant_on_a_symmetric_grid(tta, h, w):
    tile, overlap = 64, 16                                  # L = tile + k (tile - overlap) on both axes
    scene = torch.rand(2, h, w, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    out = _toy_scene_probs(scene, tile, overlap, tta)
    for g in siamese.TTA_TRANSFORMS[tta]:
        got = _toy_scene_probs(f(scene, g), tile, overlap, tta)
        assert float((got - f(out, g)).abs().max()) < 1e-12, g
    # without the average the toy network is not equivariant (the check above has teeth)
    plain = _toy_scene_probs(scene, tile, overlap, None)
    assert float((_toy_scene_probs(f(scene, 1), tile, overlap, None) - f(plain, 1)).abs().max()) > 1e-3


def _eng(k=1, c=3):
    return siamese.SiameseEngine(torch.device("cpu"), c, k)


U8 = torch.zeros(40, 50, 3, dtype=torch.uint8)


@pytest.mark.parametrize("engines,kw,match", [
    ([], {}, "non-empty list"),
    ("one", {}, "non-empty list"),
    (["x"], {}, "SiameseEngine"),
    (None, {"tta": "rot90"}, "tta must be"),
    (None, {"tta": ["flips"]}, "tta must be"),
    (None, {"tile": 24}, "multiple of 16"),
    (None, {"tile": 64, "overlap": 64}, "overlap"),
    (None, {"batch": 0}, "batch"),
])
def test_ensemble_arguments_are_checked_before_any_work(engines, kw, match):
    eng = _eng()
    if engines is None:
        engines = [eng]
    with pytest.raises(ValueError, match=match):
        siamese.predict_scene_ensemble(engines, U8, U8, **kw)
    assert eng._n is None and eng.training


def test_ensemble_members_must_match():
    a = _eng(1)
    for b in (_eng(2), _eng(1, c=2)):
        with pytest.raises(ValueError, match="ensemble members must share"):
            siamese.predict_scene_ensemble([a, b], U8, U8)
    with pytest.raises(ValueError, match="engines must be"):
        siamese.predict_scene_ensemble(a, U8, U8)
    with pytest.raises(ValueError, match="tta must be"):
        siamese.SiameseEngine.predict_scene.__wrapped__(a, U8, U8, tta="d8")


def test_tta_entry_points_check_their_arguments_without_a_gpu(lib_path):
    from gan_aug_pfa_b200 import _lib
    h = _lib.lib()
    fake = ctypes.c_void_p(16)
    ok = (300, 420, 128, 128, 96, 96, 3, 5)
    for d in (-1, 8):
        assert h.gap_scene_gather_tta(fake, fake, 1, 3, *ok, 0, 4, d, fake, fake, None) == -1
        assert b"d must be 0..7" in h.gap_last_error_string()
        assert h.gap_scene_blend_tta(fake, 2, *ok, 0, 4, d, 1, fake, fake, None) == -1
        assert b"d must be 0..7" in h.gap_last_error_string()
    assert h.gap_scene_gather_tta(fake, fake, 1, 5, *ok, 0, 4, 4, fake, fake, None) == -1          # 5 channels
    assert h.gap_scene_blend_tta(fake, 17, *ok, 0, 4, 4, 0, fake, fake, None) == -1                # 17 classes
    assert h.gap_scene_blend_tta(None, 2, *ok, 0, 4, 4, 0, fake, fake, None) == -1


def test_ops_reject_a_bad_transform_or_a_wrong_extent():
    from gan_aug_pfa_b200 import ops
    grid = ((40, 48, 48, 1), (100, 64, 48, 2))            # ey = 48, ex = 64
    img = torch.zeros(40, 100, 3, dtype=torch.uint8)
    o = torch.zeros(2, 48, 64, 4, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="d must be"):
        ops.scene_gather(img, img, grid, 0, o, o, d=8)
    with pytest.raises(ValueError, match=r"\[batch, 64, 48, 4\]"):
        ops.scene_gather(img, img, grid, 0, o, o, d=4)
    lg = torch.zeros(2, 2, 48, 64)
    acc, ws = torch.zeros(2, 40, 100), torch.zeros(40, 100)
    with pytest.raises(ValueError, match=r"\(K,\) 64, 48"):
        ops.scene_blend(lg, grid, 0, acc, ws, d=5, first_pass=False)
    with pytest.raises(ValueError, match="d must be"):
        ops.scene_blend(lg, grid, 0, acc, ws, d=True)
