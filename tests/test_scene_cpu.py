"""Sliding-window scene inference without a GPU: the tile grid and the blending window that csrc/scene.cu must follow,
the fp64 reference blend the GPU tests use against an independent per-pixel loop, and the argument checks of
SiameseEngine.predict_scene and of the scene entry points."""
import ctypes
import math

import numpy as np
import pytest
import torch

from gan_aug_pfa_b200 import siamese
from gan_aug_pfa_b200.siamese import scene_axis, scene_window
from scene_ref import blend_ref, cut_tiles, tile_origins


@pytest.mark.parametrize("length,tile,overlap", [
    (7, 64, 16),            # shorter than 16
    (1, 16, 0),
    (100, 256, 64),         # shorter than the tile, not a multiple of 16
    (256, 256, 64),         # exactly one tile
    (257, 256, 64),         # one pixel more: the second tile is snapped to the edge
    (192 * 5, 256, 64),     # a multiple of the step
    (192 * 5 + 64, 256, 64),
    (1000, 128, 0),         # plain stitching
    (300, 64, 48),          # overlap = tile - 16
    (8192, 512, 64),
])
def test_tile_grid_covers_every_pixel_inside_the_scene(length, tile, overlap):
    origins, ext = scene_axis(length, tile, overlap)
    assert ext % 16 == 0 and ext >= 16
    if length <= tile:
        assert origins == [0] and ext == -(-length // 16) * 16 and ext - length < 16
    else:
        step = tile - overlap
        assert ext == tile
        assert len(origins) == math.ceil((length - tile) / step) + 1
        assert origins[-1] == length - tile                               # snapped to the edge
        assert all(0 <= o and o + ext <= length for o in origins)         # no tile reads outside the scene
        assert origins == sorted(origins)
        assert all(b - a <= step for a, b in zip(origins, origins[1:]))
        assert all(o == i * step for i, o in enumerate(origins[:-1]))
    covered = np.zeros(length, dtype=bool)
    for o in origins:
        covered[o:o + ext] = True
    assert covered.all()


def test_window_matches_its_formula():
    for e in (16, 48, 128, 512):
        g = scene_window(e)
        sigma = e / 8
        want = [math.exp(-(t + 0.5 - e / 2) ** 2 / (2 * sigma ** 2)) for t in range(e)]
        assert g.dtype == torch.float64 and g.shape == (e,)
        assert np.allclose(g.numpy(), want, rtol=1e-15, atol=0)
        assert torch.equal(g, g.flip(0))                         # symmetric about the tile centre
        assert g.min() == pytest.approx(math.exp(-(e / 2 - 0.5) ** 2 / (2 * sigma ** 2)))
        assert float(g.min() ** 2) > math.exp(-17)               # every covered pixel has a positive weight


def _numpy_blend(tile_logits, h, w, tile, overlap):
    """Independent per-pixel loop: for each pixel, every tile that covers it, in tile-index order."""
    z = tile_logits.double().numpy()
    n_t, k, ey, ex = z.shape
    oy, _ = scene_axis(h, tile, overlap)
    ox, _ = scene_axis(w, tile, overlap)
    sy, sx = ey / 8, ex / 8
    out = np.zeros((k, h, w))
    for y in range(h):
        for x in range(w):
            num, den = np.zeros(k), 0.0
            t = 0
            for y0 in oy:
                for x0 in ox:
                    if y0 <= y < y0 + ey and x0 <= x < x0 + ex:
                        ty, tx = y - y0, x - x0
                        wt = math.exp(-(ty + 0.5 - ey / 2) ** 2 / (2 * sy * sy)) * \
                            math.exp(-(tx + 0.5 - ex / 2) ** 2 / (2 * sx * sx))
                        v = z[t, :, ty, tx]
                        if k == 1:
                            p = 1 / (1 + np.exp(-v))
                        else:
                            e = np.exp(v - v.max())
                            p = e / e.sum()
                        num += wt * p
                        den += wt
                    t += 1
            out[:, y, x] = num / den
    return out


@pytest.mark.parametrize("k,h,w,tile,overlap", [(1, 37, 50, 16, 8), (3, 40, 29, 32, 16), (2, 9, 70, 32, 0),
                                                 (7, 33, 33, 16, 0)])
def test_reference_blend_matches_a_per_pixel_loop(k, h, w, tile, overlap):
    origins, (ey, ex) = tile_origins(h, w, tile, overlap)
    g = torch.Generator().manual_seed(k * 100 + h)
    z = torch.randn(len(origins), k, ey, ex, generator=g, dtype=torch.float64) * 4
    got = blend_ref(z, h, w, tile, overlap)
    want = _numpy_blend(z, h, w, tile, overlap)
    assert np.allclose(got.numpy(), want, rtol=0, atol=1e-13)
    if k > 1:
        assert torch.allclose(got.sum(0), torch.ones(h, w, dtype=torch.float64))


def test_overlap_zero_is_plain_stitching():
    h, w, tile = 40, 70, 32
    scene = torch.randn(3, h, w, dtype=torch.float64)
    tiles = cut_tiles(scene, tile, 0)
    assert tiles.shape == (len(tile_origins(h, w, tile, 0)[0]), 3, 32, 32)
    p = blend_ref(tiles, h, w, tile, 0)
    assert torch.allclose(p, torch.softmax(scene, 0), rtol=0, atol=1e-15)


def test_cut_tiles_replicates_the_edge():
    scene = torch.arange(3 * 7 * 20, dtype=torch.float32).view(3, 7, 20)
    t = cut_tiles(scene, 16, 4)               # y: one 16-row tile over 7 rows; x: origins 0, 4
    assert t.shape == (2, 3, 16, 16)
    assert torch.equal(t[0, :, :7], scene[:, :, :16])
    assert torch.equal(t[0, :, 7:], scene[:, 6:7, :16].expand(3, 9, 16))
    assert torch.equal(t[1, :, :7], scene[:, :, 4:20])


# ------------------------------------------------------------------------------------------------
# argument checks: ValueError before any work, on an engine built on the CPU
# ------------------------------------------------------------------------------------------------
def _eng(c=3, k=2):
    return siamese.SiameseEngine(torch.device("cpu"), c, k)


U8 = torch.zeros(40, 50, 3, dtype=torch.uint8)
F32 = torch.zeros(3, 40, 50)


@pytest.mark.parametrize("kw,match", [
    ({"tile": 8}, "multiple of 16"), ({"tile": 24}, "multiple of 16"), ({"tile": 0}, "multiple of 16"),
    ({"tile": 64.0}, "must be an int"), ({"overlap": -1}, "overlap"), ({"tile": 64, "overlap": 64}, "overlap"),
    ({"batch": 0}, "batch"), ({"batch": True}, "must be an int"),
])
def test_predict_scene_rejects_bad_grid_arguments(kw, match):
    with pytest.raises(ValueError, match=match):
        _eng().predict_scene(U8, U8, **kw)


@pytest.mark.parametrize("a,b,match", [
    (U8.to(torch.int16), U8.to(torch.int16), "uint8"),
    (F32.double(), F32.double(), "uint8"),
    (U8[..., 0], U8[..., 0], "uint8"),
    (U8[None], U8[None], "uint8"),
    (torch.zeros(40, 50, 4, dtype=torch.uint8), torch.zeros(40, 50, 4, dtype=torch.uint8), "4 channels"),
    (F32[:2], F32[:2], "2 channels"),
    (U8, U8[:39], "same dtype and shape"),
    (U8, F32, "same dtype and shape"),
    (torch.zeros(0, 50, 3, dtype=torch.uint8), torch.zeros(0, 50, 3, dtype=torch.uint8), "empty"),
])
def test_predict_scene_rejects_bad_inputs(a, b, match):
    with pytest.raises(ValueError, match=match):
        _eng().predict_scene(a, b)


@pytest.mark.parametrize("labels", [torch.zeros(40, 50, dtype=torch.int32), torch.zeros(40, 49, dtype=torch.int64),
                                    torch.zeros(1, 40, 50, dtype=torch.int64), [[0]]])
def test_predict_scene_rejects_bad_labels(labels):
    with pytest.raises(ValueError, match="labels must be an int64"):
        _eng(3, 1).predict_scene(U8, U8, labels=labels)


def test_fp32_scene_must_be_on_the_engine_device():
    eng = _eng()
    eng.dev = torch.device("cuda:0")          # an engine of a CUDA device, without making it current (no GPU here)
    with pytest.raises(ValueError, match="must be on the engine's device"):
        siamese.SiameseEngine.predict_scene.__wrapped__(eng, F32, F32)


def test_scene_entry_points_check_their_arguments_without_a_gpu(lib_path):
    from gan_aug_pfa_b200 import _lib
    h = _lib.lib()
    fake = ctypes.c_void_p(16)
    # a consistent grid: 300 x 420 at tile 128, overlap 32 -> y (300, 128, 96, 3), x (420, 128, 96, 5)
    ok = (300, 420, 128, 128, 96, 96, 3, 5)
    assert h.gap_scene_gather(fake, fake, 1, 5, *ok, 0, 4, fake, fake, None) == -1          # 5 channels
    assert h.gap_scene_gather(None, fake, 1, 3, *ok, 0, 4, fake, fake, None) == -1
    assert h.gap_scene_gather(fake, fake, 1, 3, *ok, 15, 4, fake, fake, None) == -1         # tile0 past the grid
    assert h.gap_scene_gather(fake, fake, 1, 3, 300, 420, 128, 128, 96, 96, 2, 5, 0, 4, fake, fake, None) == -1
    assert h.gap_scene_gather(fake, fake, 1, 3, 300, 420, 120, 128, 96, 96, 3, 5, 0, 4, fake, fake, None) == -1
    assert b"gap_scene_gather: bad arguments" in h.gap_last_error_string()
    assert h.gap_scene_gather(fake, fake, 1, 3, *ok, 0, 4, ctypes.c_void_p(18), fake, None) == -1   # not 8-byte aligned
    assert b"8-byte aligned" in h.gap_last_error_string()
    assert h.gap_scene_blend(fake, 0, *ok, 0, 4, fake, fake, None) == -1
    assert h.gap_scene_blend(fake, 17, *ok, 0, 4, fake, fake, None) == -1
    assert h.gap_scene_blend(fake, 2, *ok, 0, 0, fake, fake, None) == -1
    assert h.gap_scene_blend(fake, 2, 100, 420, 128, 128, 128, 96, 2, 5, 0, 4, fake, fake, None) == -1   # one tile fits
    assert h.gap_scene_finalize(fake, fake, 2, 0, fake, 0, None, -100, None, None) == -1
    assert h.gap_scene_finalize(fake, fake, 2, 64, fake, 0, fake, -100, None, None) == -1   # labels without counts
    assert b"gap_scene_finalize: bad arguments" in h.gap_last_error_string()
