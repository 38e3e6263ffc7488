"""The generator's sliding-window scene inference without a GPU: the tile grid with the generator's alignment (and the
unchanged grid of predict_scene), the fp64 reference blend and uint8 rule the GPU tests use against independent loops,
the argument checks of GeneratorEngine.translate_scene and of its entry points."""
import ctypes
import math

import numpy as np
import pytest
import torch

from gan_aug_pfa_b200 import pix2pix, siamese
from gan_aug_pfa_b200.scene import _scene_grid, scene_axis
from gan_aug_pfa_b200.spec import GeneratorSpec
from translate_ref import blend_image_ref, cut_tiles, near_integer, tile_origins, u8_ref

LENGTHS = (1, 7, 128, 129, 300, 333, 1000)


def _axis_before(length, tile, overlap):
    """scene_axis as predict_scene introduced it (alignment 16)."""
    if length <= tile:
        return [0], -(-length // 16) * 16
    step = tile - overlap
    n = -(-(length - tile) // step) + 1
    return [min(i * step, length - tile) for i in range(n)], tile


@pytest.mark.parametrize("length", LENGTHS)
@pytest.mark.parametrize("tile,overlap", [(128, 0), (128, 32), (128, 64), (128, 127), (256, 0), (256, 64),
                                          (256, 200), (64, 16), (16, 0)])
def test_default_alignment_keeps_the_grid_of_predict_scene(length, tile, overlap):
    assert scene_axis(length, tile, overlap) == _axis_before(length, tile, overlap)
    assert siamese.scene_axis(length, tile, overlap) == _axis_before(length, tile, overlap)
    got = _scene_grid(length, length + 5, tile, overlap)
    assert got == siamese._scene_grid(length, length + 5, tile, overlap)
    for (ln, ext, step, n), L in zip(got, (length, length + 5)):
        origins, e = _axis_before(L, tile, overlap)
        assert (ln, ext, n) == (L, e, len(origins))
        assert step == (tile - overlap if n > 1 else e)


@pytest.mark.parametrize("align", [128, 256])
@pytest.mark.parametrize("length", LENGTHS)
@pytest.mark.parametrize("mult,overlap", [(1, 0), (1, 32), (1, 64), (2, 0), (2, 64), (2, 100)])
def test_aligned_grid_covers_every_pixel(align, length, mult, overlap):
    tile = align * mult
    origins, ext = scene_axis(length, tile, overlap, align)
    assert ext % align == 0 and ext >= align and ext <= tile
    if length <= tile:
        assert origins == [0] and ext == -(-length // align) * align and ext - length < align
    else:
        step = tile - overlap
        assert ext == tile and origins == _axis_before(length, tile, overlap)[0]
        assert len(origins) == math.ceil((length - tile) / step) + 1
        assert origins[-1] == length - tile
        assert all(0 <= o and o + ext <= length for o in origins)
    covered = np.zeros(length, dtype=bool)
    for o in origins:
        covered[o:o + ext] = True
    assert covered.all()
    (ln, e, s, n), _ = _scene_grid(length, 3, tile, overlap, align)
    assert (ln, e, n) == (length, ext, len(origins)) and s == (tile - overlap if n > 1 else ext)


def _numpy_blend(tile_vals, h, w, tile, overlap, align):
    """Independent per-pixel loop: for each pixel, every tile that covers it, in tile-index order."""
    v = tile_vals.double().numpy()
    n_t, c, ey, ex = v.shape
    oy, _ = scene_axis(h, tile, overlap, align)
    ox, _ = scene_axis(w, tile, overlap, align)
    out = np.zeros((c, h, w))
    for y in range(h):
        for x in range(w):
            num, den = np.zeros(c), 0.0
            t = 0
            for y0 in oy:
                for x0 in ox:
                    if y0 <= y < y0 + ey and x0 <= x < x0 + ex:
                        ty, tx = y - y0, x - x0
                        wt = math.exp(-(ty + 0.5 - ey / 2) ** 2 / (2 * (ey / 8) ** 2)) * \
                            math.exp(-(tx + 0.5 - ex / 2) ** 2 / (2 * (ex / 8) ** 2))
                        num += wt * v[t, :, ty, tx]
                        den += wt
                    t += 1
            out[:, y, x] = num / den
    return out


@pytest.mark.parametrize("c,h,w,tile,overlap,align", [(1, 37, 50, 32, 8, 32), (3, 40, 29, 32, 16, 32),
                                                       (4, 9, 70, 32, 0, 32), (2, 70, 45, 64, 24, 32)])
def test_reference_image_blend_matches_a_per_pixel_loop(c, h, w, tile, overlap, align):
    origins, (ey, ex) = tile_origins(h, w, tile, overlap, align)
    g = torch.Generator().manual_seed(c * 100 + h)
    v = torch.rand(len(origins), c, ey, ex, generator=g, dtype=torch.float64) * 2 - 1
    got = blend_image_ref(v, h, w, tile, overlap, align)
    want = _numpy_blend(v, h, w, tile, overlap, align)
    assert np.allclose(got.numpy(), want, rtol=0, atol=1e-13)
    assert got.min() >= -1 and got.max() <= 1                      # a convex combination of the tile values


def test_overlap_zero_stitches_the_tiles():
    h, w, tile, align = 40, 70, 32, 32
    scene = torch.rand(3, h, w, dtype=torch.float64) * 2 - 1
    got = blend_image_ref(cut_tiles(scene, tile, 0, align), h, w, tile, 0, align)
    assert torch.allclose(got, scene, rtol=0, atol=1e-15)


def test_u8_reference_is_the_truncating_rule():
    g = torch.Generator().manual_seed(3)
    v = torch.cat([torch.rand(4000, generator=g, dtype=torch.float64) * 2.2 - 1.1,
                   torch.tensor([-1.0, 1.0, 0.0, -2.0, 2.0], dtype=torch.float64),
                   torch.arange(256, dtype=torch.float64) / 255 * 2 - 1])
    want = [min(max(int(math.floor((x * 0.5 + 0.5) * 255)), 0), 255) for x in v.tolist()]
    assert u8_ref(v).tolist() == want
    assert u8_ref(torch.tensor([1.0])).item() == 255 and u8_ref(torch.tensor([-1.0])).item() == 0
    # exact integers of (v * 0.5 + 0.5) * 255 are what may round either way in fp32
    assert bool(near_integer(torch.arange(256, dtype=torch.float64) / 255 * 2 - 1).all())
    assert not bool(near_integer(torch.tensor([(10.5 / 255) * 2 - 1], dtype=torch.float64)).any())


# ------------------------------------------------------------------------------------------------
# argument checks: ValueError before any work, on an engine built on the CPU
# ------------------------------------------------------------------------------------------------
def _eng(ic=3, oc=3, num_downs=7):
    return pix2pix.GeneratorEngine(torch.device("cpu"), ic, oc, num_downs, init=False)


U8 = torch.zeros(40, 50, 3, dtype=torch.uint8)
F32 = torch.zeros(3, 40, 50)


@pytest.mark.parametrize("kw,match", [
    ({"tile": 64}, "multiple of 2"), ({"tile": 192}, "multiple of 2"), ({"tile": 0}, "multiple of 2"),
    ({"tile": -128}, "multiple of 2"), ({"tile": 128.0}, "must be an int"), ({"tile": 8192}, "at most"),
    ({"overlap": -1}, "overlap"), ({"tile": 128, "overlap": 128}, "overlap"), ({"overlap": 300}, "overlap"),
    ({"batch": 0}, "batch"), ({"batch": -2}, "batch"), ({"batch": True}, "must be an int"),
])
def test_translate_scene_rejects_bad_grid_arguments(kw, match):
    with pytest.raises(ValueError, match=match):
        _eng().translate_scene(U8, **kw)


def test_tile_must_match_the_depth_of_the_generator():
    with pytest.raises(ValueError, match="2\\^8 = 256"):
        _eng(num_downs=8).translate_scene(U8, tile=128)


@pytest.mark.parametrize("img,match", [
    (U8.to(torch.int16), "uint8"), (F32.double(), "uint8"), (U8[..., 0], "uint8"), (U8[None], "uint8"),
    (np.zeros((40, 50, 3), dtype=np.uint8), "uint8"),
    (torch.zeros(40, 50, 4, dtype=torch.uint8), "4 channels"), (F32[:2], "2 channels"),
    (torch.zeros(0, 50, 3, dtype=torch.uint8), "empty"), (torch.zeros(3, 40, 0), "empty"),
])
def test_translate_scene_rejects_bad_inputs(img, match):
    with pytest.raises(ValueError, match=match):
        _eng().translate_scene(img)


def test_channel_count_is_the_engine_input_nc():
    with pytest.raises(ValueError, match="expected input_nc = 1"):
        _eng(1, 3).translate_scene(U8)


def test_fp32_scene_must_be_on_the_engine_device():
    eng = _eng()
    eng.dev = torch.device("cuda:0")          # an engine of a CUDA device, without making it current (no GPU here)
    with pytest.raises(ValueError, match="must be on the engine's device"):
        pix2pix.GeneratorEngine.translate_scene.__wrapped__(eng, F32)


def test_a_stand_alone_block_engine_has_no_image_output():
    chain = [(512, 512, 512, False, False), (512, 512, 512, False, True)]
    eng = pix2pix.GeneratorEngine(torch.device("cpu"), init=False, spec=GeneratorSpec.for_block_chain(chain))
    assert eng.virtual0
    with pytest.raises(ValueError, match="stand-alone"):
        eng.translate_scene(torch.zeros(512, 40, 50))


def test_scene_image_entry_points_check_their_arguments_without_a_gpu(lib_path):
    from gan_aug_pfa_b200 import _lib
    h = _lib.lib()
    fake = ctypes.c_void_p(16)
    # a consistent grid: 300 x 420 at tile 128, overlap 32 -> y (300, 128, 96, 3), x (420, 128, 96, 5)
    ok = (300, 420, 128, 128, 96, 96, 3, 5)
    g1 = h.gap_scene_gather_one
    for c in (0, 5):
        assert g1(fake, 1, c, *ok, 0, 4, fake, None) == -1
        assert b"c must be 1..4" in h.gap_last_error_string()
    assert g1(None, 1, 3, *ok, 0, 4, fake, None) == -1
    assert b"gap_scene_gather_one: bad arguments" in h.gap_last_error_string()
    assert g1(fake, 1, 3, *ok, 0, 4, None, None) == -1
    assert g1(fake, 1, 3, *ok, 15, 4, fake, None) == -1                 # tile0 past the grid
    assert g1(fake, 1, 3, *ok, 0, 0, fake, None) == -1                  # batch 0
    assert g1(fake, 1, 3, 300, 420, 128, 128, 96, 96, 2, 5, 0, 4, fake, None) == -1     # too few tiles
    assert g1(fake, 1, 3, 300, 420, 120, 128, 96, 96, 3, 5, 0, 4, fake, None) == -1     # extent not a multiple of 16
    assert b"gap_scene_gather_one: bad arguments" in h.gap_last_error_string()
    assert g1(fake, 1, 3, *ok, 0, 4, ctypes.c_void_p(20), None) == -1   # not 8-byte aligned
    assert b"8-byte aligned" in h.gap_last_error_string()
    bi = h.gap_scene_blend_image
    for c in (0, 5):
        assert bi(fake, c, *ok, 0, 4, fake, fake, None) == -1
        assert b"c must be 1..4" in h.gap_last_error_string()
    for args in ((None, 3, *ok, 0, 4, fake, fake), (fake, 3, *ok, 0, 4, None, fake), (fake, 3, *ok, 0, 4, fake, None),
                 (fake, 3, *ok, -1, 4, fake, fake), (fake, 3, *ok, 0, 0, fake, fake),
                 (fake, 3, 100, 420, 128, 128, 128, 96, 2, 5, 0, 4, fake, fake),      # one tile fits the y axis
                 (fake, 3, 300, 420, 128, 128, 96, 96, 3, 6, 0, 4, fake, fake)):      # one tile too many in x
        assert bi(*args, None) == -1
        assert b"gap_scene_blend_image: bad arguments" in h.gap_last_error_string()
    assert bi(ctypes.c_void_p(24), 3, *ok, 0, 4, fake, fake, None) == -1
    assert b"16-byte aligned" in h.gap_last_error_string()
    big = (20000, 20000, 8192, 8192, 8192, 8192, 3, 3)
    assert bi(fake, 3, *big, 0, 4, fake, fake, None) == -1
    assert b"exceeds" in h.gap_last_error_string()
    fi = h.gap_scene_finalize_image
    for c in (0, 5):
        assert fi(fake, fake, c, 64, fake, 0, None) == -1
        assert b"c must be 1..4" in h.gap_last_error_string()
    for args in ((None, fake, 3, 64, fake, 0), (fake, None, 3, 64, fake, 0), (fake, fake, 3, 64, None, 1),
                 (fake, fake, 3, 0, fake, 0)):
        assert fi(*args, None) == -1
        assert b"gap_scene_finalize_image: bad arguments" in h.gap_last_error_string()


def test_gather_one_launcher_checks_before_any_cuda_call():
    from gan_aug_pfa_b200 import ops
    grid = _scene_grid(40, 50, 128, 32, 128)
    out = torch.zeros(2, 128, 128, 4, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="1 to 4 channels"):
        ops.scene_gather_one(torch.zeros(40, 50, 5, dtype=torch.uint8), grid, 0, out)
    with pytest.raises(ValueError, match="out must be"):
        ops.scene_gather_one(U8, grid, 0, out[..., :3])
    with pytest.raises(ValueError, match="tile0"):
        ops.scene_gather_one(U8, grid, 1, out)
    with pytest.raises(ValueError, match="CUDA"):
        ops.scene_gather_one(U8, grid, 0, out)
    acc, ws = torch.zeros(3, 40, 50), torch.zeros(40, 50)
    with pytest.raises(ValueError, match="fake must be"):
        ops.scene_blend_image(torch.zeros(2, 128, 128, 3), grid, 0, acc, ws)
    with pytest.raises(ValueError, match="acc must be"):
        ops.scene_blend_image(torch.zeros(2, 128, 128, 4), grid, 0, torch.zeros(5, 40, 50), ws)
    with pytest.raises(ValueError, match="image must be"):
        ops.scene_finalize_image(acc, ws, torch.zeros(40, 50, 2, dtype=torch.uint8), False)
    with pytest.raises(ValueError, match="CUDA"):
        ops.scene_finalize_image(acc, ws, torch.zeros(40, 50, 3, dtype=torch.uint8), False)
