"""Change objects (objects.change_objects, csrc/objects.cu) on the GPU: exact equality of pred, ids, objects, confusion
and object_counts with the scipy reference of tests/objects_ref.py on random maps around the percolation thresholds,
a spiral through every block, checkerboards, degenerate shapes, batches with objects on the sample borders, K = 1, 2,
7 and 16, min_area and min_overlap; sentinel guard bands around every buffer of the entry points; determinism; the
one host synchronisation; a 4096 x 4096 map; and predict_scene -> change_objects end to end."""
import warnings

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from gan_aug_pfa_b200 import models as M  # noqa: E402
from gan_aug_pfa_b200 import ops  # noqa: E402
from gan_aug_pfa_b200.objects import change_objects  # noqa: E402
from gan_aug_pfa_b200.siamese import SiameseEngine  # noqa: E402
from objects_ref import change_objects_ref  # noqa: E402

DEV = torch.device("cuda:0")


def _random_map(shape, k, density, seed):
    g = torch.Generator().manual_seed(seed)
    kk = max(k, 2)
    on = torch.rand(shape, generator=g) < density
    cls = torch.randint(1, kk, shape, generator=g)
    return (on * cls).to(torch.uint8)


def _random_labels(shape, k, density, seed, ignore=-100):
    g = torch.Generator().manual_seed(seed)
    lab = _random_map(shape, k, density, seed + 1).long()
    lab[torch.rand(shape, generator=g) < 0.05] = ignore
    lab[torch.rand(shape, generator=g) < 0.01] = max(k, 2) + 3          # outside the classes: background, uncounted
    return lab


def _check(pred, k, labels=None, on_device=True, **kw):
    r = change_objects(pred.to(DEV) if on_device else pred, k,
                       labels=None if labels is None else labels.to(DEV), **kw)
    want = change_objects_ref(pred.numpy(), k, labels=None if labels is None else labels.numpy(), **kw)
    assert r.pred.shape == pred.shape and r.pred.dtype == torch.uint8
    assert r.ids.shape == pred.shape and r.ids.dtype == torch.int32
    assert r.objects.dtype == torch.int64 and r.objects.shape[1] == 7
    assert np.array_equal(r.ids.cpu().numpy(), want["ids"])
    assert np.array_equal(r.objects.cpu().numpy(), want["objects"])
    assert np.array_equal(r.pred.cpu().numpy(), want["pred"])
    if labels is None:
        assert r.confusion is None and r.object_counts is None
    else:
        assert np.array_equal(r.confusion.cpu().numpy(), want["confusion"])
        assert np.array_equal(r.object_counts.cpu().numpy(), want["object_counts"])
    return r


CASES = [(1, 0.45, 0, 0.0), (1, 0.6, 3, 0.5), (2, 0.1, 1, 1.0), (2, 0.45, 0, 0.5), (2, 0.6, 5, 0.0),
         (7, 0.45, 2, 1.0), (7, 0.6, 0, 0.5), (16, 0.6, 1, 0.0), (16, 0.1, 0, 1.0)]


@pytest.mark.parametrize("connectivity", [4, 8])
@pytest.mark.parametrize("k,density,min_area,min_overlap", CASES)
def test_random_maps_match_the_reference(k, density, min_area, min_overlap, connectivity):
    shape = (301, 417)                                                    # not multiples of the 32 x 32 block
    seed = int(k * 100 + density * 10 + connectivity)
    pred = _random_map(shape, k, density, seed)
    labels = _random_labels(shape, k, density, seed + 7)
    _check(pred, k, labels, min_area=min_area, connectivity=connectivity, min_overlap=min_overlap)
    _check(pred, k, min_area=min_area, connectivity=connectivity)


@pytest.mark.parametrize("connectivity", [4, 8])
def test_batches_never_join_across_the_sample_border(connectivity):
    n, h, w = 3, 70, 90
    pred = _random_map((n, h, w), 2, 0.6, 5)
    pred[:, 0, :] = 1                                                     # every sample's first and last rows full
    pred[:, -1, :] = 1
    labels = _random_labels((n, h, w), 2, 0.5, 6)
    labels[:, -1, :] = 1
    labels[:, 0, :] = 1
    r = _check(pred, 2, labels, connectivity=connectivity, min_area=2, min_overlap=0.5)
    assert set(r.objects[:, 0].tolist()) == {0, 1, 2}


def _spiral(size):
    """A one-pixel-wide square spiral with one-pixel gaps between its turns: one object through every block, whose
    union chains are as deep as they get."""
    m = np.zeros((size, size), np.uint8)
    y = x = 0
    m[0, 0] = 1
    steps = [size - 1, size - 1, size - 1]
    while steps[-1] - 2 > 0:
        steps += [steps[-1] - 2] * 2
    for i, n in enumerate(steps):
        dy, dx = ((0, 1), (1, 0), (0, -1), (-1, 0))[i % 4]
        for _ in range(n):
            y, x = y + dy, x + dx
            m[y, x] = 1
    return torch.from_numpy(m)


@pytest.mark.parametrize("connectivity", [4, 8])
def test_a_spiral_through_every_block(connectivity):
    pred = _spiral(203)
    r = _check(pred, 1, connectivity=connectivity)
    if connectivity == 4:
        assert r.objects.shape[0] == 1 and int(r.objects[0, 2]) == int(pred.sum())
    labels = pred.long().flip(1).contiguous()
    _check(pred, 1, labels, connectivity=connectivity, min_overlap=0.5)


@pytest.mark.parametrize("connectivity", [4, 8])
def test_a_checkerboard(connectivity):
    pred = (torch.arange(97)[:, None] + torch.arange(131)[None, :]) % 2
    pred = (pred * 3).to(torch.uint8)
    r = _check(pred, 4, pred.long(), connectivity=connectivity)
    assert r.objects.shape[0] == (1 if connectivity == 8 else int((pred > 0).sum()))


@pytest.mark.parametrize("shape", [(1, 1), (1, 777), (555, 1), (33, 33), (2, 1, 40), (4, 40, 1)])
@pytest.mark.parametrize("fill", ["full", "empty", "single", "random"])
def test_degenerate_shapes(shape, fill):
    if fill == "full":
        pred = torch.full(shape, 2, dtype=torch.uint8)
    elif fill == "empty":
        pred = torch.zeros(shape, dtype=torch.uint8)
    elif fill == "single":
        pred = torch.zeros(shape, dtype=torch.uint8)
        pred.view(-1)[pred.numel() // 2] = 1
    else:
        pred = _random_map(shape, 3, 0.5, 11)
    labels = _random_labels(shape, 3, 0.5, 12)
    for conn in (4, 8):
        _check(pred, 3, labels, connectivity=conn)
        _check(pred, 3, labels, connectivity=conn, min_area=2, min_overlap=1.0)


def test_host_input_and_ignore_index():
    shape = (120, 130)
    pred = _random_map(shape, 7, 0.5, 21)
    labels = _random_labels(shape, 7, 0.5, 22, ignore=255)
    _check(pred, 7, labels, on_device=False, ignore_index=255, min_area=2)


def test_out_of_range_pred_raises_after_the_count():
    pred = _random_map((50, 60), 2, 0.5, 3)
    pred[7, 9] = 2
    with pytest.raises(ValueError, match="values >= 2"):
        change_objects(pred.to(DEV), 2)
    with pytest.raises(ValueError, match="values >= 2"):
        change_objects(pred.to(DEV), 1)
    change_objects(pred.to(DEV), 3)


# ------------------------------------------------------------------------------------------------
# the entry points inside sentinel guard bands
# ------------------------------------------------------------------------------------------------
G = 64


def _guarded(numel, dtype, fill):
    buf = torch.full((numel + 2 * G,), fill, device=DEV, dtype=dtype)
    return buf, buf[G:G + numel]


@pytest.mark.parametrize("k", [1, 7])
def test_entry_points_write_nothing_outside_their_buffers(k):
    n, h, w = 2, 67, 101
    px = n * h * w
    kk = max(k, 2)
    pred = _random_map((n, h, w), k, 0.5, 31)
    labels = _random_labels((n, h, w), k, 0.5, 32)
    want = change_objects_ref(pred.numpy(), k, labels=labels.numpy(), min_area=2, min_overlap=0.5)
    bufs = {}

    def g(name, numel, dtype, fill):
        bufs[name] = _guarded(numel, dtype, fill) + (fill,)
        return bufs[name][1]

    src = g("src", px, torch.uint8, 0xAB)
    src.copy_(pred.view(-1).to(DEV))
    lsrc = g("lsrc", px, torch.int64, -7777)
    lsrc.copy_(labels.view(-1).to(DEV))
    parent, ids = g("parent", px, torch.int32, -55), g("ids", px, torch.int32, -55)
    info = g("info", 2, torch.int32, -55)
    chunk = g("chunk", -(-px // ops.OBJECTS_CHUNK), torch.int32, -55)
    out = g("out", px, torch.uint8, 0xCD)
    lparent, larea = g("lparent", px, torch.int32, -55), g("larea", px, torch.int32, -55)
    loverlap = g("loverlap", px, torch.int32, -55)
    ops.objects_label(src, n, h, w, k, 8, parent, ids, info=info)
    ops.objects_number(src, parent, ids, 2, chunk, info)
    ops.objects_label(lsrc, n, h, w, k, 8, lparent, larea, classes=out)
    count, bad = info.tolist()
    assert bad == 0 and count == len(want["objects"])
    objects = g("objects", count * 7, torch.int64, -99)
    overlap = g("overlap", count, torch.int32, -55)
    conf = g("conf", 4 if k == 1 else k * k, torch.int64, -99)
    oc = g("oc", kk * 4, torch.int64, -99)
    ops.objects_finish(src, parent, ids, n, h, w, k, count, out, objects, overlap, lparent, larea, loverlap, 0.5, conf,
                       oc)
    torch.cuda.synchronize()
    for name, (buf, _, fill) in bufs.items():
        assert bool((buf[:G] == fill).all() and (buf[-G:] == fill).all()), name
    assert np.array_equal(ids.cpu().numpy(), want["ids"].ravel())
    assert np.array_equal(out.cpu().numpy(), want["pred"].ravel())
    assert np.array_equal(objects.view(count, 7).cpu().numpy(), want["objects"])
    assert np.array_equal(conf.cpu().numpy(), want["confusion"].ravel())
    assert np.array_equal(oc.view(kk, 4).cpu().numpy(), want["object_counts"])
    assert torch.equal(src.cpu(), pred.view(-1))                          # the input is not modified


# ------------------------------------------------------------------------------------------------
# determinism, synchronisation, size
# ------------------------------------------------------------------------------------------------
def test_two_runs_are_bit_identical_and_synchronise_once():
    shape = (2, 700, 900)
    pred = _random_map(shape, 7, 0.6, 41).to(DEV)
    labels = _random_labels(shape, 7, 0.6, 42).to(DEV)
    kw = dict(labels=labels, min_area=3, min_overlap=0.5)
    a = change_objects(pred, 7, **kw)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("warn")
    try:
        with warnings.catch_warnings(record=True) as caught:
            warnings.simplefilter("always")
            b = change_objects(pred, 7, **kw)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    syncs = [c for c in caught if "synchroniz" in str(c.message)]
    assert len(syncs) == 1, [str(c.message) for c in caught]
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_a_4096_map_against_the_reference():
    shape = (4096, 4096)
    pred = _random_map(shape, 2, 0.45, 51)
    labels = _random_labels(shape, 2, 0.45, 52)
    _check(pred, 2, labels, min_area=4, min_overlap=0.5)


# ------------------------------------------------------------------------------------------------
# predict_scene -> change_objects
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 7])
def test_predict_scene_then_change_objects(k):
    h, w = 300, 420
    torch.manual_seed(0)
    sd = {kk: v.detach().clone() for kk, v in M.SiameseUNet(3, k).state_dict().items()}
    eng = SiameseEngine(DEV, 3, k)
    eng.load_state_dict(sd)
    g = torch.Generator().manual_seed(5)
    u1, u2 = (torch.randint(0, 256, (h, w, 3), generator=g, dtype=torch.uint8) for _ in range(2))
    lab = _random_labels((h, w), k, 0.3, 9).to(DEV)
    r = eng.predict_scene(u1, u2, tile=128, overlap=32, batch=4, labels=lab)
    o0 = change_objects(r.pred, k, labels=lab)
    assert torch.equal(o0.confusion, r.confusion)
    assert torch.equal(o0.pred, r.pred)
    _check(r.pred.cpu(), k, lab.cpu(), min_area=16, min_overlap=0.5)
