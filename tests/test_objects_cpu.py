"""Change objects without a GPU: the scipy reference of tests/objects_ref.py on hand-made maps, the argument checks of
objects.change_objects (raised before any work is enqueued) and of the gap_objects_* entry points, and the formulas
of metrics.object_metrics."""
import ctypes

import numpy as np
import pytest
import torch

from gan_aug_pfa_b200 import metrics, objects, ops
from objects_ref import change_objects_ref, components


def test_reference_numbers_objects_by_first_pixel_across_classes():
    pred = np.array([[0, 2, 2, 0, 1],
                     [1, 0, 0, 0, 1],
                     [1, 1, 0, 2, 0],
                     [0, 0, 2, 0, 0]], np.uint8)
    r8 = change_objects_ref(pred, 3, connectivity=8)
    assert r8["ids"].tolist() == [[0, 1, 1, 0, 2],
                                  [3, 0, 0, 0, 2],
                                  [3, 3, 0, 4, 0],
                                  [0, 0, 4, 0, 0]]
    assert r8["objects"].tolist() == [[0, 2, 2, 0, 1, 0, 2],
                                      [0, 1, 2, 0, 4, 1, 4],
                                      [0, 1, 3, 1, 0, 2, 1],
                                      [0, 2, 2, 2, 2, 3, 3]]
    r4 = change_objects_ref(pred, 3, connectivity=4)       # the diagonal pair of class 2 splits
    assert r4["ids"][2, 3] == 4 and r4["ids"][3, 2] == 5 and len(r4["objects"]) == 5
    assert (r4["pred"] == pred).all() and r4["confusion"] is None


def test_reference_checkerboard_and_samples():
    cb = (np.indices((6, 7)).sum(0) % 2).astype(np.uint8)
    assert len(change_objects_ref(cb, 2, connectivity=8)["objects"]) == 1
    assert len(change_objects_ref(cb, 2, connectivity=4)["objects"]) == int(cb.sum())
    two = np.ones((2, 3, 3), np.uint8)                      # components never cross the sample border
    r = change_objects_ref(two, 2)
    assert r["objects"].tolist() == [[0, 1, 9, 0, 0, 2, 2], [1, 1, 9, 0, 0, 2, 2]]
    assert components(two.astype(np.int64), 2, 8)[1].min() == 2


def test_reference_min_area_confusion_and_counts():
    pred = np.array([[1, 1, 0, 0, 2],
                     [1, 1, 0, 0, 0],
                     [0, 0, 0, 2, 2],
                     [1, 0, 0, 2, 2]], np.uint8)
    lab = np.array([[1, 1, 0, -100, 2],
                    [1, 0, 0, 0, 0],
                    [0, 0, 0, 0, 0],
                    [0, 0, 0, 2, 2]], np.int64)
    r = change_objects_ref(pred, 3, labels=lab, min_area=2, min_overlap=0.5)
    assert r["pred"].tolist() == [[1, 1, 0, 0, 0],
                                  [1, 1, 0, 0, 0],
                                  [0, 0, 0, 2, 2],
                                  [0, 0, 0, 2, 2]]
    assert r["objects"].tolist() == [[0, 1, 4, 0, 0, 1, 1], [0, 2, 4, 2, 3, 3, 4]]
    want = np.zeros((3, 3), np.int64)
    for y, p in zip(lab.ravel(), r["pred"].ravel()):
        if y != -100:
            want[y, p] += 1
    assert (r["confusion"] == want).all()
    # reference: class 1 one object (3 px, all predicted 1: detected); class 2 the corner pixel (predicted 0 after
    # filtering: missed) and the bottom pair (detected).  predicted: class 1 (4 px, 3 labelled 1 >= 2: matched),
    # class 2 (4 px, 2 labelled 2 >= 2: matched)
    assert r["object_counts"].tolist() == [[0, 0, 0, 0], [1, 1, 1, 1], [2, 1, 1, 1]]
    strict = change_objects_ref(pred, 3, labels=lab, min_area=2, min_overlap=1.0)
    assert strict["object_counts"].tolist() == [[0, 0, 0, 0], [1, 1, 1, 0], [2, 1, 1, 0]]


def test_reference_single_logit_map():
    pred = np.array([[1, 0, 1], [1, 0, 0]], np.uint8)
    lab = np.array([[1, 1, 0], [0, 0, 2]], np.int64)        # 2 is outside {0, 1}: not counted, background
    r = change_objects_ref(pred, 1, labels=lab)
    assert r["confusion"].tolist() == [1, 2, 1, 1]          # TP, FP, FN, TN
    assert r["object_counts"].tolist() == [[0, 0, 0, 0], [1, 1, 2, 1]]


# ------------------------------------------------------------------------------------------------
# argument checks: ValueError before any launch
# ------------------------------------------------------------------------------------------------
@pytest.fixture
def no_launch(monkeypatch):
    def boom(*a, **k):
        raise AssertionError("work was enqueued")
    for name in ("objects_label", "objects_number", "objects_finish"):
        monkeypatch.setattr(ops, name, boom)


GOOD = torch.zeros(5, 6, dtype=torch.uint8)


@pytest.mark.parametrize("kwargs", [
    dict(pred=GOOD.float()),
    dict(pred=GOOD[None, None]),
    dict(pred=torch.zeros(5, dtype=torch.uint8)),
    dict(pred=torch.zeros(0, 6, dtype=torch.uint8)),
    dict(pred=GOOD.numpy()),
    dict(n_classes=0),
    dict(n_classes=17),
    dict(n_classes=2.0),
    dict(n_classes=True),
    dict(labels=torch.zeros(5, 6, dtype=torch.int32)),
    dict(labels=torch.zeros(5, 7, dtype=torch.int64)),
    dict(labels=torch.zeros(1, 5, 6, dtype=torch.int64)),
    dict(connectivity=6),
    dict(connectivity=0),
    dict(min_area=-1),
    dict(min_area=1.5),
    dict(min_overlap=-0.1),
    dict(min_overlap=1.01),
    dict(min_overlap=float("nan")),
    dict(ignore_index=0.5),
    dict(pred=torch.zeros(1, dtype=torch.uint8).expand(2, 2 ** 15, 2 ** 15)),     # 2^31 pixels
])
def test_bad_arguments_raise_before_any_work(no_launch, kwargs):
    args = dict(pred=GOOD, n_classes=2)
    args.update(kwargs)
    with pytest.raises(ValueError):
        objects.change_objects(args.pop("pred"), args.pop("n_classes"), **args)


def test_entry_points_reject_bad_arguments_without_a_gpu(lib_path):
    from gan_aug_pfa_b200 import _lib
    h = _lib.lib()
    p = ctypes.c_void_p(16)
    assert h.gap_objects_label(p, 0, 1, 4, 4, 17, -100, 8, None, p, p, p, None) != 0
    assert b"k must be" in h.gap_last_error_string()
    assert h.gap_objects_label(p, 0, 1, 4, 4, 2, -100, 6, None, p, p, p, None) != 0
    assert b"connectivity" in h.gap_last_error_string()
    assert h.gap_objects_label(p, 0, 2, 2 ** 15, 2 ** 15, 2, -100, 8, None, p, p, p, None) != 0
    assert h.gap_objects_label(p, 1, 1, 4, 4, 2, -100, 8, None, p, p, p, None) != 0       # labels need classes
    assert h.gap_objects_number(p, p, p, 16, -1, p, p, None) != 0
    assert h.gap_objects_finish(p, p, p, 1, 4, 4, 2, 3, p, None, p, p, None, p, 0.5, p, p, None) != 0
    assert b"go together" in h.gap_last_error_string()
    assert h.gap_objects_finish(p, p, p, 1, 4, 4, 2, 3, p, p, p, p, p, p, 1.5, p, p, None) != 0
    assert b"min_overlap" in h.gap_last_error_string()


def test_object_metrics_formulas():
    counts = torch.tensor([[0, 0, 0, 0], [4, 3, 5, 2], [0, 0, 2, 0], [3, 1, 0, 0]])
    m = metrics.object_metrics(counts)
    s = 1e-6
    f = np.float32
    for i, (ref, det, prd, mat) in enumerate(counts[1:].tolist()):
        p = (f(mat) + f(s)) / (f(prd) + f(s))
        r = (f(det) + f(s)) / (f(ref) + f(s))
        f1 = (f(2) * p * r + f(s)) / (p + r + f(s))
        assert m["precision"][i] == pytest.approx(float(p), rel=1e-6)
        assert m["recall"][i] == pytest.approx(float(r), rel=1e-6)
        assert m["f1"][i] == pytest.approx(float(f1), rel=1e-6)
    assert len(m["precision"]) == 3
    assert m["precision"][0] == pytest.approx(0.4) and m["recall"][0] == pytest.approx(0.75)
    assert m["precision"][2] == pytest.approx(1.0) and m["recall"][2] == pytest.approx(1 / 3)
    one = metrics.object_metrics(np.array([[0, 0, 0, 0], [2, 1, 4, 4]]))    # K = 1: one change class
    assert one["precision"] == [pytest.approx(1.0)] and one["recall"] == [pytest.approx(0.5)]
