"""Multi-class Siamese U-Net without a GPU: seeded weights of SiameseUNet(3, K) against a torch restatement of the
reference's construction order, the class-count rejections, the loss-kind pairings, the checkpoint class-count
check, and the argument checks of the multi-class head entry points."""
import ctypes
import hashlib
from types import SimpleNamespace

import pytest
import torch
import torch.nn as nn

from gan_aug_pfa_b200 import models as M
from gan_aug_pfa_b200 import checkpoint, ops, siamese, spec


def _digest(sd):
    return [(k, tuple(v.shape), str(v.dtype), hashlib.sha256(v.detach().contiguous().numpy().tobytes()).hexdigest())
            for k, v in sd.items()]


def _dc(cin, cout):
    return nn.Sequential(nn.Conv2d(cin, cout, 3, padding=1, bias=False), nn.BatchNorm2d(cout), nn.ReLU(inplace=True),
                         nn.Conv2d(cout, cout, 3, padding=1, bias=False), nn.BatchNorm2d(cout), nn.ReLU(inplace=True))


class _Gate(nn.Module):
    def __init__(self, fg, fl, fi):
        super().__init__()
        self.W_g = nn.Sequential(nn.Conv2d(fg, fi, 1, bias=True), nn.BatchNorm2d(fi))
        self.W_x = nn.Sequential(nn.Conv2d(fl, fi, 1, bias=True), nn.BatchNorm2d(fi))
        self.psi = nn.Sequential(nn.Conv2d(fi, 1, 1, bias=True), nn.BatchNorm2d(1), nn.Sigmoid())


class _TorchSiamese(nn.Module):
    """SiameseUNet.__init__ (models.py:47-90) restated with plain torch layers: construction order = RNG order."""

    def __init__(self, n_channels, n_classes):
        super().__init__()
        self.dconv_down1, self.dconv_down2 = _dc(n_channels, 64), _dc(64, 128)
        self.dconv_down3, self.dconv_down4 = _dc(128, 256), _dc(256, 512)
        self.bottleneck = _dc(512, 1024)
        self.att3, self.att2 = _Gate(2048, 1024, 512), _Gate(512, 512, 256)
        self.att1, self.att_last = _Gate(256, 256, 128), _Gate(128, 128, 64)
        self.dconv_up3, self.dconv_up2 = _dc(2048 + 1024, 512), _dc(512 + 512, 256)
        self.dconv_up1, self.dconv_last = _dc(256 + 256, 128), _dc(128 + 128, 64)
        self.conv_last = nn.Conv2d(64, n_classes, 1)


@pytest.mark.parametrize("k", [2, 7, 16])
def test_seeded_state_dicts_match_a_torch_restatement(k):
    torch.manual_seed(5)
    ref = _TorchSiamese(3, k).state_dict()
    torch.manual_seed(5)
    sd = spec.SiameseSpec(3, k).default_state_dict()
    assert _digest(sd) == _digest(ref)
    torch.manual_seed(5)
    mod = M.SiameseUNet(3, k).state_dict()
    assert _digest(mod) == _digest(ref)
    assert sd["conv_last.weight"].shape == (k, 64, 1, 1) and sd["conv_last.bias"].shape == (k,)


@pytest.mark.parametrize("k", [0, 17, 2.0, "2", None, True])
def test_class_counts_outside_1_to_16_are_rejected_at_construction(k):
    with pytest.raises(NotImplementedError, match="1 to 16 classes"):
        M.SiameseUNet(3, k)
    with pytest.raises(NotImplementedError, match="1 to 16 classes"):
        siamese.SiameseEngine(torch.device("cpu"), 3, k)


def test_engine_registers_the_k_class_head():
    eng = siamese.SiameseEngine(torch.device("cpu"), 3, 7)
    assert tuple(eng.param("conv_last.weight").shape) == (7, 64, 1, 1)
    assert tuple(eng.param("conv_last.bias").shape) == (7,)
    assert eng.store.off("conv_last.weight") > eng.store.off("att3.W_g.0.weight")     # inside the reduced tail
    one = siamese.SiameseEngine(torch.device("cpu"), 3, 1)
    assert tuple(one.param("conv_last.weight").shape) == (1, 64, 1, 1)
    assert one.store.segs["conv_last.weight"][1] == 64 and one.store.segs["conv_last.bias"][1] == 1


@pytest.mark.parametrize("k,kind", [(1, "ce"), (2, "combined"), (7, "focal_dice"), (16, "combined")])
def test_loss_kind_and_class_count_pairings(k, kind):
    eng = siamese.SiameseEngine(torch.device("cpu"), 3, k)
    lab = torch.zeros(1, 16, 16, dtype=torch.int64)
    with pytest.raises(ValueError, match="kind='ce' with n_classes > 1"):
        eng.loss_and_grad(lab, kind)
    x = torch.zeros(1, 3, 16, 16)
    with pytest.raises(ValueError, match="kind='ce' with n_classes > 1"):
        eng.train_step(x, x, lab, kind=kind)


def test_ce_rejects_unknown_keywords_and_wrong_weight_lengths():
    eng = siamese.SiameseEngine(torch.device("cpu"), 3, 3)
    lab = torch.zeros(1, 16, 16, dtype=torch.int64)
    with pytest.raises(ValueError, match="class_weight and ignore_index"):
        eng.loss_and_grad(lab, "ce", pos_weight=9.0)
    with pytest.raises(ValueError, match="class_weight has 2 entries; n_classes = 3"):
        eng.loss_and_grad(lab, "ce", class_weight=[1.0, 2.0])


def test_checkpoint_class_count_mismatch_is_refused_and_legacy_reads_as_one():
    base = {"format": checkpoint.FORMAT, "kind": "siamese", "channels": {"n_channels": 3}}
    with pytest.raises(ValueError, match="n_classes=2; this one has n_classes=7"):
        checkpoint.load_siamese_state(SimpleNamespace(n_channels=3, n_classes=7), dict(base, n_classes=2))
    # a checkpoint without the field was written by an n_classes = 1 engine
    with pytest.raises(ValueError, match="n_classes=1; this one has n_classes=2"):
        checkpoint.load_siamese_state(SimpleNamespace(n_channels=3, n_classes=2), base)
    loaded = []
    eng = SimpleNamespace(n_channels=3, n_classes=1)
    orig = checkpoint._load_net
    checkpoint._load_net = lambda e, d: loaded.append(d)
    try:
        assert checkpoint.load_siamese_state(eng, dict(base, net="N", extra={"e": 1}), restore_rng=False) == {"e": 1}
    finally:
        checkpoint._load_net = orig
    assert loaded == ["N"]


def test_siamese_state_records_the_class_count():
    eng = siamese.SiameseEngine(torch.device("cpu"), 3, 5)
    orig = torch.cuda.synchronize
    torch.cuda.synchronize = lambda *a: None
    try:
        st = checkpoint.siamese_state(eng)
    finally:
        torch.cuda.synchronize = orig
    assert st["n_classes"] == 5 and st["channels"] == {"n_channels": 3}


def test_head_entry_points_check_arguments_without_a_gpu(lib_path):
    from gan_aug_pfa_b200 import _lib
    h = _lib.lib()
    fake = ctypes.c_void_p(1 << 20)          # never dereferenced: validation fails first
    for k in (0, 17):
        assert h.gap_conv1x1_ck_fwd(fake, 64, fake, fake, k, 1, 64, fake, None, None) == -1
        assert b"k must be 1..16" in h.gap_last_error_string()
        assert h.gap_conv1x1_ck_dgrad(fake, fake, k, 1, 64, fake, 64, None) == -1
        assert b"k must be 1..16" in h.gap_last_error_string()
        assert h.gap_conv1x1_ck_wgrad(fake, fake, 64, k, 1, 64, fake, None, None) == -1
        assert b"k must be 1..16" in h.gap_last_error_string()
        assert h.gap_seg_ce_loss(fake, fake, k, 1, 64, None, -100, fake, fake, fake, 1.0, fake, None) == -1
        assert b"k must be 1..16" in h.gap_last_error_string()
        assert h.gap_seg_confusion_ck(fake, fake, k, 1, 64, -100, fake, None) == -1
        assert b"k must be 1..16" in h.gap_last_error_string()
    assert h.gap_conv1x1_ck_fwd(None, 64, fake, fake, 2, 1, 64, fake, None, None) == -1
    assert h.gap_conv1x1_ck_fwd(fake, 60, fake, fake, 2, 1, 64, fake, None, None) == -1        # ldx < 64
    assert h.gap_conv1x1_ck_fwd(fake, 72, fake, None, 2, 1, 64, fake, None, None) == -1        # no bias
    assert h.gap_conv1x1_ck_dgrad(fake, fake, 2, 1, 64, fake, 68, None) == -1                 # ldg % 8
    assert h.gap_conv1x1_ck_wgrad(fake, fake, 64, 2, 0, 64, fake, None, None) == -1           # n = 0
    assert h.gap_seg_ce_loss(fake, fake, 2, 1, 64, None, -100, fake, None, fake, 1.0, fake, None) == -1   # no counter
    assert h.gap_seg_confusion_ck(fake, fake, 2, 1, 0, -100, fake, None) == -1
    assert b"gap_seg_confusion_ck: bad arguments" in h.gap_last_error_string()


def test_ops_wrappers_check_head_arguments_before_any_cuda_call():
    bf = torch.bfloat16
    x = torch.zeros(2, 4, 4, 64, dtype=bf)
    w, b = torch.zeros(3, 64), torch.zeros(3)
    with pytest.raises(ValueError, match="number of classes must be an int in 1..16"):
        ops.conv1x1_ck_fwd(x, torch.zeros(17, 64), torch.zeros(17), torch.zeros(2, 17, 4, 4))
    with pytest.raises(ValueError, match=r"x must be NHWC bf16 \[n, h, w, 64\]"):
        ops.conv1x1_ck_fwd(torch.zeros(2, 4, 4, 32, dtype=bf), w, b, torch.zeros(2, 3, 4, 4))
    with pytest.raises(ValueError, match="out must be contiguous fp32 class planes"):
        ops.conv1x1_ck_fwd(x, w, b, torch.zeros(2, 3, 4, 5))
    with pytest.raises(ValueError, match="weight must be contiguous fp32"):
        ops.conv1x1_ck_fwd(x, torch.zeros(2, 64), b, torch.zeros(2, 3, 4, 4))
    with pytest.raises(ValueError, match="pred must be contiguous uint8"):
        ops.conv1x1_ck_fwd(x, w, b, torch.zeros(2, 3, 4, 4), torch.zeros(2, 4, 4, dtype=torch.int64))
    with pytest.raises(ValueError, match="needs CUDA tensors"):
        ops.conv1x1_ck_fwd(x, w, b, torch.zeros(2, 3, 4, 4))
    with pytest.raises(ValueError, match="dl must be contiguous fp32 class planes"):
        ops.conv1x1_ck_dgrad(torch.zeros(2, 3, 4, 4, dtype=torch.float64), w, x)
    with pytest.raises(ValueError, match="needs CUDA tensors"):
        ops.conv1x1_ck_dgrad(torch.zeros(2, 3, 4, 4), w, x)
    with pytest.raises(ValueError, match="db must be contiguous fp32"):
        ops.conv1x1_ck_wgrad(torch.zeros(2, 3, 4, 4), x, w, torch.zeros(4))
    lg, lab = torch.zeros(2, 3, 4, 4), torch.zeros(2, 4, 4, dtype=torch.int64)
    s2, bad, loss = torch.zeros(2, dtype=torch.float64), torch.zeros(1, dtype=torch.int64), torch.zeros(1, dtype=torch.float64)
    with pytest.raises(ValueError, match="labels must be contiguous int64"):
        ops.seg_ce_loss(lg, lab.int(), None, -100, s2, bad, None, 1.0, loss)
    with pytest.raises(ValueError, match=r"class_weight must be contiguous fp32 \[3\]"):
        ops.seg_ce_loss(lg, lab, torch.ones(2), -100, s2, bad, None, 1.0, loss)
    with pytest.raises(ValueError, match="bad_labels must be int64"):
        ops.seg_ce_loss(lg, lab, None, -100, s2, bad.float(), None, 1.0, loss)
    with pytest.raises(ValueError, match="needs CUDA tensors"):
        ops.seg_ce_loss(lg, lab, None, -100, s2, bad, lg.clone(), 1.0, loss)
    with pytest.raises(ValueError, match=r"counts must be a contiguous int64 \[n=2, 3, 3\]"):
        ops.seg_confusion_ck(lg, lab, -100, torch.zeros(2, 4, dtype=torch.int64))
    with pytest.raises(ValueError, match="needs CUDA tensors"):
        ops.seg_confusion_ck(lg, lab, -100, torch.zeros(2, 3, 3, dtype=torch.int64))


def test_multiclass_metrics_formulas_on_a_known_matrix():
    from gan_aug_pfa_b200 import metrics
    c = torch.tensor([[[5, 1, 0], [2, 3, 1], [0, 0, 0]], [[1, 0, 0], [0, 1, 0], [0, 0, 0]]])
    m = metrics.multiclass_metrics(c, smooth=1e-6)
    tot = c.sum(0)             # [[6,1,0],[2,4,1],[0,0,0]]
    tp0, fp0, fn0 = 6.0, 2.0, 1.0
    assert m["precision"][0] == pytest.approx((tp0 + 1e-6) / (tp0 + fp0 + 1e-6), rel=1e-6)
    assert m["recall"][0] == pytest.approx((tp0 + 1e-6) / (tp0 + fn0 + 1e-6), rel=1e-6)
    assert m["iou"][1] == pytest.approx((4 + 1e-6) / (4 + 1 + 3 + 1e-6), rel=1e-6)
    assert m["iou"][2] == pytest.approx(1e-6 / (1 + 1e-6), rel=1e-6)    # never labelled, predicted once
    assert m["accuracy"] == pytest.approx((10 + 1e-6) / (int(tot.sum()) + 1e-6), rel=1e-6)
    assert m["mean_iou"] == pytest.approx(sum(m["iou"]) / 3, rel=1e-6)
