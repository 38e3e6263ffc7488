"""Multi-class Dice losses without a GPU: the torch reference of kind="ce_dice" / "softmax_focal_dice" (the definition
the native kernels are tested against) reduces to the reference's own CombinedLoss-style CE + Dice and FocalDiceLoss
at K = 2; the loss-kind pairings and keyword checks of the engine; the argument checks of the criteria, the ops
wrapper and the C entry point."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from gan_aug_pfa_b200 import losses, ops, siamese
from oracle import pix2pix_oracle as O


def softmax_dice_ref(z, y, kind, w_point=0.5, gamma=2.0, smooth=1.0, weight=None, ignore_index=-100):
    """kind="ce_dice": w_point * CE + (1 - w_point) * Dice; kind="softmax_focal_dice": w_point * Focal + (1 - w_point)
    * Dice, on logits z [n, K, h, w] against labels y [n, h, w], p = softmax(z).  Counted pixels V: y != ignore_index
    and 0 <= y < K; every sum runs over V across the whole batch.
      Dice  = 1 - 1/(K-1) sum_{k=1..K-1} (2 I_k + s) / (P_k + T_k + s),  I_k = sum p_k [y=k], P_k = sum p_k,
              T_k = sum [y=k]  (class 0 excluded)
      CE    = nn.CrossEntropyLoss(weight, ignore_index): sum w[y] (-log p_y) / sum w[y]
      Focal = sum a[y] (1 - p_y)^gamma (-log p_y) / |V|,  a = weight (None: all 1)"""
    k = z.shape[1]
    valid = (y != ignore_index) & (y >= 0) & (y < k)
    yc = torch.where(valid, y, torch.zeros_like(y))
    vm = valid.to(z.dtype)
    logp = torch.log_softmax(z, 1)
    p = logp.exp()
    onehot = F.one_hot(yc, k).permute(0, 3, 1, 2).to(z.dtype) * vm[:, None]
    inter = (p * onehot).sum((0, 2, 3))
    psum = (p * vm[:, None]).sum((0, 2, 3))
    tsum = onehot.sum((0, 2, 3))
    dice = 1 - ((2 * inter + smooth) / (psum + tsum + smooth))[1:].mean()
    nll = -logp.gather(1, yc[:, None])[:, 0]
    w = torch.ones_like(nll) if weight is None else weight.to(z.dtype)[yc]
    if kind == "ce_dice":
        point = (w * nll * vm).sum() / (w * vm).sum()
    else:
        r = (p * (1 - F.one_hot(yc, k).permute(0, 3, 1, 2).to(z.dtype))).sum(1)     # 1 - p_y without cancellation
        mod = r ** gamma if gamma != 0 else torch.ones_like(r)
        point = (w * mod * nll * vm).sum() / vm.sum()
    return w_point * point + (1 - w_point) * dice


def _k2_case(seed):
    g = torch.Generator().manual_seed(seed)
    z = torch.randn(3, 2, 11, 13, generator=g, dtype=torch.float64) * 2
    y = (torch.rand(3, 11, 13, generator=g) < 0.2).long()
    return z, y


@pytest.mark.parametrize("beta,gamma,fa,smooth", [(0.5, 2.0, 0.75, 1.0), (0.3, 0.5, 0.25, 1e-3), (0.8, 0.0, 0.6, 2.0)])
def test_softmax_focal_dice_at_k2_is_the_reference_focal_dice_loss(beta, gamma, fa, smooth):
    z, y = _k2_case(1)
    za = z.clone().requires_grad_(True)
    got = softmax_dice_ref(za, y, "softmax_focal_dice", beta, gamma, smooth, torch.tensor([1 - fa, fa]))
    got.backward()
    zb = z.clone().requires_grad_(True)
    want = O.focal_dice_loss((zb[:, 1] - zb[:, 0])[:, None], y, beta, gamma, fa, smooth)
    want.backward()
    assert abs(float(got.detach()) - float(want.detach())) <= 1e-10 * abs(float(want))
    assert float((za.grad - zb.grad).norm()) <= 1e-10 * float(zb.grad.norm())


@pytest.mark.parametrize("alpha,smooth", [(0.5, 1.0), (0.2, 1e-3), (1.0, 1.0), (0.0, 3.0)])
def test_ce_dice_at_k2_is_cross_entropy_plus_the_reference_dice_loss(alpha, smooth):
    z, y = _k2_case(2)
    za = z.clone().requires_grad_(True)
    got = softmax_dice_ref(za, y, "ce_dice", alpha, smooth=smooth)
    got.backward()
    zb = z.clone().requires_grad_(True)
    want = alpha * F.cross_entropy(zb, y) + (1 - alpha) * O.dice_loss((zb[:, 1] - zb[:, 0])[:, None], y.double(), smooth)
    want.backward()
    assert abs(float(got.detach()) - float(want.detach())) <= 1e-10 * abs(float(want))
    assert float((za.grad - zb.grad).norm()) <= 1e-10 * float(zb.grad.norm())


def test_ce_term_is_torch_cross_entropy_with_weights_and_ignored_pixels():
    g = torch.Generator().manual_seed(3)
    z = torch.randn(2, 5, 9, 7, generator=g, dtype=torch.float64)
    y = torch.randint(0, 5, (2, 9, 7), generator=g)
    y[torch.rand(2, 9, 7, generator=g) < 0.3] = 255
    w = torch.rand(5, generator=g, dtype=torch.float64) + 0.5
    got = softmax_dice_ref(z, y, "ce_dice", 1.0, weight=w, ignore_index=255)
    want = F.cross_entropy(z, y, weight=w, ignore_index=255)
    assert abs(float(got) - float(want)) <= 1e-12 * abs(float(want))


# ------------------------------------------------------------------------------------------------
# engine: kinds, pairings and keywords (all raise before any CUDA work)
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["ce_dice", "softmax_focal_dice"])
def test_dice_kinds_need_more_than_one_class(kind):
    eng = siamese.SiameseEngine(torch.device("cpu"), 3, 1)
    lab = torch.zeros(1, 16, 16, dtype=torch.int64)
    with pytest.raises(ValueError, match="kind='ce' with n_classes > 1 \\(or 'ce_dice', 'softmax_focal_dice'\\)"):
        eng.loss_and_grad(lab, kind)
    x = torch.zeros(1, 3, 16, 16)
    with pytest.raises(ValueError, match="does not apply to n_classes = 1"):
        eng.train_step(x, x, lab, kind=kind)


@pytest.mark.parametrize("k", [2, 16])
def test_binary_kinds_with_several_classes_keep_the_pairing_message(k):
    eng = siamese.SiameseEngine(torch.device("cpu"), 3, k)
    lab = torch.zeros(1, 16, 16, dtype=torch.int64)
    for kind in ("combined", "focal_dice"):
        with pytest.raises(ValueError, match="kind='ce' with n_classes > 1"):
            eng.loss_and_grad(lab, kind)


@pytest.mark.parametrize("kind,bad", [("ce_dice", {"beta": 0.5}), ("ce_dice", {"gamma": 2.0}),
                                      ("softmax_focal_dice", {"alpha": 0.5}), ("softmax_focal_dice", {"pos_weight": 9.0})])
def test_dice_kinds_reject_unknown_keywords(kind, bad):
    eng = siamese.SiameseEngine(torch.device("cpu"), 3, 3)
    lab = torch.zeros(1, 16, 16, dtype=torch.int64)
    with pytest.raises(ValueError, match=f"kind='{kind}' takes"):
        eng.loss_and_grad(lab, kind, **bad)
    x = torch.zeros(1, 3, 16, 16)
    with pytest.raises(ValueError, match=f"kind='{kind}' takes"):      # before the forward is enqueued
        eng.train_step(x, x, lab, kind=kind, **bad)


@pytest.mark.parametrize("kind", ["ce_dice", "softmax_focal_dice"])
def test_dice_kinds_check_weights_and_ranges(kind):
    eng = siamese.SiameseEngine(torch.device("cpu"), 3, 3)
    lab = torch.zeros(1, 16, 16, dtype=torch.int64)
    with pytest.raises(ValueError, match="class_weight has 2 entries; n_classes = 3"):
        eng.loss_and_grad(lab, kind, class_weight=[1.0, 2.0])
    with pytest.raises(ValueError, match="class_weight has 4 entries; n_classes = 3"):
        eng.loss_and_grad(lab, kind, class_weight=torch.ones(4))
    for s in (0.0, -1.0, float("nan")):
        with pytest.raises(ValueError, match="smooth must be > 0"):
            eng.loss_and_grad(lab, kind, smooth=s)
    wkey = "alpha" if kind == "ce_dice" else "beta"
    for v in (-0.1, 1.5):
        with pytest.raises(ValueError, match="point-term weight must be in \\[0, 1\\]"):
            eng.loss_and_grad(lab, kind, **{wkey: v})
    if kind == "softmax_focal_dice":
        with pytest.raises(ValueError, match="gamma must be >= 0"):
            eng.loss_and_grad(lab, kind, gamma=-0.5)


# ------------------------------------------------------------------------------------------------
# criteria, ops wrapper and C entry point
# ------------------------------------------------------------------------------------------------
def test_criteria_check_arguments_without_a_device():
    import gan_aug_pfa_b200 as pkg
    assert pkg.CEDiceLoss is losses.CEDiceLoss and pkg.SoftmaxFocalDiceLoss is losses.SoftmaxFocalDiceLoss
    with pytest.raises(ValueError, match="smooth must be > 0"):
        losses.CEDiceLoss(smooth=0.0)
    with pytest.raises(ValueError, match="point-term weight"):
        losses.CEDiceLoss(alpha=1.1)
    with pytest.raises(ValueError, match="gamma must be >= 0"):
        losses.SoftmaxFocalDiceLoss(gamma=-1.0)
    with pytest.raises(ValueError, match="one entry per class"):
        losses.SoftmaxFocalDiceLoss(weight=[1.0])
    crit = losses.SoftmaxFocalDiceLoss(weight=[0.25, 0.75, 1.0])
    assert crit.weight.dtype == torch.float32 and "weight" in dict(crit.named_buffers())
    lab = torch.zeros(2, 4, 4, dtype=torch.int64)
    with pytest.raises(ValueError, match="needs CUDA tensors"):
        crit(torch.zeros(2, 3, 4, 4), lab)
    with pytest.raises(ValueError, match="K in 2..16"):
        crit(torch.zeros(2, 1, 4, 4), lab)
    with pytest.raises(ValueError, match="K in 2..16"):
        crit(torch.zeros(2, 17, 4, 4), lab)
    with pytest.raises(ValueError, match="K in 2..16"):
        crit(torch.zeros(2, 3, 16), lab)
    with pytest.raises(ValueError, match="fp32 and labels int64"):
        crit(torch.zeros(2, 3, 4, 4, dtype=torch.float64), lab)
    with pytest.raises(ValueError, match="fp32 and labels int64"):
        crit(torch.zeros(2, 3, 4, 4), lab.int())
    with pytest.raises(ValueError, match=r"labels must be \[n=2, h=4, w=4\]"):
        crit(torch.zeros(2, 3, 4, 4), torch.zeros(2, 4, 5, dtype=torch.int64))
    with pytest.raises(ValueError, match="weight has 3 entries; the logits have 4 classes"):
        crit(torch.zeros(2, 4, 4, 4), lab)


def test_ops_wrapper_checks_arguments_before_any_cuda_call():
    lg, lab = torch.zeros(2, 3, 4, 4), torch.zeros(2, 4, 4, dtype=torch.int64)
    sums, bad = torch.zeros(ops.DICE_SUMS, dtype=torch.float64), torch.zeros(1, dtype=torch.int64)
    loss = torch.zeros(1, dtype=torch.float64)
    call = lambda **kw: ops.seg_softmax_dice_loss(**dict(dict(logits=lg, labels=lab, mode=1, w_point=0.5, gamma=2.0,  # noqa: E731
                                                               smooth=1.0, class_weight=None, ignore_index=-100,
                                                               sums=sums, bad_labels=bad, grad=None, grad_scale=1.0,
                                                               loss=loss), **kw))
    with pytest.raises(ValueError, match="mode must be 0"):
        call(mode=2)
    with pytest.raises(ValueError, match="smooth must be > 0"):
        call(smooth=-1.0)
    with pytest.raises(ValueError, match="gamma must be >= 0"):
        call(gamma=-1.0)
    with pytest.raises(ValueError, match="point-term weight"):
        call(w_point=2.0)
    with pytest.raises(ValueError, match="number of classes must be in 2..16"):
        call(logits=torch.zeros(2, 1, 4, 4))
    with pytest.raises(ValueError, match="labels must be contiguous int64"):
        call(labels=lab.int())
    with pytest.raises(ValueError, match=r"class_weight must be contiguous fp32 \[3\]"):
        call(class_weight=torch.ones(2))
    with pytest.raises(ValueError, match=r"sums must be fp64 \[>= 8\]"):
        call(sums=torch.zeros(7, dtype=torch.float64))
    with pytest.raises(ValueError, match="grad must be contiguous fp32 class planes"):
        call(grad=torch.zeros(2, 3, 4, 5))
    with pytest.raises(ValueError, match="bad_labels must be int64"):
        call(bad_labels=bad.float())
    with pytest.raises(ValueError, match="needs CUDA tensors"):
        call()


def test_entry_point_checks_arguments_without_a_gpu(lib_path):
    from gan_aug_pfa_b200 import _lib
    h = _lib.lib()
    fake = ctypes.c_void_p(1 << 20)          # never dereferenced: validation fails first

    def call(k=3, mode=1, w_point=0.5, gamma=2.0, smooth=1.0, sums=fake, bad=fake, loss=fake, n=1):
        return h.gap_seg_softmax_dice(fake, fake, k, n, 64, mode, w_point, gamma, smooth, None, -100, sums, bad, None,
                                      1.0, loss, None)

    for k in (0, 1, 17):
        assert call(k=k) == -1
        assert b"k must be 2..16" in h.gap_last_error_string()
    for kw in (dict(mode=2), dict(sums=None), dict(bad=None), dict(loss=None), dict(n=0)):
        assert call(**kw) == -1
        assert b"gap_seg_softmax_dice: bad arguments" in h.gap_last_error_string()
    for kw in (dict(smooth=0.0), dict(smooth=float("nan")), dict(gamma=-0.5), dict(w_point=-0.1), dict(w_point=1.5)):
        assert call(**kw) == -1
        assert b"smooth > 0, gamma >= 0 and 0 <= w_point <= 1" in h.gap_last_error_string()
