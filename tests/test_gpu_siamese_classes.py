"""Multi-class Siamese U-Net (SiameseUNet(n_channels, K), K = 2..16) on the native kernels: known-answer tests of the
K-class head, the softmax cross-entropy and the confusion matrix against torch; the K = 1 path left as it was; the
engine, the drop-in module and the checkpoints against the oracle.

Network tolerances follow tests/test_gpu_siamese.py: the native network keeps bf16 activations, so its logits, loss
and gradients must lie within 1.5x the distance of torch's own bf16 autocast run from the fp32 oracle, measured here
on the same fixture."""
import io

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

from gan_aug_pfa_b200 import checkpoint, metrics, ops  # noqa: E402
from gan_aug_pfa_b200 import models as M  # noqa: E402
from gan_aug_pfa_b200.siamese import SiameseEngine  # noqa: E402
from oracle import pix2pix_oracle as O  # noqa: E402

DEV = torch.device("cuda:0")
NAN = float("nan")


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _guarded(numel, guard, dtype, fill):
    buf = torch.full((numel + 2 * guard,), fill, device=DEV, dtype=dtype)
    return buf, buf[guard:guard + numel]


# ------------------------------------------------------------------------------------------------
# head kernels
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [2, 3, 7, 16])
def test_head_kernels_against_torch(k):
    g = torch.Generator().manual_seed(10 + k)
    n, h, w = 3, 7, 13                    # 273 pixels: not a multiple of any CTA tile, odd plane size
    ld = 80                               # the head input is a channel slice of a wider buffer
    xs = torch.randn(n, h, w, ld, generator=g).to(torch.bfloat16)
    xs[..., :8] = NAN
    xs[..., 72:] = NAN
    xd = xs.to(DEV)[..., 8:72]
    x = xs[..., 8:72].float()
    wt = torch.randn(k, 64, generator=g) / 8
    b = torch.randn(k, generator=g)
    wt[1] = wt[0]                         # classes 0 and 1 tie everywhere: argmax must say 0 where they lead
    b[1] = b[0]
    wb = wt.to(torch.bfloat16).float()
    ref = torch.einsum("nhwc,kc->nkhw", x.double(), wb.double()).float() + b.view(1, k, 1, 1)
    numel, G = n * k * h * w, 67
    buf, out = _guarded(numel, G, torch.float32, NAN)
    pbuf, pred = _guarded(n * h * w, G, torch.uint8, 0xEE)
    ops.conv1x1_ck_fwd(xd, wt.to(DEV), b.to(DEV), out.view(n, k, h, w), pred.view(n, h, w))
    got = out.view(n, k, h, w).cpu()
    assert rel(got, ref) < 4e-3
    assert torch.isnan(buf[:G]).all() and torch.isnan(buf[G + numel:]).all()
    assert (pbuf[:G] == 0xEE).all() and (pbuf[G + n * h * w:] == 0xEE).all()
    assert torch.equal(pred.view(n, h, w).cpu().long(), torch.argmax(got, dim=1))
    assert (got[:, 0] == got[:, 1]).all()          # the constructed ties are exact ...
    assert (pred.cpu() != 1).all()                  # ... and resolved to the lower index
    # input gradient: written into channels 8..71 of an 80-channel NaN-filled buffer
    dl = torch.randn(n, k, h, w, generator=g)
    gbuf = torch.full((n, h, w, ld), NAN, device=DEV, dtype=torch.bfloat16)
    ops.conv1x1_ck_dgrad(dl.to(DEV), wt.to(DEV), gbuf[..., 8:72])
    gref = torch.einsum("nkhw,kc->nhwc", dl.double(), wb.double())
    assert rel(gbuf[..., 8:72].cpu().float(), gref) < 4e-3
    assert torch.isnan(gbuf[..., :8]).all() and torch.isnan(gbuf[..., 72:]).all()
    # weight and bias gradients, accumulated onto ones
    dw = torch.ones(k, 64, device=DEV)
    db = torch.ones(k, device=DEV)
    ops.conv1x1_ck_wgrad(dl.to(DEV), xd, dw, db)
    wref = torch.einsum("nkhw,nhwc->kc", dl.double(), x.double()) + 1.0
    assert rel(dw.cpu(), wref) < 2e-4
    assert rel(db.cpu(), dl.double().sum((0, 2, 3)) + 1.0) < 2e-4


def test_head_at_full_size_with_a_large_gradient_sum():
    """batch 4 @512^2 (1,048,576 pixels): the weight gradient sums a million products per entry."""
    g = torch.Generator(device=DEV).manual_seed(3)
    k, n, h, w = 7, 4, 512, 512
    x = torch.randn(n, h, w, 64, device=DEV, generator=g).to(torch.bfloat16)
    dl = torch.randn(n, k, h, w, device=DEV, generator=g) * 1e-3
    dw = torch.zeros(k, 64, device=DEV)
    db = torch.zeros(k, device=DEV)
    ops.conv1x1_ck_wgrad(dl, x, dw, db)
    wref = torch.einsum("nkp,npc->kc", dl.double().view(n, k, -1), x.double().view(n, -1, 64))
    assert rel(dw, wref) < 2e-4
    assert rel(db, dl.double().sum((0, 2, 3))) < 2e-4


# ------------------------------------------------------------------------------------------------
# cross-entropy and confusion matrix
# ------------------------------------------------------------------------------------------------
def _ce(logits, labels, weight, ignore_index, grad_scale=1.0):
    k = logits.shape[1]
    sums = torch.zeros(2, device=DEV, dtype=torch.float64)
    bad = torch.zeros(1, device=DEV, dtype=torch.int64)
    loss = torch.zeros(1, device=DEV, dtype=torch.float64)
    grad = torch.full_like(logits, NAN)
    cw = None if weight is None else weight.to(DEV)
    ops.seg_ce_loss(logits, labels, cw, ignore_index, sums, bad, grad, grad_scale, loss)
    assert k == grad.shape[1]
    return float(loss), grad.cpu(), int(bad)


@pytest.mark.parametrize("k", [2, 7, 16])
@pytest.mark.parametrize("weighted", [False, True])
def test_cross_entropy_matches_torch(k, weighted):
    g = torch.Generator().manual_seed(20 + k)
    n, h, w = 3, 17, 23
    logits = torch.randn(n, k, h, w, generator=g) * 3
    labels = torch.randint(0, k, (n, h, w), generator=g)
    labels[torch.rand(n, h, w, generator=g) < 0.2] = -100            # ignored pixels
    weight = torch.rand(k, generator=g) * 2 + 0.1 if weighted else None
    xr = logits.double().requires_grad_(True)
    ref = F.cross_entropy(xr, labels, weight=None if weight is None else weight.double(), ignore_index=-100)
    ref.backward()
    loss, grad, bad = _ce(logits.to(DEV), labels.to(DEV), weight, -100)
    assert abs(loss - float(ref)) <= 1e-6 * abs(float(ref))
    assert rel(grad, xr.grad) < 1e-5
    assert bad == 0
    # grad_scale and another ignore_index
    lab2 = labels.clone()
    lab2[lab2 == -100] = 255
    loss2, grad2, _ = _ce(logits.to(DEV), lab2.to(DEV), weight, 255, grad_scale=0.25)
    assert abs(loss2 - float(ref)) <= 1e-6 * abs(float(ref))
    assert rel(grad2, 0.25 * xr.grad) < 1e-5


def test_cross_entropy_counts_out_of_range_labels_and_ignores_them():
    g = torch.Generator().manual_seed(7)
    k, n, h, w = 5, 2, 16, 16
    logits = torch.randn(n, k, h, w, generator=g)
    labels = torch.randint(0, k, (n, h, w), generator=g)
    flat = labels.view(-1)
    planted = torch.tensor([3, 40, 41, 200, 511])
    flat[planted] = torch.tensor([k, -1, 99, -7, k + 3])
    clean = labels.clone()
    clean.view(-1)[planted] = -100
    weight = torch.tensor([1.0, 2.0, 0.5, 1.5, 3.0])
    xr = logits.double().requires_grad_(True)
    ref = F.cross_entropy(xr, clean, weight=weight.double())
    ref.backward()
    loss, grad, bad = _ce(logits.to(DEV), labels.to(DEV), weight, -100)
    assert bad == len(planted)
    assert abs(loss - float(ref)) <= 1e-6 * abs(float(ref))
    assert rel(grad, xr.grad) < 1e-5


def test_cross_entropy_of_an_all_ignored_batch_is_nan_like_torch():
    logits = torch.randn(2, 3, 8, 8)
    labels = torch.full((2, 8, 8), -100)
    xr = logits.clone().requires_grad_(True)
    ref = F.cross_entropy(xr, labels)
    ref.backward()
    loss, grad, bad = _ce(logits.to(DEV), labels.to(DEV), None, -100)
    assert torch.isnan(ref) and loss != loss
    assert torch.equal(grad, xr.grad) and bad == 0


@pytest.mark.parametrize("k", [2, 7, 16])
def test_confusion_matrix_and_metrics(k):
    g = torch.Generator().manual_seed(30 + k)
    n, h, w = 3, 31, 45
    logits = torch.randn(n, k, h, w, generator=g).to(torch.bfloat16).float()    # coarse values: exact ties occur
    logits[:, 1] = torch.where(torch.rand(n, h, w, generator=g) < 0.3, logits[:, 0], logits[:, 1])
    labels = torch.randint(0, k, (n, h, w), generator=g)
    labels[torch.rand(n, h, w, generator=g) < 0.1] = -100
    labels[0, 0, :3] = torch.tensor([k, -2, 1000])                  # out of range: not counted
    pred = torch.argmax(logits, dim=1)
    want = torch.zeros(n, k, k, dtype=torch.int64)
    for i in range(n):
        m = (labels[i] >= 0) & (labels[i] < k)
        want[i] = torch.bincount(labels[i][m] * k + pred[i][m], minlength=k * k).view(k, k)
    got = metrics.confusion_matrix(logits.to(DEV), labels.to(DEV))
    assert torch.equal(got.cpu(), want)
    metrics.confusion_matrix(logits.to(DEV), labels.to(DEV), out=got)              # accumulates
    assert torch.equal(got.cpu(), 2 * want)
    mm = metrics.multiclass_metrics(want)
    c = want.sum(0).float()
    tp = c.diagonal()
    fp, fn = c.sum(0) - tp, c.sum(1) - tp
    s = 1e-6
    p = (tp + s) / (tp + fp + s)
    r = (tp + s) / (tp + fn + s)
    iou = (tp + s) / (tp + fp + fn + s)
    assert mm["precision"] == pytest.approx(p.tolist(), rel=1e-6)
    assert mm["recall"] == pytest.approx(r.tolist(), rel=1e-6)
    assert mm["f1"] == pytest.approx(((2 * p * r + s) / (p + r + s)).tolist(), rel=1e-6)
    assert mm["iou"] == pytest.approx(iou.tolist(), rel=1e-6)
    assert mm["mean_iou"] == pytest.approx(float(iou.mean()), rel=1e-6)
    assert mm["accuracy"] == pytest.approx(float((tp.sum() + s) / (c.sum() + s)), rel=1e-6)


# ------------------------------------------------------------------------------------------------
# K = 1 keeps its kernels
# ------------------------------------------------------------------------------------------------
def test_single_class_engine_uses_no_multiclass_kernel(monkeypatch):
    def boom(*a, **kw):
        raise AssertionError("a multi-class kernel was launched for n_classes = 1")

    for name in ("conv1x1_ck_fwd", "conv1x1_ck_dgrad", "conv1x1_ck_wgrad", "seg_ce_loss", "seg_confusion_ck"):
        monkeypatch.setattr(ops, name, boom)
    torch.manual_seed(0)
    m = M.SiameseUNet(3, 1)
    eng = SiameseEngine(DEV)
    eng.load_state_dict({k: v.detach() for k, v in m.state_dict().items()})
    g = torch.Generator().manual_seed(1)
    x1, x2 = (torch.rand(2, 3, 32, 32, generator=g) * 2 - 1).to(DEV), (torch.rand(2, 3, 32, 32, generator=g) * 2 - 1).to(DEV)
    lab = (torch.rand(2, 32, 32, generator=g) < 0.2).long().to(DEV)
    eng.train_step(x1, x2, lab)
    logits = eng.forward(x1, x2)
    assert tuple(logits.shape) == (2, 32, 32) and tuple(eng.dlogits.shape) == (2, 32, 32)
    again = torch.empty(2 * 32 * 32, device=DEV)
    ops.conv1x1_cout1_fwd(eng._last, eng.store.seg(eng.store.p, "conv_last.weight"), eng.param("conv_last.bias"), again)
    assert torch.equal(logits.reshape(-1), again)
    eng.backward()
    out = m.to(DEV)(x1, x2)
    assert tuple(out.shape) == (2, 1, 32, 32)


# ------------------------------------------------------------------------------------------------
# network level against the oracle
# ------------------------------------------------------------------------------------------------
def _fixture(k, n=2, hw=128, seed=0):
    g = torch.Generator().manual_seed(100 + k + seed)
    x1 = torch.rand(n, 3, hw, hw, generator=g) * 2 - 1
    x2 = torch.rand(n, 3, hw, hw, generator=g) * 2 - 1
    lab = torch.randint(0, k, (n, hw, hw), generator=g)
    lab[torch.rand(n, hw, hw, generator=g) < 0.05] = -100
    weight = torch.linspace(0.5, 2.0, k)
    return x1, x2, lab, weight


def _oracle(sd, x1, x2, lab, weight, bf16=False):
    """fp32 oracle on the GPU (TF32 off), or the same under torch's bf16 autocast: logits, loss, gradients."""
    sd = {kk: v.detach().clone().to(DEV) for kk, v in sd.items()}
    names = O.param_names(sd)
    for kk in names:
        sd[kk].requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
        out = O.siamese_forward(sd, x1.to(DEV), x2.to(DEV), True, {})
    out = out.float()
    loss = F.cross_entropy(out, lab.to(DEV), weight=weight.to(DEV))
    grads = torch.autograd.grad(loss, [sd[kk] for kk in names])
    return out.detach(), float(loss), torch.cat([gg.reshape(-1) for gg in grads]).detach(), names


@pytest.mark.parametrize("k", [2, 7])
def test_engine_and_dropin_match_the_oracle(k):
    x1, x2, lab, weight = _fixture(k)
    torch.manual_seed(0)
    m = M.SiameseUNet(3, k)
    sd0 = {kk: v.detach().clone() for kk, v in m.state_dict().items()}
    ref_out, ref_loss, ref_g, names = _oracle(sd0, x1, x2, lab, weight)
    y_out, y_loss, y_g, _ = _oracle(sd0, x1, x2, lab, weight, bf16=True)
    yard_out, yard_g = rel(y_out, ref_out), rel(y_g, ref_g)
    yard_loss = max(abs(y_loss - ref_loss), 1e-3 * abs(ref_loss))
    # drop-in module: the reference's loop body with nn.CrossEntropyLoss(weight) and AdamW
    m = m.to(DEV)
    m.train()
    crit = nn.CrossEntropyLoss(weight=weight.to(DEV))
    opt = torch.optim.AdamW(m.parameters(), lr=1.0152e-4, weight_decay=1.118e-5)
    losses = []
    for step in range(3):
        opt.zero_grad()
        out = m(x1.to(DEV), x2.to(DEV))
        assert tuple(out.shape) == (2, k, 128, 128)
        loss = crit(out, lab.to(DEV))
        loss.backward()
        if step == 0:
            assert rel(out.detach(), ref_out) < 1.5 * yard_out, (rel(out.detach(), ref_out), yard_out)
            assert abs(float(loss) - ref_loss) < 1.5 * yard_loss
            got_g = torch.cat([dict(m.named_parameters())[kk].grad.reshape(-1) for kk in names])
            assert rel(got_g, ref_g) < 1.5 * yard_g, (rel(got_g, ref_g), yard_g)
        opt.step()
        losses.append(float(loss))
    # the oracle's own three steps (fp32, same AdamW)
    sd = {kk: v.clone().to(DEV) for kk, v in sd0.items()}
    ost = O.AdamState(sd, O.param_names(sd), 1.0152e-4, (0.9, 0.999), 1e-8, 1.118e-5, decoupled=True)
    crit_o = lambda o, t: F.cross_entropy(o, t, weight=weight.to(DEV))       # noqa: E731
    want = [O.siamese_train_step(sd, ost, x1.to(DEV), x2.to(DEV), lab.to(DEV), criterion=crit_o) for _ in range(3)]
    for got_l, ref_l in zip(losses, want):
        assert abs(got_l - ref_l) < max(1.5 * yard_loss, 3e-2 * ref_l), (losses, want)
    # the engine's fused step gives the drop-in loop's losses
    eng = SiameseEngine(DEV, 3, k)
    eng.load_state_dict(sd0)
    seq = [float(eng.train_step(x1.to(DEV), x2.to(DEV), lab.to(DEV), kind="ce", class_weight=weight.tolist()).cpu())
           for _ in range(3)]
    assert seq == pytest.approx(losses, rel=2e-3)
    assert int(eng.bad_labels) == 0
    # eval: predict() is the argmax of the eval-mode logits
    m.eval()
    with torch.no_grad():
        ev = m(x1.to(DEV), x2.to(DEV))
    pred = m._engine_obj.predict(x1.to(DEV), x2.to(DEV))
    assert pred.dtype == torch.uint8 and torch.equal(pred.long(), ev.argmax(1))
    eng.training = False
    pe = eng.predict(x1.to(DEV), x2.to(DEV))
    assert eng.training is False and pe.shape == (2, 128, 128)


def test_class_weight_as_a_device_tensor_and_the_pairing_errors():
    k = 3
    x1, x2, lab, weight = _fixture(k, hw=32)
    torch.manual_seed(0)
    sd = M.SiameseUNet(3, k).state_dict()
    a, b = SiameseEngine(DEV, 3, k), SiameseEngine(DEV, 3, k)
    a.load_state_dict(sd)
    b.load_state_dict(sd)
    la = float(a.train_step(x1.to(DEV), x2.to(DEV), lab.to(DEV), class_weight=weight.to(DEV)).cpu())
    lb = float(b.train_step(x1.to(DEV), x2.to(DEV), lab.to(DEV), kind="ce", class_weight=tuple(weight.tolist())).cpu())
    assert la == lb
    with pytest.raises(ValueError, match="kind='ce' with n_classes > 1"):
        a.train_step(x1.to(DEV), x2.to(DEV), lab.to(DEV), kind="combined")


def test_multiclass_engine_resumes_from_a_checkpoint():
    k = 7
    g = torch.Generator().manual_seed(4)
    data = [((torch.rand(2, 3, 32, 32, generator=g) * 2 - 1).to(DEV), (torch.rand(2, 3, 32, 32, generator=g) * 2 - 1).to(DEV),
             torch.randint(0, k, (2, 32, 32), generator=g).to(DEV)) for _ in range(4)]
    torch.manual_seed(0)
    a = SiameseEngine(DEV, 3, k)
    a.load_state_dict({kk: v.detach() for kk, v in M.SiameseUNet(3, k).state_dict().items()})
    for bt in data[:2]:
        a.train_step(*bt)
    buf = io.BytesIO()
    checkpoint.save(buf, checkpoint.siamese_state(a))
    want = [float(a.train_step(*bt).cpu()) for bt in data[2:]]
    buf.seek(0)
    state = checkpoint.load(buf)
    assert state["n_classes"] == k
    r = SiameseEngine(DEV, 3, k)
    checkpoint.load_siamese_state(r, state)
    got = [float(r.train_step(*bt).cpu()) for bt in data[2:]]
    assert got == pytest.approx(want, rel=5e-3)
    with pytest.raises(ValueError, match="n_classes=7; this one has n_classes=2"):
        checkpoint.load_siamese_state(SiameseEngine(DEV, 3, 2), state)


def test_batch4_512_step_is_finite_and_matches_the_oracle_loss():
    k = 7
    x1, x2, lab, weight = _fixture(k, n=4, hw=512, seed=1)
    torch.manual_seed(0)
    sd0 = {kk: v.detach().clone() for kk, v in M.SiameseUNet(3, k).state_dict().items()}
    with torch.no_grad():
        ref = F.cross_entropy(O.siamese_forward({kk: v.to(DEV) for kk, v in sd0.items()}, x1.to(DEV), x2.to(DEV), True, {}),
                              lab.to(DEV), weight=weight.to(DEV))
        with torch.autocast("cuda", dtype=torch.bfloat16):
            yo = O.siamese_forward({kk: v.to(DEV) for kk, v in sd0.items()}, x1.to(DEV), x2.to(DEV), True, {})
        yard = F.cross_entropy(yo.float(), lab.to(DEV), weight=weight.to(DEV))
    eng = SiameseEngine(DEV, 3, k)
    eng.load_state_dict(sd0)
    loss = float(eng.train_step(x1.to(DEV), x2.to(DEV), lab.to(DEV), class_weight=weight).cpu())
    assert torch.isfinite(eng.store.p).all() and torch.isfinite(eng.logits).all()
    bound = 1.5 * max(abs(float(yard) - float(ref)), 1e-3 * float(ref))
    assert abs(loss - float(ref)) < bound, (loss, float(ref), float(yard))

