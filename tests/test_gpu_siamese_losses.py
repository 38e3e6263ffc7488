"""Multi-class Dice losses on the native kernels (gap_seg_softmax_dice): known-answer tests of kind="ce_dice" and
"softmax_focal_dice" against the fp64 torch reference of tests/test_siamese_losses_cpu.py, graph capture, and the
engine and the drop-in criteria (losses.py) against the oracle.

Network tolerances follow tests/test_gpu_siamese_classes.py: the native network keeps bf16 activations, so its logits,
loss and gradients must lie within 1.5x the distance of torch's own bf16 autocast run from the fp32 oracle."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from gan_aug_pfa_b200 import losses, ops  # noqa: E402
from gan_aug_pfa_b200 import models as M  # noqa: E402
from gan_aug_pfa_b200.siamese import SiameseEngine  # noqa: E402
from oracle import pix2pix_oracle as O  # noqa: E402
from test_siamese_losses_cpu import softmax_dice_ref  # noqa: E402

DEV = torch.device("cuda:0")
NAN = float("nan")
MODE = {"ce_dice": 0, "softmax_focal_dice": 1}


def rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


@pytest.fixture(autouse=True)
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _native(logits, labels, kind, w_point, gamma, smooth, weight, ignore_index, grad_scale=1.0, guard=61):
    """(loss, gradient, bad-label count) of one gap_seg_softmax_dice call; the gradient sits inside NaN guard bands."""
    numel = logits.numel()
    buf = torch.full((numel + 2 * guard,), NAN, device=DEV)
    grad = buf[guard:guard + numel].view(logits.shape)
    sums = torch.full((ops.DICE_SUMS,), NAN, device=DEV, dtype=torch.float64)     # zeroed by the call
    bad = torch.zeros(1, device=DEV, dtype=torch.int64)
    loss = torch.zeros(1, device=DEV, dtype=torch.float64)
    cw = None if weight is None else weight.to(DEV)
    ops.seg_softmax_dice_loss(logits.to(DEV), labels.to(DEV), MODE[kind], w_point, gamma, smooth, cw, ignore_index,
                              sums, bad, grad, grad_scale, loss)
    assert torch.isnan(buf[:guard]).all() and torch.isnan(buf[guard + numel:]).all()
    return float(loss), grad.cpu(), int(bad)


def _case(k, seed):
    """n = 3, 37 x 29 (3219 pixels): ignored labels, planted out-of-range labels, confident pixels (+-30 logits, right
    and wrong), and for K > 2 a class that never occurs."""
    g = torch.Generator().manual_seed(seed)
    n, h, w = 3, 37, 29
    logits = torch.randn(n, k, h, w, generator=g) * 3
    hi = max(k - 1, 2)                                      # labels 0 .. K-2: class K-1 is absent (K > 2)
    labels = torch.randint(0, hi, (n, h, w), generator=g)
    labels[torch.rand(n, h, w, generator=g) < 0.15] = -100
    conf = torch.rand(n, h, w, generator=g) < 0.2
    c = torch.randint(0, k, (n, h, w), generator=g)
    conf_logits = torch.full((n, k, h, w), -30.0).scatter_(1, c[:, None], 30.0)
    logits = torch.where(conf[:, None], conf_logits, logits)
    right = conf & (torch.rand(n, h, w, generator=g) < 0.7) & (labels >= 0)
    c2 = torch.where(labels >= 0, labels, torch.zeros_like(labels))      # most confident pixels are right
    logits = torch.where(right[:, None], torch.full((n, k, h, w), -30.0).scatter_(1, c2[:, None], 30.0), logits)
    flat = labels.view(-1)
    planted = torch.tensor([5, 77, 400, 1999, 3000])
    flat[planted] = torch.tensor([k, -1, 99, -7, k + 5])
    return logits, labels, len(planted)


CASES = [("ce_dice", 0.0), ("softmax_focal_dice", 0.0), ("softmax_focal_dice", 0.5), ("softmax_focal_dice", 2.0)]


@pytest.mark.parametrize("k", [2, 3, 7, 16])
@pytest.mark.parametrize("kind,gamma", CASES)
@pytest.mark.parametrize("weighted", [False, True])
@pytest.mark.parametrize("smooth", [1.0, 1.96e-6])
def test_kernel_matches_the_fp64_reference(k, kind, gamma, weighted, smooth):
    logits, labels, nbad = _case(k, 40 + k)
    g = torch.Generator().manual_seed(k)
    weight = torch.rand(k, generator=g) * 2 + 0.1 if weighted else None
    w_point = 0.4
    z = logits.double().requires_grad_(True)
    clean = labels.clone()
    clean[(clean < 0) | (clean >= k)] = -100
    ref = softmax_dice_ref(z, clean, kind, w_point, gamma, smooth, None if weight is None else weight.double())
    ref.backward()
    loss, grad, bad = _native(logits, labels, kind, w_point, gamma, smooth, weight, -100)
    assert bad == nbad
    assert abs(loss - float(ref)) <= 1e-5 * abs(float(ref)), (loss, float(ref))
    assert rel(grad, z.grad) <= 1e-5, rel(grad, z.grad)
    assert (grad.permute(1, 0, 2, 3)[:, (labels < 0) | (labels >= k)] == 0).all()     # uncounted pixels: zero
    # another ignore_index and a gradient scale
    lab2 = labels.clone()
    lab2[lab2 == -100] = 255
    loss2, grad2, _ = _native(logits, lab2, kind, w_point, gamma, smooth, weight, 255, grad_scale=0.25)
    assert abs(loss2 - float(ref)) <= 1e-5 * abs(float(ref))
    assert rel(grad2, 0.25 * z.grad) <= 1e-5


@pytest.mark.parametrize("kind", ["ce_dice", "softmax_focal_dice"])
def test_all_ignored_batch_gives_nan_and_a_zero_gradient(kind):
    logits = torch.randn(2, 4, 8, 8)
    labels = torch.full((2, 8, 8), -100)
    loss, grad, bad = _native(logits, labels, kind, 0.5, 2.0, 1.0, None, -100)
    assert loss != loss and bad == 0
    assert (grad == 0).all()


def test_loss_without_a_gradient_buffer():
    logits, labels, _ = _case(7, 3)
    want, _, _ = _native(logits, labels, "softmax_focal_dice", 0.5, 2.0, 1.0, None, -100)
    sums = torch.zeros(ops.DICE_SUMS, device=DEV, dtype=torch.float64)
    bad = torch.zeros(1, device=DEV, dtype=torch.int64)
    loss = torch.zeros(1, device=DEV, dtype=torch.float64)
    ops.seg_softmax_dice_loss(logits.to(DEV), labels.to(DEV), 1, 0.5, 2.0, 1.0, None, -100, sums, bad, None, 1.0, loss)
    assert float(loss) == pytest.approx(want, rel=1e-12)          # the fp64 atomics may add in another order


# ------------------------------------------------------------------------------------------------
# no host synchronisation: the engine's loss_and_grad replays inside a CUDA graph
# ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["ce_dice", "softmax_focal_dice"])
def test_loss_and_grad_replays_in_a_cuda_graph(kind):
    k, n, hw = 7, 2, 32
    eng = SiameseEngine(DEV, 3, k)
    eng._alloc(n, hw, hw)
    g = torch.Generator(device=DEV).manual_seed(9)
    lab = torch.randint(0, k, (n, hw, hw), device=DEV, generator=g)
    lab[0, 0, :4] = -100
    kw = dict(class_weight=torch.linspace(0.5, 2.0, k, device=DEV), smooth=1.0)
    eng.logits.copy_(torch.randn(eng.logits.shape, device=DEV, generator=g))
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        eng.loss_and_grad(lab, kind, **kw)                # warm-up outside the capture
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = eng.loss_and_grad(lab, kind, **kw)
    new = torch.randn(eng.logits.shape, device=DEV, generator=g) * 2
    eng.logits.copy_(new)
    graph.replay()
    torch.cuda.synchronize()
    got_loss, got_grad = float(out), eng.dlogits.clone()
    eng.dlogits.fill_(NAN)
    want_loss = float(eng.loss_and_grad(lab, kind, **kw))
    assert got_loss == pytest.approx(want_loss, rel=1e-12)         # the fp64 atomics may add in another order
    assert rel(got_grad, eng.dlogits) <= 1e-6


# ------------------------------------------------------------------------------------------------
# network level against the oracle
# ------------------------------------------------------------------------------------------------
def _fixture(k, n=2, hw=128, seed=0):
    g = torch.Generator().manual_seed(200 + k + seed)
    x1 = torch.rand(n, 3, hw, hw, generator=g) * 2 - 1
    x2 = torch.rand(n, 3, hw, hw, generator=g) * 2 - 1
    # change is rare: about 10 % of the pixels carry a class > 0
    lab = torch.randint(1, k, (n, hw, hw), generator=g) * (torch.rand(n, hw, hw, generator=g) < 0.1)
    lab[torch.rand(n, hw, hw, generator=g) < 0.05] = -100
    weight = torch.linspace(0.5, 2.0, k)
    return x1, x2, lab, weight


KINDS = {"ce_dice": (losses.CEDiceLoss, dict(alpha=0.5, smooth=1.0)),
         "softmax_focal_dice": (losses.SoftmaxFocalDiceLoss, dict(beta=0.5, gamma=2.0, smooth=1.0))}


def _torch_crit(kind, kw, weight):
    w_point = kw.get("alpha", kw.get("beta"))
    return lambda o, t: softmax_dice_ref(o.float(), t, kind, w_point, kw.get("gamma", 0.0), kw["smooth"], weight)


def _oracle(sd, x1, x2, lab, crit, bf16=False):
    sd = {kk: v.detach().clone().to(DEV) for kk, v in sd.items()}
    names = O.param_names(sd)
    for kk in names:
        sd[kk].requires_grad_(True)
    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=bf16):
        out = O.siamese_forward(sd, x1.to(DEV), x2.to(DEV), True, {})
    out = out.float()
    loss = crit(out, lab.to(DEV))
    grads = torch.autograd.grad(loss, [sd[kk] for kk in names])
    return out.detach(), float(loss), torch.cat([gg.reshape(-1) for gg in grads]).detach(), names


@pytest.mark.parametrize("k", [2, 7])
@pytest.mark.parametrize("kind", ["ce_dice", "softmax_focal_dice"])
def test_engine_and_dropin_match_the_oracle(k, kind):
    x1, x2, lab, weight = _fixture(k)
    cls, kw = KINDS[kind]
    tcrit = _torch_crit(kind, kw, weight.to(DEV))
    torch.manual_seed(0)
    m = M.SiameseUNet(3, k)
    sd0 = {kk: v.detach().clone() for kk, v in m.state_dict().items()}
    ref_out, ref_loss, ref_g, names = _oracle(sd0, x1, x2, lab, tcrit)
    y_out, y_loss, y_g, _ = _oracle(sd0, x1, x2, lab, tcrit, bf16=True)
    yard_out, yard_g = rel(y_out, ref_out), rel(y_g, ref_g)
    yard_loss = max(abs(y_loss - ref_loss), 1e-3 * abs(ref_loss))
    # drop-in module with the native criterion and AdamW
    m = m.to(DEV)
    m.train()
    crit = cls(weight=weight, **kw).to(DEV)
    opt = torch.optim.AdamW(m.parameters(), lr=1.0152e-4, weight_decay=1.118e-5)
    got_losses = []
    for step in range(3):
        opt.zero_grad()
        out = m(x1.to(DEV), x2.to(DEV))
        loss = crit(out, lab.to(DEV))
        assert loss.dim() == 0 and loss.dtype == torch.float32
        loss.backward()
        if step == 0:
            assert rel(out.detach(), ref_out) < 1.5 * yard_out, (rel(out.detach(), ref_out), yard_out)
            assert abs(float(loss) - ref_loss) < 1.5 * yard_loss, (float(loss), ref_loss, yard_loss)
            got_g = torch.cat([dict(m.named_parameters())[kk].grad.reshape(-1) for kk in names])
            assert rel(got_g, ref_g) < 1.5 * yard_g, (rel(got_g, ref_g), yard_g)
        opt.step()
        got_losses.append(float(loss))
    assert int(crit.bad_labels) == 0
    # the oracle's own three steps (fp32, same AdamW)
    sd = {kk: v.clone().to(DEV) for kk, v in sd0.items()}
    ost = O.AdamState(sd, O.param_names(sd), 1.0152e-4, (0.9, 0.999), 1e-8, 1.118e-5, decoupled=True)
    want = [O.siamese_train_step(sd, ost, x1.to(DEV), x2.to(DEV), lab.to(DEV), criterion=tcrit) for _ in range(3)]
    for got_l, ref_l in zip(got_losses, want):
        assert abs(got_l - ref_l) < max(1.5 * yard_loss, 3e-2 * ref_l), (got_losses, want)
    # the engine's fused step gives the drop-in loop's losses
    eng = SiameseEngine(DEV, 3, k)
    eng.load_state_dict(sd0)
    seq = [float(eng.train_step(x1.to(DEV), x2.to(DEV), lab.to(DEV), kind=kind, class_weight=weight.tolist(),
                                **kw).cpu()) for _ in range(3)]
    assert seq == pytest.approx(got_losses, rel=2e-3)
    assert int(eng.bad_labels) == 0


def test_criterion_without_grad_and_with_a_scaled_backward():
    logits, labels, _ = _case(3, 5)
    crit = losses.SoftmaxFocalDiceLoss(beta=0.3, gamma=0.5, weight=[1.0, 2.0, 0.5]).to(DEV)
    lg = logits.to(DEV)
    with torch.no_grad():
        a = crit(lg, labels.to(DEV))
    z = lg.clone().requires_grad_(True)
    b = crit(z, labels.to(DEV))
    (3.0 * b).backward()
    assert float(a) == pytest.approx(float(b), rel=1e-6)
    zr = logits.double().requires_grad_(True)
    clean = labels.clone()
    clean[(clean < 0) | (clean >= 3)] = -100
    ref = softmax_dice_ref(zr, clean, "softmax_focal_dice", 0.3, 0.5, 1.0, torch.tensor([1.0, 2.0, 0.5]).double())
    (3.0 * ref).backward()
    assert abs(float(b) - float(ref)) <= 1e-5 * abs(float(ref))
    assert rel(z.grad.cpu(), zr.grad) <= 1e-5
    assert int(crit.bad_labels) == 10                  # five planted labels, counted by both calls


@pytest.mark.parametrize("kind", ["ce_dice", "softmax_focal_dice"])
def test_batch4_512_step_is_finite_and_matches_the_oracle_loss(kind):
    k = 7
    x1, x2, lab, weight = _fixture(k, n=4, hw=512, seed=1)
    _, kw = KINDS[kind]
    tcrit = _torch_crit(kind, kw, weight.to(DEV))
    torch.manual_seed(0)
    sd0 = {kk: v.detach().clone() for kk, v in M.SiameseUNet(3, k).state_dict().items()}
    with torch.no_grad():
        ref = tcrit(O.siamese_forward({kk: v.to(DEV) for kk, v in sd0.items()}, x1.to(DEV), x2.to(DEV), True, {}),
                    lab.to(DEV))
        with torch.autocast("cuda", dtype=torch.bfloat16):
            yo = O.siamese_forward({kk: v.to(DEV) for kk, v in sd0.items()}, x1.to(DEV), x2.to(DEV), True, {})
        yard = tcrit(yo.float(), lab.to(DEV))
    eng = SiameseEngine(DEV, 3, k)
    eng.load_state_dict(sd0)
    loss = float(eng.train_step(x1.to(DEV), x2.to(DEV), lab.to(DEV), kind=kind, class_weight=weight, **kw).cpu())
    assert torch.isfinite(eng.store.p).all() and torch.isfinite(eng.logits).all()
    bound = 1.5 * max(abs(float(yard) - float(ref)), 1e-3 * float(ref))
    assert abs(loss - float(ref)) < bound, (loss, float(ref), float(yard))
