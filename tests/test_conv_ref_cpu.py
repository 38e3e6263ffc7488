"""The per-element bound of tests/conv_ref.py on both sides, without a GPU: it accepts a CPU emulation of the
implicit-GEMM kernels (fp32 accumulation from the bf16 operands, then round-to-nearest-even to bf16) on every geometry
and epilogue the GPU tests use, and it rejects small, local mutations of that emulation at the largest K those tests
use (8192 = 16 taps x 512 channels; 4096 = 4 taps x 1024 channels for the four-phase geometry)."""
import pytest
import torch
import torch.nn.functional as F
from torch.nn import grad as G

import conv_ref as R
from gan_aug_pfa_b200 import ops

SMS = 148


def _bf(t):
    return t.to(torch.bfloat16)


def _emul_conv(x, w, stride, pad):
    return _bf(R.nhwc(F.conv2d(x.float(), w.float(), None, stride, pad)))


def _rand(g, *shape, scale=1.0):
    return _bf(torch.randn(*shape, generator=g) * scale)


def _rejects(got, exp, what):
    with pytest.raises(AssertionError, match="outside the bound"):
        R.assert_within(got, exp, what)


@pytest.fixture(scope="module")
def k8192():
    """Conv2d 512 -> 64, k4 s1 p1, 17x17 -> 16x16 (two 16 x 8 M tiles), batch 1: K = 8192."""
    g = torch.Generator().manual_seed(1)
    x = _rand(g, 1, 512, 17, 17)
    w = _rand(g, 64, 512, 4, 4, scale=(16 * 512) ** -0.5)
    exp = R.Expect(*R.conv_fwd(x, w, 1, 1))
    return x, w, exp, _emul_conv(x, w, 1, 1)


def _tile0_pixels(n, gh, gw, ctot, n_out):
    """[n, gh, gw] bool: the output points of M tile 0 under the host code's tile shape."""
    cfg = R.fprop_config(n, gh, gw, ops.geom_conv_fwd(4, 1, 1), n_out, ctot, SMS)
    bw, bh = 1 << cfg["log_bw"], 1 << cfg["log_bh"]
    m = torch.zeros(n, gh, gw, dtype=torch.bool)
    m[:cfg["bni"], :bh, :bw] = True
    assert int(m.sum()) == 128
    return m


def test_bound_accepts_the_emulation_at_k8192(k8192):
    x, w, exp, got = k8192
    worst = R.assert_within(got, exp, "emulation")
    assert worst <= 1.0


def test_bound_rejects_one_zeroed_chunk_of_one_tile(k8192):
    x, w, exp, got = k8192
    bad = got.clone()
    tile = _tile0_pixels(1, 16, 16, 512, 64)
    bad[..., 16:32][tile] = 0
    _rejects(bad, exp, "zeroed chunk")


def test_bound_rejects_one_dropped_k_slice_in_one_chunk_of_one_tile(k8192):
    """The smallest K error a tile bug makes: one tap's 64-channel slice missing from one 16-column chunk of one
    128-pixel M tile, 1/128 of K."""
    x, w, exp, got = k8192
    wm = w.clone()
    wm[16:32, 128:192, 2, 1] = 0
    mut = _emul_conv(x, wm, 1, 1)
    bad = got.clone()
    tile = _tile0_pixels(1, 16, 16, 512, 64)
    bad[..., 16:32][tile] = mut[..., 16:32][tile]
    assert int((bad != got).sum()) > 0
    _rejects(bad, exp, "dropped K slice")


def test_bound_rejects_one_row_shifted_by_one_pixel(k8192):
    x, w, exp, got = k8192
    bad = got.clone()
    bad[0, 4] = torch.roll(got[0, 4], 1, dims=0)
    _rejects(bad, exp, "shifted row")


def test_bound_rejects_one_phase_with_swapped_taps():
    """ConvTranspose2d 1024 -> 64 through the four phases (K = 4 taps x 1024): phase (0, *) reads kernel rows 3 and 1
    for its taps th = 0 and 1; swapping them changes only the even output rows."""
    g = torch.Generator().manual_seed(2)
    x = _rand(g, 1, 1024, 6, 6)
    w = _rand(g, 1024, 64, 4, 4, scale=(4 * 1024) ** -0.5)
    exp = R.Expect(*R.convT_fwd(x, w))
    got = _bf(R.nhwc(F.conv_transpose2d(x.float(), w.float(), None, 2, 1)))
    R.assert_within(got, exp, "emulation")
    ws = w.clone()
    ws[:, :, [1, 3]] = w[:, :, [3, 1]]
    swapped = _bf(R.nhwc(F.conv_transpose2d(x.float(), ws.float(), None, 2, 1)))
    bad = got.clone()
    bad[:, 0::2] = swapped[:, 0::2]
    assert torch.equal(bad[:, 1::2], got[:, 1::2])
    _rejects(bad, exp, "swapped phase taps")


def test_guard_check_rejects_one_changed_guard_element():
    for lo, hi, where in ((16, 48, "past the slot"), (8, 32, "before the slot")):
        gb = R.Guarded((2, 3, 5, 272), torch.bfloat16, "cpu", lo=lo, hi=hi, fill=float("nan"), guard_fill=R.SENTINEL)
        gb.view.copy_(torch.randn(2, 3, 5, 272))
        gb.check("untouched")
        if where == "past the slot":
            gb.buf[2, 1, 3, lo + 272 + 5] = 0.0
        else:
            gb.buf[1, 2, 0, lo - 1] = R.SENTINEL / 2
        with pytest.raises(AssertionError, match=where):
            gb.check("mutated")
    gb = R.Guarded((4, 16, 64), torch.float32, "cpu", lo=0, hi=16)
    gb.view.zero_()
    gb.buf[-1, 0, 0] += 1.0         # the guard row after the slot
    with pytest.raises(AssertionError, match="guard entry after"):
        gb.check("fp32 rows")


# ---- the bound accepts the emulation of every geometry and epilogue the GPU tests use ------------------------------
def test_bound_accepts_every_geometry():
    g = torch.Generator().manual_seed(3)
    x = _rand(g, 3, 128, 12, 10)
    for k, s, p in ((1, 1, 0), (3, 1, 1), (4, 1, 1), (4, 2, 1)):
        w = _rand(g, 80, 128, k, k, scale=(k * k * 128) ** -0.5)
        R.assert_within(_emul_conv(x, w, s, p), R.Expect(*R.conv_fwd(x, w, s, p)), f"k{k}s{s}")
    # stride-1 and stride-2 dgrad (the second is the four-phase geometry)
    w = _rand(g, 128, 48, 4, 4, scale=(16 * 128) ** -0.5)
    for s, hw in ((1, (13, 11)), (2, (24, 20))):
        got = _bf(R.nhwc(G.conv2d_input((3, 48) + hw, w.float(), x.float(), s, 1)))
        R.assert_within(got, R.Expect(*R.conv_dgrad(x, w, hw, s, 1)), f"dgrad s{s}")
    # weight gradient: fp32 output, K = pixels
    dy = _rand(g, 3, 64, 6, 5)
    got = G.conv2d_weight(x.float(), (64, 128, 4, 4), dy.float(), 2, 1).permute(0, 2, 3, 1).reshape(64, 16, 128)
    R.assert_within(got, R.Expect(*R.wgrad(x, dy, 4, 2, 1)), "wgrad", dtype=torch.float32)


def test_bound_accepts_every_epilogue():
    g = torch.Generator().manual_seed(4)
    x = _rand(g, 2, 256, 8, 8)
    w = _rand(g, 96, 256, 3, 3, scale=(9 * 256) ** -0.5)
    acc = R.nhwc(F.conv2d(x.float(), w.float(), None, 1, 1))            # fp32 accumulator
    base = R.Expect(*R.conv_fwd(x, w, 1, 1))
    sc, b = torch.rand(96, generator=g) + 0.5, torch.randn(96, generator=g)
    v = acc * sc + b
    e = base.scale(sc).bias(b)
    for act, fn in ((0, lambda t: t), (1, lambda t: F.leaky_relu(t, 0.2)), (2, F.relu), (3, torch.tanh),
                    (4, torch.sigmoid)):
        R.assert_within(_bf(fn(v)), e.act(act), f"act {act} bf16")
        R.assert_within(fn(v), e.act(act), f"act {act} fp32")
    prev = _rand(g, *acc.shape)
    R.assert_within(_bf(acc + prev.float()), base.accumulate(prev), "accumulate")
    # backward-fused: d = mask ? g + g2 : slope * g from the fp32 accumulator, one rounding
    y, g2 = _rand(g, *acc.shape), _rand(g, *acc.shape)
    bsc, bsh = torch.rand(96, generator=g) + 0.5, torch.randn(96, generator=g) * 0.3
    d = torch.where(y.float() * bsc + bsh > 0, acc + g2.float(), 0.2 * acc)
    taken, other, amb = base.bwd(y, 0.2, bsc, bsh, g2)
    R.assert_within(_bf(d), taken, "bwd", alt=(other, amb))
    # a mask decision taken the other way on an unambiguous element is rejected
    i = int(((~amb) & (y.float() * bsc + bsh > 0)).flatten().nonzero()[0])
    bad = _bf(d).flatten().clone()
    bad[i] = _bf(0.2 * acc.flatten()[i])
    if abs(float(acc.flatten()[i] + g2.float().flatten()[i] - 0.2 * acc.flatten()[i])) > 1e-2:
        _rejects(bad.view_as(d), taken, "flipped mask")


def test_stats_check_both_sides():
    g = torch.Generator().manual_seed(5)
    out = _rand(g, 4, 6, 6, 48)
    o = out.double().reshape(-1, 48)
    st = torch.cat([o.sum(0), (o * o).sum(0)])
    R.assert_stats(st, out)
    st[48 + 7] *= 1 + 1e-4
    with pytest.raises(AssertionError, match="channel 7"):
        R.assert_stats(st, out)


def test_config_mirror_branches():
    """The host-code mirror reproduces the configurations the GPU cases name (148 SMs)."""
    c = R.fprop_config(5, 4, 4, ops.geom_conv_fwd(4, 2, 1), 512, 512, SMS)
    assert (c["block_n"], c["mt"], c["halo"]) == (64, 1, False)
    c = R.fprop_config(2, 20, 20, ops.geom_conv_fwd(3, 1, 1), 64, 64, SMS)
    assert (c["halo"], c["log_bw"], c["log_bh"]) == (True, 4, 3)
    c = R.fprop_config(2, 20, 12, ops.geom_conv_fwd(3, 1, 1), 64, 64, SMS)
    assert (c["halo"], c["log_bw"], c["log_bh"]) == (True, 3, 4)
    c = R.fprop_config(2, 20, 20, ops.geom_conv_fwd(3, 1, 1), 128, 64, SMS)
    assert not c["halo"]
    assert R.fprop_config(1, 8, 8, ops.geom_phase_k4s2p1(), 272, 256, SMS)["block_n"] == 144
    assert R.fprop_config(1, 8, 8, ops.geom_phase_k4s2p1(), 640, 256, SMS)["block_n"] == 224
    assert R.wgrad_config(512, 320, 16) == dict(block_n=256, mt=2, tpc=1)
