"""Every launch configuration of the implicit-GEMM engine against fp64, element by element (tests/conv_ref.py).

gap_conv_gemm picks, from the shape, the M tile shape (several images per tile, one row per tile, tall and narrow,
halo 16x8 / 8x16), the N tile (block_n, n_tiles, the under-filled cost model), two M tiles per item and the
accumulator stages, CTA pairs, the store path (vec_ok 2 / 1 / 0, fast or generic) and one of three epilogues
(<0> plain, <1> backward-fused, <2> accumulate); gap_conv_wgrad picks block_n, mt, taps per CTA, split-K, one or two
producer lanes and the vector or scalar reduction.  Each case below names the branch it is there for; knobs force the
branches no small shape reaches, and the fixture restores the defaults.

Every output, and every y / g2 / prev / source operand, is a channel slot of a wider buffer with guard channels on
both sides and a guard image before and after (conv_ref.Guarded): a stray write lands in memory the test owns and shows
up as a changed guard.  Outputs start as NaN, so an element the kernel never writes fails the fp64 comparison.  A
failure names the element, its M tile and N tile under the host code's choice (conv_ref.fprop_config), and the ratio
of its error to its bound."""
import pytest
import torch

pytestmark = pytest.mark.gpu

from gan_aug_pfa_b200 import _lib, ops  # noqa: E402
import conv_ref as R  # noqa: E402
from test_gpu_conv import pack_conv, pack_phase  # noqa: E402

DEV = "cuda:0"
NAN = float("nan")
DEVICE_REF_MACS = 1e8      # larger references run in fp64 on the device, to keep the CPU time bounded


@pytest.fixture
def restore_knobs():
    """Restores every launch knob to its default after a test that forces some (run_fprop / run_wgrad knobs=...)."""
    yield
    for k, v in {**R.FPROP_DEFAULTS, **R.WGRAD_DEFAULTS}.items():
        _lib.debug_set(k, v)


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _bf(t):
    return t.to(torch.bfloat16)


def _hi(lo, c, mult=8, extra=128):
    """Right guard width: at least `extra` channels (a stray chunk of up to 112 columns stays inside) and a row length
    that is a multiple of `mult`."""
    return extra + (-(lo + c + extra)) % mult


def _slot(shape, dtype, align, fill, guard=R.SENTINEL):
    """A guarded NHWC slot whose first element is `align` bytes aligned (and no more) and whose row length is a multiple
    of 16 elements when align == 32, else of 8."""
    lo = align // torch.tensor([], dtype=dtype).element_size()
    return R.Guarded(shape, dtype, DEV, lo=lo, hi=_hi(lo, shape[-1], 16 if align == 32 else 8), fill=fill,
                     guard_fill=guard)


def _source(x_nhwc, align=16):
    """The source operand as a slot of a wider NaN-guarded buffer: src_ld > src_c."""
    gb = R.Guarded(tuple(x_nhwc.shape), torch.bfloat16, DEV, lo=8 if align == 16 else 16, hi=56, fill=NAN,
                   guard_fill=NAN)
    gb.view.copy_(x_nhwc)
    return gb


# ---- geometries: NCHW operands, packed weights, grid, output size and the fp64 reference --------------------------
def _problem(kind, n, cin, n_out, h, w, g):
    if kind in ("k1", "k3s1", "k4s1", "k4s2", "convT_dgrad"):
        k, s, p = {"k1": (1, 1, 0), "k3s1": (3, 1, 1), "k4s1": (4, 1, 1), "k4s2": (4, 2, 1),
                   "convT_dgrad": (4, 2, 1)}[kind]
        x = _bf(torch.randn(n, cin, h, w, generator=g))
        wt = _bf(torch.randn(n_out, cin, k, k, generator=g) / (k * k * cin) ** 0.5)
        oh, ow = (h + 2 * p - k) // s + 1, (w + 2 * p - k) // s + 1
        return dict(x=x, wpk=pack_conv(wt), geom=ops.geom_conv_fwd(k, s, p), grid=(oh, ow), out_hw=(oh, ow),
                    ref=lambda xx, ww=wt: R.conv_fwd(xx, ww.to(xx.device), s, p), macs=n * oh * ow * n_out * k * k * cin)
    if kind == "dgrad_s1":         # x plays dY of a Conv2d(n_out -> cin, k4, s1, p1) over an (h+1) x (w+1) input
        x = _bf(torch.randn(n, cin, h, w, generator=g))
        wt = _bf(torch.randn(cin, n_out, 4, 4, generator=g) / (16 * cin) ** 0.5)
        wf = wt.flip(2, 3).permute(1, 2, 3, 0).reshape(1, n_out, 16 * cin).contiguous()
        hw = (h + 1, w + 1)
        return dict(x=x, wpk=wf, geom=ops.geom_conv_dgrad_s1(4, 1), grid=hw, out_hw=hw,
                    ref=lambda xx, ww=wt: R.conv_dgrad(xx, ww.to(xx.device), hw, 1, 1),
                    macs=n * hw[0] * hw[1] * n_out * 16 * cin)
    if kind in ("phase", "dgrad_s2"):   # ConvTranspose2d forward == Conv2d(n_out -> cin, k4 s2 p1) dgrad
        x = _bf(torch.randn(n, cin, h, w, generator=g))
        wt = _bf(torch.randn(cin, n_out, 4, 4, generator=g) / (4 * cin) ** 0.5)
        return dict(x=x, wpk=pack_phase(wt.permute(1, 0, 2, 3)), geom=ops.geom_phase_k4s2p1(), grid=(h, w),
                    out_hw=(2 * h, 2 * w), ref=lambda xx, ww=wt: R.convT_fwd(xx, ww.to(xx.device)),
                    macs=n * h * w * 4 * n_out * 4 * cin)
    raise ValueError(kind)


def run_fprop(kind, n, cin, n_out, h, w, *, seed=0, srcs=1, act=0, act2=None, bias=False, scale=False, stats=False,
              accumulate=False, out_f32=False, align=32, bwd=None, knobs=None, expect=None):
    """One gap_conv_gemm launch inside guard bands, checked element by element against fp64.  bwd = dict(c0, bn, g2,
    ld32) selects the backward-fused epilogue; expect = {config key: value} asserts the host code's choice (mirror)."""
    g = torch.Generator().manual_seed(seed)
    pr = _problem(kind, n, cin, n_out, h, w, g)
    cfg = R.fprop_config(n, pr["grid"][0], pr["grid"][1], pr["geom"], n_out, cin, _sms(), accumulate, knobs)
    for k, v in (expect or {}).items():
        assert cfg[k] == v, f"the case no longer reaches its branch: {k} = {cfg[k]}, wanted {v} ({cfg})"
    xd = R.nhwc(pr["x"]).to(DEV)
    if srcs == 2:
        c1 = 64 if cin > 64 else cin // 2
        sources = [_source(xd[..., :c1]), _source(xd[..., c1:], align=32)]
    else:
        sources = [_source(xd)]
    oh, ow = pr["out_hw"]
    odt = torch.float32 if out_f32 else torch.bfloat16
    prev = _bf(torch.randn(n, oh, ow, n_out, generator=g)) if accumulate else None
    out = _slot((n, oh, ow, n_out), odt, align, NAN)
    if accumulate:
        out.view.copy_(prev.to(DEV))
    out2 = _slot((n, oh, ow, n_out), torch.bfloat16, align, NAN) if act2 is not None else None
    sc = (torch.rand(n_out, generator=g) + 0.5) if scale else None
    b = torch.randn(n_out, generator=g) if bias else None
    c0 = bwd.get("c0", 0) if bwd else 0
    nb = n_out - c0
    st = None
    if stats:
        st = R.Guarded((1, 2 * nb), torch.float64, DEV, lo=16, hi=16, fill=0.0)
    kw = {}
    guards = [("out", out)] + [(f"src{i}", s) for i, s in enumerate(sources)]
    if bwd is not None:
        ya = 32 if bwd.get("ld32", True) else 16
        y = _bf(torch.randn(n, oh, ow, nb, generator=g))
        yb = _slot((n, oh, ow, nb), torch.bfloat16, ya, NAN, guard=NAN)
        yb.view.copy_(y.to(DEV))
        guards.append(("y", yb))
        d = dict(y=yb.view, slope=0.2, c0=c0)
        bsc = bsh = g2 = None
        if bwd.get("bn", True):
            bsc, bsh = torch.rand(nb, generator=g) + 0.5, torch.randn(nb, generator=g) * 0.3
            d.update(scale=bsc.to(DEV), shift=bsh.to(DEV))
        if bwd.get("g2", True):
            g2 = _bf(torch.randn(n, oh, ow, nb, generator=g))
            gb2 = _slot((n, oh, ow, nb), torch.bfloat16, ya, NAN, guard=NAN)
            gb2.view.copy_(g2.to(DEV))
            guards.append(("g2", gb2))
            d["g2"] = gb2.view
        kw["bwd"] = d
    if knobs:
        for k_, v_ in knobs.items():
            _lib.debug_set(k_, v_)
    ops.conv_gemm([s.view for s in sources], pr["wpk"].to(DEV), pr["geom"], out.view, n_out, pr["grid"], act=act,
                  out2=out2.view if out2 else None, act2=act2 if act2 is not None else 0,
                  bias=b.to(DEV) if bias else None, stats=st.view.reshape(-1) if stats else None,
                  scale=sc.to(DEV) if scale else None, accumulate=accumulate, **kw)
    torch.cuda.synchronize()
    for name, gb in guards + ([("out2", out2)] if out2 else []) + ([("stats", st)] if st else []):
        gb.check(f"{name} guard")

    ref_dev = DEV if pr["macs"] > DEVICE_REF_MACS else "cpu"
    base = R.Expect(*pr["ref"](pr["x"].to(ref_dev)))
    locate = R.fprop_locator(cfg, pr["geom"].n_phase)
    got = out.view
    if bwd is not None:
        lo = R.Expect(base.ref[..., :c0], base.s[..., :c0])
        taken, other, amb = R.Expect(base.ref[..., c0:], base.s[..., c0:]).bwd(y, 0.2, bsc, bsh, g2)
        cat = lambda a, b_: torch.cat([a, b_], -1)  # noqa: E731
        exp = R.Expect(cat(lo.ref, taken.ref), cat(lo.s, taken.s))
        alt = R.Expect(cat(lo.ref, other.ref), cat(lo.s, other.s))
        mask = cat(torch.zeros_like(lo.ref, dtype=torch.bool), amb)
        R.assert_within(got, exp, f"{kind} backward-fused output", locate=locate, alt=(alt, mask))
        assert float(amb.double().mean()) < 0.01
        if stats:
            R.assert_stats(st.view.reshape(-1), got[..., c0:], y, "backward-fused stats")
        return cfg
    e = base
    if scale:
        e = e.scale(sc)
    if bias:
        e = e.bias(b)
    e1 = e.act(act)
    if accumulate:
        e1 = e1.accumulate(prev)
    R.assert_within(got, e1, f"{kind} output", locate=locate)
    if out2:
        R.assert_within(out2.view, e.act(act2), f"{kind} out2", locate=locate)
    if stats:
        assert act == 0
        R.assert_stats(st.view.reshape(-1), got, None, "stats")
    return cfg


LRELU, RELU, TANH, SIGMOID = ops.ACT_LRELU, ops.ACT_RELU, ops.ACT_TANH, ops.ACT_SIGMOID

FPROP_CASES = [
    # ---- M tile shape (log_bw / log_bh / images per tile)
    ("mtile_gw_ge_128_one_row_per_tile", dict(kind="k1", n=1, cin=64, n_out=64, h=3, w=130,
                                              expect=dict(log_bw=7, log_bh=0))),
    ("mtile_gw_le_3_tall_narrow", dict(kind="k3s1", n=2, cin=64, n_out=48, h=40, w=3,
                                       expect=dict(log_bw=2, log_bh=5, halo=False))),
    ("mtile_32_images_per_tile_n_not_multiple", dict(kind="k4s2", n=37, cin=128, n_out=80, h=4, w=4,
                                                     expect=dict(bni=32))),
    ("mtile_1x1_grid_128_images_per_tile", dict(kind="k4s2", n=130, cin=64, n_out=64, h=2, w=2,
                                                expect=dict(bni=128))),
    ("halo_16x8", dict(kind="k3s1", n=2, cin=128, n_out=64, h=20, w=20, expect=dict(halo=True, log_bw=4))),
    ("halo_8x16", dict(kind="k3s1", n=2, cin=64, n_out=48, h=20, w=12, expect=dict(halo=True, log_bw=3))),
    ("halo_stride2_two_groups", dict(kind="k4s2", n=2, cin=64, n_out=128, h=34, w=40, expect=dict(halo=True))),
    ("halo_dgrad_s1_four_taps", dict(kind="dgrad_s1", n=2, cin=64, n_out=64, h=17, w=19, expect=dict(halo=True))),
    ("halo_phase", dict(kind="phase", n=2, cin=128, n_out=64, h=10, w=16, expect=dict(halo=True))),
    ("halo_off_npad_times_taps_gt_256", dict(kind="k3s1", n=2, cin=64, n_out=128, h=20, w=20,
                                             expect=dict(halo=False))),
    ("halo_knob_off", dict(kind="k3s1", n=2, cin=128, n_out=64, h=20, w=20, knobs=dict(fprop_halo=0),
                           expect=dict(halo=False))),
    # ---- N tile (block_n = roundup16(n_pad / n_tiles); the under-filled cost model)
    ("ntile_16", dict(kind="k1", n=3, cin=64, n_out=16, h=9, w=14, expect=dict(block_n=16))),
    ("ntile_144", dict(kind="k3s1", n=2, cin=64, n_out=144, h=12, w=20, expect=dict(block_n=144))),
    ("ntile_256_full_launch", dict(kind="k1", n=37, cin=64, n_out=256, h=32, w=32, expect=dict(block_n=256))),
    ("ntile_272_two_tiles_of_144", dict(kind="k1", n=3, cin=64, n_out=272, h=10, w=10,
                                        expect=dict(block_n=144, n_tiles=2))),
    ("ntile_640_three_tiles_of_224", dict(kind="k4s2", n=2, cin=128, n_out=640, h=8, w=12,
                                          expect=dict(block_n=224, n_tiles=3))),
    ("ntile_1024", dict(kind="k1", n=10, cin=64, n_out=1024, h=32, w=32, expect=dict(block_n=256, n_tiles=4))),
    ("costmodel_block_n_64_512to512_4x4_batch5", dict(kind="k4s2", n=5, cin=512, n_out=512, h=8, w=8,
                                                      expect=dict(block_n=64, mt=1))),
    ("costmodel_block_n_128", dict(kind="k4s2", n=32, cin=64, n_out=1024, h=16, w=16,
                                   expect=dict(block_n=128, halo=False))),
    ("costmodel_mt2_one_acc_stage", dict(kind="phase", n=4, cin=64, n_out=512, h=32, w=32,
                                         expect=dict(mt=2, block_n=256, acc_stages=1))),
    ("costmodel_mt2_two_acc_stages", dict(kind="k1", n=32, cin=64, n_out=128, h=32, w=32,
                                          expect=dict(mt=2, block_n=128, acc_stages=2))),
    ("forced_block_n_64", dict(kind="k4s1", n=2, cin=128, n_out=256, h=9, w=11, knobs=dict(fprop_block_n=64),
                               expect=dict(block_n=64, n_tiles=4))),
    ("forced_block_n_128_ragged_last_tile", dict(kind="k1", n=3, cin=64, n_out=144, h=10, w=10,
                                                 knobs=dict(fprop_block_n=128), expect=dict(block_n=128, n_tiles=2))),
    ("forced_mt2_odd_m_tiles_missing_partner", dict(kind="k3s1", n=3, cin=64, n_out=128, h=20, w=20,
                                                    knobs=dict(fprop_mt=2), expect=dict(mt=2, m_tiles_pp=15))),
    ("forced_mt2_block_n_256_one_acc_stage", dict(kind="k4s1", n=3, cin=128, n_out=256, h=17, w=17,
                                                  knobs=dict(fprop_mt=2, fprop_block_n=256), expect=dict(mt=2, acc_stages=1))),
    ("forced_mt1", dict(kind="k1", n=32, cin=64, n_out=128, h=32, w=32, knobs=dict(fprop_mt=1),
                        expect=dict(mt=1))),
    ("forced_two_stages_long_k", dict(kind="k4s2", n=2, cin=512, n_out=256, h=16, w=16,
                                      knobs=dict(fprop_stages=2))),
    ("forced_pairs_ntile_144", dict(kind="k1", n=25, cin=64, n_out=144, h=32, w=32, knobs=dict(fprop_pair=2, fprop_mt=1),
                                    expect=dict(pair=True))),
    # ---- store paths and epilogue <0>
    ("store_vec_ok_1_generic", dict(kind="k3s1", n=2, cin=64, n_out=80, h=12, w=9, align=16, act=LRELU)),
    ("store_vec_ok_0_generic", dict(kind="k3s1", n=2, cin=64, n_out=80, h=12, w=9, align=8, act=RELU)),
    ("store_out2_fast", dict(kind="k4s2", n=2, cin=128, n_out=64, h=16, w=16, act=LRELU, act2=RELU)),
    ("store_out2_generic", dict(kind="k4s2", n=2, cin=128, n_out=64, h=16, w=16, align=16, act=LRELU, act2=RELU)),
    ("store_tanh_bf16_generic", dict(kind="phase", n=2, cin=128, n_out=48, h=6, w=7, act=TANH, bias=True)),
    ("store_sigmoid_bf16_generic", dict(kind="k3s1", n=2, cin=64, n_out=16, h=9, w=9, act=SIGMOID, bias=True)),
    ("store_fp32_tanh", dict(kind="k4s2", n=2, cin=128, n_out=64, h=16, w=16, act=TANH, out_f32=True)),
    ("store_fp32_identity_bias", dict(kind="k1", n=2, cin=64, n_out=48, h=8, w=8, bias=True, out_f32=True)),
    ("epi0_bias_scale_stats", dict(kind="k4s2", n=3, cin=128, n_out=272, h=16, w=16, bias=True, scale=True,
                                   stats=True)),
    ("epi0_stats_halo", dict(kind="k3s1", n=2, cin=64, n_out=64, h=20, w=20, stats=True, expect=dict(halo=True))),
    # ---- epilogue <2> (accumulate)
    ("epi2_accumulate_vector", dict(kind="k3s1", n=2, cin=64, n_out=64, h=20, w=20, accumulate=True, act=LRELU)),
    ("epi2_accumulate_scalar_ragged_chunk", dict(kind="k1", n=2, cin=64, n_out=24, h=8, w=8, accumulate=True)),
    ("epi2_accumulate_unaligned", dict(kind="k1", n=2, cin=128, n_out=64, h=8, w=8, accumulate=True, align=16)),
    # ---- geometries: two sources (src_ld > src_c for every source)
    ("two_sources_k3s1", dict(kind="k3s1", n=2, cin=192, n_out=64, h=12, w=12, srcs=2)),
    ("two_sources_phase", dict(kind="phase", n=2, cin=256, n_out=128, h=8, w=8, srcs=2)),
    ("two_sources_convT_dgrad", dict(kind="convT_dgrad", n=2, cin=128, n_out=256, h=16, w=16, srcs=2)),
]


@pytest.mark.parametrize("case", [c for _, c in FPROP_CASES], ids=[i for i, _ in FPROP_CASES])
def test_fprop_config(case, restore_knobs):
    run_fprop(**case)


# ---- epilogue <1>: backward-fused (activation + BatchNorm backward on channels >= c0) ------------------------------
BWD_CASES = [
    ("n128_bn_g2_c0_0", dict(kind="dgrad_s2", n=3, cin=128, n_out=128, h=8, w=8, bwd=dict(c0=0))),
    ("n256_dgrad_s1_c0_64", dict(kind="dgrad_s1", n=2, cin=128, n_out=256, h=9, w=9, bwd=dict(c0=64))),
    ("n272_bn_g2_c0_0", dict(kind="dgrad_s2", n=2, cin=128, n_out=272, h=8, w=8, bwd=dict(c0=0),
                             expect=dict(block_n=144, n_tiles=2))),
    ("n272_no_bn_no_g2_c0_64", dict(kind="dgrad_s2", n=2, cin=128, n_out=272, h=8, w=8,
                                    bwd=dict(c0=64, bn=False, g2=False))),
    ("n272_c0_160_across_n_tiles", dict(kind="dgrad_s2", n=2, cin=128, n_out=272, h=8, w=8, bwd=dict(c0=160))),
    ("n272_ld32_off", dict(kind="dgrad_s2", n=2, cin=128, n_out=272, h=8, w=8, bwd=dict(c0=0, ld32=False))),
    ("n272_convT_dgrad_no_g2", dict(kind="convT_dgrad", n=2, cin=256, n_out=272, h=12, w=12,
                                    bwd=dict(c0=0, g2=False))),
    ("n640_bn_g2_c0_0", dict(kind="dgrad_s2", n=2, cin=128, n_out=640, h=8, w=8, bwd=dict(c0=0),
                             expect=dict(block_n=224, n_tiles=3))),
    ("n640_no_bn_c0_64_ld32_off", dict(kind="dgrad_s2", n=2, cin=128, n_out=640, h=8, w=8,
                                       bwd=dict(c0=64, bn=False, ld32=False))),
    ("n640_dgrad_s1", dict(kind="dgrad_s1", n=2, cin=128, n_out=640, h=7, w=9, bwd=dict(c0=0, g2=False))),
    ("n272_pairs", dict(kind="dgrad_s2", n=40, cin=64, n_out=272, h=16, w=16, bwd=dict(c0=0),
                        knobs=dict(fprop_pair=2), expect=dict(pair=True, block_n=144))),
    ("n640_pairs_c0_64", dict(kind="dgrad_s2", n=16, cin=64, n_out=640, h=16, w=16, bwd=dict(c0=64),
                              knobs=dict(fprop_pair=2), expect=dict(pair=True, block_n=224))),
]


@pytest.mark.parametrize("case", [c for _, c in BWD_CASES], ids=[i for i, _ in BWD_CASES])
def test_backward_fused_epilogue(case, restore_knobs):
    run_fprop(stats=True, **case)


# ---- weight gradient ------------------------------------------------------------------------------------------------
def run_wgrad(kind, n, cin, cout, h, w, *, seed=0, m_rows=0, twice=False, knobs=None, expect=None):
    """Conv2d weight gradient dW[cout][tap][cin] (fp32) inside guard rows and channels, against fp64."""
    k, s, p = {"k1": (1, 1, 0), "k3s1": (3, 1, 1), "k4s1": (4, 1, 1), "k4s2": (4, 2, 1)}[kind]
    cfg = R.wgrad_config(cout, cin, k * k, knobs)
    for kk, v in (expect or {}).items():
        assert cfg[kk] == v, f"the case no longer reaches its branch: {kk} = {cfg[kk]}, wanted {v} ({cfg})"
    g = torch.Generator().manual_seed(seed)
    ho, wo = (h + 2 * p - k) // s + 1, (w + 2 * p - k) // s + 1
    x = _bf(torch.randn(n, cin, h, w, generator=g))
    dy = _bf(torch.randn(n, cout, ho, wo, generator=g))
    xs, dys = _source(R.nhwc(x).to(DEV)), _source(R.nhwc(dy).to(DEV), align=32)
    out = R.Guarded((cout, k * k, cin), torch.float32, DEV, lo=16, hi=16, fill=0.0)
    if knobs:
        for k_, v_ in knobs.items():
            _lib.debug_set(k_, v_)
    calls = 2 if twice else 1
    for _ in range(calls):
        ops.conv_wgrad(dys.view, xs.view, out.view, (k, k), s, (-p, -p), k * k * out.ld, out.ld, m_rows=m_rows)
    torch.cuda.synchronize()
    for name, gb in (("dW", out), ("x", xs), ("dy", dys)):
        gb.check(f"{name} guard")
    macs = n * ho * wo * cout * cin * k * k
    dev = DEV if macs > DEVICE_REF_MACS else "cpu"
    ref, sabs = R.wgrad(x.to(dev), dy.to(dev), k, s, p)
    exp = R.Expect(calls * ref, calls * sabs)
    if m_rows:
        exp.ref[m_rows:] = 0
        exp.s[m_rows:] = 0
    R.assert_within(out.view, exp, f"{kind} wgrad", dtype=torch.float32, locate=R.wgrad_locator(cfg))


WGRAD_CASES = [
    ("default_k4s2_mt2", dict(kind="k4s2", n=2, cin=128, cout=256, h=16, w=16, expect=dict(mt=2))),
    ("default_k3s1", dict(kind="k3s1", n=2, cin=64, cout=64, h=20, w=20)),
    ("default_k1", dict(kind="k1", n=3, cin=256, cout=128, h=9, w=7)),
    ("n_c_320_ragged_last_n_tile", dict(kind="k4s2", n=2, cin=320, cout=128, h=12, w=12,
                                        expect=dict(block_n=256))),
    ("m_rows_lt_m_c", dict(kind="k4s1", n=2, cin=64, cout=128, h=9, w=9, m_rows=37)),
    ("accumulates_second_call", dict(kind="k4s2", n=2, cin=64, cout=128, h=16, w=16, twice=True)),
    ("forced_block_n_64", dict(kind="k4s2", n=2, cin=256, cout=128, h=8, w=8, knobs=dict(wgrad_block_n=64))),
    ("forced_block_n_128", dict(kind="k3s1", n=2, cin=320, cout=128, h=8, w=8, knobs=dict(wgrad_block_n=128))),
    ("forced_block_n_256_mt1", dict(kind="k4s2", n=2, cin=256, cout=256, h=8, w=8,
                                    knobs=dict(wgrad_block_n=256, wgrad_mt=1))),
    ("forced_mt2_single_m_tile", dict(kind="k3s1", n=2, cin=64, cout=128, h=10, w=10, knobs=dict(wgrad_mt=2))),
    ("forced_tpc_3_ragged_tap_group", dict(kind="k4s2", n=2, cin=64, cout=128, h=12, w=12,
                                           knobs=dict(wgrad_tpc=3, wgrad_mt=1, wgrad_block_n=64))),
    ("forced_tpc_4", dict(kind="k3s1", n=2, cin=128, cout=128, h=10, w=10, knobs=dict(wgrad_tpc=4, wgrad_mt=1))),
    ("forced_splits_1", dict(kind="k4s2", n=4, cin=64, cout=128, h=32, w=32, knobs=dict(wgrad_splits=1))),
    ("forced_splits_2", dict(kind="k4s2", n=4, cin=64, cout=128, h=32, w=32, knobs=dict(wgrad_splits=2))),
    ("forced_splits_7", dict(kind="k4s2", n=4, cin=64, cout=128, h=32, w=32, knobs=dict(wgrad_splits=7))),
    ("forced_splits_max_one_pixel_tile_each", dict(kind="k3s1", n=3, cin=64, cout=64, h=16, w=16,
                                                   knobs=dict(wgrad_splits=1 << 20))),
    ("forced_single_producer", dict(kind="k4s2", n=2, cin=64, cout=128, h=16, w=16, knobs=dict(wgrad_dual=0))),
    ("forced_dual_producer_one_tap", dict(kind="k1", n=2, cin=128, cout=128, h=8, w=8, knobs=dict(wgrad_dual=1))),
    ("forced_scalar_reduction", dict(kind="k4s2", n=2, cin=320, cout=128, h=12, w=12,
                                     knobs=dict(wgrad_scalar_red=1))),
]


@pytest.mark.parametrize("case", [c for _, c in WGRAD_CASES], ids=[i for i, _ in WGRAD_CASES])
def test_wgrad_config(case, restore_knobs):
    run_wgrad(**case)


# ---- batch-64 shapes of test_gpu_batch64.py, one per geometry (fp64 reference on the device) ------------------------
B64_FPROP = [
    ("k4s2_fwd_128to256_64", dict(kind="k4s2", n=64, cin=128, n_out=256, h=64, w=64, stats=True)),
    ("dgrad_s2_256to512_32", dict(kind="dgrad_s2", n=64, cin=512, n_out=256, h=16, w=16)),
    ("patchgan_k4s1_fwd", dict(kind="k4s1", n=64, cin=256, n_out=512, h=32, w=32)),
    ("patchgan_dgrad_s1", dict(kind="dgrad_s1", n=64, cin=512, n_out=256, h=31, w=31)),
    ("convT_fwd_1024to512_8", dict(kind="phase", n=64, cin=1024, n_out=512, h=8, w=8, stats=True)),
    ("convT_dgrad_1024to256_16", dict(kind="convT_dgrad", n=64, cin=256, n_out=1024, h=32, w=32)),
]


@pytest.mark.parametrize("case", [c for _, c in B64_FPROP], ids=[i for i, _ in B64_FPROP])
def test_batch64_fprop(case, restore_knobs):
    run_fprop(**case)


def test_batch64_wgrad(restore_knobs):
    run_wgrad("k4s2", 64, 128, 256, 64, 64)

