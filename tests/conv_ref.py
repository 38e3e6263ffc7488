"""fp64 reference of the implicit-GEMM convolutions (gap_conv_gemm, gap_conv_wgrad) with a per-element error bound,
guard-banded buffers that expose stray writes, and a mirror of the host code's launch-configuration choice that names
the tile a failing element belongs to.  Tests import it; the product never does.

Every reference is computed in float64 from the same bf16-rounded operands the kernel reads, together with
S = the same operation on |a| and |b| (the per-element sum of absolute products).  An output element passes when

    |got - ref| <= eps_out * |ref| + 2^-14 * S  (+ 2^-18 after Tanh / Sigmoid)

- eps_out * |ref| is the output rounding: round-to-nearest-even to bf16 is 2^-9 relative, doubled (2^-8); fp32
  outputs (weight gradients, out_f32) take 2^-23.
- 2^-14 * S covers the fp32 accumulation: random-sign rounding errors come to ~2^-24 * S, and even an adder that
  truncates stays orders of magnitude below 2^-14 * S.  It stays well below the effect of losing one 64-channel slice
  of K, which costs ~8 / K of S per element (1e-3 * S at K = 8192).
- 2^-18 is the fp32 error of tanhf / __expf on outputs of magnitude <= 1.
The epilogue carries S along: scale s -> |s| * S, activation with slope a -> |a| * S on the negative side (S near 0,
where the sign can flip), accumulate -> |prev| + S, backward-fused mask -> S + |g2| or |slope| * S."""
import math

import torch
import torch.nn.functional as F
from torch.nn import grad as G

U_ACC = 2.0 ** -14
U_FN = 2.0 ** -18
SENTINEL = -448.0          # exact in bf16 and fp32
SLOPES = {0: 1.0, 1: 0.2, 2: 0.0}       # ops.ACT_NONE / ACT_LRELU / ACT_RELU: negative-side slope
ACT_TANH, ACT_SIGMOID = 3, 4


def out_eps(dtype):
    return 2.0 ** -8 if dtype == torch.bfloat16 else 2.0 ** -23


def nhwc(t):
    return t.permute(0, 2, 3, 1)


def _pair(fn, a, b):
    a, b = a.double(), b.double()
    return fn(a, b), fn(a.abs(), b.abs())


# ---- references: NCHW operands in, (ref, S) out in the kernel's layout ------------------------------------------
def conv_fwd(x, w, stride, pad):
    """Conv2d forward (k1/k3/k4, stride 1/2), and ConvTranspose2d dgrad (k4 s2 p1 over dY): NHWC [n, oh, ow, cout]."""
    r, s = _pair(lambda a, b: F.conv2d(a, b, None, stride, pad), x, w)
    return nhwc(r), nhwc(s)


def conv_dgrad(dy, w, in_hw, stride, pad):
    """Conv2d dgrad (stride 1 with flipped taps, stride 2 through the four phases): NHWC [n, ih, iw, cin]."""
    shape = (dy.shape[0], w.shape[1]) + tuple(in_hw)
    r, s = _pair(lambda a, b: G.conv2d_input(shape, b, a, stride, pad), dy, w)
    return nhwc(r), nhwc(s)


def convT_fwd(x, w):
    """ConvTranspose2d(k4, s2, p1) forward, w [cin, cout, 4, 4]: NHWC [n, 2h, 2w, cout]."""
    r, s = _pair(lambda a, b: F.conv_transpose2d(a, b, None, 2, 1), x, w)
    return nhwc(r), nhwc(s)


def wgrad(x, dy, k, stride, pad):
    """Conv2d weight gradient in the kernel's [cout][kh*kw][cin] layout."""
    shape = (dy.shape[1], x.shape[1], k, k)
    r, s = _pair(lambda a, b: G.conv2d_weight(a, shape, b, stride, pad), x, dy)
    co, ci = shape[:2]
    return r.permute(0, 2, 3, 1).reshape(co, k * k, ci), s.permute(0, 2, 3, 1).reshape(co, k * k, ci)


# ---- expected values and the bound ----------------------------------------------------------------------------------
class Expect:
    """ref, S and the extra absolute term of one output tensor; the epilogue steps return new instances."""

    def __init__(self, ref, s, extra=0.0):
        self.ref, self.s, self.extra = ref, s, extra

    def scale(self, sc):
        sc = sc.double().to(self.ref.device)
        return Expect(self.ref * sc, self.s * sc.abs(), self.extra)

    def bias(self, b):
        return Expect(self.ref + b.double().to(self.ref.device), self.s, self.extra)

    def act(self, act):
        r, s = self.ref, self.s
        if act in SLOPES:
            a = SLOPES[act]
            neg = r < -U_ACC * s          # certainly negative in the kernel too
            return Expect(torch.where(r > 0, r, a * r), torch.where(neg, a * s, s), self.extra)
        if act == ACT_TANH:
            return Expect(torch.tanh(r), s, self.extra + U_FN)
        if act == ACT_SIGMOID:
            return Expect(torch.sigmoid(r), s / 4, self.extra + U_FN)
        raise ValueError(act)

    def accumulate(self, prev):
        p = prev.double().to(self.ref.device)
        return Expect(self.ref + p, self.s + p.abs(), self.extra)

    def bwd(self, y, slope, scale=None, shift=None, g2=None):
        """d = (y*scale + shift > 0) ? g (+ g2) : slope * g.  Returns (taken, other, ambiguous): the branch the fp64
        mask takes, the other one, and the elements whose mask argument is within 1e-3 of 0 (either branch counts)."""
        yh = y.double().to(self.ref.device)
        if scale is not None:
            yh = yh * scale.double().to(yh.device) + shift.double().to(yh.device)
        gg = 0.0 if g2 is None else g2.double().to(yh.device)
        on_r, on_s = self.ref + gg, self.s + (gg.abs() if g2 is not None else 0.0)
        off_r, off_s = slope * self.ref, abs(slope) * self.s
        m = yh > 0
        taken = Expect(torch.where(m, on_r, off_r), torch.where(m, on_s, off_s), self.extra)
        other = Expect(torch.where(m, off_r, on_r), torch.where(m, off_s, on_s), self.extra)
        return taken, other, yh.abs() < 1e-3

    def bound(self, dtype):
        return out_eps(dtype) * self.ref.abs() + U_ACC * self.s + self.extra


def ratio(got, exp, dtype):
    """|got - ref| / bound per element (inf where got is NaN / inf)."""
    g = got.double().to(exp.ref.device)
    err = (g - exp.ref).abs()
    r = torch.where(err == 0, torch.zeros_like(err), err / exp.bound(dtype))     # a ReLU zero has a zero bound
    return torch.where(torch.isfinite(g), r, torch.full_like(r, math.inf))


def assert_within(got, exp, what, dtype=None, locate=None, alt=None):
    """Per-element check of `got` against `exp`.  alt = (expect2, mask): on `mask` the nearer of the two expectations
    counts.  On failure the message names the worst element (its index, and through `locate` its tile) and the ratio
    of its error to its bound."""
    dtype = dtype or got.dtype
    r = ratio(got, exp, dtype)
    if alt is not None:
        e2, mask = alt
        r = torch.where(mask.to(r.device), torch.minimum(r, ratio(got, e2, dtype)), r)
    worst = float(r.max())
    if worst <= 1.0:
        return worst
    flat = int(r.argmax())
    idx = []
    for d in reversed(r.shape):
        idx.append(flat % d)
        flat //= d
    idx = tuple(reversed(idx))
    n_bad = int((r > 1).sum())
    g = float(got[idx])
    msg = (f"{what}: {n_bad} of {r.numel()} elements outside the bound; worst at {idx}: got {g:.6g}, "
           f"ref {float(exp.ref[idx]):.6g}, S {float(exp.s[idx]):.4g}, |err| / bound = {worst:.3g}")
    if locate is not None:
        msg += f" ({locate(idx)})"
    raise AssertionError(msg)


def assert_stats(stats, out, y=None, what="stats"):
    """Per-channel BatchNorm sums of the epilogue against fp64 sums of the stored bf16 output: [sum o | sum o^2], or,
    for the backward-fused epilogue, [sum d | sum d*y].  Each is within 1e-5 of the sum of the absolute terms (fp32
    partial sums over 32 rows carry <= 31 * 2^-24 of it; products of two bf16 values are exact in fp32)."""
    o = out.double().reshape(-1, out.shape[-1])
    second = o * o if y is None else o * y.double().to(o.device).reshape(o.shape)
    c = o.shape[1]
    st = stats.double().to(o.device)
    for name, got, ref, mag in (("sum", st[:c], o.sum(0), o.abs().sum(0)),
                                ("sum2", st[c:], second.sum(0), second.abs().sum(0))):
        r = (got - ref).abs() / (1e-5 * mag).clamp_min(1e-30)
        if float(r.max()) > 1:
            ch = int(r.argmax())
            raise AssertionError(f"{what} {name}: channel {ch}: got {float(got[ch]):.9g}, ref {float(ref[ch]):.9g}, "
                                 f"|err| / (1e-5 sum|.|) = {float(r.max()):.3g}")


# ---- guard-banded buffers -----------------------------------------------------------------------------------------
class Guarded:
    """A [d0, ..., c] slot inside a [d0 + 2, ..., lo + c + hi] buffer: one guard entry of the first dimension before
    and after (a guard image, or a guard weight row) and `lo` / `hi` guard channels on each side.  Everything outside
    the slot holds `fill`; check() reports the first guard element that changed."""

    def __init__(self, shape, dtype, device, lo=16, hi=48, fill=SENTINEL, guard_fill=None):
        self.shape, self.lo, self.hi = tuple(shape), lo, hi
        full = (shape[0] + 2,) + tuple(shape[1:-1]) + (lo + shape[-1] + hi,)
        gf = fill if guard_fill is None else guard_fill
        self.buf = torch.full(full, gf, dtype=dtype, device=device)
        self.view = self.buf[1:shape[0] + 1, ..., lo:lo + shape[-1]]
        if gf != fill:
            self.view.fill_(fill)
        self._ref = self.buf.clone()

    @property
    def ld(self):
        return self.buf.shape[-1]

    def check(self, what):
        ib = {2: torch.int16, 4: torch.int32, 8: torch.int64}[self.buf.element_size()]
        diff = self.buf.view(ib) != self._ref.view(ib)
        diff[1:self.shape[0] + 1, ..., self.lo:self.lo + self.shape[-1]] = False
        if bool(diff.any()):
            idx = tuple(int(i) for i in diff.nonzero()[0])
            c = idx[-1] - self.lo
            where = (f"{c - self.shape[-1]} channels past the slot" if c >= self.shape[-1] else
                     f"{-c} channels before the slot" if c < 0 else "inside the channel range")
            first = idx[0] - 1
            ent = "guard entry before" if first < 0 else ("guard entry after" if first >= self.shape[0] else
                                                           f"entry {first}")
            raise AssertionError(f"{what}: {int(diff.sum())} guard elements changed; first at {ent}, "
                                 f"index {idx[1:-1]}, {where}: {float(self.buf[idx]):.6g}")


# ---- the host code's launch configuration (conv_fprop.cu gap_conv_gemm, conv_wgrad.cu gap_conv_wgrad) ------------
def _ilog2_ceil(v):
    return max(0, math.ceil(math.log2(v))) if v > 1 else 0


FPROP_DEFAULTS = dict(fprop_pair=1, fprop_halo=1, fprop_ld32=1, fprop_balance=1, fprop_block_n=0, fprop_mt=0,
                      fprop_stages=0)
WGRAD_DEFAULTS = dict(wgrad_block_n=0, wgrad_mt=0, wgrad_tpc=0, wgrad_splits=0, wgrad_dual=-1, wgrad_scalar_red=0,
                      wgrad_acc_cols=512)


def fprop_config(n, gh, gw, geom, n_out, ctot, sms, accumulate=False, knobs=None):
    """The tile shape, halo mode, N tile, M tiles per item, accumulator stages and CTA-pair choice of gap_conv_gemm for
    a launch of geometry `geom` (ops.Geometry) over an n x gh x gw grid."""
    kb = dict(FPROP_DEFAULTS, **(knobs or {}))
    n_phase, taps_h, taps_w, in_stride = geom.n_phase, geom.taps_h, geom.taps_w, geom.in_stride
    log_bw = min(7, _ilog2_ceil(gw))
    log_bh = min(7 - log_bw, _ilog2_ceil(gh))
    halo_taps = taps_h // in_stride
    halo = kb["fprop_halo"] != 0 and halo_taps >= 2 and taps_h % in_stride == 0
    if halo:
        if gw >= 16 and gh >= 8:
            log_bw, log_bh = 4, 3
        elif gw >= 8 and gh >= 16:
            log_bw, log_bh = 3, 4
        else:
            halo = False
    n_pad = (n_out + 15) // 16 * 16
    if halo and min(n_pad, 256) * halo_taps > 256:
        halo = False
        log_bw = min(7, _ilog2_ceil(gw))
        log_bh = min(7 - log_bw, _ilog2_ceil(gh))
    bw, bh = 1 << log_bw, 1 << log_bh
    bni = 128 // (bw * bh)
    tiles_w, tiles_h, tiles_n = -(-gw // bw), -(-gh // bh), -(-n // bni)
    m_pp = tiles_w * tiles_h * tiles_n
    m_tiles = m_pp * n_phase
    n_tiles = -(-n_pad // 256)
    block_n = (-(-n_pad // n_tiles) + 15) // 16 * 16
    model_mt = 0
    if kb["fprop_block_n"] > 0:
        block_n = kb["fprop_block_n"]
        n_tiles = -(-n_pad // block_n)
    elif not halo and m_tiles * n_tiles < 2 * sms:
        wide, best = block_n, None
        for bn in (wide, 128, 64):
            if bn > wide or (bn != wide and wide % bn != 0):
                continue
            for mt_c in (1, 2):
                if mt_c == 2 and m_pp < 2:
                    continue
                items = -(-m_pp // mt_c) * n_phase * -(-n_pad // bn)
                cost = -(-items // sms) * max(130 + 280 * mt_c + 80 * bn // 64, 2 * mt_c * bn + 100)
                if best is None or cost < best:
                    best, block_n, model_mt = cost, bn, mt_c
        n_tiles = -(-n_pad // block_n)
    k_iters = taps_h * taps_w * (ctot // 64)
    mt = 2 if (m_pp >= 2 and (m_tiles // 2) * n_tiles >= 2 * sms) else 1
    if mt == 2 and 2 * block_n > 256 and k_iters < 128:
        mt = 1
    if model_mt > 0:
        mt = model_mt
    if kb["fprop_mt"] > 0:
        mt = min(kb["fprop_mt"], 2)
    pk = kb["fprop_pair"]
    pair = pk != 0 and sms % 2 == 0 and block_n % 16 == 0 and block_n >= 32 and not accumulate
    if pair and pk != 2 and not (block_n == 256 and n_phase == 1 and k_iters >= 64):
        pair = False
    if pair and -(-m_pp // (2 * mt)) * n_phase * n_tiles < sms // 2:
        pair = False
    return dict(log_bw=log_bw, log_bh=log_bh, bni=bni, tiles_w=tiles_w, tiles_h=tiles_h, m_tiles_pp=m_pp, halo=halo,
                block_n=block_n, n_tiles=n_tiles, mt=mt, acc_stages=2 if mt * block_n <= 256 else 1, pair=pair)


def fprop_locator(cfg, n_phase):
    """Maps an NHWC output index (n, y, x, c) to its output phase, M tile and N tile under `cfg`."""
    def locate(idx):
        n, y, x, c = idx
        ph, pw = (y % 2, x % 2) if n_phase == 4 else (0, 0)
        gy, gx = (y // 2, x // 2) if n_phase == 4 else (y, x)
        tw, th, tn = gx >> cfg["log_bw"], gy >> cfg["log_bh"], n // cfg["bni"]
        mi = (tn * cfg["tiles_h"] + th) * cfg["tiles_w"] + tw
        return (f"phase {ph * 2 + pw}, M tile {mi} of {cfg['m_tiles_pp']} (row {gy % (1 << cfg['log_bh'])}, col "
                f"{gx % (1 << cfg['log_bw'])}, image {n % cfg['bni']} of the tile), N tile {c // cfg['block_n']} "
                f"(block_n {cfg['block_n']}, column {c % cfg['block_n']}), mt {cfg['mt']}, halo {int(cfg['halo'])}, "
                f"pair {int(cfg['pair'])}")
    return locate


def wgrad_config(m_c, n_c, n_taps, knobs=None):
    """block_n, M tiles per CTA and taps per CTA of gap_conv_wgrad."""
    kb = dict(WGRAD_DEFAULTS, **(knobs or {}))
    block_n = kb["wgrad_block_n"] or min(256, n_c)
    mt = min(kb["wgrad_mt"], 2) if kb["wgrad_mt"] > 0 else (2 if m_c >= 256 else 1)
    tpc = min(max(1, kb["wgrad_acc_cols"] // (mt * block_n)), n_taps)
    while tpc > 1 and ((mt * 2 + tpc * (block_n // 64)) * 8192 > 72 * 1024 or n_taps % tpc != 0):
        tpc -= 1
    if kb["wgrad_tpc"] > 0:
        tpc = min(kb["wgrad_tpc"], n_taps)
    return dict(block_n=block_n, mt=mt, tpc=tpc)


def wgrad_locator(cfg):
    def locate(idx):
        m, tap, c = idx
        return (f"M tile {m // (128 * cfg['mt'])} (mt {cfg['mt']}), tap group {tap // cfg['tpc']} (tpc {cfg['tpc']}), "
                f"N tile {c // cfg['block_n']} (block_n {cfg['block_n']})")
    return locate
