"""Host-side launchers: torch tensors in, C-ABI calls out.

PyTorch is used for device memory and streams only; every computation below is a ``gap_*`` call
into libgap_b200.so.  Activations are NHWC bf16 tensors (possibly channel slices of a wider
buffer: ``x[..., a:b]`` keeps the parent's pixel stride).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_SIGMOID, ACT_TANH  # noqa: F401


# bench.py sets PROFILE to a list to time every GEMM launch with CUDA events:
# entries are (kernel name, algorithmic FLOPs, start event, end event).
PROFILE = None


def _timed(name: str, flops: float, fn) -> None:
    if PROFILE is None:
        fn()
        return
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    fn()
    e1.record()
    PROFILE.append((name, flops, e0, e1))


def _stream() -> C.c_void_p:
    """The current stream of the CURRENT device: the engines pin the current device to their own for the duration of
    every entry point (pix2pix._on_device), so this is the stream of the tensors being launched on."""
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _nhwc_view(t: torch.Tensor, dtype=torch.bfloat16) -> tuple[int, int, int, int, int]:
    """Return (n, h, w, c, pixel_stride) of an NHWC bf16 tensor that may be a channel slice."""
    if t.dtype != dtype or t.dim() != 4 or not t.is_cuda:
        raise ValueError(f"expected a CUDA NHWC bf16 tensor, got {t.dtype} {tuple(t.shape)} {t.device}")
    n, h, w, c = t.shape
    sn, sh, sw, sc = t.stride()
    if c > 1 and sc != 1:
        raise ValueError("NHWC tensor must be channel-contiguous")
    ld = sw
    if (w > 1 and sh != w * ld and h > 1) or (n > 1 and sn != h * w * ld):
        raise ValueError(f"NHWC tensor must be dense in n/h/w (strides {t.stride()})")
    return n, h, w, c, ld


@dataclass(frozen=True)
class Geometry:
    """Iteration geometry of one gap_conv_gemm call (see gap_b200.h)."""
    n_phase: int
    taps_h: int
    taps_w: int
    in_stride: int
    in_off_h: tuple[int, int]
    in_off_w: tuple[int, int]
    out_stride: int


def geom_conv_fwd(k: int, stride: int, pad: int) -> Geometry:
    """Conv2d forward (models.py:177,223,230,238,243,9,12) and ConvTranspose2d dgrad."""
    return Geometry(1, k, k, stride, (-pad, -pad), (-pad, -pad), 1)


def geom_conv_dgrad_s1(k: int, pad: int) -> Geometry:
    """Stride-1 Conv2d dgrad: a stride-1 conv over dY with flipped taps and pad k-1-pad."""
    return Geometry(1, k, k, 1, (-(k - 1 - pad),) * 2, (-(k - 1 - pad),) * 2, 1)


def geom_phase_k4s2p1() -> Geometry:
    """ConvTranspose2d(k4,s2,p1) forward (models.py:184,189,194) and Conv2d(k4,s2,p1) dgrad:
    four output-parity phases of 2x2 taps; phase (ph,pw), tap (th,tw) uses kernel element
    (3-ph-2*th, 3-pw-2*tw)."""
    return Geometry(4, 2, 2, 1, (-1, 0), (-1, 0), 2)


def conv_gemm(srcs: Sequence[torch.Tensor], wpk: torch.Tensor, geom: Geometry, out: torch.Tensor,
              n_out: int, grid_hw: tuple[int, int], *, act: int = ACT_NONE,
              out2: Optional[torch.Tensor] = None, act2: int = ACT_NONE,
              bias: Optional[torch.Tensor] = None, stats: Optional[torch.Tensor] = None,
              flops: Optional[float] = None, bwd: Optional[dict] = None, scale: Optional[torch.Tensor] = None,
              accumulate: bool = False) -> None:
    """Launch the implicit-GEMM engine.  ``wpk`` is [n_phase, rows, taps*ctot] bf16.  ``flops`` overrides
    the algorithmic FLOP count reported to the profiler (layers that pad channels pass the true one).
    ``accumulate``: add the result to what ``out`` already holds instead of overwriting it."""
    a = _lib.ConvGemmArgs()
    n = ih = iw = None
    for i in range(2):
        if i < len(srcs):
            sn, sh, sw, sc, ld = _nhwc_view(srcs[i])
            if n is None:
                n, ih, iw = sn, sh, sw
            elif (n, ih, iw) != (sn, sh, sw):
                raise ValueError("concatenated sources must share n/h/w")
            a.src[i] = srcs[i].data_ptr()
            a.src_c[i] = sc
            a.src_ld[i] = ld
        else:
            a.src[i] = None
            a.src_c[i] = 0
            a.src_ld[i] = 0
    a.n, a.ih, a.iw = n, ih, iw
    a.gh, a.gw = grid_hw
    a.n_phase = geom.n_phase
    a.taps_h, a.taps_w = geom.taps_h, geom.taps_w
    a.in_stride = geom.in_stride
    a.in_off_h[0], a.in_off_h[1] = geom.in_off_h
    a.in_off_w[0], a.in_off_w[1] = geom.in_off_w
    a.out_stride = geom.out_stride
    if wpk.dtype != torch.bfloat16 or wpk.dim() != 3 or not wpk.is_contiguous():
        raise ValueError("wpk must be a contiguous [n_phase, rows, K] bf16 tensor")
    ctot = sum(int(s.shape[3]) for s in srcs)
    if wpk.shape[0] != geom.n_phase or wpk.shape[2] != geom.taps_h * geom.taps_w * ctot:
        raise ValueError(f"wpk shape {tuple(wpk.shape)} does not match geometry/channels {ctot}")
    a.wpk = wpk.data_ptr()
    a.w_rows = wpk.shape[1]
    a.n_out = n_out
    on, oh, ow, oc, old = _nhwc_view(out, out.dtype if out.dtype == torch.float32 else torch.bfloat16)
    a.out_f32 = 1 if out.dtype == torch.float32 else 0
    if on != n or oc < n_out:
        raise ValueError("output tensor does not match")
    a.oh, a.ow = oh, ow
    a.out = out.data_ptr()
    a.out_ld = old
    a.act = act
    if out2 is not None:
        o2n, o2h, o2w, o2c, o2ld = _nhwc_view(out2)
        if (o2n, o2h, o2w) != (on, oh, ow) or o2c < n_out:
            raise ValueError("out2 does not match out")
        a.out2 = out2.data_ptr()
        a.out2_ld = o2ld
    else:
        a.out2 = None
        a.out2_ld = 0
    a.act2 = act2
    if bias is not None:
        if bias.dtype != torch.float32 or bias.numel() < n_out:
            raise ValueError("bias must be fp32 with >= n_out elements")
        a.bias = bias.data_ptr()
    else:
        a.bias = None
    c0 = int(bwd.get("c0", 0)) if bwd is not None else 0
    if scale is not None:
        if scale.dtype != torch.float32 or scale.numel() < n_out:
            raise ValueError("scale must be fp32 with >= n_out elements")
        a.scale = scale.data_ptr()
    else:
        a.scale = None
    a.accumulate = 1 if accumulate else 0
    if stats is not None:
        if stats.dtype != torch.float64 or stats.numel() != 2 * (n_out - c0):
            raise ValueError("stats must be fp64 [2*(n_out - c0)]")
        a.stats = stats.data_ptr()
    else:
        a.stats = None
    if bwd is not None:
        # backward-fused epilogue: see gap_conv_gemm_args.bwd_* in gap_b200.h
        y = bwd["y"]
        yn, yh, yw, yc, yld = _nhwc_view(y)
        if (yn, yh, yw) != (on, oh, ow) or yc != n_out - c0:
            raise ValueError("bwd y must be [n, oh, ow, n_out - c0]")
        a.bwd_y, a.bwd_y_ld = y.data_ptr(), yld
        sc, sh = bwd.get("scale"), bwd.get("shift")
        a.bwd_scale = None if sc is None else sc.data_ptr()
        a.bwd_shift = None if sh is None else sh.data_ptr()
        g2 = bwd.get("g2")
        if g2 is not None:
            gn, gh_, gw_, gc, gld = _nhwc_view(g2)
            if (gn, gh_, gw_, gc) != (on, oh, ow, n_out - c0):
                raise ValueError("bwd g2 must match y")
            a.bwd_g2, a.bwd_g2_ld = g2.data_ptr(), gld
        else:
            a.bwd_g2, a.bwd_g2_ld = None, 0
        a.bwd_slope = float(bwd.get("slope", 0.0))
        a.bwd_c0 = c0
    else:
        a.bwd_y = None
    if flops is None:
        flops = 2.0 * n * grid_hw[0] * grid_hw[1] * geom.n_phase * n_out * geom.taps_h * geom.taps_w * ctot
    _timed("conv_fprop_kernel", flops,
           lambda: _lib.check(_lib.lib().gap_conv_gemm(C.byref(a), _stream()), "gap_conv_gemm"))


def conv_wgrad(mop: torch.Tensor, nop: torch.Tensor, out: torch.Tensor, taps: tuple[int, int], stride: int,
               off: tuple[int, int], ld_m: int, ld_tap: int, m_rows: int = 0,
               flops: Optional[float] = None) -> None:
    """out[m*ld_m + tap*ld_tap + c] += sum_pix mop[pix, m] * nop[gather(pix, tap), c]   (fp32 out)."""
    a = _lib.WgradArgs()
    n, gh, gw, mc, mld = _nhwc_view(mop)
    n2, nh, nw, nc, nld = _nhwc_view(nop)
    if n != n2:
        raise ValueError("mop / nop batch mismatch")
    if out.dtype != torch.float32 or not out.is_cuda:
        raise ValueError("wgrad output must be a CUDA fp32 tensor")
    a.mop, a.m_c, a.m_ld = mop.data_ptr(), mc, mld
    a.m_rows = m_rows
    a.nop, a.n_c, a.n_ld = nop.data_ptr(), nc, nld
    a.n, a.gh, a.gw, a.nh, a.nw = n, gh, gw, nh, nw
    a.taps_h, a.taps_w = taps
    a.stride = stride
    a.off_h, a.off_w = off
    a.out = out.data_ptr()
    a.ld_m, a.ld_tap = ld_m, ld_tap
    if flops is None:
        flops = 2.0 * n * gh * gw * (m_rows if m_rows > 0 else mc) * nc * taps[0] * taps[1]
    _timed("conv_wgrad_kernel", flops,
           lambda: _lib.check(_lib.lib().gap_conv_wgrad(C.byref(a), _stream()), "gap_conv_wgrad"))


# ------------------------------------------------------------------------------------------------
# thin wrappers over the elementwise / reduction entry points
# ------------------------------------------------------------------------------------------------
def _ptr(t: Optional[torch.Tensor]):
    return None if t is None else C.c_void_p(t.data_ptr())


def _rows_ld(t: torch.Tensor) -> tuple[int, int, int]:
    """(pixels, channels, pixel stride) of a channel-contiguous [..., C] tensor dense in the rest."""
    c = t.shape[-1]
    ld = t.stride(-2) if t.dim() >= 2 else c
    return t.numel() // c, c, ld


def nchw_to_nhwc_bf16(x: torch.Tensor, out: torch.Tensor) -> None:
    n, c, h, w = x.shape
    if x.dtype != torch.float32 or not x.is_contiguous():
        raise ValueError("expected a contiguous fp32 NCHW tensor")
    _lib.check(_lib.lib().gap_nchw_f32_to_nhwc_bf16(_ptr(x), _ptr(out), n, c, h, w, out.stride(2), _stream()),
               "gap_nchw_f32_to_nhwc_bf16")


def nhwc_to_nchw_f32(x: torch.Tensor, out: torch.Tensor, c: int, c_total: Optional[int] = None, c_off: int = 0) -> None:
    n, h, w, _ = x.shape
    _lib.check(_lib.lib().gap_nhwc_to_nchw_f32(_ptr(x), 1 if x.dtype == torch.float32 else 0, _ptr(out), n, c, h, w,
                                               x.stride(2), c if c_total is None else c_total, c_off, _stream()),
               "gap_nhwc_to_nchw_f32")


def tanh_bwd(gout_nchw: torch.Tensor, y_nhwc_f32: torch.Tensor, dpre: torch.Tensor) -> None:
    n, c, h, w = gout_nchw.shape
    _lib.check(_lib.lib().gap_tanh_bwd(_ptr(gout_nchw), _ptr(y_nhwc_f32), y_nhwc_f32.stride(2), _ptr(dpre),
                                       dpre.stride(2), n, c, h, w, _stream()), "gap_tanh_bwd")


def gen_out_bwd(fake_f32: torch.Tensor, real: torch.Tensor, dfake_d: Optional[torch.Tensor], l1_scale: float,
                dpre: torch.Tensor, loss_acc: torch.Tensor) -> None:
    """L1 * lambda + Tanh backward.  ``real`` is real_B either as fp32 NCHW (what the reference's DataLoader yields) or
    as the raw uint8 [n, h, w, C] image (normalised in the kernel like dataset.py does); C = 1..4 channels, which
    ``fake_f32`` / ``dfake_d`` / ``dpre`` hold in the first C of their channel slots."""
    n, h, w, slots = fake_f32.shape
    if real.dtype == torch.uint8:
        c = real.shape[-1]
        if real.dim() != 4 or tuple(real.shape[:3]) != (n, h, w) or not real.is_contiguous():
            raise ValueError("uint8 real_B must be contiguous [n, h, w, C]")
        fn, name = _lib.lib().gap_gen_out_bwd_u8, "gap_gen_out_bwd_u8"
    else:
        c = real.shape[1]
        fn, name = _lib.lib().gap_gen_out_bwd, "gap_gen_out_bwd"
    if not 1 <= c <= slots:
        raise ValueError(f"real_B has {c} channels; the generator output holds {slots} channel slots")
    _lib.check(fn(_ptr(fake_f32), fake_f32.stride(2), _ptr(real), h * w, _ptr(dfake_d),
                  0 if dfake_d is None else dfake_d.stride(2), l1_scale, _ptr(dpre), dpre.stride(2), n * h * w, c,
                  _ptr(loss_acc), _stream()), name)


def gan_losses(acc4: torch.Tensor, count: int, l1_weight: float, numel: int, out2: torch.Tensor) -> None:
    """[loss_D, loss_G] of train_gan.py:61,68-69 from the iteration's four fp64 loss sums (re-zeroed)."""
    if acc4.dtype != torch.float64 or out2.dtype != torch.float64 or acc4.numel() < 4 or out2.numel() < 2:
        raise ValueError("acc4 / out2 must be fp64 with 4 / 2 elements")
    _lib.check(_lib.lib().gap_gan_losses(_ptr(acc4), float(count), float(l1_weight), float(numel), _ptr(out2), _stream()),
               "gap_gan_losses")


def bce_logits_const(logits: torch.Tensor, target: float, grad_scale: float, dlogits: Optional[torch.Tensor],
                     loss_acc: torch.Tensor) -> None:
    _lib.check(_lib.lib().gap_bce_logits_const(_ptr(logits), logits.numel(), target, grad_scale, _ptr(dlogits),
                                               0 if dlogits is None else dlogits.stride(2), _ptr(loss_acc), _stream()),
               "gap_bce_logits_const")


def bce_logits_const_f32(logits: torch.Tensor, target: float, grad_scale: float, dlogits: Optional[torch.Tensor],
                         loss_acc: torch.Tensor, dbias: Optional[torch.Tensor] = None) -> None:
    """BCEWithLogitsLoss vs a constant target (train_gan.py:58,60,67): fp32 gradient (+ the producing conv's
    bias gradient)."""
    if dlogits is not None and (dlogits.dtype != torch.float32 or dlogits.numel() != logits.numel()):
        raise ValueError("dlogits must be fp32 with the shape of logits")
    _lib.check(_lib.lib().gap_bce_logits_const_f32(_ptr(logits), logits.numel(), target, grad_scale, _ptr(dlogits),
                                                   _ptr(loss_acc), _ptr(dbias), _stream()), "gap_bce_logits_const_f32")


def sum_f32(x: torch.Tensor, out: torch.Tensor) -> None:
    _lib.check(_lib.lib().gap_sum_f32(_ptr(x), x.numel(), _ptr(out), _stream()), "gap_sum_f32")


def _pre(pre: Optional[tuple], c: int):
    """(scale, shift, slope) of a fused input transform LeakyReLU_slope(x*scale + shift) -> ctypes arguments."""
    if pre is None:
        return None, None, 0.0
    sc, sh, slope = pre
    if sc.dtype != torch.float32 or sh.dtype != torch.float32 or sc.numel() < c or sh.numel() < c:
        raise ValueError("pre = (scale, shift, slope) needs fp32 vectors with >= c elements")
    return _ptr(sc), _ptr(sh), float(slope)


def cout1_conv_fwd(x: torch.Tensor, w: torch.Tensor, bias: Optional[torch.Tensor], z_ws: torch.Tensor,
                   logits: torch.Tensor, ksize: int = 4, pad: int = 1, pre: Optional[tuple] = None) -> None:
    """Conv2d(C -> 1, k4, s1, p1) + bias (models.py:243): x NHWC bf16, w bf16 [16*C] ([kh][kw][c]), logits fp32
    [n, oh, ow(, 1)].  pre = (scale, shift, slope): x is the raw conv output below and BatchNorm + LeakyReLU
    (models.py:239-240) are applied while it is read."""
    n, ih, iw, c, ld = _nhwc_view(x)
    if z_ws.dtype != torch.float32 or z_ws.numel() < n * ih * iw * 16 or logits.dtype != torch.float32:
        raise ValueError("z_ws / logits must be fp32 (z_ws >= n*ih*iw*16 elements)")
    if w.dtype != torch.bfloat16 or w.numel() != ksize * ksize * c:
        raise ValueError("w must be bf16 [k*k*C]")
    if logits.numel() != n * (ih + 2 * pad - ksize + 1) * (iw + 2 * pad - ksize + 1):
        raise ValueError("logits shape mismatch")
    sc, sh, slope = _pre(pre, c)
    _lib.check(_lib.lib().gap_cout1_conv_fwd(_ptr(x), ld, n, ih, iw, c, _ptr(w), _ptr(bias), ksize, pad, _ptr(z_ws),
                                             _ptr(logits), sc, sh, slope, _stream()), "gap_cout1_conv_fwd")


def cout1_conv_dgrad(dlogits: torch.Tensor, w: torch.Tensor, gx: torch.Tensor, ksize: int = 4, pad: int = 1,
                     bwd: Optional[dict] = None) -> None:
    """Input gradient of Conv2d(C -> 1, k4, s1).  ``bwd`` = dict(y, scale, shift, slope, sums) fuses the activation
    backward of the layer below and its BatchNorm-backward sums into the kernel (see gap_cout1_conv_dgrad_bwd)."""
    n, ih, iw, c, ld = _nhwc_view(gx)
    oh, ow = ih + 2 * pad - ksize + 1, iw + 2 * pad - ksize + 1
    if dlogits.dtype != torch.float32 or dlogits.numel() != n * oh * ow:
        raise ValueError("dlogits must be fp32 [n, oh, ow]")
    if bwd is None:
        _lib.check(_lib.lib().gap_cout1_conv_dgrad(_ptr(dlogits), n, oh, ow, _ptr(w), ksize, pad, c, _ptr(gx), ld, ih, iw,
                                                   _stream()), "gap_cout1_conv_dgrad")
        return
    y = bwd["y"]
    yn, yh, yw, yc, yld = _nhwc_view(y)
    if (yn, yh, yw, yc) != (n, ih, iw, c) or bwd["sums"].dtype != torch.float64 or bwd["sums"].numel() != 2 * c:
        raise ValueError("bwd y must match gx and sums must be fp64 [2c]")
    _lib.check(_lib.lib().gap_cout1_conv_dgrad_bwd(_ptr(dlogits), n, oh, ow, _ptr(w), ksize, pad, c, _ptr(gx), ld, ih, iw,
                                                   _ptr(y), yld, _ptr(bwd["scale"]), _ptr(bwd["shift"]),
                                                   float(bwd.get("slope", 0.0)), _ptr(bwd["sums"]), _stream()),
               "gap_cout1_conv_dgrad_bwd")


def cout1_conv_wgrad(dlogits: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, ksize: int = 4, pad: int = 1,
                     pre: Optional[tuple] = None) -> None:
    n, ih, iw, c, ld = _nhwc_view(x)
    oh, ow = ih + 2 * pad - ksize + 1, iw + 2 * pad - ksize + 1
    if dlogits.dtype != torch.float32 or dlogits.numel() != n * oh * ow:
        raise ValueError("dlogits must be fp32 [n, oh, ow]")
    if dw.dtype != torch.float32 or dw.numel() != ksize * ksize * c:
        raise ValueError("dw must be fp32 [k*k*C]")
    sc, sh, slope = _pre(pre, c)
    _lib.check(_lib.lib().gap_cout1_conv_wgrad(_ptr(dlogits), n, oh, ow, _ptr(x), ld, ih, iw, c, ksize, pad, _ptr(dw),
                                               sc, sh, slope, _stream()), "gap_cout1_conv_wgrad")


def thin_conv_fwd(s0: torch.Tensor, s1: Optional[torch.Tensor], wpk: torch.Tensor, bias: Optional[torch.Tensor],
                  out1: torch.Tensor, act1: int = ACT_NONE, out2: Optional[torch.Tensor] = None,
                  act2: int = ACT_NONE) -> None:
    """Conv2d(k4,s2,p1) over one or two 4-slot NHWC sources (1..4 channels each, unused slots zero) -> cw = 64/128
    channels, fused bias + activation(s); wpk bf16 [cw, 16*CT] with CT = 4 (one source) or 8 (two), zero in the
    columns of unused slots."""
    n, h, w, _, ld0 = _nhwc_view(s0)
    ld1 = 0
    if s1 is not None:
        n1, h1, w1, _, ld1 = _nhwc_view(s1)
        if (n1, h1, w1) != (n, h, w):
            raise ValueError("sources must share n/h/w")
    on, oh, ow, cw, ldo1 = _nhwc_view(out1)
    if (on, oh, ow) != (n, h // 2, w // 2):
        raise ValueError("out1 shape mismatch")
    ct = 8 if s1 is not None else 4
    if wpk.dtype != torch.bfloat16 or wpk.numel() != cw * 16 * ct or not wpk.is_contiguous():
        raise ValueError(f"wpk must be contiguous bf16 [{cw}, {16 * ct}]")
    ldo2 = 0
    if out2 is not None:
        o2 = _nhwc_view(out2)
        if o2[:4] != (on, oh, ow, cw):
            raise ValueError("out2 shape mismatch")
        ldo2 = o2[4]
    if bias is not None and (bias.dtype != torch.float32 or bias.numel() < cw):
        raise ValueError("bias must be fp32 [cw]")
    _lib.check(_lib.lib().gap_thin_conv_fwd(_ptr(s0), ld0, _ptr(s1), ld1, n, h, w, _ptr(wpk), _ptr(bias), cw, _ptr(out1),
                                            ldo1, act1, _ptr(out2), ldo2, act2, _stream()), "gap_thin_conv_fwd")


def thin_conv_wgrad(wide: torch.Tensor, s0: torch.Tensor, s1: Optional[torch.Tensor], dw: torch.Tensor, ld_m: int,
                    dbias: Optional[torch.Tensor] = None, c0: int = 3, c1: Optional[int] = None) -> None:
    """dw[cw][(kh*4+kw)*c + ch] += sum_pix wide[pix][cw] * thin[2*pix+tap-1][ch] (fp32 master layout, row stride
    ld_m); dbias[cw] += sum_pix wide[pix][cw].  c0 / c1: channels of the two sources (c1 defaults to 3 with a second
    source, 0 without); c = c0 + c1, and source 1's channel s is master channel c0 + s."""
    n, oh, ow, cw, ldw = _nhwc_view(wide)
    n0, h, w, _, ld0 = _nhwc_view(s0)
    if (n0, h, w) != (n, 2 * oh, 2 * ow):
        raise ValueError("thin source must be at twice the resolution of the wide tensor")
    ld1 = 0
    if s1 is not None:
        n1, h1, w1, _, ld1 = _nhwc_view(s1)
        if (n1, h1, w1) != (n, h, w):
            raise ValueError("sources must share n/h/w")
    if c1 is None:
        c1 = 3 if s1 is not None else 0
    if not 1 <= c0 <= 4 or (s1 is not None and not 1 <= c1 <= 4) or (s1 is None and c1 != 0):
        raise ValueError(f"channels per source must be 1..4 (c1 = 0 without a second source), got c0={c0} c1={c1}")
    c = c0 + c1
    if dw.dtype != torch.float32 or dw.numel() < (cw - 1) * ld_m + 16 * c:
        raise ValueError("dw too small")
    if (c0, c1) == (3, 3 if s1 is not None else 0):
        _lib.check(_lib.lib().gap_thin_conv_wgrad(_ptr(wide), ldw, _ptr(s0), ld0, _ptr(s1), ld1, n, h, w, cw, _ptr(dw),
                                                  ld_m, _ptr(dbias), _stream()), "gap_thin_conv_wgrad")
        return
    _lib.check(_lib.lib().gap_thin_conv_wgrad_c(_ptr(wide), ldw, _ptr(s0), ld0, c0, _ptr(s1), ld1, c1, n, h, w, cw,
                                                _ptr(dw), ld_m, _ptr(dbias), _stream()), "gap_thin_conv_wgrad_c")


def u8_hwc_to_nhwc_bf16(x: torch.Tensor, out: torch.Tensor) -> None:
    """uint8 [n,h,w,C] (C = 1..4) -> normalised NHWC bf16 with 4 channel slots, slots >= C zero (dataset.py:155-159 on
    the device)."""
    c = x.shape[-1]
    if x.dtype != torch.uint8 or not 1 <= c <= 4 or not x.is_contiguous() or not x.is_cuda:
        raise ValueError(f"expected a contiguous CUDA uint8 [n,h,w,C] tensor with C = 1..4, got {x.dtype} {tuple(x.shape)}")
    if c == 3:
        _lib.check(_lib.lib().gap_u8_hwc_to_nhwc_bf16(_ptr(x), _ptr(out), out.stride(2), x.numel() // 3, _stream()),
                   "gap_u8_hwc_to_nhwc_bf16")
        return
    _lib.check(_lib.lib().gap_u8_hwc_to_nhwc_bf16_c(_ptr(x), c, _ptr(out), out.stride(2), x.numel() // c, _stream()),
               "gap_u8_hwc_to_nhwc_bf16_c")


def resize_u8_to_nhwc_bf16(x: torch.Tensor, out: Optional[torch.Tensor], out_nchw_f32: Optional[torch.Tensor] = None) -> None:
    """dataset.py's ToTensor + JointResize(BILINEAR, antialias) + JointNormalize on the device: uint8 [n,ih,iw,C]
    (C = 1..4) -> NHWC bf16 [n,oh,ow,4 slots] (slots >= C zero) and / or the fp32 NCHW [n,C,oh,ow] tensor the reference's
    DataLoader yields (the output tensors' h / w are the target size)."""
    if x.dtype != torch.uint8 or x.dim() != 4 or not 1 <= x.shape[-1] <= 4 or not x.is_contiguous() or not x.is_cuda:
        raise ValueError("expected a contiguous CUDA uint8 [n,h,w,C] tensor with C = 1..4")
    n, c = x.shape[0], x.shape[-1]
    ld = 0
    if out is not None:
        on, oh, ow, _, ld = _nhwc_view(out)
        if on != n or out.shape[-1] < 4:
            raise ValueError("output must be NHWC bf16 [n, oh, ow, >=4]")
    if out_nchw_f32 is not None:
        f = out_nchw_f32
        if f.dtype != torch.float32 or f.dim() != 4 or f.shape[0] != n or f.shape[1] != c or not f.is_contiguous() or not f.is_cuda:
            raise ValueError(f"out_nchw_f32 must be a contiguous CUDA fp32 [n,{c},oh,ow] tensor")
        if out is not None and (f.shape[2], f.shape[3]) != (oh, ow):
            raise ValueError("both outputs must have the same size")
        oh, ow = f.shape[2], f.shape[3]
    if out is None and out_nchw_f32 is None:
        raise ValueError("no output given")
    if c == 3:
        _lib.check(_lib.lib().gap_resize_u8_to_nhwc_bf16(_ptr(x), n, x.shape[1], x.shape[2], oh, ow, _ptr(out), ld,
                                                         _ptr(out_nchw_f32), _stream()), "gap_resize_u8_to_nhwc_bf16")
        return
    _lib.check(_lib.lib().gap_resize_u8_to_nhwc_bf16_c(_ptr(x), c, n, x.shape[1], x.shape[2], oh, ow, _ptr(out), ld,
                                                       _ptr(out_nchw_f32), _stream()), "gap_resize_u8_to_nhwc_bf16_c")


def resize_nearest_i64(x: torch.Tensor, out: torch.Tensor) -> None:
    """JointResize's label half (dataset.py:143-146): nearest-neighbour resize of an int64 [n,ih,iw] map into [n,oh,ow]."""
    if x.dtype != torch.int64 or out.dtype != torch.int64 or x.dim() != 3 or out.dim() != 3 or x.shape[0] != out.shape[0] \
            or not (x.is_contiguous() and out.is_contiguous() and x.is_cuda and out.is_cuda):
        raise ValueError("expected contiguous CUDA int64 [n,h,w] tensors")
    _lib.check(_lib.lib().gap_resize_nearest_i64(_ptr(x), x.shape[0], x.shape[1], x.shape[2], out.shape[1], out.shape[2],
                                                 _ptr(out), _stream()), "gap_resize_nearest_i64")


def thin_convT_fwd(wide: torch.Tensor, wcol: torch.Tensor, bias: Optional[torch.Tensor], act: int,
                   out_bf16: Optional[torch.Tensor], out_f32: Optional[torch.Tensor],
                   out_u8: Optional[torch.Tensor] = None, co: int = 3) -> None:
    """ConvTranspose2d(cw -> co, k4, s2, p1) (+bias, Tanh), co = 1..4, into 4-slot NHWC outputs (slots >= co written
    as zero); wcol bf16 [16*co = tap*co + c, cw]; out_u8 uint8 [n, 2ih, 2iw, co]."""
    if not 1 <= co <= 4:
        raise ValueError(f"co must be 1..4, got {co}")
    n, ih, iw, cw, ldw = _nhwc_view(wide)
    if wcol.dtype != torch.bfloat16 or tuple(wcol.shape) != (16 * co, cw) or not wcol.is_contiguous():
        raise ValueError(f"wcol must be contiguous bf16 [{16 * co}, {cw}]")
    for o, dt in ((out_bf16, torch.bfloat16), (out_f32, torch.float32)):
        if o is not None and (o.dtype != dt or tuple(o.shape[:3]) != (n, 2 * ih, 2 * iw) or o.shape[3] < 4):
            raise ValueError("output must be [n, 2ih, 2iw, >=4]")
    if out_u8 is not None and (out_u8.dtype != torch.uint8 or tuple(out_u8.shape) != (n, 2 * ih, 2 * iw, co)
                               or not out_u8.is_contiguous()):
        raise ValueError(f"out_u8 must be a contiguous uint8 [{n}, {2 * ih}, {2 * iw}, {co}] tensor")
    args = (n, ih, iw, cw) + (() if co == 3 else (co,)) + (
        _ptr(wcol), _ptr(bias), act, _ptr(out_bf16), 0 if out_bf16 is None else out_bf16.stride(2), _ptr(out_f32),
        0 if out_f32 is None else out_f32.stride(2), _ptr(out_u8), _stream())
    if co == 3:
        _lib.check(_lib.lib().gap_thin_convT_fwd(_ptr(wide), ldw, *args), "gap_thin_convT_fwd")
    else:
        _lib.check(_lib.lib().gap_thin_convT_fwd_c(_ptr(wide), ldw, *args), "gap_thin_convT_fwd_c")


def bn_finalize(stats, count, gamma, beta, eps, momentum, repeat, running_mean, running_var, nbt, scale, shift,
                save_mean, save_invstd) -> None:
    c = scale.numel()
    _lib.check(_lib.lib().gap_bn_finalize(_ptr(stats), c, float(count), _ptr(gamma), _ptr(beta), eps, momentum, repeat,
                                          _ptr(running_mean), _ptr(running_var), _ptr(nbt), _ptr(scale), _ptr(shift),
                                          _ptr(save_mean), _ptr(save_invstd), _stream()), "gap_bn_finalize")


def bn_eval_scale_shift(gamma, beta, running_mean, running_var, eps, scale, shift) -> None:
    _lib.check(_lib.lib().gap_bn_eval_scale_shift(scale.numel(), _ptr(gamma), _ptr(beta), _ptr(running_mean),
                                                  _ptr(running_var), eps, _ptr(scale), _ptr(shift), _stream()),
               "gap_bn_eval_scale_shift")


def bn_act(y: torch.Tensor, scale, shift, out1: torch.Tensor, act1: int, out2: Optional[torch.Tensor] = None,
           act2: int = ACT_NONE) -> None:
    pixels, c, ld = _rows_ld(y)
    _lib.check(_lib.lib().gap_bn_act(_ptr(y), ld, _ptr(scale), _ptr(shift), pixels, c, _ptr(out1), out1.stride(-2),
                                     act1, _ptr(out2), 0 if out2 is None else out2.stride(-2), act2, _stream()),
               "gap_bn_act")


def bn_bwd_reduce(y, g1, g2, slope, scale, shift, mean, invstd, sums) -> None:
    pixels, c, ld = _rows_ld(y)
    _lib.check(_lib.lib().gap_bn_bwd_reduce(_ptr(y), ld, _ptr(g1), g1.stride(-2), _ptr(g2),
                                            0 if g2 is None else g2.stride(-2), slope, _ptr(scale), _ptr(shift),
                                            _ptr(mean), _ptr(invstd), pixels, c, _ptr(sums), _stream()),
               "gap_bn_bwd_reduce")


def bn_bwd_apply(y, g1, g2, slope, scale, shift, mean, invstd, sums, count, dy) -> None:
    pixels, c, ld = _rows_ld(y)
    _lib.check(_lib.lib().gap_bn_bwd_apply(_ptr(y), ld, _ptr(g1), g1.stride(-2), _ptr(g2),
                                           0 if g2 is None else g2.stride(-2), slope, _ptr(scale), _ptr(shift),
                                           _ptr(mean), _ptr(invstd), pixels, c, _ptr(sums), float(count), _ptr(dy),
                                           dy.stride(-2), _stream()), "gap_bn_bwd_apply")


def bn_param_grads(sums, dgamma, dbeta) -> None:
    _lib.check(_lib.lib().gap_bn_param_grads(_ptr(sums), sums.numel() // 2, _ptr(dgamma), _ptr(dbeta), _stream()),
               "gap_bn_param_grads")


def bn_bwd_finalize(raw, mean, invstd, dgamma, dbeta, sums) -> None:
    """raw [sum d, sum d*y] (re-zeroed) -> sums [sum d, sum d*xhat]; dgamma / dbeta accumulated (may be None)."""
    _lib.check(_lib.lib().gap_bn_bwd_finalize(_ptr(raw), _ptr(mean), _ptr(invstd), mean.numel(), _ptr(dgamma),
                                              _ptr(dbeta), _ptr(sums), _stream()), "gap_bn_bwd_finalize")


def colsum_bf16(x: torch.Tensor, c: int, out: torch.Tensor) -> None:
    pixels = x.numel() // x.shape[-1]
    _lib.check(_lib.lib().gap_colsum_bf16(_ptr(x), x.stride(-2), pixels, c, _ptr(out), _stream()), "gap_colsum_bf16")


def _in_view(y: torch.Tensor) -> tuple[int, int, int, int]:
    """(n, h*w, c, pixel stride) of an InstanceNorm input; a 1x1 map has no spatial statistics (torch raises too)."""
    n, h, w, c, ld = _nhwc_view(y)
    if h * w < 2:
        raise ValueError(f"InstanceNorm2d needs more than one spatial element per channel, got input size {tuple(y.shape)}")
    return n, h * w, c, ld


def _in_same(y: torch.Tensor, *others: Optional[torch.Tensor]) -> None:
    for t in others:
        if t is not None and (t.dtype != torch.bfloat16 or tuple(t.shape) != tuple(y.shape)):
            raise ValueError(f"expected a bf16 tensor of shape {tuple(y.shape)}, got {t.dtype} {tuple(t.shape)}")


def _in_vecs(n: int, c: int, *vecs: torch.Tensor) -> None:
    for v in vecs:
        if v.dtype != torch.float32 or v.numel() != n * c:
            raise ValueError(f"per-(image, channel) vectors must be fp32 [{n}][{c}]")


def in_stats(y: torch.Tensor, sums: torch.Tensor) -> None:
    """sums [2][N*C] fp64 += per-(image, channel) [sum y, sum y^2] of the NHWC bf16 tensor y."""
    n, hw, c, ld = _in_view(y)
    if sums.dtype != torch.float64 or sums.numel() != 2 * n * c:
        raise ValueError(f"sums must be fp64 [2 * {n} * {c}]")
    _lib.check(_lib.lib().gap_in_stats(_ptr(y), ld, n, hw, c, _ptr(sums), _stream()), "gap_in_stats")


def in_act(y: torch.Tensor, scale, shift, out1: torch.Tensor, act1: int, out2: Optional[torch.Tensor] = None,
           act2: int = ACT_NONE) -> None:
    """out1 = act1(y*scale + shift), out2 = act2(same) with per-(image, channel) scale / shift [N][C]."""
    n, hw, c, ld = _in_view(y)
    _in_same(y, out1, out2)
    _in_vecs(n, c, scale, shift)
    _lib.check(_lib.lib().gap_in_act(_ptr(y), ld, n, hw, c, _ptr(scale), _ptr(shift), _ptr(out1), out1.stride(-2), act1,
                                     _ptr(out2), 0 if out2 is None else out2.stride(-2), act2, _stream()), "gap_in_act")


def in_bwd_reduce(y, g1, g2, slope, scale, shift, sums) -> None:
    n, hw, c, ld = _in_view(y)
    _in_same(y, g1, g2)
    _in_vecs(n, c, scale, shift)
    if sums.dtype != torch.float64 or sums.numel() != 2 * n * c:
        raise ValueError(f"sums must be fp64 [2 * {n} * {c}]")
    _lib.check(_lib.lib().gap_in_bwd_reduce(_ptr(y), ld, _ptr(g1), g1.stride(-2), _ptr(g2),
                                            0 if g2 is None else g2.stride(-2), slope, _ptr(scale), _ptr(shift), n, hw, c,
                                            _ptr(sums), _stream()), "gap_in_bwd_reduce")


def in_bwd_apply(y, g1, g2, slope, scale, shift, sums, dy, dbias: Optional[torch.Tensor] = None) -> None:
    """dy = InstanceNorm backward of the activated gradient; dbias (fp32 [C], optional) += its per-channel sum."""
    n, hw, c, ld = _in_view(y)
    _in_same(y, g1, g2, dy)
    _in_vecs(n, c, scale, shift)
    if sums.dtype != torch.float64 or sums.numel() != 2 * n * c:
        raise ValueError(f"sums must be fp64 [2 * {n} * {c}]")
    if dbias is not None and (dbias.dtype != torch.float32 or dbias.numel() != c):
        raise ValueError(f"dbias must be fp32 [{c}]")
    _lib.check(_lib.lib().gap_in_bwd_apply(_ptr(y), ld, _ptr(g1), g1.stride(-2), _ptr(g2),
                                           0 if g2 is None else g2.stride(-2), slope, _ptr(scale), _ptr(shift), n, hw, c,
                                           _ptr(sums), _ptr(dy), dy.stride(-2), _ptr(dbias), _stream()),
               "gap_in_bwd_apply")


def adam_flat(p, g, m, v, lr, beta1, beta2, eps, weight_decay, decoupled, step, grad_scale=1.0) -> None:
    _lib.check(_lib.lib().gap_adam_flat(_ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), lr, beta1, beta2, eps,
                                        weight_decay, 1 if decoupled else 0, step, grad_scale, _stream()),
               "gap_adam_flat")


def adam_flat_devstep(p, g, m, v, lr, beta1, beta2, eps, weight_decay, decoupled, step_dev, grad_scale=1.0) -> None:
    """Adam / AdamW with the step counter in device memory (int32 tensor), for CUDA-graph replay."""
    _lib.check(_lib.lib().gap_adam_flat_devstep(_ptr(p), _ptr(g), _ptr(m), _ptr(v), p.numel(), lr, beta1, beta2, eps,
                                                weight_decay, 1 if decoupled else 0, _ptr(step_dev), grad_scale, _stream()),
               "gap_adam_flat_devstep")


def pack_weights(w: torch.Tensor, w_off: int, out: torch.Tensor, mode: int, n_phase: int, rows: int, rows_pad: int,
                 taps: tuple[int, int], c: int, c_pad: int, krow: int, strides: tuple[int, int, int, int],
                 kdim: int = 0) -> None:
    """``w`` is a flat fp32 buffer, ``w_off`` the element offset of this layer's weights in it."""
    src = C.c_void_p(w.data_ptr() + 4 * w_off)
    _lib.check(_lib.lib().gap_pack_weights(src, _ptr(out), mode, n_phase, rows, rows_pad, taps[0], taps[1], c, c_pad,
                                           krow, strides[0], strides[1], strides[2], strides[3], kdim, _stream()),
               "gap_pack_weights")


class PackPlan:
    """All fp32-master -> bf16-operand repacks of one network as ONE launch (gap_pack_weights_multi).

    ``add`` takes the arguments of :func:`pack_weights`; ``run`` launches.  Padding elements of the
    operands are never written, so the operand buffers must be zero-initialised by the owner."""

    def __init__(self) -> None:
        self.entries: list[_lib.PackEntry] = []
        self.total_tiles = 0
        self._table = None
        self._keep = []

    def add(self, w: torch.Tensor, w_off: int, out: torch.Tensor, mode: int, n_phase: int, rows: int, rows_pad: int,
            taps: tuple[int, int], c: int, c_pad: int, krow: int, strides: tuple[int, int, int, int],
            out_off: int = 0) -> None:
        """``out_off`` (elements) shifts the destination inside each operand row (channel-slot packing)."""
        if mode not in (0, 1, 2):
            raise ValueError("PackPlan supports modes 0-2")
        last = out_off + ((n_phase - 1) * rows_pad + rows - 1) * krow + (taps[0] * taps[1] - 1) * c_pad + c - 1
        if out.dtype != torch.bfloat16 or not out.is_contiguous() or last >= out.numel():
            raise ValueError("operand buffer is too small for this entry")
        e = _lib.PackEntry()
        e.w = w.data_ptr() + 4 * w_off
        e.out = out.data_ptr() + 2 * out_off
        e.mode, e.n_phase, e.rows, e.rows_pad = mode, n_phase, rows, rows_pad
        e.taps_h, e.taps_w, e.c, e.c_pad, e.krow = taps[0], taps[1], c, c_pad, krow
        e.tiles_r, e.tiles_c = (rows + 63) // 64, (c + 63) // 64
        e.tile_begin = self.total_tiles
        e.s_r, e.s_c, e.s_kh, e.s_kw = strides
        self.total_tiles += n_phase * taps[0] * taps[1] * e.tiles_r * e.tiles_c
        self.entries.append(e)
        self._keep.append((w, out))
        self._table = None

    def run(self) -> None:
        if not self.entries:
            return
        if self._table is None:
            arr = (_lib.PackEntry * len(self.entries))(*self.entries)
            raw = bytes(arr)
            dev = self._keep[0][1].device
            self._table = torch.frombuffer(bytearray(raw), dtype=torch.uint8).to(dev)
        _lib.check(_lib.lib().gap_pack_weights_multi(_ptr(self._table), len(self.entries), self.total_tiles, _stream()),
                   "gap_pack_weights_multi")


# ------------------------------------------------------------------------------------------------
# Siamese U-Net extras (gap_b200.h "Siamese U-Net extras")
# ------------------------------------------------------------------------------------------------
def _px(t: torch.Tensor) -> int:
    return t.numel() // t.shape[-1]


def im2col_k3s1p1_c3(x: torch.Tensor, col: torch.Tensor) -> None:
    n, h, w, _, ld = _nhwc_view(x)
    _lib.check(_lib.lib().gap_im2col_k3s1p1_c3(_ptr(x), ld, _ptr(col), n, h, w, _stream()), "gap_im2col_k3s1p1_c3")


def im2col_k3s1p1(x: torch.Tensor, col: torch.Tensor, c: int) -> None:
    """col[pix][(kh*3+kw)*c + ch] (9*c values, zero padded to 64) of the first c = 1..4 channel slots of x."""
    if not 1 <= c <= 4:
        raise ValueError(f"c must be 1..4, got {c}")
    if c == 3:
        im2col_k3s1p1_c3(x, col)
        return
    n, h, w, _, ld = _nhwc_view(x)
    _lib.check(_lib.lib().gap_im2col_k3s1p1_c(_ptr(x), ld, c, _ptr(col), n, h, w, _stream()), "gap_im2col_k3s1p1_c")


def maxpool2x2_fwd(x: torch.Tensor, out: torch.Tensor) -> None:
    n, h, w, c, ld = _nhwc_view(x)
    _lib.check(_lib.lib().gap_maxpool2x2_fwd(_ptr(x), ld, _ptr(out), out.stride(2), n, h, w, c, _stream()),
               "gap_maxpool2x2_fwd")


def maxpool2x2_bwd(x: torch.Tensor, gout: torch.Tensor, gin: torch.Tensor, accumulate: bool) -> None:
    n, h, w, c, ld = _nhwc_view(x)
    _lib.check(_lib.lib().gap_maxpool2x2_bwd(_ptr(x), ld, _ptr(gout), gout.stride(2), _ptr(gin), gin.stride(2), n, h, w, c,
                                             1 if accumulate else 0, _stream()), "gap_maxpool2x2_bwd")


def upsample2x_fwd(x: torch.Tensor, out: torch.Tensor) -> None:
    n, h, w, c, ld = _nhwc_view(x)
    _lib.check(_lib.lib().gap_upsample_bilinear2x_fwd(_ptr(x), ld, _ptr(out), out.stride(2), n, h, w, c, _stream()),
               "gap_upsample_bilinear2x_fwd")


def upsample2x_bwd(gout: torch.Tensor, gin: torch.Tensor, accumulate: bool) -> None:
    n, h, w, c, ld = _nhwc_view(gin)
    _lib.check(_lib.lib().gap_upsample_bilinear2x_bwd(_ptr(gout), gout.stride(2), _ptr(gin), ld, n, h, w, c,
                                                      1 if accumulate else 0, _stream()), "gap_upsample_bilinear2x_bwd")


def dropout_(x: torch.Tensor, p_drop: float, seed: int, offset: int) -> None:
    """In-place nn.Dropout(p) with a regenerable mask (same (seed, offset) -> same mask; used on the gradient too)."""
    _lib.check(_lib.lib().gap_dropout_bf16(_ptr(x), x.stride(-2), _px(x), x.shape[-1], p_drop, seed & (2**64 - 1),
                                           offset & (2**64 - 1), _stream()), "gap_dropout_bf16")


def att_add_relu_fwd(yg, scg, shg, yx, scx, shx, s) -> None:
    _lib.check(_lib.lib().gap_att_add_relu_fwd(_ptr(yg), _ptr(scg), _ptr(shg), _ptr(yx), _ptr(scx), _ptr(shx), _ptr(s),
                                               _px(s), s.shape[-1], _stream()), "gap_att_add_relu_fwd")


def relu_bwd(s: torch.Tensor, gs: torch.Tensor, d: torch.Tensor) -> None:
    _lib.check(_lib.lib().gap_relu_bwd(_ptr(s), _ptr(gs), _ptr(d), s.numel(), _stream()), "gap_relu_bwd")


def lrelu_bwd(y: torch.Tensor, g: torch.Tensor, slope: float, d: torch.Tensor, accumulate: bool) -> None:
    """d (+)= (y > 0) ? g : slope*g on NHWC bf16 tensors / channel slices of the same shape."""
    _lib.check(_lib.lib().gap_lrelu_bwd_bf16(_ptr(y), y.stride(-2), _ptr(g), g.stride(-2), slope, _ptr(d), d.stride(-2),
                                             _px(y), y.shape[-1], 1 if accumulate else 0, _stream()), "gap_lrelu_bwd_bf16")


def att_gate_fwd(ypsi, scale, shift, psi, x, out) -> None:
    _lib.check(_lib.lib().gap_att_gate_fwd(_ptr(ypsi), _ptr(scale), _ptr(shift), _ptr(psi), _ptr(x), x.stride(-2), _ptr(out),
                                           out.stride(-2), _px(x), x.shape[-1], _stream()), "gap_att_gate_fwd")


def att_gate_bwd(gout, x, psi, gx, accumulate: bool, dz) -> None:
    _lib.check(_lib.lib().gap_att_gate_bwd(_ptr(gout), gout.stride(-2), _ptr(x), x.stride(-2), _ptr(psi), _ptr(gx),
                                           gx.stride(-2), 1 if accumulate else 0, _ptr(dz), _px(x), x.shape[-1], _stream()),
               "gap_att_gate_bwd")


def vec_stats(y: torch.Tensor, stats: torch.Tensor) -> None:
    _lib.check(_lib.lib().gap_vec_stats(_ptr(y), y.numel(), _ptr(stats), _stream()), "gap_vec_stats")


def vec_bn_bwd(y, dz, scale, mean, invstd, sums, dy) -> None:
    _lib.check(_lib.lib().gap_vec_bn_bwd(_ptr(y), _ptr(dz), y.numel(), _ptr(scale), _ptr(mean), _ptr(invstd), _ptr(sums),
                                         _ptr(dy), _stream()), "gap_vec_bn_bwd")


def conv1x1_cout1_fwd(x, w, bias, out) -> None:
    _lib.check(_lib.lib().gap_conv1x1_cout1_fwd(_ptr(x), x.stride(-2), _ptr(w), _ptr(bias), _ptr(out), _px(x), x.shape[-1],
                                                _stream()), "gap_conv1x1_cout1_fwd")


def conv1x1_cout1_dgrad(dl, w, gx) -> None:
    _lib.check(_lib.lib().gap_conv1x1_cout1_dgrad(_ptr(dl), _ptr(w), _ptr(gx), gx.stride(-2), _px(gx), gx.shape[-1],
                                                  _stream()), "gap_conv1x1_cout1_dgrad")


def conv1x1_cout1_wgrad(dl, x, dw, db) -> None:
    _lib.check(_lib.lib().gap_conv1x1_cout1_wgrad(_ptr(dl), _ptr(x), x.stride(-2), _px(x), x.shape[-1], _ptr(dw), _ptr(db),
                                                  _stream()), "gap_conv1x1_cout1_wgrad")


def seg_loss(logits: torch.Tensor, labels: torch.Tensor, mode: int, w_point: float, w_dice: float, pos_weight: float,
             smooth: float, gamma: float, focal_alpha: float, sums4: torch.Tensor, grad: Optional[torch.Tensor],
             grad_scale: float, loss: torch.Tensor) -> None:
    """CombinedLoss (mode 0) / FocalDiceLoss (mode 1) of train.py:82-128 with the gradient w.r.t. the logits."""
    if logits.dtype != torch.float32 or labels.dtype != torch.int64 or logits.numel() != labels.numel():
        raise ValueError("logits must be fp32 and labels int64 with the same number of elements")
    _lib.check(_lib.lib().gap_seg_loss(_ptr(logits), _ptr(labels), logits.numel(), mode, w_point, w_dice, pos_weight, smooth,
                                       gamma, focal_alpha, _ptr(sums4), _ptr(grad), grad_scale, _ptr(loss), _stream()),
               "gap_seg_loss")


def seg_confusion(logits: torch.Tensor, labels: torch.Tensor, counts: torch.Tensor) -> None:
    """counts[n, 4] (int64, accumulated) += per-sample [TP, FP, FN, TN] of sigmoid(logits) > 0.5 vs {0,1} labels
    (evaluate.py:34-46).  logits fp32 [n, ...]; labels int64 or fp32 with the same number of elements."""
    n = logits.shape[0]
    if logits.dtype != torch.float32 or not logits.is_contiguous() or not labels.is_contiguous():
        raise ValueError("logits must be contiguous fp32, labels contiguous")
    if labels.dtype not in (torch.int64, torch.float32) or labels.numel() != logits.numel():
        raise ValueError("labels must be int64 or fp32 with as many elements as logits")
    if counts.dtype != torch.int64 or tuple(counts.shape) != (n, 4) or not counts.is_contiguous():
        raise ValueError("counts must be a contiguous int64 [n, 4] tensor")
    if not (logits.is_cuda and labels.is_cuda and counts.is_cuda):
        raise ValueError("seg_confusion needs CUDA tensors (there is no CPU path)")
    _lib.check(_lib.lib().gap_seg_confusion(_ptr(logits), _ptr(labels), 1 if labels.dtype == torch.int64 else 0, n,
                                            logits.numel() // n, _ptr(counts), _stream()), "gap_seg_confusion")


# ------------------------------------------------------------------------------------------------
# Multi-class head of SiameseUNet(n_channels, n_classes), K = 1..16 (gap_b200.h "Multi-class head"): fp32 class
# planes [n][K][h][w]; head input NHWC bf16 [n][h][w][64]
# ------------------------------------------------------------------------------------------------
MAX_CLASSES = 16


def _check_k(k: int, what: str) -> None:
    if not isinstance(k, int) or not 1 <= k <= MAX_CLASSES:
        raise ValueError(f"{what}: the number of classes must be an int in 1..{MAX_CLASSES}, got {k!r}")


def _head_input(x: torch.Tensor, what: str) -> tuple[int, int]:
    """(n, hw) of an NHWC bf16 [n, h, w, 64] head input (a channel slice of a wider buffer is fine)."""
    if x.dim() != 4 or x.shape[-1] != 64 or x.dtype != torch.bfloat16 or x.stride(-1) != 1:
        raise ValueError(f"{what}: x must be NHWC bf16 [n, h, w, 64], got {tuple(x.shape)} {x.dtype}")
    n, h, w, _ = x.shape
    if x.stride(1) != w * x.stride(2) or x.stride(0) != h * x.stride(1) or x.stride(2) % 8 or x.data_ptr() % 16:
        raise ValueError(f"{what}: x must have 16-byte aligned rows of a whole number of 8-element vectors")
    return n, h * w


def _planes(t: torch.Tensor, n: int, k: int, hw: int, what: str, name: str) -> None:
    if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != n * k * hw or t.shape[0] != n:
        raise ValueError(f"{what}: {name} must be contiguous fp32 class planes [n={n}, K={k}, h, w], got "
                         f"{tuple(t.shape)} {t.dtype}")


def _head_weight(w: torch.Tensor, k: int, what: str) -> None:
    if w.dtype != torch.float32 or not w.is_contiguous() or w.numel() != k * 64:
        raise ValueError(f"{what}: the weight must be contiguous fp32 [K={k}, 64], got {tuple(w.shape)} {w.dtype}")


def _cuda(what: str, *ts: Optional[torch.Tensor]) -> None:
    if not all(t.is_cuda for t in ts if t is not None):
        raise ValueError(f"{what} needs CUDA tensors (there is no CPU path)")


def conv1x1_ck_fwd(x: torch.Tensor, w: torch.Tensor, bias: torch.Tensor, out: torch.Tensor,
                   pred: Optional[torch.Tensor] = None) -> None:
    """out [n, K, h, w] fp32 = Conv2d(64 -> K, 1)(x) + bias; pred (uint8 [n, h, w], optional) = argmax over K."""
    what = "conv1x1_ck_fwd"
    n, hw = _head_input(x, what)
    k = out.shape[1] if out.dim() == 4 else -1
    _check_k(k, what)
    _planes(out, n, k, hw, what, "out")
    _head_weight(w, k, what)
    if bias.dtype != torch.float32 or not bias.is_contiguous() or bias.numel() != k:
        raise ValueError(f"{what}: bias must be contiguous fp32 [{k}]")
    if pred is not None and (pred.dtype != torch.uint8 or not pred.is_contiguous() or pred.numel() != n * hw):
        raise ValueError(f"{what}: pred must be contiguous uint8 [n, h, w]")
    _cuda(what, x, w, bias, out, pred)
    _lib.check(_lib.lib().gap_conv1x1_ck_fwd(_ptr(x), x.stride(2), _ptr(w), _ptr(bias), k, n, hw, _ptr(out), _ptr(pred),
                                             _stream()), "gap_conv1x1_ck_fwd")


def conv1x1_ck_dgrad(dl: torch.Tensor, w: torch.Tensor, gx: torch.Tensor) -> None:
    """gx [n, h, w, 64] bf16 (written) = sum_c dl[:, c] * w[c]."""
    what = "conv1x1_ck_dgrad"
    n, hw = _head_input(gx, what)
    k = dl.shape[1] if dl.dim() == 4 else -1
    _check_k(k, what)
    _planes(dl, n, k, hw, what, "dl")
    _head_weight(w, k, what)
    _cuda(what, dl, w, gx)
    _lib.check(_lib.lib().gap_conv1x1_ck_dgrad(_ptr(dl), _ptr(w), k, n, hw, _ptr(gx), gx.stride(2), _stream()),
               "gap_conv1x1_ck_dgrad")


def conv1x1_ck_wgrad(dl: torch.Tensor, x: torch.Tensor, dw: torch.Tensor, db: Optional[torch.Tensor]) -> None:
    """dw [K, 64] += sum_pix dl[c, pix] * x[pix]; db [K] += sum_pix dl[c, pix] (fp32, accumulated)."""
    what = "conv1x1_ck_wgrad"
    n, hw = _head_input(x, what)
    k = dl.shape[1] if dl.dim() == 4 else -1
    _check_k(k, what)
    _planes(dl, n, k, hw, what, "dl")
    _head_weight(dw, k, what)
    if db is not None and (db.dtype != torch.float32 or not db.is_contiguous() or db.numel() != k):
        raise ValueError(f"{what}: db must be contiguous fp32 [{k}]")
    _cuda(what, dl, x, dw, db)
    _lib.check(_lib.lib().gap_conv1x1_ck_wgrad(_ptr(dl), _ptr(x), x.stride(2), k, n, hw, _ptr(dw), _ptr(db), _stream()),
               "gap_conv1x1_ck_wgrad")


def _labels(labels: torch.Tensor, n: int, hw: int, what: str) -> None:
    if labels.dtype != torch.int64 or not labels.is_contiguous() or labels.numel() != n * hw:
        raise ValueError(f"{what}: labels must be contiguous int64 [n, h, w] matching the logits")


def seg_ce_loss(logits: torch.Tensor, labels: torch.Tensor, class_weight: Optional[torch.Tensor], ignore_index: int,
                sums2: torch.Tensor, bad_labels: torch.Tensor, grad: Optional[torch.Tensor], grad_scale: float,
                loss: torch.Tensor) -> None:
    """nn.CrossEntropyLoss(weight=class_weight, ignore_index=ignore_index) on fp32 class planes [n, K, h, w] against
    int64 labels [n, h, w]: loss (fp64 [1], written) and grad = grad_scale * d(loss)/d(logits).  bad_labels (int64 [1])
    counts the labels outside [0, K) that are not ignore_index; they contribute nothing."""
    what = "seg_ce_loss"
    if logits.dim() != 4:
        raise ValueError(f"{what}: logits must be class planes [n, K, h, w], got {tuple(logits.shape)}")
    n, k = logits.shape[0], logits.shape[1]
    hw = logits.shape[2] * logits.shape[3]
    _check_k(k, what)
    _planes(logits, n, k, hw, what, "logits")
    _labels(labels, n, hw, what)
    if grad is not None:
        _planes(grad, n, k, hw, what, "grad")
    if class_weight is not None and (class_weight.dtype != torch.float32 or not class_weight.is_contiguous()
                                     or class_weight.numel() != k):
        raise ValueError(f"{what}: class_weight must be contiguous fp32 [{k}]")
    if sums2.dtype != torch.float64 or sums2.numel() < 2 or loss.dtype != torch.float64 or loss.numel() < 1:
        raise ValueError(f"{what}: sums2 must be fp64 [2] and loss fp64 [1]")
    if bad_labels.dtype != torch.int64 or bad_labels.numel() < 1:
        raise ValueError(f"{what}: bad_labels must be int64 [1]")
    _cuda(what, logits, labels, class_weight, sums2, bad_labels, grad, loss)
    _lib.check(_lib.lib().gap_seg_ce_loss(_ptr(logits), _ptr(labels), k, n, hw, _ptr(class_weight), int(ignore_index),
                                          _ptr(sums2), _ptr(bad_labels), _ptr(grad), grad_scale, _ptr(loss), _stream()),
               "gap_seg_ce_loss")


DICE_SUMS = 3 * (MAX_CLASSES - 1) + 2      # fp64 workspace of seg_softmax_dice_loss for any K


def check_dice_args(what: str, w_point, gamma, smooth) -> None:
    """The keyword ranges of the softmax Dice losses (ValueError otherwise)."""
    if not 0.0 <= float(w_point) <= 1.0:
        raise ValueError(f"{what}: the point-term weight must be in [0, 1], got {w_point!r}")
    if not float(gamma) >= 0.0:
        raise ValueError(f"{what}: gamma must be >= 0, got {gamma!r}")
    if not float(smooth) > 0.0:
        raise ValueError(f"{what}: smooth must be > 0, got {smooth!r}")


def seg_softmax_dice_loss(logits: torch.Tensor, labels: torch.Tensor, mode: int, w_point: float, gamma: float,
                          smooth: float, class_weight: Optional[torch.Tensor], ignore_index: int, sums: torch.Tensor,
                          bad_labels: torch.Tensor, grad: Optional[torch.Tensor], grad_scale: float,
                          loss: torch.Tensor) -> None:
    """w_point * Point + (1 - w_point) * Dice on fp32 class planes [n, K, h, w] (K = 2..16) against int64 labels
    [n, h, w]; Dice = 1 - mean over classes 1..K-1 of (2 I_k + smooth) / (P_k + T_k + smooth) over the whole batch.
    mode 0: Point = nn.CrossEntropyLoss(weight=class_weight, ignore_index); mode 1: Point = the softmax focal loss
    mean a[y] (1 - p_y)^gamma (-log p_y), a = class_weight.  loss (fp64 [1]) is written, grad = grad_scale *
    d(loss)/d(logits); sums is an fp64 workspace of >= 3(K-1)+2; bad_labels (int64 [1]) counts the labels outside
    [0, K) that are not ignore_index (they contribute nothing)."""
    what = "seg_softmax_dice_loss"
    if mode not in (0, 1):
        raise ValueError(f"{what}: mode must be 0 (cross-entropy) or 1 (focal), got {mode!r}")
    check_dice_args(what, w_point, gamma, smooth)
    if logits.dim() != 4:
        raise ValueError(f"{what}: logits must be class planes [n, K, h, w], got {tuple(logits.shape)}")
    n, k = logits.shape[0], logits.shape[1]
    hw = logits.shape[2] * logits.shape[3]
    if not 2 <= k <= MAX_CLASSES:
        raise ValueError(f"{what}: the number of classes must be in 2..{MAX_CLASSES}, got {k}")
    _planes(logits, n, k, hw, what, "logits")
    _labels(labels, n, hw, what)
    if grad is not None:
        _planes(grad, n, k, hw, what, "grad")
    if class_weight is not None and (class_weight.dtype != torch.float32 or not class_weight.is_contiguous()
                                     or class_weight.numel() != k):
        raise ValueError(f"{what}: class_weight must be contiguous fp32 [{k}]")
    if sums.dtype != torch.float64 or sums.numel() < 3 * (k - 1) + 2 or loss.dtype != torch.float64 or loss.numel() < 1:
        raise ValueError(f"{what}: sums must be fp64 [>= {3 * (k - 1) + 2}] and loss fp64 [1]")
    if bad_labels.dtype != torch.int64 or bad_labels.numel() < 1:
        raise ValueError(f"{what}: bad_labels must be int64 [1]")
    _cuda(what, logits, labels, class_weight, sums, bad_labels, grad, loss)
    _lib.check(_lib.lib().gap_seg_softmax_dice(_ptr(logits), _ptr(labels), k, n, hw, mode, w_point, gamma, smooth,
                                               _ptr(class_weight), int(ignore_index), _ptr(sums), _ptr(bad_labels),
                                               _ptr(grad), grad_scale, _ptr(loss), _stream()), "gap_seg_softmax_dice")


def seg_confusion_ck(logits: torch.Tensor, labels: torch.Tensor, ignore_index: int, counts: torch.Tensor) -> None:
    """counts [n, K, K] (int64, accumulated) += per-sample confusion matrix: rows = label, columns = argmax over the
    K planes of logits [n, K, h, w]; labels equal to ignore_index or outside [0, K) are skipped."""
    what = "seg_confusion_ck"
    if logits.dim() != 4:
        raise ValueError(f"{what}: logits must be class planes [n, K, h, w], got {tuple(logits.shape)}")
    n, k = logits.shape[0], logits.shape[1]
    hw = logits.shape[2] * logits.shape[3]
    _check_k(k, what)
    _planes(logits, n, k, hw, what, "logits")
    _labels(labels, n, hw, what)
    if counts.dtype != torch.int64 or tuple(counts.shape) != (n, k, k) or not counts.is_contiguous():
        raise ValueError(f"{what}: counts must be a contiguous int64 [n={n}, {k}, {k}] tensor")
    _cuda(what, logits, labels, counts)
    _lib.check(_lib.lib().gap_seg_confusion_ck(_ptr(logits), _ptr(labels), k, n, hw, int(ignore_index), _ptr(counts),
                                               _stream()), "gap_seg_confusion_ck")


# ------------------------------------------------------------------------------------------------
# Sliding-window scene inference (gap_b200.h "Sliding-window inference"): a tile grid is (ay, ax), each axis the tuple
# (len, ext, step, n) of scene._scene_grid
# ------------------------------------------------------------------------------------------------
def _scene_grid_args(grid, what: str) -> tuple:
    (h, ey, sy, ny), (w, ex, sx, nx) = grid
    if ey % 16 or ex % 16 or min(h, w, ey, ex, sy, sx, ny, nx) < 1:
        raise ValueError(f"{what}: bad tile grid {grid!r}")
    return h, w, ey, ex, sy, sx, ny, nx


def _scene_input(x: torch.Tensor, c: int, h: int, w: int, what: str, name: str) -> bool:
    """True for a uint8 [h, w, c] scene, False for an fp32 [c, h, w] one (ValueError otherwise)."""
    if x.dtype == torch.uint8 and tuple(x.shape) == (h, w, c) and x.is_contiguous():
        return True
    if x.dtype == torch.float32 and tuple(x.shape) == (c, h, w) and x.is_contiguous():
        return False
    raise ValueError(f"{what}: {name} must be a contiguous uint8 [{h}, {w}, {c}] or fp32 [{c}, {h}, {w}] scene, got "
                     f"{x.dtype} {tuple(x.shape)}")


def _tta_extent(d, ey: int, ex: int, what: str) -> Tuple[int, int]:
    """The extent of the dihedral transform d (0..7, d = 4 s + 2 v + u) of an [ey, ex] tile: [ex, ey] when s = 1."""
    if isinstance(d, bool) or not isinstance(d, int) or not 0 <= d <= 7:
        raise ValueError(f"{what}: d must be an int in 0..7, got {d!r}")
    return (ex, ey) if d & 4 else (ey, ex)


def scene_gather(img1: torch.Tensor, img2: torch.Tensor, grid, tile0: int, out1: torch.Tensor, out2: torch.Tensor,
                 d: int = 0) -> None:
    """Tiles tile0 .. tile0 + batch - 1 of both scenes (uint8 [H, W, C] normalised as dataset.py does, or fp32 [C, H, W]
    rounded to bf16) -> out1 / out2, dense NHWC bf16 [batch, E_y, E_x, 4]; slots >= C and tiles past the grid are zero.
    d (0..7): each tile is replaced by its dihedral transform d = 4 s + 2 v + u (transposed if s, then rows flipped if
    v, then columns flipped if u), so out1 / out2 are [batch, E_x, E_y, 4] when s = 1."""
    what = "scene_gather"
    h, w, ey, ex, sy, sx, ny, nx = _scene_grid_args(grid, what)
    oy, ox = _tta_extent(d, ey, ex, what)
    c = img1.shape[-1] if img1.dtype == torch.uint8 else img1.shape[0]
    if not 1 <= c <= 4:
        raise ValueError(f"{what}: scenes of 1 to 4 channels are supported, got {c}")
    u8 = _scene_input(img1, c, h, w, what, "img1")
    if _scene_input(img2, c, h, w, what, "img2") != u8:
        raise ValueError(f"{what}: img1 and img2 must have the same dtype")
    batch = out1.shape[0]
    for name, o in (("out1", out1), ("out2", out2)):
        if o.dtype != torch.bfloat16 or tuple(o.shape) != (batch, oy, ox, 4) or not o.is_contiguous():
            raise ValueError(f"{what}: {name} must be a contiguous bf16 [batch, {oy}, {ox}, 4] tensor, got "
                             f"{o.dtype} {tuple(o.shape)}")
        if o.data_ptr() % 8:
            raise ValueError(f"{what}: {name} must be 8-byte aligned (each 4-slot pixel is one 8-byte store)")
    if not 0 <= tile0 < ny * nx:
        raise ValueError(f"{what}: tile0 = {tile0} outside the {ny * nx} tiles of the grid")
    _cuda(what, img1, img2, out1, out2)
    _lib.check(_lib.lib().gap_scene_gather_tta(_ptr(img1), _ptr(img2), int(u8), c, h, w, ey, ex, sy, sx, ny, nx,
                                               int(tile0), batch, d, _ptr(out1), _ptr(out2), _stream()),
               "gap_scene_gather_tta")


def scene_blend(logits: torch.Tensor, grid, tile0: int, acc: torch.Tensor, wsum: torch.Tensor, d: int = 0,
                first_pass: bool = True) -> None:
    """Window-weighted probabilities of one batch of tile logits (fp32 [batch, E_y, E_x] for K = 1, [batch, K, E_y, E_x]
    for K > 1) -> acc [K, H, W] += w * p, wsum [H, W] += w (fp32) at every scene pixel the batch covers.
    d (0..7): the logits are those of scene_gather(..., d)'s transformed tiles ([.., E_x, E_y] when d >= 4) and are
    mapped back by the inverse transform.  first_pass: a pixel's sums may start from zero at its first covering tile
    (the accumulators need no clearing); False for every later pass over the grid, which adds onto acc / wsum."""
    what = "scene_blend"
    h, w, ey, ex, sy, sx, ny, nx = _scene_grid_args(grid, what)
    oy, ox = _tta_extent(d, ey, ex, what)
    k = 1 if logits.dim() == 3 else (logits.shape[1] if logits.dim() == 4 else -1)
    _check_k(k, what)
    batch = logits.shape[0]
    if logits.dtype != torch.float32 or not logits.is_contiguous() or tuple(logits.shape[-2:]) != (oy, ox):
        raise ValueError(f"{what}: logits must be contiguous fp32 [batch, (K,) {oy}, {ox}], got {logits.dtype} "
                         f"{tuple(logits.shape)}")
    if acc.dtype != torch.float32 or tuple(acc.shape) != (k, h, w) or not acc.is_contiguous():
        raise ValueError(f"{what}: acc must be a contiguous fp32 [{k}, {h}, {w}] tensor")
    if wsum.dtype != torch.float32 or tuple(wsum.shape) != (h, w) or not wsum.is_contiguous():
        raise ValueError(f"{what}: wsum must be a contiguous fp32 [{h}, {w}] tensor")
    if not 0 <= tile0 < ny * nx:
        raise ValueError(f"{what}: tile0 = {tile0} outside the {ny * nx} tiles of the grid")
    _cuda(what, logits, acc, wsum)
    _lib.check(_lib.lib().gap_scene_blend_tta(_ptr(logits), k, h, w, ey, ex, sy, sx, ny, nx, int(tile0), batch, d,
                                              int(bool(first_pass)), _ptr(acc), _ptr(wsum), _stream()),
               "gap_scene_blend_tta")


def scene_finalize(acc: torch.Tensor, wsum: torch.Tensor, pred: torch.Tensor, write_probs: bool,
                   labels: Optional[torch.Tensor] = None, ignore_index: int = -100,
                   counts: Optional[torch.Tensor] = None) -> None:
    """pred (uint8 [H, W]) = argmax of acc / wsum over K (K = 1: > 0.5); write_probs: acc becomes the probabilities in
    place.  With labels (int64 [H, W]) counts (int64, accumulated) += the [K, K] confusion matrix (K = 1: [TP, FP, FN,
    TN]) over pixels whose label is not ignore_index and lies in [0, K) ({0, 1} for K = 1)."""
    what = "scene_finalize"
    if acc.dim() != 3:
        raise ValueError(f"{what}: acc must be fp32 [K, H, W], got {tuple(acc.shape)}")
    k, h, w = acc.shape
    _check_k(k, what)
    if acc.dtype != torch.float32 or not acc.is_contiguous():
        raise ValueError(f"{what}: acc must be a contiguous fp32 [K, H, W] tensor")
    if wsum.dtype != torch.float32 or tuple(wsum.shape) != (h, w) or not wsum.is_contiguous():
        raise ValueError(f"{what}: wsum must be a contiguous fp32 [{h}, {w}] tensor")
    if pred.dtype != torch.uint8 or tuple(pred.shape) != (h, w) or not pred.is_contiguous():
        raise ValueError(f"{what}: pred must be a contiguous uint8 [{h}, {w}] tensor")
    if (labels is None) != (counts is None):
        raise ValueError(f"{what}: labels and counts go together")
    if labels is not None:
        if labels.dtype != torch.int64 or tuple(labels.shape) != (h, w) or not labels.is_contiguous():
            raise ValueError(f"{what}: labels must be a contiguous int64 [{h}, {w}] tensor")
        shape = (4,) if k == 1 else (k, k)
        if counts.dtype != torch.int64 or tuple(counts.shape) != shape or not counts.is_contiguous():
            raise ValueError(f"{what}: counts must be a contiguous int64 {list(shape)} tensor")
    _cuda(what, acc, wsum, pred, labels, counts)
    _lib.check(_lib.lib().gap_scene_finalize(_ptr(acc), _ptr(wsum), k, h * w, _ptr(pred), int(bool(write_probs)),
                                             _ptr(labels), int(ignore_index), _ptr(counts), _stream()),
               "gap_scene_finalize")


def scene_gather_one(img: torch.Tensor, grid, tile0: int, out: torch.Tensor) -> None:
    """Tiles tile0 .. tile0 + batch - 1 of one scene (uint8 [H, W, C] normalised as dataset.py does, or fp32 [C, H, W]
    rounded to bf16) -> out, dense NHWC bf16 [batch, E_y, E_x, 4] (the generator's input batch); slots >= C and tiles
    past the grid are zero."""
    what = "scene_gather_one"
    h, w, ey, ex, sy, sx, ny, nx = _scene_grid_args(grid, what)
    c = (img.shape[-1] if img.dtype == torch.uint8 else img.shape[0]) if img.dim() == 3 else 0
    if not 1 <= c <= 4:
        raise ValueError(f"{what}: scenes of 1 to 4 channels are supported, got {img.dtype} {tuple(img.shape)}")
    u8 = _scene_input(img, c, h, w, what, "img")
    batch = out.shape[0]
    if out.dtype != torch.bfloat16 or tuple(out.shape) != (batch, ey, ex, 4) or not out.is_contiguous():
        raise ValueError(f"{what}: out must be a contiguous bf16 [batch, {ey}, {ex}, 4] tensor, got {out.dtype} "
                         f"{tuple(out.shape)}")
    if out.data_ptr() % 8:
        raise ValueError(f"{what}: out must be 8-byte aligned (each 4-slot pixel is one 8-byte store)")
    if not 0 <= tile0 < ny * nx:
        raise ValueError(f"{what}: tile0 = {tile0} outside the {ny * nx} tiles of the grid")
    _cuda(what, img, out)
    _lib.check(_lib.lib().gap_scene_gather_one(_ptr(img), int(u8), c, h, w, ey, ex, sy, sx, ny, nx, int(tile0), batch,
                                               _ptr(out), _stream()), "gap_scene_gather_one")


SCENE_MAX_WINDOW = 12288        # ey + ex of gap_scene_blend_image: its window table lives in shared memory


def scene_blend_image(fake: torch.Tensor, grid, tile0: int, acc: torch.Tensor, wsum: torch.Tensor) -> None:
    """Window-weighted generator outputs of one batch of tiles (fp32 [batch, E_y, E_x, 4], channels >= C unused) ->
    acc [C, H, W] += w * v, wsum [H, W] += w (fp32) at every scene pixel the batch covers; C = acc.shape[0] in 1..4."""
    what = "scene_blend_image"
    h, w, ey, ex, sy, sx, ny, nx = _scene_grid_args(grid, what)
    if acc.dim() != 3 or not 1 <= acc.shape[0] <= 4:
        raise ValueError(f"{what}: acc must be fp32 [C, {h}, {w}] with C in 1..4, got {tuple(acc.shape)}")
    c = acc.shape[0]
    if acc.dtype != torch.float32 or tuple(acc.shape) != (c, h, w) or not acc.is_contiguous():
        raise ValueError(f"{what}: acc must be a contiguous fp32 [{c}, {h}, {w}] tensor")
    if wsum.dtype != torch.float32 or tuple(wsum.shape) != (h, w) or not wsum.is_contiguous():
        raise ValueError(f"{what}: wsum must be a contiguous fp32 [{h}, {w}] tensor")
    batch = fake.shape[0] if fake.dim() == 4 else 0
    if fake.dtype != torch.float32 or tuple(fake.shape) != (batch, ey, ex, 4) or not fake.is_contiguous() or batch < 1:
        raise ValueError(f"{what}: fake must be a contiguous fp32 [batch, {ey}, {ex}, 4] tensor, got {fake.dtype} "
                         f"{tuple(fake.shape)}")
    if fake.data_ptr() % 16:
        raise ValueError(f"{what}: fake must be 16-byte aligned (each 4-slot pixel is one 16-byte load)")
    if ey + ex > SCENE_MAX_WINDOW:
        raise ValueError(f"{what}: tile extents {ey} + {ex} exceed {SCENE_MAX_WINDOW}")
    if not 0 <= tile0 < ny * nx:
        raise ValueError(f"{what}: tile0 = {tile0} outside the {ny * nx} tiles of the grid")
    _cuda(what, fake, acc, wsum)
    _lib.check(_lib.lib().gap_scene_blend_image(_ptr(fake), c, h, w, ey, ex, sy, sx, ny, nx, int(tile0), batch,
                                                _ptr(acc), _ptr(wsum), _stream()), "gap_scene_blend_image")


def scene_finalize_image(acc: torch.Tensor, wsum: torch.Tensor, image: torch.Tensor, write_float: bool) -> None:
    """image (uint8 [H, W, C]) = uint8(clamp((v * 0.5 + 0.5) * 255, 0, 255)), truncated, of v = acc / wsum;
    write_float: acc (fp32 [C, H, W]) becomes v in place."""
    what = "scene_finalize_image"
    if acc.dim() != 3 or not 1 <= acc.shape[0] <= 4:
        raise ValueError(f"{what}: acc must be fp32 [C, H, W] with C in 1..4, got {tuple(acc.shape)}")
    c, h, w = acc.shape
    if acc.dtype != torch.float32 or not acc.is_contiguous():
        raise ValueError(f"{what}: acc must be a contiguous fp32 [C, H, W] tensor")
    if wsum.dtype != torch.float32 or tuple(wsum.shape) != (h, w) or not wsum.is_contiguous():
        raise ValueError(f"{what}: wsum must be a contiguous fp32 [{h}, {w}] tensor")
    if image.dtype != torch.uint8 or tuple(image.shape) != (h, w, c) or not image.is_contiguous():
        raise ValueError(f"{what}: image must be a contiguous uint8 [{h}, {w}, {c}] tensor")
    _cuda(what, acc, wsum, image)
    _lib.check(_lib.lib().gap_scene_finalize_image(_ptr(acc), _ptr(wsum), c, h * w, _ptr(image),
                                                   int(bool(write_float)), _stream()), "gap_scene_finalize_image")


# ------------------------------------------------------------------------------------------------
# Change objects (gap_b200.h "Change objects"): connected components of a class map [n, h, w], flat int32 buffers of
# n*h*w pixels
# ------------------------------------------------------------------------------------------------
OBJECTS_CHUNK = 4096            # pixels per entry of gap_objects_number's chunk scratch


def _flat(t: Optional[torch.Tensor], numel: int, dtype, what: str, name: str) -> None:
    if t is not None and (t.dtype != dtype or t.numel() != numel or not t.is_contiguous()):
        raise ValueError(f"{what}: {name} must be a contiguous {dtype} tensor of {numel} elements, got {t.dtype} "
                         f"{tuple(t.shape)}")


def objects_label(src: torch.Tensor, n: int, h: int, w: int, k: int, connectivity: int, parent: torch.Tensor,
                  area: torch.Tensor, classes: Optional[torch.Tensor] = None, info: Optional[torch.Tensor] = None,
                  ignore_index: int = -100) -> None:
    """Components of a uint8 pred (info: int32 [2], info[1] counts values >= max(k, 2)) or of int64 labels (classes:
    uint8, the label class or 255 for ignore_index / out-of-range labels): parent <- each pixel's root, area <- the
    pixel count at each root (int32, n*h*w each)."""
    what = "objects_label"
    _check_k(k, what)
    px = n * h * w
    i64 = src.dtype == torch.int64
    _flat(src, px, torch.int64 if i64 else torch.uint8, what, "src")
    for name, t, dt in (("parent", parent, torch.int32), ("area", area, torch.int32), ("classes", classes, torch.uint8),
                        ("info", info, torch.int32)):
        _flat(t, 2 if name == "info" else px, dt, what, name)
    if i64 != (classes is not None) or (not i64 and info is None):
        raise ValueError(f"{what}: int64 labels need classes, a uint8 pred needs info")
    _cuda(what, src, parent, area, classes, info)
    _lib.check(_lib.lib().gap_objects_label(_ptr(src), int(i64), n, h, w, k, int(ignore_index), int(connectivity),
                                            _ptr(classes), _ptr(parent), _ptr(area), _ptr(info), _stream()),
               "gap_objects_label")


def objects_number(pred: torch.Tensor, parent: torch.Tensor, area_ids: torch.Tensor, min_area: int,
                   chunk: torch.Tensor, info: torch.Tensor) -> None:
    """Roots of non-zero class with area >= min_area get ids 1..count in raster order (area_ids[root], 0 for the
    others); info[0] <- count.  chunk: int32 scratch of ceil(pixels / OBJECTS_CHUNK)."""
    what = "objects_number"
    px = pred.numel()
    _flat(pred, px, torch.uint8, what, "pred")
    _flat(parent, px, torch.int32, what, "parent")
    _flat(area_ids, px, torch.int32, what, "area_ids")
    _flat(chunk, -(-px // OBJECTS_CHUNK), torch.int32, what, "chunk")
    _flat(info, 2, torch.int32, what, "info")
    _cuda(what, pred, parent, area_ids, chunk, info)
    _lib.check(_lib.lib().gap_objects_number(_ptr(pred), _ptr(parent), _ptr(area_ids), px, int(min_area), _ptr(chunk),
                                             _ptr(info), _stream()), "gap_objects_number")


def objects_finish(pred: torch.Tensor, parent: torch.Tensor, ids: torch.Tensor, n: int, h: int, w: int, k: int,
                   count: int, pred_out: torch.Tensor, objects: torch.Tensor, overlap: Optional[torch.Tensor] = None,
                   lparent: Optional[torch.Tensor] = None, larea: Optional[torch.Tensor] = None,
                   loverlap: Optional[torch.Tensor] = None, min_overlap: float = 0.0,
                   confusion: Optional[torch.Tensor] = None, object_counts: Optional[torch.Tensor] = None) -> None:
    """ids of every pixel, pred_out (pred with dropped objects zeroed) and objects (int64 [count, 7]); with the label
    map's lparent / larea (and its classes in pred_out on entry): confusion and object_counts (see gap_b200.h)."""
    what = "objects_finish"
    _check_k(k, what)
    px = n * h * w
    kk = max(k, 2)
    for name, t, numel, dt in (("pred", pred, px, torch.uint8), ("parent", parent, px, torch.int32),
                               ("ids", ids, px, torch.int32), ("pred_out", pred_out, px, torch.uint8),
                               ("objects", objects, count * 7, torch.int64), ("overlap", overlap, count, torch.int32),
                               ("lparent", lparent, px, torch.int32), ("larea", larea, px, torch.int32),
                               ("loverlap", loverlap, px, torch.int32),
                               ("confusion", confusion, 4 if k == 1 else k * k, torch.int64),
                               ("object_counts", object_counts, kk * 4, torch.int64)):
        _flat(t, numel, dt, what, name)
    labelled = (lparent, larea, loverlap, confusion, object_counts, overlap)
    if any(t is None for t in labelled) and any(t is not None for t in labelled):
        raise ValueError(f"{what}: lparent, larea, loverlap, overlap, confusion and object_counts go together")
    _cuda(what, pred, parent, ids, pred_out, objects, *labelled)
    _lib.check(_lib.lib().gap_objects_finish(_ptr(pred), _ptr(parent), _ptr(ids), n, h, w, k, int(count),
                                             _ptr(pred_out), _ptr(overlap), _ptr(objects), _ptr(lparent), _ptr(larea),
                                             _ptr(loverlap), float(min_overlap), _ptr(confusion),
                                             _ptr(object_counts), _stream()), "gap_objects_finish")
