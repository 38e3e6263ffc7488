"""Native Siamese U-Net engine: SiameseUNet (models.py:47-145) forward / backward and one train.py
iteration (train.py:137-146), sequenced as C-ABI kernel launches over the same tcgen05 conv kernels as
the Pix2Pix engines.

What it mirrors in the reference:
  * double_conv (models.py:7-15), AttentionGate (models.py:18-44), SiameseUNet (models.py:47-145)
  * CombinedLoss / FocalDiceLoss (train.py:82-128), AdamW (train.py:295), train_one_epoch's loop body

Data layout: activations NHWC bf16; the two encoder branches write their skip features straight into the
channel slots of the concatenated skip buffers S_k = [conv_k(x1) | conv_k(x2)] and the decoder inputs live in
D_k = [upsample(prev) | attention(S_k)], so no torch.cat ever copies.  The shared encoder runs twice, so its
BatchNorm layers keep one set of saved statistics per pass (and update their running buffers twice, like the
reference).  Single-channel maps (psi, logits) are fp32.

Classes: n_classes = K = 1..16.  The logits and their gradient are fp32 class planes [n][K][h][w] (NCHW, what
nn.CrossEntropyLoss and torch.argmax(dim=1) expect; for K = 1 the same memory as the [n][h][w] map, which keeps its
shape).  K = 1 runs the single-channel conv_last kernels and the sigmoid losses; K > 1 runs the gap_conv1x1_ck_* head
kernels and softmax cross-entropy (`kind="ce"`), or softmax cross-entropy / focal loss with a multi-class Dice term
(`kind="ce_dice"` / `"softmax_focal_dice"`, gap_seg_softmax_dice).
"""
from __future__ import annotations

from typing import Callable, Dict, List, NamedTuple, Optional, Tuple

import torch

from . import ops
from .ops import ACT_NONE, ACT_RELU
from .pix2pix import BN_EPS, BN_MOMENTUM, _BN, _Net, _on_device
from .scene import _scene_grid, scene_axis, scene_window  # noqa: F401  (predict_scene's grid and window)

ENC = (("dconv_down1", 64), ("dconv_down2", 128), ("dconv_down3", 256), ("dconv_down4", 512), ("bottleneck", 1024))
MAX_CLASSES = ops.MAX_CLASSES
MULTI_KINDS = ("ce", "ce_dice", "softmax_focal_dice")       # loss kinds of n_classes > 1
SINGLE_KINDS = ("combined", "focal_dice")                   # loss kinds of n_classes = 1
DICE_KW = {"ce_dice": {"alpha": 0.5, "smooth": 1.0, "class_weight": None, "ignore_index": -100},
           "softmax_focal_dice": {"beta": 0.5, "gamma": 2.0, "smooth": 1.0, "class_weight": None, "ignore_index": -100}}
DEC = (("att3", "dconv_up3", 2048, 1024, 512), ("att2", "dconv_up2", 512, 512, 256), ("att1", "dconv_up1", 256, 256, 128),
       ("att_last", "dconv_last", 128, 128, 64))      # (gate, block, F_g, F_l, block out channels)


def check_n_classes(n_classes) -> None:
    """NotImplementedError unless n_classes is an int in 1..16 (the classes the native head kernels cover)."""
    if isinstance(n_classes, bool) or not isinstance(n_classes, int) or not 1 <= n_classes <= MAX_CLASSES:
        raise NotImplementedError(f"n_classes = {n_classes!r} is not implemented natively: 1 to {MAX_CLASSES} classes "
                                  "are")


class SceneResult(NamedTuple):
    """predict_scene's result; fields that were not asked for are None.
    pred: uint8 [H, W] class map (K = 1: 0/1).  probs: fp32 [K, H, W] blended probabilities (K = 1: the sigmoid).
    confusion: int64 [K, K] (rows = label, columns = prediction) or, K = 1, [TP, FP, FN, TN]."""
    pred: torch.Tensor
    probs: Optional[torch.Tensor]
    confusion: Optional[torch.Tensor]


def _k(name: str, leaf: str) -> str:
    """state_dict key of `leaf` inside the sub-module `name` ("" = the engine's root module is that sub-module)."""
    return leaf if not name else name + "." + leaf


class _Saved:
    """BatchNorm statistics of one layer evaluation (the shared encoder evaluates each layer twice)."""

    def __init__(self, c: int, dev) -> None:
        self.scale = torch.empty(c, device=dev)
        self.shift = torch.empty(c, device=dev)
        self.mean = torch.empty(c, device=dev)
        self.invstd = torch.empty(c, device=dev)


class SiameseEngine(_Net):
    """SiameseUNet(n_channels, n_classes), n_channels = 1..4 (default 3), n_classes = 1..16 (default 1)."""

    def __init__(self, device, n_channels: int = 3, n_classes: int = 1) -> None:
        super().__init__(device)
        check_n_classes(n_classes)
        if not isinstance(n_channels, int) or not 1 <= n_channels <= 4:
            raise NotImplementedError(f"n_channels = {n_channels!r} is not implemented natively: images of 1 to 4 "
                                      "channels are")
        self.n_channels, self.n_classes = n_channels, n_classes
        self.key_order: List[str] = []
        self.conv_meta: Dict[str, Tuple[int, int, int]] = {}      # conv key -> (cout, cin, k)
        # ---- registration in the reference's module order (models.py:54-90) = state_dict order
        cin = n_channels
        for name, c in ENC:
            self._reg_double_conv(name, cin, c)
            cin = c
        for gate, _, fg, fl, _ in DEC:
            self._reg_gate(gate, fg, fl, fl // 2)
        for _, block, fg, fl, cout in DEC:
            self._reg_double_conv(block, fg + fl, cout)
        self._reg("conv_last.weight", n_classes * 64, (n_classes, 64, 1, 1), (64, 1, 1, 1))
        self._reg_vec("conv_last.bias", n_classes)
        self.key_order += ["conv_last.weight", "conv_last.bias"]
        self.store.allocate(device)
        for bn in self.bns.values():
            bn.allocate(device)
        # ---- packed bf16 operands (zero-filled once)
        bf = dict(device=device, dtype=torch.bfloat16)
        self.w_fwd: Dict[str, torch.Tensor] = {}
        self.w_dg: Dict[str, torch.Tensor] = {}
        for key, (co, ci, k) in self.conv_meta.items():
            if ci <= 4:
                self.w_fwd[key] = torch.zeros(1, co, 64, **bf)          # im2col form, K = 9*ci padded to 64; no dgrad
                continue
            self.w_fwd[key] = torch.zeros(1, co, k * k * ci, **bf)
            self.w_dg[key] = torch.zeros(1, ci, k * k * co, **bf)
        self._plan = None
        self._n = None
        self._tape: List[Callable[[], None]] = []
        self._marks: Dict[int, int] = {}     # tape index -> flat-buffer offset from which every gradient is final once
        #                                      that entry has run (the backward pass finalises the buffer tail first)
        self.reducer = None                  # parallel.TailReducer when data parallel (see train_step)
        # cross-entropy (n_classes > 1): fp64 workspace, and the count of labels outside [0, K) that are not
        # ignore_index (they contribute nothing to the loss; the count is never reset by the engine)
        self.ce_sums = torch.zeros(2, device=device, dtype=torch.float64)
        self.dice_sums = torch.zeros(ops.DICE_SUMS, device=device, dtype=torch.float64)     # the Dice kinds' sums
        self.bad_labels = torch.zeros(1, device=device, dtype=torch.int64)
        self._cw_cache = (None, None)

    # -- registration ------------------------------------------------------------------------------
    def _reg_convk(self, key: str, cout: int, cin: int, k: int, bias: bool) -> None:
        if cin <= 4:      # the image-side first conv: [cout][(kh*3+kw)*cin + c] padded to 64
            self._reg(key + ".weight", cout * 64, (cout, cin, k, k), (64, 1, cin * k, cin))
        else:             # [cout][kh][kw][cin]
            self._reg(key + ".weight", cout * k * k * cin, (cout, cin, k, k), (k * k * cin, 1, k * cin, cin))
        self.conv_meta[key] = (cout, cin, k)
        self.key_order.append(key + ".weight")
        if bias:
            self._reg_vec(key + ".bias", cout)
            self.key_order.append(key + ".bias")

    def _reg_bn_keys(self, prefix: str, c: int) -> None:
        self._reg_bn(prefix, c)
        self.key_order += [prefix + s for s in (".weight", ".bias", ".running_mean", ".running_var", ".num_batches_tracked")]

    def _reg_double_conv(self, name: str, cin: int, cout: int) -> None:
        self._reg_convk(name + ".0", cout, cin, 3, False)
        self._reg_bn_keys(name + ".1", cout)
        self._reg_convk(name + ".3", cout, cout, 3, False)
        self._reg_bn_keys(name + ".4", cout)

    def _reg_gate(self, name: str, fg: int, fl: int, fint: int) -> None:
        self._reg_convk(_k(name, "W_g.0"), fint, fg, 1, True)
        self._reg_bn_keys(_k(name, "W_g.1"), fint)
        self._reg_convk(_k(name, "W_x.0"), fint, fl, 1, True)
        self._reg_bn_keys(_k(name, "W_x.1"), fint)
        self._reg(_k(name, "psi.0.weight"), fint, (1, fint, 1, 1), (fint, 1, 1, 1))
        self._reg_vec(_k(name, "psi.0.bias"), 1)
        self.key_order += [_k(name, "psi.0.weight"), _k(name, "psi.0.bias")]
        self._reg_bn_keys(_k(name, "psi.1"), 1)

    # -- operands ------------------------------------------------------------------------------------
    def repack(self) -> None:
        if self._plan is None:
            plan = ops.PackPlan()
            p, off = self.store.p, self.store.off
            for key, (co, ci, k) in self.conv_meta.items():
                o = off(key + ".weight")
                if ci <= 4:
                    plan.add(p, o, self.w_fwd[key], 0, 1, co, co, (1, 1), 64, 64, 64, (64, 1, 0, 0))
                    continue
                kk = k * k
                plan.add(p, o, self.w_fwd[key], 0, 1, co, co, (k, k), ci, ci, kk * ci, (kk * ci, 1, k * ci, ci))
                plan.add(p, o, self.w_dg[key], 1, 1, ci, ci, (k, k), co, co, kk * co, (1, kk * ci, k * ci, ci))
            self._plan = plan
        self._plan.run()

    # -- buffers -------------------------------------------------------------------------------------
    def _alloc(self, n: int, h: int, w: int) -> None:
        if self._n == (n, h, w):
            return
        if h % 16 or w % 16:
            raise ValueError(f"input {h}x{w} must be divisible by 16")
        dev = self.dev
        bf = dict(device=dev, dtype=torch.bfloat16)
        z = lambda hh, ww, c: torch.zeros(n, hh, ww, c, **bf)
        self.x_in = [z(h, w, 4), z(h, w, 4)]
        self.col = [z(h, w, 64), z(h, w, 64)]
        self.S, self.gS = [], []            # concatenated skip features of levels 1..4 and the bottleneck pair
        for lvl, (_, c) in enumerate(ENC):
            hh, ww = h >> lvl, w >> lvl
            self.S.append(z(hh, ww, 2 * c))
            self.gS.append(z(hh, ww, 2 * c))
        self.D, self.gD = [], []            # decoder inputs [upsampled | attended skip]
        for i, (_, _, fg, fl, _) in enumerate(DEC):
            lvl = 3 - i
            hh, ww = h >> lvl, w >> lvl
            self.D.append(z(hh, ww, fg + fl))
            self.gD.append(z(hh, ww, fg + fl))
        planes = (n, h, w) if self.n_classes == 1 else (n, self.n_classes, h, w)
        self.logits = torch.empty(*planes, device=dev)
        self.dlogits = torch.zeros(*planes, device=dev)
        self.tmp: Dict[Tuple[int, ...], torch.Tensor] = {}
        self.saved: Dict[Tuple[str, int], _Saved] = {}
        self.loss_sums = torch.zeros(4, device=dev, dtype=torch.float64)
        self.loss_out = torch.zeros(1, device=dev, dtype=torch.float64)
        self._n = (n, h, w)

    def _scratch(self, tag: str, shape, dtype=torch.bfloat16) -> torch.Tensor:
        key = (tag, tuple(shape), dtype)
        t = self.tmp.get(key)
        if t is None:
            t = torch.empty(*shape, device=self.dev, dtype=dtype)
            self.tmp[key] = t
        return t

    def _sv(self, name: str, pass_id: int, c: int) -> _Saved:
        key = (name, pass_id)
        if key not in self.saved:
            self.saved[key] = _Saved(c, self.dev)
        return self.saved[key]

    # -- BatchNorm of one evaluation -----------------------------------------------------------------
    def _bn_stats(self, bn: _BN, sv: _Saved, count: int) -> None:
        gamma, beta = self.param(bn.name + ".weight"), self.param(bn.name + ".bias")
        if self.training:
            ops.bn_finalize(bn.stats, count, gamma, beta, BN_EPS, BN_MOMENTUM, 1, bn.running_mean, bn.running_var, bn.nbt,
                            sv.scale, sv.shift, sv.mean, sv.invstd)
        else:
            ops.bn_eval_scale_shift(gamma, beta, bn.running_mean, bn.running_var, BN_EPS, sv.scale, sv.shift)

    def _bn_bwd(self, bn: _BN, sv: _Saved, y: torch.Tensor, g: torch.Tensor, slope: float, dy: torch.Tensor) -> None:
        count = y.numel() // y.shape[-1]
        ops.bn_bwd_reduce(y, g, None, slope, sv.scale, sv.shift, sv.mean, sv.invstd, bn.sums)
        ops.bn_bwd_apply(y, g, None, slope, sv.scale, sv.shift, sv.mean, sv.invstd, bn.sums, count, dy)
        ops.bn_param_grads(bn.sums, self.grad(bn.name + ".weight"), self.grad(bn.name + ".bias"))

    # -- layers --------------------------------------------------------------------------------------
    def _conv_bn_relu(self, x: torch.Tensor, key: str, out: torch.Tensor, pass_id: int, gx: Optional[torch.Tensor],
                      gout: torch.Tensor, gx_accumulate: bool = False, gout_premasked: bool = False,
                      below: Optional[dict] = None) -> dict:
        """out = ReLU(BN(conv3x3(x))) (models.py:9-14).  gout: gradient buffer of `out`; gx: gradient buffer of `x`
        (None: the network input).  gout_premasked: the consumer's dgrad epilogue already applied this layer's ReLU
        backward and accumulated its BatchNorm sums (bn.sums holds [sum d, sum d*y]).  below: the record of the
        conv-BN-ReLU layer that produced `x`; when given, this layer's dgrad does the same for it."""
        co, ci, k = self.conv_meta[key]
        bn = self.bns[key[:-1] + str(int(key[-1]) + 1)]
        n, h, w, _ = out.shape
        y = self._scratch(f"y.{key}.{pass_id}", (n, h, w, co))
        sv = self._sv(bn.name, pass_id, co)
        if not self.training:
            # eval (train.py:151, evaluate.py:146): BatchNorm folds into the conv epilogue; nothing is kept for backward
            self._bn_stats(bn, sv, n * h * w)
            if ci <= 4:
                ops.conv_gemm([x], self.w_fwd[key], ops.geom_conv_fwd(1, 1, 0), out, co, (h, w), act=ACT_RELU,
                              scale=sv.scale, bias=sv.shift, flops=2.0 * n * h * w * co * 9 * ci)
            else:
                ops.conv_gemm([x], self.w_fwd[key], ops.geom_conv_fwd(3, 1, 1), out, co, (h, w), act=ACT_RELU,
                              scale=sv.scale, bias=sv.shift)
            return {"bn": bn, "sv": sv, "y": y}
        stats = bn.stats
        if ci <= 4:
            ops.conv_gemm([x], self.w_fwd[key], ops.geom_conv_fwd(1, 1, 0), y, co, (h, w), stats=stats,
                          flops=2.0 * n * h * w * co * 9 * ci)
        else:
            ops.conv_gemm([x], self.w_fwd[key], ops.geom_conv_fwd(3, 1, 1), y, co, (h, w), stats=stats)
        self._bn_stats(bn, sv, n * h * w)
        ops.bn_act(y, sv.scale, sv.shift, out, ACT_RELU)

        def backward() -> None:
            # (one dy buffer per layer evaluation: the weight gradient runs on the side stream and may still be reading
            # it when the next layer's backward starts)
            dy = self._scratch(f"dy.{key}.{pass_id}", (n, h, w, co))
            if gout_premasked:
                ops.bn_bwd_finalize(bn.sums, sv.mean, sv.invstd, self.grad(bn.name + ".weight"),
                                    self.grad(bn.name + ".bias"), bn.sums2)
                ops.bn_bwd_apply(y, gout, None, 1.0, sv.scale, sv.shift, sv.mean, sv.invstd, bn.sums2, n * h * w, dy)
            else:
                self._bn_bwd(bn, sv, y, gout, 0.0, dy)
            wseg = self.store.seg(self.store.g, key + ".weight")
            # weight gradients are off the critical path: they run on the side stream (tensor-bound) underneath the
            # HBM-bound BatchNorm / pooling / gate passes of the layers that follow
            if ci <= 4:
                self._fork_wgrad(lambda: ops.conv_wgrad(dy, x, wseg, (1, 1), 1, (0, 0), 64, 0,
                                                        flops=2.0 * n * h * w * co * 9 * ci))
                return
            self._fork_wgrad(lambda: ops.conv_wgrad(dy, x, wseg, (3, 3), 1, (-1, -1), 9 * ci, ci))
            if gx is None:
                return
            if gx_accumulate:       # gx already holds the other consumers' contributions: added in the epilogue
                ops.conv_gemm([dy], self.w_dg[key], ops.geom_conv_dgrad_s1(3, 1), gx, ci, (h, w), accumulate=True)
            elif below is not None:
                b = below
                ops.conv_gemm([dy], self.w_dg[key], ops.geom_conv_dgrad_s1(3, 1), gx, ci, (h, w), stats=b["bn"].sums,
                              bwd={"y": b["y"], "scale": b["sv"].scale, "shift": b["sv"].shift, "slope": 0.0})
            else:
                ops.conv_gemm([dy], self.w_dg[key], ops.geom_conv_dgrad_s1(3, 1), gx, ci, (h, w))

        self._tape.append(backward)
        return {"bn": bn, "sv": sv, "y": y}

    def _double_conv(self, x, name: str, out, pass_id: int, gx, gout, gx_accumulate: bool = False) -> None:
        co = self.conv_meta[name + ".0"][0]
        n, h, w, _ = out.shape
        mid = self._scratch(f"mid.{name}.{pass_id}", (n, h, w, co))
        gmid = self._scratch(f"gmid.{name}.{pass_id}", (n, h, w, co))
        # the second conv's dgrad epilogue applies the first layer's ReLU backward and BatchNorm-backward sums
        rec = self._conv_bn_relu(x, name + ".0", mid, pass_id, gx, gmid, gx_accumulate, gout_premasked=True)
        self._conv_bn_relu(mid, name + ".3", out, pass_id, gmid, gout, below=rec)

    def _conv1x1_bn(self, x: torch.Tensor, key: str, gx: torch.Tensor) -> Tuple[torch.Tensor, _Saved]:
        """y = conv1x1(x) + bias with BatchNorm statistics (AttentionGate W_g / W_x, models.py:21-29).  The gradient
        with respect to x is ADDED to gx (both gate inputs have other consumers)."""
        co, ci, _ = self.conv_meta[key]
        bn = self.bns[key[:-1] + "1"]
        n, h, w, _ = x.shape
        y = self._scratch(f"y.{key}", (n, h, w, co))
        sv = self._sv(bn.name, 0, co)
        ops.conv_gemm([x], self.w_fwd[key], ops.geom_conv_fwd(1, 1, 0), y, co, (h, w), bias=self.param(key + ".bias"),
                      stats=bn.stats if self.training else None)
        self._bn_stats(bn, sv, n * h * w)

        def backward(d: torch.Tensor) -> None:
            dy = self._scratch("dy", (n, h, w, co))
            self._bn_bwd(bn, sv, y, d, 1.0, dy)
            ops.conv_wgrad(dy, x, self.store.seg(self.store.g, key + ".weight"), (1, 1), 1, (0, 0), ci, 0)
            # (the conv bias feeds a training-mode BatchNorm, which subtracts the batch mean: its gradient, the
            # per-channel sum of dy, is identically zero -- autograd's value for it is rounding noise of relative size
            # 1e-7, tests/test_oracle_vs_reference.py pins that -- so it stays at the zero zero_grad() wrote instead of
            # costing a pass over dy)
            ops.conv_gemm([dy], self.w_dg[key], ops.geom_conv_fwd(1, 1, 0), gx, ci, (h, w), accumulate=True)

        return y, sv, backward

    def _gate(self, name: str, g: torch.Tensor, gg: torch.Tensor, x: torch.Tensor, gxs: torch.Tensor, out: torch.Tensor,
              gout: torch.Tensor) -> None:
        """out = x * Sigmoid(BN(psi(ReLU(BN(W_g g) + BN(W_x x)))))   (AttentionGate.forward, models.py:39-44).
        gg / gxs: gradient buffers of g / x; gout: gradient buffer of out.  The gate writes the FIRST contribution to
        gxs (through x * psi); the W_g / W_x input gradients are added to gg / gxs."""
        n, h, w, fl = x.shape
        fint = self.conv_meta[_k(name, "W_g.0")][0]
        pix = n * h * w
        yg, svg, bwd_g = self._conv1x1_bn(g, _k(name, "W_g.0"), gg)
        yx, svx, bwd_x = self._conv1x1_bn(x, _k(name, "W_x.0"), gxs)
        s = self._scratch(f"s.{name}", (n, h, w, fint))
        ops.att_add_relu_fwd(yg, svg.scale, svg.shift, yx, svx.scale, svx.shift, s)
        ypsi = self._scratch(f"ypsi.{name}", (pix,), torch.float32)
        psi = self._scratch(f"psi.{name}", (pix,), torch.float32)
        wpsi, bpsi = self.store.seg(self.store.p, _k(name, "psi.0.weight")), self.param(_k(name, "psi.0.bias"))
        ops.conv1x1_cout1_fwd(s, wpsi, bpsi, ypsi)
        bn = self.bns[_k(name, "psi.1")]
        sv = self._sv(bn.name, 0, 1)
        if self.training:
            ops.vec_stats(ypsi, bn.stats)
        self._bn_stats(bn, sv, pix)
        ops.att_gate_fwd(ypsi, sv.scale, sv.shift, psi, x, out)

        def backward() -> None:
            dz = self._scratch("dz", (pix,), torch.float32)
            dyp = self._scratch("dyp", (pix,), torch.float32)
            ops.att_gate_bwd(gout, x, psi, gxs, False, dz)
            ops.vec_bn_bwd(ypsi, dz, sv.scale, sv.mean, sv.invstd, bn.sums, dyp)
            ops.bn_param_grads(bn.sums, self.grad(bn.name + ".weight"), self.grad(bn.name + ".bias"))
            ops.conv1x1_cout1_wgrad(dyp, s, self.store.seg(self.store.g, _k(name, "psi.0.weight")),
                                    self.grad(_k(name, "psi.0.bias")))
            gs = self._scratch("gs", (n, h, w, fint))
            ops.conv1x1_cout1_dgrad(dyp, wpsi, gs)
            d = self._scratch("d", (n, h, w, fint))
            ops.relu_bwd(s, gs, d)
            bwd_x(d)
            bwd_g(d)

        self._tape.append(backward)

    # -- forward ---------------------------------------------------------------------------------------
    def _encode(self, p: int, x: Optional[torch.Tensor]) -> None:
        """forward_encoder (models.py:92-102) for branch p: 4 x (double_conv + MaxPool2d(2)) + bottleneck; the features
        land in the channel slots p of the concatenated skip buffers S[0..4].  x: the fp32 NCHW input, or None when
        x_in[p] already holds it (staged by the scene gather)."""
        n = self.x_in[p].shape[0]
        if x is not None:
            if x.shape[1] != self.n_channels:
                raise ValueError(f"input has {x.shape[1]} channels, expected n_channels = {self.n_channels}")
            ops.nchw_to_nhwc_bf16(x.contiguous().float(), self.x_in[p])
        ops.im2col_k3s1p1(self.x_in[p], self.col[p], self.n_channels)
        src, gsrc = self.col[p], None
        for lvl, (name, c) in enumerate(ENC):
            out = self.S[lvl][..., p * c:(p + 1) * c]
            gout = self.gS[lvl][..., p * c:(p + 1) * c]
            if p == 0:      # pass 0's entries run last in backward: after them this level's segments are final
                self._marks[len(self._tape)] = self.store.off(name + ".0.weight")
            self._double_conv(src, name, out, p, gsrc, gout)
            if lvl < 4:
                nh, nw = out.shape[1] // 2, out.shape[2] // 2
                pooled = self._scratch(f"pool.{lvl}.{p}", (n, nh, nw, c))
                gpooled = self._scratch(f"gpool.{lvl}.{p}", (n, nh, nw, c))
                ops.maxpool2x2_fwd(out, pooled)
                # the skip tensor already holds the decoder's gradient when the pool backward runs: accumulate
                self._tape.append(lambda o=out, gp=gpooled, go=gout: ops.maxpool2x2_bwd(o, gp, go, True))
                src, gsrc = pooled, gpooled

    @_on_device
    def forward_encoder(self, x: torch.Tensor) -> List[torch.Tensor]:
        """SiameseUNet.forward_encoder(x) (models.py:92-102) on its own: returns (conv1, conv2, conv3, conv4, bottleneck)
        as NHWC bf16 views.  backward_encoder() expects the gradients of those five tensors in self.gS[lvl][..., :c]."""
        n, _, h, w = x.shape
        self._alloc(n, h, w)
        self._tape = []
        self._marks = {}
        self._encode(0, x)
        return [self.S[lvl][..., :c] for lvl, (_, c) in enumerate(ENC)]

    @_on_device
    def backward_encoder(self) -> None:
        for idx in range(len(self._tape) - 1, -1, -1):
            self._tape[idx]()
        self._join_wgrad()
        self._tape = []

    @_on_device
    def forward(self, x1: torch.Tensor, x2: torch.Tensor, pred: Optional[torch.Tensor] = None) -> torch.Tensor:
        """x1, x2: fp32 NCHW on the device.  Returns fp32 logits [n, h, w] (n_classes = 1) or class planes
        [n, K, h, w] (n_classes = K > 1); pred (uint8 [n, h, w], K > 1 only) receives the argmax class map."""
        n, _, h, w = x1.shape
        self._alloc(n, h, w)
        return self._forward_from((x1, x2), pred)

    def _forward_from(self, xs, pred: Optional[torch.Tensor] = None) -> torch.Tensor:
        """forward() from the inputs on: xs = (x1, x2) fp32 NCHW, converted into x_in as each encoder pass starts, or
        (None, None) when x_in already holds the batch (the staged path of predict_scene)."""
        self._tape = []
        self._marks = {}
        for p, x in enumerate(xs):
            self._encode(p, x)
        prev, gprev = self.S[4], self.gS[4]          # bottleneck pair (2048 channels)
        self._marks[len(self._tape)] = self.store.off(DEC[0][0] + ".W_g.0.weight")   # gates, decoder blocks, conv_last
        for i, (gate, block, fg, fl, cout) in enumerate(DEC):
            lvl = 3 - i
            d, gd = self.D[i], self.gD[i]
            up, gup = d[..., :fg], gd[..., :fg]
            ops.upsample2x_fwd(prev, up)
            # the block's first conv writes gd completely; the gate then adds W_g's input gradient to gup
            self._tape.append(lambda gu=gup, gp=gprev: ops.upsample2x_bwd(gu, gp, False))
            self._gate(gate, up, gup, self.S[lvl], self.gS[lvl], d[..., fg:], gd[..., fg:])
            nb, hh, ww, _ = d.shape
            out = self._scratch(f"dec.{block}", (nb, hh, ww, cout))
            gout = self._scratch(f"gdec.{block}", (nb, hh, ww, cout))
            self._double_conv(d, block, out, 0, gd, gout)
            prev, gprev = out, gout
        self._last, self._glast = prev, gprev
        if self.n_classes == 1:
            ops.conv1x1_cout1_fwd(prev, self.store.seg(self.store.p, "conv_last.weight"), self.param("conv_last.bias"),
                                  self.logits.view(-1))
        else:
            ops.conv1x1_ck_fwd(prev, self.store.seg(self.store.p, "conv_last.weight"), self.param("conv_last.bias"),
                               self.logits, pred)
        return self.logits

    @_on_device
    def predict(self, x1: torch.Tensor, x2: torch.Tensor, out_u8: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Eval-mode forward (BatchNorm with the running statistics) that returns the uint8 class map [n, h, w]: the
        argmax over the K class planes, ties to the lowest class as torch.argmax(dim=1).  n_classes > 1 only."""
        if self.n_classes == 1:
            raise ValueError("predict() returns the argmax over n_classes > 1 planes; with n_classes = 1 threshold the "
                             "logits of forward()")
        n, _, h, w = x1.shape
        if out_u8 is None:
            out_u8 = torch.empty(n, h, w, device=self.dev, dtype=torch.uint8)
        was = self.training
        self.training = False
        try:
            self.forward(x1, x2, pred=out_u8)
        finally:
            self.training = was
            self._tape = []
        return out_u8

    def _scene_input(self, x, name: str):
        """(is_uint8, h, w) of a predict_scene input, ValueError unless it is uint8 [H, W, C] (host or device) or fp32
        [C, H, W] on the engine's device, with C = n_channels."""
        if not isinstance(x, torch.Tensor) or x.dim() != 3:
            raise ValueError(f"{name} must be a uint8 [H, W, C] or fp32 [C, H, W] tensor, got "
                             f"{getattr(x, 'shape', type(x))}")
        if x.dtype == torch.uint8:
            h, w, c = x.shape
        elif x.dtype == torch.float32:
            c, h, w = x.shape
            if x.device.type != self.dev.type or (self.dev.index is not None and x.device.index != self.dev.index):
                raise ValueError(f"{name}: an fp32 [C, H, W] scene must be on the engine's device {self.dev}, got "
                                 f"{x.device}")
        else:
            raise ValueError(f"{name} must be uint8 [H, W, C] or fp32 [C, H, W], got {x.dtype}")
        if c != self.n_channels:
            raise ValueError(f"{name} has {c} channels, expected n_channels = {self.n_channels}")
        if h < 1 or w < 1:
            raise ValueError(f"{name} is empty: {tuple(x.shape)}")
        return x.dtype == torch.uint8, h, w

    @_on_device
    def predict_scene(self, img1: torch.Tensor, img2: torch.Tensor, tile: int = 256, overlap: int = 64, batch: int = 8,
                      return_probs: bool = False, labels: Optional[torch.Tensor] = None,
                      ignore_index: int = -100) -> SceneResult:
        """A change map of a whole scene of any size at its own resolution, by sliding-window inference.

        img1, img2: the two images of the scene, either uint8 [H, W, C] as PIL / numpy give them (host or device;
        normalised on the device as dataset.py's ToTensor + Normalize(0.5, 0.5); a host scene is copied to the device
        once) or fp32 [C, H, W] on the device, already normalised (what forward() takes).  C = n_channels, the same
        shape for both, any H, W >= 1.

        The scene is cut into tiles of tile x tile pixels that overlap by `overlap` (scene_axis: an axis shorter than
        the tile gets one tile of its own length rounded up to 16, padded by repeating the edge), and the tiles run
        `batch` at a time through the eval-mode network (BatchNorm with the running statistics, as predict()).  Their
        softmax (K = 1: sigmoid) probabilities are blended with the Gaussian window of scene_window:
        p = sum_tiles w * p_tile / sum_tiles w, summed in ascending tile index, so the result does not depend on
        `batch`.  pred is the argmax of p (ties to the lowest class) or, for K = 1, p > 0.5.

        return_probs: also return p (fp32 [K, H, W]).  labels (int64 [H, W]): also return the confusion counts of pred
        against them at full resolution: [K, K] (rows = label; metrics.multiclass_metrics takes it) or, for K = 1,
        [TP, FP, FN, TN] (metrics.metrics_from_counts); pixels labelled ignore_index or outside [0, K) ({0, 1} for
        K = 1) are not counted.

        Memory: (K + 1) * 4 bytes per scene pixel of accumulators (which become probs), and the engine's activation
        buffers sized for `batch` tiles; like any call at a new shape this may re-allocate them.  Everything runs on
        the current stream without a host synchronisation.  The `training` flag is restored afterwards and no
        parameter, gradient or BatchNorm buffer changes.  Bad arguments raise ValueError before any work is enqueued."""
        for name, v in (("tile", tile), ("overlap", overlap), ("batch", batch)):
            if isinstance(v, bool) or not isinstance(v, int):
                raise ValueError(f"{name} must be an int, got {v!r}")
        if tile < 16 or tile % 16:
            raise ValueError(f"tile must be a multiple of 16 and at least 16, got {tile}")
        if not 0 <= overlap < tile:
            raise ValueError(f"overlap must be in [0, tile = {tile}), got {overlap}")
        if batch < 1:
            raise ValueError(f"batch must be >= 1, got {batch}")
        u8, h, w = self._scene_input(img1, "img1")
        if self._scene_input(img2, "img2")[0] != u8 or img2.shape != img1.shape:
            raise ValueError(f"img1 and img2 must have the same dtype and shape, got {img1.dtype} "
                             f"{tuple(img1.shape)} and {img2.dtype} {tuple(img2.shape)}")
        if labels is not None and (not isinstance(labels, torch.Tensor) or labels.dtype != torch.int64
                                   or tuple(labels.shape) != (h, w)):
            raise ValueError(f"labels must be an int64 [{h}, {w}] tensor, got "
                             f"{getattr(labels, 'dtype', type(labels))} {tuple(getattr(labels, 'shape', ()))}")
        k = self.n_classes
        grid = _scene_grid(h, w, tile, overlap)
        (_, ey, _, ny), (_, ex, _, nx) = grid
        img1, img2 = img1.to(self.dev).contiguous(), img2.to(self.dev).contiguous()
        if labels is not None:
            labels = labels.to(self.dev).contiguous()
        acc = torch.empty(k, h, w, device=self.dev)              # every pixel is written by the batch of its first tile
        wsum = torch.empty(h, w, device=self.dev)
        pred = torch.empty(h, w, device=self.dev, dtype=torch.uint8)
        conf = None
        if labels is not None:
            conf = torch.zeros((4,) if k == 1 else (k, k), device=self.dev, dtype=torch.int64)
        was = self.training
        self.training = False
        try:
            self._alloc(batch, ey, ex)
            for t0 in range(0, ny * nx, batch):                 # the last batch is padded with zero tiles
                ops.scene_gather(img1, img2, grid, t0, self.x_in[0], self.x_in[1])
                self._forward_from((None, None))
                ops.scene_blend(self.logits, grid, t0, acc, wsum)
            ops.scene_finalize(acc, wsum, pred, return_probs, labels, ignore_index, conf)
        finally:
            self.training = was
            self._tape = []
        return SceneResult(pred, acc if return_probs else None, conf)

    # -- backward --------------------------------------------------------------------------------------
    @_on_device
    def backward(self) -> None:
        """Consumes self.dlogits (fp32 [n, h, w] or [n, K, h, w]); accumulates every parameter gradient."""
        if self.n_classes == 1:
            dl = self.dlogits.view(-1)
            ops.conv1x1_cout1_wgrad(dl, self._last, self.store.seg(self.store.g, "conv_last.weight"),
                                    self.grad("conv_last.bias"))
            ops.conv1x1_cout1_dgrad(dl, self.store.seg(self.store.p, "conv_last.weight"), self._glast)
        else:
            ops.conv1x1_ck_wgrad(self.dlogits, self._last, self.store.seg(self.store.g, "conv_last.weight"),
                                 self.grad("conv_last.bias"))
            ops.conv1x1_ck_dgrad(self.dlogits, self.store.seg(self.store.p, "conv_last.weight"), self._glast)
        for idx in range(len(self._tape) - 1, -1, -1):
            self._tape[idx]()
            if self.reducer is not None and idx in self._marks:
                self._join_wgrad()          # the segments' side-stream weight gradients are part of what gets reduced
                self.reducer.ready_from(self._marks[idx])
        self._join_wgrad()
        self._tape = []

    # -- one training iteration (train.py:137-146) ------------------------------------------------------
    def _class_weight(self, class_weight) -> Optional[torch.Tensor]:
        if class_weight is None:
            return None
        if isinstance(class_weight, torch.Tensor) and class_weight.device == self.dev:
            return class_weight.detach().float().contiguous()
        key = tuple(float(v) for v in (class_weight.tolist() if isinstance(class_weight, torch.Tensor) else class_weight))
        if self._cw_cache[0] != key:         # one upload per distinct weight vector, not one per step
            self._cw_cache = (key, torch.tensor(key, device=self.dev, dtype=torch.float32))
        return self._cw_cache[1]

    def _check_kind(self, kind: str) -> None:
        k = self.n_classes
        if (kind in MULTI_KINDS and k == 1) or (kind in SINGLE_KINDS and k > 1):
            raise ValueError(f"loss kind {kind!r} does not apply to n_classes = {k}: use kind='ce' with n_classes > 1 "
                             "(or 'ce_dice', 'softmax_focal_dice') and 'combined' or 'focal_dice' with n_classes = 1")

    def _dice_args(self, kind: str, kw: dict) -> dict:
        """The keywords of a Dice kind with their defaults, checked (ValueError) before any launch."""
        unknown = set(kw) - set(DICE_KW[kind])
        if unknown:
            raise ValueError(f"kind={kind!r} takes {', '.join(DICE_KW[kind])}, not {sorted(unknown)}")
        args = dict(DICE_KW[kind], **kw)
        w_point = args["alpha"] if kind == "ce_dice" else args["beta"]
        ops.check_dice_args(f"kind={kind!r}", w_point, args.get("gamma", 0.0), args["smooth"])
        cw = self._class_weight(args["class_weight"])
        if cw is not None and cw.numel() != self.n_classes:
            raise ValueError(f"class_weight has {cw.numel()} entries; n_classes = {self.n_classes}")
        return dict(mode=0 if kind == "ce_dice" else 1, w_point=float(w_point), gamma=float(args.get("gamma", 0.0)),
                    smooth=float(args["smooth"]), class_weight=cw, ignore_index=int(args["ignore_index"]))

    def loss_and_grad(self, labels: torch.Tensor, kind: Optional[str] = None, **kw) -> torch.Tensor:
        """The loss on self.logits; writes d(loss)/d(logits) into self.dlogits and returns the loss as a device fp64
        scalar tensor.  n_classes = 1: kind "combined" (CombinedLoss, train.py:82-105; the default) or "focal_dice"
        (FocalDiceLoss, train.py:108-128).  n_classes > 1: kind "ce" (the default), nn.CrossEntropyLoss(
        weight=class_weight, ignore_index=ignore_index) with class_weight a length-K sequence or device tensor;
        kind "ce_dice" (alpha * CE + (1 - alpha) * Dice; alpha=0.5, smooth=1.0, class_weight, ignore_index) or
        "softmax_focal_dice" (beta * Focal + (1 - beta) * Dice; beta=0.5, gamma=2.0, smooth=1.0, class_weight as the
        focal per-class factor, ignore_index), the K-class forms of CombinedLoss and FocalDiceLoss.  Their Dice term is
        1 - the mean over classes 1..K-1 (class 0, "no change", is excluded) of (2 I_k + smooth) / (P_k + T_k + smooth),
        summed over this batch.  Data parallel: each rank's Dice uses its own batch (as the binary "combined" and
        "focal_dice" do) and the gradients are averaged by the reducer; there is no cross-rank Dice."""
        k = self.n_classes
        if kind is None:
            kind = "combined" if k == 1 else "ce"
        self._check_kind(kind)
        if kind == "ce":
            unknown = set(kw) - {"class_weight", "ignore_index"}
            if unknown:
                raise ValueError(f"kind='ce' takes class_weight and ignore_index, not {sorted(unknown)}")
            cw = self._class_weight(kw.get("class_weight"))
            if cw is not None and cw.numel() != k:
                raise ValueError(f"class_weight has {cw.numel()} entries; n_classes = {k}")
            ops.seg_ce_loss(self.logits, labels.contiguous(), cw, int(kw.get("ignore_index", -100)), self.ce_sums,
                            self.bad_labels, self.dlogits, 1.0, self.loss_out)
        elif kind in DICE_KW:
            a = self._dice_args(kind, kw)
            ops.seg_softmax_dice_loss(self.logits, labels.contiguous(), a["mode"], a["w_point"], a["gamma"], a["smooth"],
                                      a["class_weight"], a["ignore_index"], self.dice_sums, self.bad_labels, self.dlogits,
                                      1.0, self.loss_out)
        elif kind == "combined":
            alpha = kw.get("alpha", 0.5)
            ops.seg_loss(self.logits, labels, 0, alpha, 1.0 - alpha, kw.get("pos_weight", 9.0), kw.get("smooth", 1.0), 0.0,
                         0.0, self.loss_sums, self.dlogits, 1.0, self.loss_out)
        elif kind == "focal_dice":
            beta = kw.get("beta", 0.5)
            ops.seg_loss(self.logits, labels, 1, beta, 1.0 - beta, 1.0, kw.get("smooth", 1.0), kw.get("gamma", 2.0),
                         kw.get("focal_alpha", 0.75), self.loss_sums, self.dlogits, 1.0, self.loss_out)
        else:
            raise ValueError(f"unknown loss {kind!r}")
        return self.loss_out

    @_on_device
    def train_step(self, img1: torch.Tensor, img2: torch.Tensor, labels: torch.Tensor, lr: float = 1.0152e-4,
                   weight_decay: float = 1.118e-5, kind: Optional[str] = None, grad_scale: float = 1.0, allreduce=None,
                   **loss_kw) -> torch.Tensor:
        """zero_grad -> forward -> criterion -> backward -> AdamW step (train.py:140-144).  Data parallel: set
        `self.reducer = parallel.TailReducer(self.store.g)` (or pass `allreduce`) and grad_scale = 1 / world.  kind: see
        loss_and_grad ("combined" for n_classes = 1, "ce" for n_classes > 1 by default)."""
        if kind is None:
            kind = "combined" if self.n_classes == 1 else "ce"
        self._check_kind(kind)                  # the pairing error before any work is enqueued
        if kind in DICE_KW:
            self._dice_args(kind, loss_kw)      # and the keyword errors of the Dice kinds
        self.training = True
        self.zero_grad()
        self.forward(img1, img2)
        loss = self.loss_and_grad(labels, kind, **loss_kw)
        if self.reducer is not None:        # data parallel: SUM all-reduce of the gradient tail while backward continues
            self.reducer.begin()
        self.backward()
        if self.reducer is not None:
            self.reducer.finish()
        elif allreduce is not None:
            allreduce(self.store.g)
        self.adam_step(lr, (0.9, 0.999), 1e-8, weight_decay, decoupled=True, grad_scale=grad_scale)
        return loss


class GateEngine(SiameseEngine):
    """A stand-alone AttentionGate(F_g, F_l, F_int) (models.py:18-44): the gate layers of SiameseEngine with their own
    parameter store, so `AttentionGate.forward(g, x)` computes through the same kernels."""

    def __init__(self, device, F_g: int, F_l: int, F_int: int) -> None:
        _Net.__init__(self, device)
        if F_g % 64 or F_l % 64 or F_int % 64:
            raise NotImplementedError("the native attention gate needs F_g, F_l and F_int to be multiples of 64 (the reference uses 64 ... 2048)")
        self.cfg = (F_g, F_l, F_int)
        self.key_order = []
        self.conv_meta = {}
        self._reg_gate("", F_g, F_l, F_int)
        self.store.allocate(device)
        for bn in self.bns.values():
            bn.allocate(device)
        bf = dict(device=device, dtype=torch.bfloat16)
        self.w_fwd, self.w_dg = {}, {}
        for key, (co, ci, k) in self.conv_meta.items():
            self.w_fwd[key] = torch.zeros(1, co, ci, **bf)
            self.w_dg[key] = torch.zeros(1, ci, co, **bf)
        self._plan = None
        self._n = None
        self._tape = []
        self._marks = {}
        self.reducer = None
        self.tmp, self.saved = {}, {}

    @_on_device
    def forward(self, g: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        """g [n, F_g, h, w], x [n, F_l, h, w] fp32 NCHW -> x * psi as NHWC bf16 [n, h, w, F_l]."""
        fg, fl, _ = self.cfg
        n, cg, h, w = g.shape
        if cg != fg or tuple(x.shape) != (n, fl, h, w):
            raise ValueError(f"AttentionGate expects g [n,{fg},h,w] and x [n,{fl},h,w], got {tuple(g.shape)} / {tuple(x.shape)}")
        if self._n != (n, h, w):
            bf = dict(device=self.dev, dtype=torch.bfloat16)
            self.g_in, self.gg = torch.empty(n, h, w, fg, **bf), torch.empty(n, h, w, fg, **bf)
            self.x_in2, self.gxs = torch.empty(n, h, w, fl, **bf), torch.empty(n, h, w, fl, **bf)
            self.out, self.gout = torch.empty(n, h, w, fl, **bf), torch.empty(n, h, w, fl, **bf)
            self.tmp, self.saved = {}, {}
            self._n = (n, h, w)
        self._tape = []
        ops.nchw_to_nhwc_bf16(g.contiguous().float(), self.g_in)
        ops.nchw_to_nhwc_bf16(x.contiguous().float(), self.x_in2)
        self._gate("", self.g_in, self.gg, self.x_in2, self.gxs, self.out, self.gout)
        return self.out

    @_on_device
    def backward(self) -> None:
        """Consumes self.gout (gradient of the output, NHWC bf16); leaves the input gradients in self.gg / self.gxs."""
        self.gg.zero_()
        for fn in reversed(self._tape):
            fn()
        self._tape = []
