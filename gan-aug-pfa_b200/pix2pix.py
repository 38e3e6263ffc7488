"""Native Pix2Pix engine: the U-Net generator, the PatchGAN discriminator and one GAN training
iteration, sequenced entirely as C-ABI kernel launches (libgap_b200.so).

What it mirrors in the reference:
  * UNetGenerator / UnetSkipConnectionBlock  (models.py:149-208)
  * NLayerDiscriminator                      (models.py:212-247)
  * train_gan_one_epoch's loop body          (train_gan.py:52-74), Adam(lr, betas=(0.5, 0.999))
  * generator inference under eval()/no_grad (generate_synthetic_data.py:55-68)

Data layout in HBM: activations NHWC bf16; U-Net skips live in per-level concat buffers
R_j = [ReLU(down_j) | ReLU(up_{j+1})] so torch.cat (models.py:208) never copies; master weights,
gradients and Adam moments are fp32 in flat buffers whose per-layer segments use the GEMM-native
order ([Cout][kh][kw][Cin] for Conv2d, [Cin][kh][kw][Cout] for ConvTranspose2d) and are exposed to
state_dict() as strided views with the reference's shapes.

Legal savings vs the reference's execution (SURVEY.md §8d): the second, numerically identical
generator forward (train_gan.py:65) is not recomputed (BatchNorm buffers receive both updates), and
the discriminator weight gradients of the G step (cleared by opt_d.zero_grad(), train_gan.py:55)
are not computed.
"""
from __future__ import annotations

import functools
from dataclasses import dataclass
from typing import Dict, List, NamedTuple, Optional, Tuple

import torch

from . import ops
from .ops import ACT_LRELU, ACT_NONE, ACT_RELU, ACT_TANH
from .scene import _scene_grid
from .spec import DiscriminatorSpec, GeneratorSpec

BN_EPS = 1e-5
BN_MOMENTUM = 0.1
IN_EPS = 1e-5           # nn.InstanceNorm2d default
LAMBDA_L1 = 100.0  # train_gan.py:33
# Image tensors on the hot path are NHWC bf16 with IMAGE_SLOTS channel slots: an image of 1..4 channels fills the first
# ones and the rest stay zero.  The discriminator sees cat(A, B) as two such sources.
IMAGE_SLOTS = 4


def check_image_channels(what: str, c: int) -> int:
    """`c` if it fits one 4-slot image tensor, else NotImplementedError naming the supported range."""
    if not isinstance(c, int) or not 1 <= c <= IMAGE_SLOTS:
        raise NotImplementedError(f"{what} = {c!r} is not implemented natively: images of 1 to {IMAGE_SLOTS} channels are")
    return c


def discriminator_split(input_nc: int) -> Tuple[int, int]:
    """Channels of the two sources of a discriminator over cat(A, B) with `input_nc` channels: A = the first
    ceil(input_nc / 2), B = the rest (3 | 3 for the reference's 6).  NotImplementedError outside 2..8."""
    if not isinstance(input_nc, int) or not 2 <= input_nc <= 2 * IMAGE_SLOTS:
        raise NotImplementedError(f"input_nc = {input_nc!r} is not implemented natively by the discriminator: 2 to "
                                  f"{2 * IMAGE_SLOTS} channels are (two sources of up to {IMAGE_SLOTS} channels each)")
    ca = (input_nc + 1) // 2
    return ca, input_nc - ca


class SceneImage(NamedTuple):
    """translate_scene's result.  image: uint8 [H, W, output_nc], the picture generate_synthetic_data.py saves.
    values: the blended fp32 Tanh outputs [output_nc, H, W] in [-1, 1] (return_float=True), else None."""
    image: torch.Tensor
    values: Optional[torch.Tensor]


def _pad4(n: int) -> int:
    return (n + 3) // 4 * 4


def _on_device(fn):
    """Entry points run with the engine's device current: the library launches on the thread's current device and the
    launchers pass that device's current stream, so an engine built on cuda:1 must not launch while cuda:0 is current."""
    @functools.wraps(fn)
    def wrapper(self, *a, **k):
        idx = self.dev.index
        if idx is None or torch.cuda.current_device() == idx:
            return fn(self, *a, **k)
        with torch.cuda.device(idx):
            return fn(self, *a, **k)
    return wrapper


class ParamStore:
    """Flat fp32 parameter / gradient / Adam-moment buffers with named, 16-byte-aligned segments."""

    def __init__(self) -> None:
        self.segs: Dict[str, Tuple[int, int]] = {}
        self.total = 0
        self.p = self.g = self.m = self.v = None
        self.step = 0
        self.step_dev = None

    def add(self, name: str, numel: int) -> int:
        off = self.total
        self.segs[name] = (off, numel)
        self.total += _pad4(numel)
        return off

    def allocate(self, device: torch.device) -> None:
        self.p = torch.zeros(self.total, device=device, dtype=torch.float32)
        self.g = torch.zeros_like(self.p)
        self.m = torch.zeros_like(self.p)
        self.v = torch.zeros_like(self.p)

    def seg(self, buf: torch.Tensor, name: str) -> torch.Tensor:
        off, n = self.segs[name]
        return buf[off:off + n]

    def off(self, name: str) -> int:
        return self.segs[name][0]


@dataclass
class _BN:
    """BatchNorm2d state for one layer: affine params live in the ParamStore, buffers here."""
    name: str
    c: int
    running_mean: torch.Tensor = None
    running_var: torch.Tensor = None
    nbt: torch.Tensor = None
    stats: torch.Tensor = None      # fp64 [2C] forward sums (conv epilogue)
    sums: torch.Tensor = None       # fp64 [2C] backward sums (raw [sum d, sum d*y] when a GEMM epilogue fills them)
    sums2: torch.Tensor = None      # fp64 [2C] [sum d, sum d*xhat] handed to the apply pass
    scale: torch.Tensor = None
    shift: torch.Tensor = None
    mean: torch.Tensor = None
    invstd: torch.Tensor = None

    def allocate(self, dev: torch.device) -> None:
        self.running_mean = torch.zeros(self.c, device=dev)
        self.running_var = torch.ones(self.c, device=dev)
        self.nbt = torch.zeros((), device=dev, dtype=torch.int64)
        self.stats = torch.zeros(2 * self.c, device=dev, dtype=torch.float64)
        self.sums = torch.zeros(2 * self.c, device=dev, dtype=torch.float64)
        self.sums2 = torch.zeros(2 * self.c, device=dev, dtype=torch.float64)
        self.scale = torch.empty(self.c, device=dev)
        self.shift = torch.empty(self.c, device=dev)
        self.mean = torch.empty(self.c, device=dev)
        self.invstd = torch.empty(self.c, device=dev)


@dataclass
class _IN:
    """InstanceNorm2d(affine=False) state for one layer: no parameters, no buffers; per-(image, channel) statistics of
    the current activation set, sized by the batch in _alloc."""
    name: str
    c: int
    sums: torch.Tensor = None       # fp64 [2][N*C]: forward [sum y, sum y^2], then backward [sum d, sum d*xhat]; zero at rest
    scale: torch.Tensor = None      # fp32 [N][C] = invstd
    shift: torch.Tensor = None      # fp32 [N][C] = -mean * invstd
    mean: torch.Tensor = None
    invstd: torch.Tensor = None

    def allocate(self, n: int, dev: torch.device) -> None:
        self.sums = torch.zeros(2 * n * self.c, device=dev, dtype=torch.float64)
        self.scale, self.shift, self.mean, self.invstd = (torch.empty(n, self.c, device=dev) for _ in range(4))


class _Net:
    """Shared plumbing: parameter store, BatchNorm / InstanceNorm bookkeeping, state_dict import/export."""

    def __init__(self, device: torch.device, norm: str = "batch") -> None:
        if norm not in ("batch", "instance"):
            raise ValueError(f"norm must be 'batch' or 'instance', got {norm!r}")
        self.dev = device
        self.norm = norm
        self.store = ParamStore()
        self.bns: Dict[str, _BN] = {}
        self.ins: Dict[str, _IN] = {}
        # state_dict key -> (segment name, shape, strides) for weights / biases / BN affine
        self.views: Dict[str, Tuple[str, Tuple[int, ...], Tuple[int, ...]]] = {}
        self.key_order: List[str] = []
        self.training = True
        self.grad_hook = None     # callable(segment name) fired when a gradient segment is final (data-parallel buckets)
        self.alloc_gen = 0        # bumped whenever _alloc (re)allocates the activation set: captured graphs go stale

    def _ready(self, *keys: str, side: bool = False) -> None:
        if self.grad_hook is not None:
            st = self._wgrad_stream if (side and self._wgrad_used) else None
            for k in keys:
                self.grad_hook(k, st)

    # Weight gradients are off the critical path of a backward pass (only the optimizer needs them), so they are
    # enqueued on a side stream: the block scheduler fills the SMs that the dgrad chain leaves idle (small deep layers,
    # tail waves of the persistent GEMMs) with wgrad CTAs.  Joined before anything they read is overwritten.
    overlap_wgrad = True
    _wgrad_stream = None
    _wgrad_used = False

    def _fork_wgrad(self, fn) -> None:
        if not self.overlap_wgrad:
            fn()
            return
        cur = torch.cuda.current_stream(self.dev)
        if self._wgrad_stream is None:
            self._wgrad_stream = torch.cuda.Stream(self.dev)
        self._wgrad_stream.wait_stream(cur)          # everything enqueued so far (the operands) is visible
        with torch.cuda.stream(self._wgrad_stream):
            fn()
        self._wgrad_used = True

    def _join_wgrad(self) -> None:
        if self._wgrad_used:
            torch.cuda.current_stream(self.dev).wait_stream(self._wgrad_stream)
            self._wgrad_used = False

    def grad_segments(self) -> List[Tuple[str, int, int]]:
        """(name, offset, numel) of every gradient segment in flat-buffer (= backward-completion) order."""
        return [(k, off, n) for k, (off, n) in self.store.segs.items()]

    # -- registration helpers -------------------------------------------------------------------
    def _reg(self, key: str, numel: int, shape, strides) -> None:
        self.store.add(key, numel)
        self.views[key] = (key, tuple(shape), tuple(strides))

    def _reg_conv(self, key: str, cout: int, cin: int) -> None:
        """Conv2d weight (Cout,Cin,4,4) stored [Cout][kh][kw][Cin]."""
        self._reg(key, cout * 16 * cin, (cout, cin, 4, 4), (16 * cin, 1, 4 * cin, cin))

    def _reg_convT(self, key: str, cin: int, cout: int) -> None:
        """ConvTranspose2d weight (Cin,Cout,4,4) stored [Cin][kh][kw][Cout]."""
        self._reg(key, cin * 16 * cout, (cin, cout, 4, 4), (16 * cout, 1, 4 * cout, cout))

    def _reg_small(self, key: str, rows: int, c: int, krow: int) -> None:
        """(rows, c, 4, 4) weight of a tiny-channel layer stored [rows][(kh*4+kw)*c + ch] padded to krow."""
        self._reg(key, rows * krow, (rows, c, 4, 4), (krow, 1, 4 * c, c))

    def _reg_vec(self, key: str, n: int) -> None:
        self._reg(key, n, (n,), (1,))

    def _reg_in(self, prefix: str, c: int) -> _IN:
        m = _IN(prefix, c)
        self.ins[prefix] = m
        return m

    def _reg_bn(self, prefix: str, c: int) -> _BN:
        self._reg_vec(prefix + ".weight", c)
        self._reg_vec(prefix + ".bias", c)
        bn = _BN(prefix, c)
        self.bns[prefix] = bn
        return bn

    # -- parameter views ------------------------------------------------------------------------
    def view(self, buf: torch.Tensor, key: str) -> torch.Tensor:
        seg, shape, strides = self.views[key]
        return torch.as_strided(buf, shape, strides, self.store.off(seg))

    def param(self, key: str) -> torch.Tensor:
        return self.view(self.store.p, key)

    def grad(self, key: str) -> torch.Tensor:
        return self.view(self.store.g, key)

    def state_dict(self) -> Dict[str, torch.Tensor]:
        """Reference-format state_dict (keys / shapes / dtypes of models.py; SURVEY App. C)."""
        out: Dict[str, torch.Tensor] = {}
        for key in self.key_order:
            if key in self.views:
                out[key] = self.param(key)
            else:
                prefix, leaf = key.rsplit(".", 1)
                bn = self.bns[prefix]
                out[key] = {"running_mean": bn.running_mean, "running_var": bn.running_var,
                            "num_batches_tracked": bn.nbt}[leaf]
        return out

    @_on_device
    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        mine = self.state_dict()
        missing = [k for k in mine if k not in sd]
        extra = [k for k in sd if k not in mine]
        if missing or extra:
            raise KeyError(f"state_dict mismatch: missing {missing[:4]} unexpected {extra[:4]}")
        with torch.no_grad():
            for k, dst in mine.items():
                src = sd[k]
                if tuple(src.shape) != tuple(dst.shape):
                    raise ValueError(f"{k}: shape {tuple(src.shape)} != {tuple(dst.shape)}")
                dst.copy_(src.to(self.dev))
        self.repack()

    def init_from_torch_default(self) -> None:
        """Default torch init (kaiming-uniform(a=sqrt(5)) weights, uniform bias, BN gamma=1 beta=0),
        drawn from the global RNG in the reference's module-construction order."""
        raise NotImplementedError

    def repack(self) -> None:
        raise NotImplementedError

    @_on_device
    def zero_grad(self) -> None:
        self._join_wgrad()
        self.store.g.zero_()

    # -- in-flight activation sets (autograd path: several forwards may precede one backward) --------
    _BUFFER_ATTRS: Tuple[str, ...] = ()

    def detach_buffers(self) -> dict:
        """Hand the current activation set (and the BatchNorm statistics saved for backward) to the
        caller; the next forward allocates a fresh set."""
        snap = {a: getattr(self, a) for a in self._BUFFER_ATTRS if hasattr(self, a)}
        snap["_bn"] = {k: (b.scale.clone(), b.shift.clone(), b.mean.clone(), b.invstd.clone())
                       for k, b in self.bns.items()}
        # the InstanceNorm tensors belong to the activation set: the next forward's _alloc replaces them
        snap["_in"] = {k: (m.sums, m.scale, m.shift, m.mean, m.invstd) for k, m in self.ins.items()}
        snap["_n"] = self._n
        self._n = None
        return snap

    def attach_buffers(self, snap: dict) -> None:
        for a, v in snap.items():
            if a == "_bn":
                for k, (sc, sh, mu, iv) in v.items():
                    b = self.bns[k]
                    b.scale, b.shift, b.mean, b.invstd = sc, sh, mu, iv
            elif a == "_in":
                for k, t in v.items():
                    m = self.ins[k]
                    m.sums, m.scale, m.shift, m.mean, m.invstd = t
            else:
                setattr(self, a, v)

    @_on_device
    def adam_step(self, lr: float, betas=(0.5, 0.999), eps: float = 1e-8, weight_decay: float = 0.0,
                  decoupled: bool = False, grad_scale: float = 1.0) -> None:
        self._join_wgrad()
        s = self.store
        if s.step_dev is None:
            s.step_dev = torch.full((1,), s.step, device=s.p.device, dtype=torch.int32)
        if not torch.cuda.is_current_stream_capturing():     # a capture executes nothing: replays bump the host copy
            s.step += 1
        # the step counter lives on the device (incremented by the kernel) so a captured graph can be replayed
        ops.adam_flat_devstep(s.p, s.g, s.m, s.v, lr, betas[0], betas[1], eps, weight_decay, decoupled, s.step_dev,
                              grad_scale)
        self.repack()

    # -- BatchNorm helpers -----------------------------------------------------------------------
    def _bwd_epilogue(self, bn: Optional[_BN], y: torch.Tensor, slope: float, g2=None, c0: int = 0) -> dict:
        """Arguments of the backward-fused dgrad epilogue for the layer whose output is act(BN(y)) (bn None: the
        layer has no BatchNorm and ``y`` is its activated output)."""
        d = {"y": y, "slope": slope, "g2": g2, "c0": c0}
        if bn is not None:
            d["scale"], d["shift"] = bn.scale, bn.shift
        return d

    def _bn_backward_fused(self, bn: _BN, y, d, dy, param_grads: bool = True) -> None:
        """BatchNorm backward when the producing dgrad epilogue already applied the activation backward and
        accumulated [sum d, sum d*y] into bn.sums: finalize (+ parameter gradients), then one apply pass."""
        count = y.numel() // y.shape[-1]
        dg = self.grad(bn.name + ".weight") if param_grads else None
        db = self.grad(bn.name + ".bias") if param_grads else None
        ops.bn_bwd_finalize(bn.sums, bn.mean, bn.invstd, dg, db, bn.sums2)
        ops.bn_bwd_apply(y, d, None, 1.0, bn.scale, bn.shift, bn.mean, bn.invstd, bn.sums2, count, dy)
        if param_grads:
            self._ready(bn.name + ".weight", bn.name + ".bias")

    def _bn_forward(self, bn: _BN, y: torch.Tensor, out1, act1, out2=None, act2=ACT_NONE, repeat: int = 1) -> None:
        gamma = self.param(bn.name + ".weight")
        beta = self.param(bn.name + ".bias")
        if self.training:
            count = y.numel() // y.shape[-1]
            ops.bn_finalize(bn.stats, count, gamma, beta, BN_EPS, BN_MOMENTUM, repeat, bn.running_mean,
                            bn.running_var, bn.nbt, bn.scale, bn.shift, bn.mean, bn.invstd)
            ops.bn_act(y, bn.scale, bn.shift, out1, act1, out2, act2)
            return
        ops.bn_eval_scale_shift(gamma, beta, bn.running_mean, bn.running_var, BN_EPS, bn.scale, bn.shift)
        ops.bn_act(y, bn.scale, bn.shift, out1, act1, out2, act2)

    def _bn_scale_shift(self, bn: _BN, y: torch.Tensor, repeat: int = 1) -> None:
        """BatchNorm reduced to per-channel (scale, shift) WITHOUT an apply pass: the consumer kernel normalises and
        activates while it reads the raw tensor.  Training: batch statistics from the conv epilogue's sums (+ running
        buffers, saved mean / invstd for backward); eval: running statistics."""
        gamma, beta = self.param(bn.name + ".weight"), self.param(bn.name + ".bias")
        if self.training:
            ops.bn_finalize(bn.stats, y.numel() // y.shape[-1], gamma, beta, BN_EPS, BN_MOMENTUM, repeat, bn.running_mean,
                            bn.running_var, bn.nbt, bn.scale, bn.shift, bn.mean, bn.invstd)
        else:
            ops.bn_eval_scale_shift(gamma, beta, bn.running_mean, bn.running_var, BN_EPS, bn.scale, bn.shift)

    def _bn_eval(self, bn: _BN) -> None:
        """eval-mode BatchNorm as (scale, shift) from the running statistics (generate_synthetic_data.py:55)."""
        ops.bn_eval_scale_shift(self.param(bn.name + ".weight"), self.param(bn.name + ".bias"), bn.running_mean,
                                bn.running_var, BN_EPS, bn.scale, bn.shift)

    # -- InstanceNorm helpers -------------------------------------------------------------------
    def _in_forward(self, m: _IN, y: torch.Tensor, out1, act1, out2=None, act2=ACT_NONE) -> None:
        """act(InstanceNorm(y)) into out1 (and out2): the same in train and eval mode (no running statistics)."""
        ops.in_stats(y, m.sums)
        ops.bn_finalize(m.sums, y.shape[1] * y.shape[2], None, None, IN_EPS, 0.0, 1, None, None, None, m.scale, m.shift,
                        m.mean, m.invstd)
        ops.in_act(y, m.scale, m.shift, out1, act1, out2, act2)

    def _in_backward(self, m: _IN, y, g1, g2, slope: float, dy, dbias: Optional[torch.Tensor] = None) -> None:
        """dy = InstanceNorm backward of d = act'(xhat)*g1 (+ relu'(xhat)*g2); dbias += its per-channel sum (the bias of
        the conv in front, analytically zero)."""
        ops.in_bwd_reduce(y, g1, g2, slope, m.scale, m.shift, m.sums)
        ops.in_bwd_apply(y, g1, g2, slope, m.scale, m.shift, m.sums, dy, dbias)
        ops.bn_param_grads(m.sums, None, None)      # re-zeroes the sums

    def _bn_backward(self, bn: _BN, y, g1, g2, slope: float, dy, param_grads: bool = True) -> None:
        count = y.numel() // y.shape[-1]
        ops.bn_bwd_reduce(y, g1, g2, slope, bn.scale, bn.shift, bn.mean, bn.invstd, bn.sums)
        ops.bn_bwd_apply(y, g1, g2, slope, bn.scale, bn.shift, bn.mean, bn.invstd, bn.sums, count, dy)
        if param_grads:
            ops.bn_param_grads(bn.sums, self.grad(bn.name + ".weight"), self.grad(bn.name + ".bias"))
            self._ready(bn.name + ".weight", bn.name + ".bias")
        else:
            ops.bn_param_grads(bn.sums, None, None)


# ================================================================================================
# Generator
# ================================================================================================
class GeneratorEngine(_Net):
    """UNetGenerator(input_nc, output_nc, num_downs, ngf, BatchNorm2d or InstanceNorm2d, use_dropout) with
    input_nc, output_nc in 1..4 (default 3, 3)."""

    _BUFFER_ATTRS = ("S", "x_nhwc", "A", "R", "Rin", "yd", "yu", "fake_bf", "fake_f32", "dpre", "gR", "gRin", "gA",
                     "dyu", "dyd", "xin", "out_cat")

    def __init__(self, device, input_nc: int = 3, output_nc: int = 3, num_downs: int = 7, ngf: int = 64,
                 init: bool = True, use_dropout: bool = False, dropout_seed: int = 0,
                 spec: Optional[GeneratorSpec] = None, norm: str = "batch") -> None:
        """`spec` (GeneratorSpec.for_block_chain) builds the engine of a stand-alone UnetSkipConnectionBlock instead of a
        whole UNetGenerator.  With spec.virtual0 the chain starts at an inner block: level 0 has no layers, the input
        is the block's C[0]-channel feature map and the output is torch.cat([x, model(x)], 1) (models.py:208).
        norm="instance": nn.InstanceNorm2d layers (no state) and conv biases everywhere; a given spec carries its norm."""
        super().__init__(device, spec.norm if spec is not None else norm)
        inst = self.norm == "instance"
        if inst and use_dropout:
            raise NotImplementedError("InstanceNorm2d together with use_dropout=True is not implemented natively")
        # nn.Dropout(0.5) after the up-norm of the num_downs-5 blocks at ngf*8 (models.py:156-157,197-198); their up
        # outputs are yu[j] for j = L-2 ... L-1-(num_downs-5)
        self.use_dropout = use_dropout
        self.dropout_seed = dropout_seed
        self.dropout_calls = 0          # forward counter: every forward draws fresh masks
        self._drop_off: Dict[int, int] = {}
        if spec is None:
            check_image_channels("input_nc", input_nc)
            check_image_channels("output_nc", output_nc)
            if ngf % 64 != 0 or num_downs < 5:
                raise NotImplementedError("ngf must be a multiple of 64 and num_downs >= 5")
            spec = GeneratorSpec(input_nc, output_nc, num_downs, ngf, norm=norm)
        else:
            if use_dropout:
                raise NotImplementedError("stand-alone blocks with dropout are not implemented natively")
            if any(c % 64 for c in spec.C):
                raise NotImplementedError("native blocks need channel counts that are multiples of 64 (1 to 4 at the "
                                          "image side)")
            if not spec.virtual0:
                check_image_channels("input_nc", spec.input_nc)
                check_image_channels("output_nc", spec.output_nc)
        self.spec = sp = spec
        self.input_nc, self.output_nc = sp.input_nc, sp.output_nc
        self.virtual0 = v0 = sp.virtual0
        self.L = L = sp.L
        self.C = C = sp.C
        self.k_down, self.k_dbn, self.k_up, self.k_ubn = sp.k_down, sp.k_dbn, sp.k_up, sp.k_ubn
        # flat-buffer order = order in which gradients complete in backward (DP buckets)
        ic, oc = self.input_nc, self.output_nc
        if not v0:
            self._reg_small(self.k_up[0] + ".weight", 2 * C[0], oc, 64)
            self._reg_vec(self.k_up[0] + ".bias", oc)
        # ubn / dbn: the norm layers (_BN or _IN); with InstanceNorm each conv's bias segment follows its weight
        norm_reg = self._reg_in if inst else self._reg_bn
        self.ubn: List[Optional[_BN]] = [None] * L
        self.dbn: List[Optional[_BN]] = [None] * L
        for j in range(1, L):
            cin = C[j] if j == L - 1 else 2 * C[j]
            self._reg_convT(self.k_up[j] + ".weight", cin, C[j - 1])
            if inst:
                self._reg_vec(self.k_up[j] + ".bias", C[j - 1])
            self.ubn[j] = norm_reg(self.k_ubn[j], C[j - 1])
        for j in range(L - 1, 0, -1):
            self._reg_conv(self.k_down[j] + ".weight", C[j], C[j - 1])
            if inst:
                self._reg_vec(self.k_down[j] + ".bias", C[j])
            if self.k_dbn[j] is not None:
                self.dbn[j] = norm_reg(self.k_dbn[j], C[j])
        if not v0:
            self._reg_small(self.k_down[0] + ".weight", C[0], ic, 64)
            if inst:
                self._reg_vec(self.k_down[0] + ".bias", C[0])
        self.store.allocate(device)
        for bn in self.bns.values():
            bn.allocate(device)
        self.key_order = sp.key_order()
        # packed bf16 GEMM operands
        bf = dict(device=device, dtype=torch.bfloat16)
        # (zero-filled once: the packer never writes padding elements)
        self.w_d_fwd = [None] + [torch.zeros(1, C[j], 16 * C[j - 1], **bf) for j in range(1, L)]
        self.w_d_dg = [None] + [torch.zeros(4, C[j - 1], 4 * C[j], **bf) for j in range(1, L)]
        self.w_u_fwd = [None]
        self.w_u_dg = [None]
        if not v0:
            self.w_u_T2 = torch.zeros(16 * oc, 2 * C[0], **bf)   # last ConvTranspose2d, forward: [(kh*4+kw)*oc + co][Cin]
            # thin-layer operands [rows][16 taps x 4 channel slots] (input_nc / output_nc channels, zero slots after)
            self.w_d_thin = torch.zeros(C[0], 64, **bf)          # first conv, models.py:177
            self.w_u_thin = torch.zeros(2 * C[0], 64, **bf)      # last ConvTranspose2d seen from its dgrad
        else:
            self._ident = (torch.ones(C[0], device=device), torch.zeros(C[0], device=device))
        for j in range(1, L):
            cin = C[j] if j == L - 1 else 2 * C[j]
            self.w_u_fwd.append(torch.zeros(4, C[j - 1], 4 * cin, **bf))
            self.w_u_dg.append(torch.zeros(1, cin, 16 * C[j - 1], **bf))
        self._n = None
        self._plan = None
        if init:
            self.init_from_torch_default()

    def init_from_torch_default(self) -> None:
        """Default torch init drawn from the global CPU RNG in the reference's construction order
        (spec.GeneratorSpec.default_state_dict), then copied into the flat buffers."""
        self.load_state_dict(self.spec.default_state_dict())

    def repack(self) -> None:
        """fp32 masters -> bf16 GEMM operands (one launch for the whole network)."""
        if self._plan is None:
            self._plan = self._build_pack_plan()
        self._plan.run()

    def _build_pack_plan(self) -> ops.PackPlan:
        L, C, p = self.L, self.C, self.store.p
        off = self.store.off
        plan = ops.PackPlan()
        for j in range(1, L):
            ci, co = C[j - 1], C[j]
            o = off(self.k_down[j] + ".weight")
            plan.add(p, o, self.w_d_fwd[j], 0, 1, co, co, (4, 4), ci, ci, 16 * ci, (16 * ci, 1, 4 * ci, ci))
            plan.add(p, o, self.w_d_dg[j], 2, 4, ci, ci, (2, 2), co, co, 4 * co, (1, 16 * ci, 4 * ci, ci))
        if not self.virtual0:
            k0 = off(self.k_up[0] + ".weight")
            c2, ic, oc = 2 * C[0], self.input_nc, self.output_nc
            plan.add(p, k0, self.w_u_T2, 0, 1, 16 * oc, 16 * oc, (1, 1), c2, c2, c2, (1, 64, 0, 0))
            plan.add(p, off(self.k_down[0] + ".weight"), self.w_d_thin, 0, 1, C[0], C[0], (4, 4), ic, 4, 64,
                     (64, 1, 4 * ic, ic))
            plan.add(p, k0, self.w_u_thin, 0, 1, c2, c2, (4, 4), oc, 4, 64, (64, 1, 4 * oc, oc))
        for j in range(1, L):
            ci = C[j] if j == L - 1 else 2 * C[j]
            co = C[j - 1]
            o = off(self.k_up[j] + ".weight")
            plan.add(p, o, self.w_u_fwd[j], 2, 4, co, co, (2, 2), ci, ci, 4 * ci, (1, 16 * co, 4 * co, co))
            plan.add(p, o, self.w_u_dg[j], 0, 1, ci, ci, (4, 4), co, co, 16 * co, (16 * co, 1, 4 * co, co))
        return plan

    # -- activation buffers ---------------------------------------------------------------------
    def _alloc(self, n: int, h: int, w: int) -> None:
        if self._n == (n, h, w):
            return
        L, C, v0 = self.L, self.C, self.virtual0
        depth = L - 1 if v0 else L                  # number of stride-2 down convs applied to the input
        if h % (1 << depth) or w % (1 << depth):
            raise ValueError(f"input {h}x{w} must be divisible by 2^{depth}")
        bf = dict(device=self.dev, dtype=torch.bfloat16)
        base = 0 if v0 else 1                       # S[j]: spatial size of level j's feature maps
        S = [(h >> (j + base), w >> (j + base)) for j in range(L)]
        self.S = S
        if v0:
            # stand-alone inner block: xin = the block's input, out_cat = cat([LeakyReLU(x), BN(ConvT(...))], 1); A[0] is
            # its first half (the in-place LeakyReLU of models.py:178 is what the skip carries, models.py:208)
            self.xin = torch.empty(n, h, w, C[0], **bf)
            self.out_cat = torch.empty(n, h, w, 2 * C[0], **bf)
            self.A = [self.out_cat[..., :C[0]]] + [torch.empty(n, S[j][0], S[j][1], C[j], **bf) for j in range(1, L - 1)]
            self.R = [None] + [torch.empty(n, S[j][0], S[j][1], 2 * C[j], **bf) for j in range(1, L - 1)]
        else:
            self.x_nhwc = torch.zeros(n, h, w, 4, **bf)
            self.A = [torch.empty(n, S[j][0], S[j][1], C[j], **bf) for j in range(L - 1)]
            self.R = [torch.empty(n, S[j][0], S[j][1], 2 * C[j], **bf) for j in range(L - 1)]
            self.fake_bf = torch.zeros(n, h, w, 4, **bf)
            self.fake_f32 = torch.zeros(n, h, w, 4, device=self.dev)
            self.dpre = torch.zeros(n, h, w, 4, **bf)
        self.Rin = torch.empty(n, S[L - 1][0], S[L - 1][1], C[L - 1], **bf)
        self.yd = [None] + [torch.empty(n, S[j][0], S[j][1], C[j], **bf) for j in range(1, L - 1)] + [None]
        self.yu = [None] + [torch.empty(n, S[j - 1][0], S[j - 1][1], C[j - 1], **bf) for j in range(1, L)]
        # backward scratch
        self.gR = [torch.empty(n, S[j][0], S[j][1], 2 * C[j], **bf) for j in range(L - 1)]
        self.gRin = torch.empty_like(self.Rin)
        self.gA = [torch.empty(n, S[j][0], S[j][1], C[j], **bf) for j in range(L - 1)]
        self.dyu = [None] + [torch.empty_like(self.yu[j]) for j in range(1, L)]
        self.dyd = [torch.empty(n, S[j][0], S[j][1], C[j], **bf) for j in range(L)]
        for m in self.ins.values():
            m.allocate(n, self.dev)
        self._n = (n, h, w)
        self.alloc_gen += 1

    # -- forward --------------------------------------------------------------------------------
    @_on_device
    def prepare_input(self, x_nchw: torch.Tensor) -> torch.Tensor:
        """Size the buffers for x and convert it into self.x_nhwc (NHWC bf16, 4 channel slots); returns that tensor."""
        u8_in = x_nchw.dtype == torch.uint8
        if u8_in:
            n, h, w, c = x_nchw.shape
        else:
            n, c, h, w = x_nchw.shape
        if c != self.input_nc:
            raise ValueError(f"generator input has {c} channels, expected input_nc = {self.input_nc}")
        self._alloc(n, h, w)
        if u8_in:
            ops.u8_hwc_to_nhwc_bf16(x_nchw, self.x_nhwc)
        else:
            ops.nchw_to_nhwc_bf16(x_nchw, self.x_nhwc)
        return self.x_nhwc

    @_on_device
    def forward(self, x_nchw: torch.Tensor, bn_repeat: int = 1, out_u8: Optional[torch.Tensor] = None,
                x_ready: bool = False) -> torch.Tensor:
        """x: fp32 NCHW on the device, or uint8 NHWC [n,h,w,input_nc] (normalised on the device like dataset.py:155-159).
        Returns fake as fp32 NHWC [n,h,w,4] (channels >= output_nc are zero padding); the bf16 copy is self.fake_bf.
        bn_repeat=2 folds the reference's second identical forward.  out_u8 (uint8 [n,h,w,output_nc]) additionally
        receives the image generate_synthetic_data.py:69-88 saves, written by the last layer's epilogue.  x_ready:
        prepare_input(x) has already run (the trainer converts the input before it forks the generator onto its own
        stream)."""
        self._join_wgrad()
        v0 = self.virtual0
        if v0:
            # stand-alone inner block: x is its fp32 NCHW feature map; A[0] = LeakyReLU(x) (models.py:178, in place)
            n, c, h, w = x_nchw.shape
            if c != self.C[0]:
                raise ValueError(f"block input has {c} channels, expected {self.C[0]}")
            self._alloc(n, h, w)
            ops.nchw_to_nhwc_bf16(x_nchw.contiguous().float(), self.xin)
            ops.bn_act(self.xin, self._ident[0], self._ident[1], self.A[0], ACT_LRELU)
        elif not x_ready:
            self.prepare_input(x_nchw)
        L, C, S = self.L, self.C, self.S
        g_s2 = ops.geom_conv_fwd(4, 2, 1)
        g_1x1 = ops.geom_conv_fwd(1, 1, 0)
        g_ph = ops.geom_phase_k4s2p1()
        inst = self.norm == "instance"
        bias = (lambda k: self.param(k + ".bias")) if inst else (lambda k: None)
        if not v0:
            ops.thin_conv_fwd(self.x_nhwc, None, self.w_d_thin, bias(self.k_down[0]), self.A[0], ACT_LRELU,
                              self.R[0][..., :C[0]], ACT_RELU)
        for j in range(1, L - 1):
            bn = self.dbn[j]
            if inst:        # per-image statistics: train and eval mode are the same
                ops.conv_gemm([self.A[j - 1]], self.w_d_fwd[j], g_s2, self.yd[j], C[j], S[j], bias=bias(self.k_down[j]))
                self._in_forward(bn, self.yd[j], self.A[j], ACT_LRELU, self.R[j][..., :C[j]], ACT_RELU)
                continue
            if not self.training:      # eval: BatchNorm folds into the conv epilogue (scale, shift), no extra pass
                self._bn_eval(bn)
                ops.conv_gemm([self.A[j - 1]], self.w_d_fwd[j], g_s2, self.A[j], C[j], S[j], act=ACT_LRELU,
                              out2=self.R[j][..., :C[j]], act2=ACT_RELU, scale=bn.scale, bias=bn.shift)
                continue
            ops.conv_gemm([self.A[j - 1]], self.w_d_fwd[j], g_s2, self.yd[j], C[j], S[j], stats=bn.stats)
            self._bn_forward(bn, self.yd[j], self.A[j], ACT_LRELU, self.R[j][..., :C[j]], ACT_RELU, bn_repeat)
        ops.conv_gemm([self.A[L - 2]], self.w_d_fwd[L - 1], g_s2, self.Rin, C[L - 1], S[L - 1], act=ACT_RELU,
                      bias=bias(self.k_down[L - 1]))
        for j in range(L - 1, 0, -1):
            src = self.Rin if j == L - 1 else self.R[j]
            bn = self.ubn[j]
            # the parent's in-place ReLU (models.py:180) acts on the concatenated tensor; a stand-alone block returns
            # its up-norm output un-activated
            dst, act = (self.out_cat[..., C[0]:], ACT_NONE) if (v0 and j == 1) else (self.R[j - 1][..., C[j - 1]:], ACT_RELU)
            if inst:
                ops.conv_gemm([src], self.w_u_fwd[j], g_ph, self.yu[j], C[j - 1], S[j], bias=bias(self.k_up[j]))
                self._in_forward(bn, self.yu[j], dst, act)
                continue
            if not self.training:
                self._bn_eval(bn)
                ops.conv_gemm([src], self.w_u_fwd[j], g_ph, dst, C[j - 1], S[j], act=act, scale=bn.scale, bias=bn.shift)
                continue
            ops.conv_gemm([src], self.w_u_fwd[j], g_ph, self.yu[j], C[j - 1], S[j], stats=bn.stats)
            self._bn_forward(bn, self.yu[j], dst, act, repeat=bn_repeat)
            if self._dropout_layer(j):
                # ReLU(Dropout(v)) = Dropout(ReLU(v)): the mask multiplies the slot the parent block reads
                slot = self.R[j - 1][..., C[j - 1]:]
                self._drop_off[j] = (self.dropout_calls << 40) + (j << 34)
                ops.dropout_(slot, 0.5, self.dropout_seed, self._drop_off[j])
        if v0:
            return self.out_cat
        ops.thin_convT_fwd(self.R[0], self.w_u_T2, self.param(self.k_up[0] + ".bias"), ACT_TANH, self.fake_bf, self.fake_f32,
                           out_u8, co=self.output_nc)
        self.dropout_calls += 1
        return self.fake_f32

    def _scene_input(self, img) -> Tuple[bool, int, int]:
        """(is_uint8, h, w) of a translate_scene input, ValueError unless it is uint8 [H, W, input_nc] (host or device)
        or fp32 [input_nc, H, W] on the engine's device."""
        if not isinstance(img, torch.Tensor) or img.dim() != 3:
            raise ValueError(f"img must be a uint8 [H, W, C] or fp32 [C, H, W] tensor, got "
                             f"{getattr(img, 'shape', type(img))}")
        if img.dtype == torch.uint8:
            h, w, c = img.shape
        elif img.dtype == torch.float32:
            c, h, w = img.shape
            if img.device.type != self.dev.type or (self.dev.index is not None and img.device.index != self.dev.index):
                raise ValueError(f"img: an fp32 [C, H, W] scene must be on the engine's device {self.dev}, got "
                                 f"{img.device}")
        else:
            raise ValueError(f"img must be uint8 [H, W, C] or fp32 [C, H, W], got {img.dtype}")
        if c != self.input_nc:
            raise ValueError(f"img has {c} channels, expected input_nc = {self.input_nc}")
        if h < 1 or w < 1:
            raise ValueError(f"img is empty: {tuple(img.shape)}")
        return img.dtype == torch.uint8, h, w

    @_on_device
    def translate_scene(self, img: torch.Tensor, tile: int = 256, overlap: int = 64, batch: int = 32,
                        return_float: bool = False) -> SceneImage:
        """The generator's image of a whole scene of any size at its own resolution, by sliding-window inference: the
        synthetic second image of a pair that lines up pixel for pixel with the first one and with its labels.

        img: uint8 [H, W, input_nc] as PIL / numpy give it (host or device; normalised on the device as dataset.py's
        ToTensor + Normalize(0.5, 0.5); a host scene is copied to the device once), or fp32 [input_nc, H, W] on the
        device, already normalised (what forward() takes, rounded to bf16 as forward() does).  Any H, W >= 1.

        The scene is cut into tiles of tile x tile pixels that overlap by `overlap` (scene.scene_axis: an axis shorter
        than the tile gets one tile of its own length rounded up to 2^depth, padded by repeating the edge), and the
        tiles run `batch` at a time through the eval-mode generator: BatchNorm with the running statistics, no dropout.
        Their Tanh outputs are blended with the Gaussian window of scene.scene_window, v = sum_tiles w * v_tile /
        sum_tiles w, summed in ascending tile index, so the blend does not depend on `batch`.  An InstanceNorm
        generator normalises each tile by its own statistics, which is what a generator trained on crops of the tile
        size sees.

        tile: a multiple of 2^depth, depth = the number of stride-2 levels (num_downs: 128 at 7, 256 at 8), at most
        6144.  0 <= overlap < tile, batch >= 1.  Returns SceneImage(image, values): image is uint8 [H, W, output_nc]
        = uint8(clamp((v * 0.5 + 0.5) * 255, 0, 255)), truncated as the out_u8 output of forward() and torchvision's
        to_pil_image; values (return_float=True) is v, fp32 [output_nc, H, W].

        Memory: (output_nc + 1) * 4 bytes per scene pixel of accumulators (which become `values`), output_nc bytes
        for `image`, and the generator's activation buffers sized for `batch` tiles.  Like any call at a new shape,
        this re-sizes those buffers: the next training step re-allocates them, and Pix2PixTrainer.train_step_graphed
        re-captures its graph.  Everything runs on the current stream; device inputs need no host synchronisation.
        The `training` flag is restored afterwards, and no parameter, gradient, BatchNorm buffer or dropout counter
        changes, so later training draws the dropout masks it would have drawn without this call.  Bad arguments
        raise ValueError before any work is enqueued."""
        if self.virtual0:
            raise ValueError("translate_scene needs a whole generator: a stand-alone inner block has no image output")
        for name, v in (("tile", tile), ("overlap", overlap), ("batch", batch)):
            if isinstance(v, bool) or not isinstance(v, int):
                raise ValueError(f"{name} must be an int, got {v!r}")
        align = 1 << self.L                          # the input side must divide by 2 at every stride-2 level
        if tile < align or tile % align:
            raise ValueError(f"tile must be a positive multiple of 2^{self.L} = {align}, got {tile}")
        if 2 * tile > ops.SCENE_MAX_WINDOW:
            raise ValueError(f"tile must be at most {ops.SCENE_MAX_WINDOW // 2}, got {tile}")
        if not 0 <= overlap < tile:
            raise ValueError(f"overlap must be in [0, tile = {tile}), got {overlap}")
        if batch < 1:
            raise ValueError(f"batch must be >= 1, got {batch}")
        _, h, w = self._scene_input(img)
        oc = self.output_nc
        grid = _scene_grid(h, w, tile, overlap, align)
        (_, ey, _, ny), (_, ex, _, nx) = grid
        img = img.to(self.dev).contiguous()
        acc = torch.empty(oc, h, w, device=self.dev)       # every pixel is written by the batch of its first tile
        wsum = torch.empty(h, w, device=self.dev)
        image = torch.empty(h, w, oc, device=self.dev, dtype=torch.uint8)
        was, calls = self.training, self.dropout_calls
        self.training = False
        try:
            self._alloc(batch, ey, ex)
            for t0 in range(0, ny * nx, batch):             # the last batch is padded with zero tiles
                ops.scene_gather_one(img, grid, t0, self.x_nhwc)
                self.forward(None, x_ready=True)
                ops.scene_blend_image(self.fake_f32, grid, t0, acc, wsum)
            ops.scene_finalize_image(acc, wsum, image, return_float)
        finally:
            self.training = was
            self.dropout_calls = calls
        return SceneImage(image, acc if return_float else None)

    def _dropout_layer(self, j: int) -> bool:
        """True if the block whose up-conv output is yu[j] ends in nn.Dropout(0.5) (training mode only)."""
        return self.use_dropout and self.training and (self.L - 1 - (self.L - 5)) <= j <= self.L - 2

    @_on_device
    def output_nchw(self) -> torch.Tensor:
        n, h, w = self._n
        if self.virtual0:
            out = torch.empty(n, 2 * self.C[0], h, w, device=self.dev)
            ops.nhwc_to_nchw_f32(self.out_cat, out, 2 * self.C[0])
            return out
        out = torch.empty(n, self.output_nc, h, w, device=self.dev)
        ops.nhwc_to_nchw_f32(self.fake_f32, out, self.output_nc)
        return out

    # -- backward -------------------------------------------------------------------------------
    @_on_device
    def backward(self) -> None:
        """Consumes self.dpre (gradient w.r.t. the pre-Tanh output, bf16 NHWC) and accumulates every
        parameter gradient into the flat gradient buffer."""
        L, C, S = self.L, self.C, self.S
        g_s2 = ops.geom_conv_fwd(4, 2, 1)
        g_1x1 = ops.geom_conv_fwd(1, 1, 0)
        g_ph = ops.geom_phase_k4s2p1()
        self._join_wgrad()
        v0 = self.virtual0
        gseg = lambda key: self.store.seg(self.store.g, key)
        # outermost up-conv (a stand-alone inner block starts from gR[0] = the gradient of its concatenated output)

        def _w0():
            ops.thin_conv_wgrad(self.R[0], self.dpre, None, gseg(self.k_up[0] + ".weight"), 64, c0=self.output_nc)
            ops.colsum_bf16(self.dpre, self.output_nc, self.grad(self.k_up[0] + ".bias"))
        if not v0:
            self._fork_wgrad(_w0)
            self._ready(self.k_up[0] + ".weight", self.k_up[0] + ".bias", side=True)
            ops.thin_conv_fwd(self.dpre, None, self.w_u_thin, None, self.gR[0])
        # up path, outer -> inner.  Every dgrad GEMM applies the activation backward of the layer below in its
        # epilogue and accumulates that layer's BatchNorm-backward sums (no separate reduce pass).
        inst = self.norm == "instance"
        for j in range(1, L):
            bn = self.ubn[j]
            co = C[j - 1]
            if inst:
                # InstanceNorm: the dgrad below wrote the raw gradient of ReLU(IN(yu[j])); reduce + apply here
                self._in_backward(bn, self.yu[j], self.gR[j - 1][..., co:], None, 1.0 if (v0 and j == 1) else 0.0,
                                  self.dyu[j], self.grad(self.k_up[j] + ".bias"))
                self._ready(self.k_up[j] + ".bias")
            else:
                if self._dropout_layer(j):
                    ops.dropout_(self.gR[j - 1][..., co:], 0.5, self.dropout_seed, self._drop_off[j])   # same mask as forward
                if j == 1 or self._dropout_layer(j):      # gR[0] comes from the thin-layer kernel: classic reduce + apply
                    # (slope 1: a stand-alone block's up-norm output is not followed by the parent's ReLU)
                    self._bn_backward(bn, self.yu[j], self.gR[j - 1][..., co:], None, 1.0 if (v0 and j == 1) else 0.0,
                                      self.dyu[j])
                else:
                    self._bn_backward_fused(bn, self.yu[j], self.gR[j - 1][..., co:], self.dyu[j])
            src = self.Rin if j == L - 1 else self.R[j]
            ci = src.shape[-1]
            self._fork_wgrad(lambda src=src, j=j, co=co: ops.conv_wgrad(
                src, self.dyu[j], gseg(self.k_up[j] + ".weight"), (4, 4), 2, (-1, -1), 16 * co, co))
            self._ready(self.k_up[j] + ".weight", side=True)
            if j == L - 1:
                # innermost: Rin = ReLU(conv) has no BatchNorm -> the epilogue writes dyd[L-1] directly
                ops.conv_gemm([self.dyu[j]], self.w_u_dg[j], g_s2, self.dyd[L - 1], ci, S[j],
                              bwd=self._bwd_epilogue(None, self.Rin, 0.0))
            elif inst or self._dropout_layer(j + 1):
                # the dropout mask has to hit the gradient before the ReLU / BatchNorm backward, and InstanceNorm's
                # per-image sums do not fit the epilogue: plain dgrad here
                ops.conv_gemm([self.dyu[j]], self.w_u_dg[j], g_s2, self.gR[j], ci, S[j])
            else:
                nb = self.ubn[j + 1]     # second half of gR[j] = gradient at ReLU(BN(yu[j+1]))
                ops.conv_gemm([self.dyu[j]], self.w_u_dg[j], g_s2, self.gR[j], ci, S[j], stats=nb.sums,
                              bwd=self._bwd_epilogue(nb, self.yu[j + 1], 0.0, c0=C[j]))
        for j in range(L - 1, 0, -1):
            self._fork_wgrad(lambda j=j: ops.conv_wgrad(
                self.dyd[j], self.A[j - 1], gseg(self.k_down[j] + ".weight"), (4, 4), 2, (-1, -1), 16 * C[j - 1], C[j - 1]))
            self._ready(self.k_down[j] + ".weight", side=True)
            if inst and j == L - 1:       # innermost down conv: ReLU without a norm, its bias gradient is a column sum
                self._fork_wgrad(lambda: ops.colsum_bf16(self.dyd[L - 1], C[L - 1], self.grad(self.k_down[L - 1] + ".bias")))
                self._ready(self.k_down[L - 1] + ".bias", side=True)
            jj = j - 1
            skip = self.gR[jj][..., :C[jj]]          # gradient through the ReLU'd skip copy (models.py:208)
            if jj >= 1 and inst:
                ops.conv_gemm([self.dyd[j]], self.w_d_dg[j], g_ph, self.gA[jj], C[jj], S[j])
                self._in_backward(self.dbn[jj], self.yd[jj], self.gA[jj], skip, 0.2, self.dyd[jj],
                                  self.grad(self.k_down[jj] + ".bias"))
                self._ready(self.k_down[jj] + ".bias")
            elif jj >= 1:
                bn = self.dbn[jj]
                ops.conv_gemm([self.dyd[j]], self.w_d_dg[j], g_ph, self.gA[jj], C[jj], S[j], stats=bn.sums,
                              bwd=self._bwd_epilogue(bn, self.yd[jj], 0.2, g2=skip))
                self._bn_backward_fused(bn, self.yd[jj], self.gA[jj], self.dyd[jj])
            elif v0:
                # stand-alone block: the skip half of the output IS LeakyReLU(x), so its gradient passes the LeakyReLU
                # derivative too:  dx = LeakyReLU'(x) * (dgrad + g_skip)
                ops.conv_gemm([self.dyd[j]], self.w_d_dg[j], g_ph, self.dyd[0], C[0], S[j],
                              bwd=self._bwd_epilogue(None, self.A[0], 0.2))
                ops.lrelu_bwd(self.A[0], skip, 0.2, self.dyd[0], accumulate=True)
            else:
                ops.conv_gemm([self.dyd[j]], self.w_d_dg[j], g_ph, self.dyd[0], C[0], S[j],
                              bwd=self._bwd_epilogue(None, self.A[0], 0.2, g2=skip))
        if v0:
            return
        dbias0 = self.grad(self.k_down[0] + ".bias") if inst else None
        self._fork_wgrad(lambda: ops.thin_conv_wgrad(self.dyd[0], self.x_nhwc, None, gseg(self.k_down[0] + ".weight"), 64,
                                                     dbias=dbias0, c0=self.input_nc))
        self._ready(self.k_down[0] + ".weight", *((self.k_down[0] + ".bias",) if inst else ()), side=True)


# ================================================================================================
# Discriminator
# ================================================================================================
class DiscriminatorEngine(_Net):
    """NLayerDiscriminator(input_nc, ndf, n_layers, BatchNorm2d or InstanceNorm2d) over cat(A, B), input_nc in 2..8:
    forward takes A and B as two 4-slot sources of split = (channels of A, channels of B) channels, by default
    discriminator_split(input_nc) (3 | 3 for the reference's 6)."""

    # BatchNorm + LeakyReLU of the last normalised layer (models.py:239-240) applied inside the Cout = 1 head's forward
    # and wgrad kernels instead of a separate pass that writes H (63 MB written + re-read per forward at batch 64)
    fuse_head = True

    _BUFFER_ATTRS = ("hs", "ws", "H", "y", "logits", "z_ws", "dlogits", "gH", "dy", "dfake", "_xa", "_xb")

    def __init__(self, device, input_nc: int = 6, ndf: int = 64, n_layers: int = 3, init: bool = True,
                 norm: str = "batch", split: Optional[Tuple[int, int]] = None) -> None:
        super().__init__(device, norm)
        if self.norm == "instance":
            # the head's kernels take per-channel (scale, shift) only; InstanceNorm's are per image: H is materialised
            self.fuse_head = False
        if split is None:
            split = discriminator_split(input_nc)
        else:
            split = (check_image_channels("split[0]", split[0]), check_image_channels("split[1]", split[1]))
            if sum(split) != input_nc:
                raise ValueError(f"split {split} does not add up to input_nc = {input_nc}")
        self.split = split
        if ndf % 64 != 0 or n_layers < 1:
            raise NotImplementedError("ndf must be a multiple of 64")
        self.spec = sp = DiscriminatorSpec(input_nc, ndf, n_layers, norm=self.norm)
        self.nl = n_layers
        self.C = C = sp.C
        self.k_conv, self.k_bn, self.n_conv = sp.k_conv, sp.k_bn, sp.n_conv
        self._reg_small(self.k_conv[0] + ".weight", C[0], input_nc, 128)
        self._reg_vec(self.k_conv[0] + ".bias", C[0])
        self.bn: List[Optional[_BN]] = [None] * self.n_conv
        for k in range(1, n_layers + 1):
            self._reg_conv(self.k_conv[k] + ".weight", C[k], C[k - 1])
            self.bn[k] = (self._reg_in if self.norm == "instance" else self._reg_bn)(self.k_bn[k], C[k])
        self._reg_conv(self.k_conv[-1] + ".weight", 1, C[-1])
        self._reg_vec(self.k_conv[-1] + ".bias", 1)
        self.store.allocate(device)
        for bn in self.bns.values():
            bn.allocate(device)
        self.key_order = sp.key_order()
        bf = dict(device=device, dtype=torch.bfloat16)
        self.w_fwd = [None] + [torch.zeros(1, C[k], 16 * C[k - 1], **bf) for k in range(1, n_layers + 1)]
        self.w_fwd.append(torch.zeros(1, 1, 16 * C[-1], **bf))
        self.w_dg = [None]
        # first conv seen from its input gradient: [(kh*4+kw)*c + ch][64] per source; B (channels ca..) and A (0..ca-1)
        ca, cb = split
        self.w_T2 = torch.zeros(16 * cb, C[0], **bf)
        self.w_T2a = torch.zeros(16 * ca, C[0], **bf)
        for k in range(1, n_layers + 1):
            if k < n_layers:
                self.w_dg.append(torch.zeros(4, C[k - 1], 4 * C[k], **bf))     # stride 2: four phases
            else:
                self.w_dg.append(torch.zeros(1, C[k - 1], 16 * C[k], **bf))    # stride 1: flipped taps
        self.w_dg.append(None)                                                  # Cout = 1: direct kernels, no operand
        self.w_thin = torch.zeros(C[0], 128, **bf)   # first conv: [64][16 taps x (A slots 0-3 | B slots 4-7)]
        self._n = None
        self._plan = None
        if init:
            self.init_from_torch_default()

    def stride(self, k: int) -> int:
        return 2 if k < self.nl else 1

    def init_from_torch_default(self) -> None:
        """RNG order of NLayerDiscriminator.__init__ (models.py:223-243), see spec.DiscriminatorSpec."""
        self.load_state_dict(self.spec.default_state_dict())

    def repack(self) -> None:
        if self._plan is None:
            self._plan = self._build_pack_plan()
        self._plan.run()

    def _build_pack_plan(self) -> ops.PackPlan:
        C, p, off = self.C, self.store.p, self.store.off
        plan = ops.PackPlan()
        o = off(self.k_conv[0] + ".weight")
        ca, cb = self.split
        c = ca + cb
        plan.add(p, o, self.w_thin, 0, 1, C[0], C[0], (4, 4), ca, 8, 128, (128, 1, 4 * c, c))
        plan.add(p, o + ca, self.w_thin, 0, 1, C[0], C[0], (4, 4), cb, 8, 128, (128, 1, 4 * c, c), out_off=4)
        for tap in range(16):
            plan.add(p, o + c * tap + ca, self.w_T2, 0, 1, cb, cb, (1, 1), C[0], C[0], C[0], (1, 128, 0, 0),
                     out_off=cb * tap * C[0])
            plan.add(p, o + c * tap, self.w_T2a, 0, 1, ca, ca, (1, 1), C[0], C[0], C[0], (1, 128, 0, 0),
                     out_off=ca * tap * C[0])
        for k in range(1, self.n_conv):
            ci = C[k - 1]
            co = 1 if k == self.n_conv - 1 else C[k]
            o = off(self.k_conv[k] + ".weight")
            plan.add(p, o, self.w_fwd[k], 0, 1, co, co, (4, 4), ci, ci, 16 * ci, (16 * ci, 1, 4 * ci, ci))
            if k == self.n_conv - 1:
                continue            # Cout = 1: the direct kernels read the forward operand
            if self.stride(k) == 2:
                plan.add(p, o, self.w_dg[k], 2, 4, ci, ci, (2, 2), co, co, 4 * co, (1, 16 * ci, 4 * ci, ci))
            else:
                cp = max(co, 64)
                plan.add(p, o, self.w_dg[k], 1, 1, ci, ci, (4, 4), co, cp, 16 * cp, (1, 16 * ci, 4 * ci, ci))
        return plan

    def _alloc(self, n: int, h: int, w: int) -> None:
        if self._n == (n, h, w, self.fuse_head):
            return
        C = self.C
        bf = dict(device=self.dev, dtype=torch.bfloat16)
        hs, ws = [h // 2], [w // 2]
        for k in range(1, self.n_conv):
            if self.stride(k) == 2:
                hs.append(hs[-1] // 2)
                ws.append(ws[-1] // 2)
            else:
                hs.append(hs[-1] - 1)
                ws.append(ws[-1] - 1)
        self.hs, self.ws = hs, ws
        # H[k] = LeakyReLU(BN(y[k])): the input of conv k+1.  The last one is never materialised: the Cout = 1 head
        # (forward and wgrad) normalises + activates the raw y while reading it (fuse_head).
        self.H = [None if (self.fuse_head and k == self.n_conv - 2) else torch.empty(n, hs[k], ws[k], C[k], **bf)
                  for k in range(self.n_conv - 1)]
        self.y = [None] + [torch.empty(n, hs[k], ws[k], C[k], **bf) for k in range(1, self.n_conv - 1)]
        self.logits = torch.empty(n, hs[-1], ws[-1], 1, device=self.dev)
        self.z_ws = torch.empty(n * hs[-2] * ws[-2], 16, device=self.dev)      # per-pixel tap products of the last conv
        self.dlogits = torch.zeros(n, hs[-1], ws[-1], device=self.dev)            # fp32 d(loss)/d(logits)
        self.gH = [torch.empty(n, hs[k], ws[k], C[k], **bf) for k in range(self.n_conv - 1)]
        self.dy = [torch.empty(n, hs[k], ws[k], C[k], **bf) for k in range(self.n_conv - 1)]
        self.dfake = torch.zeros(n, h, w, 4, device=self.dev)
        for m in self.ins.values():
            m.allocate(n, self.dev)
        self._n = (n, h, w, self.fuse_head)
        self.alloc_gen += 1

    @_on_device
    def forward(self, xa: torch.Tensor, xb: torch.Tensor) -> torch.Tensor:
        """xa, xb: NHWC bf16 [n,h,w,4 slots] holding split[0] / split[1] channels, the rest zero (the two halves of
        torch.cat((A, B), 1), train_gan.py:57,59,66).  Returns fp32 logits [n,h',w',1]."""
        n, h, w, _ = xa.shape
        self._join_wgrad()
        self._alloc(n, h, w)
        C = self.C
        self._xa, self._xb = xa, xb
        ops.thin_conv_fwd(xa, xb, self.w_thin, self.param(self.k_conv[0] + ".bias"), self.H[0], ACT_LRELU)
        inst = self.norm == "instance"
        for k in range(1, self.n_conv - 1):
            bn = self.bn[k]
            ops.conv_gemm([self.H[k - 1]], self.w_fwd[k], ops.geom_conv_fwd(4, self.stride(k), 1), self.y[k], C[k],
                          (self.hs[k], self.ws[k]), stats=bn.stats if (self.training and not inst) else None)
            if inst:
                self._in_forward(bn, self.y[k], self.H[k], ACT_LRELU)
            elif self.H[k] is None:
                self._bn_scale_shift(bn, self.y[k])          # applied by the head's kernels on the fly
            else:
                self._bn_forward(bn, self.y[k], self.H[k], ACT_LRELU)
        k = self.n_conv - 1
        if self.H[k - 1] is None:
            hb = self.bn[k - 1]
            ops.cout1_conv_fwd(self.y[k - 1], self.w_fwd[k].view(-1), self.param(self.k_conv[k] + ".bias"), self.z_ws,
                               self.logits, pre=(hb.scale, hb.shift, 0.2))
        else:
            ops.cout1_conv_fwd(self.H[k - 1], self.w_fwd[k].view(-1), self.param(self.k_conv[k] + ".bias"), self.z_ws,
                               self.logits)
        return self.logits

    @_on_device
    def backward(self, wgrad: bool, input_grad: bool, input_grad_a: bool = False, final_hook=None) -> Optional[torch.Tensor]:
        """Consumes self.dlogits (fp32 [n, h', w']).  wgrad=False skips every parameter gradient (the G step);
        input_grad=True returns d(loss)/d(xb) as fp32 NHWC [n,h,w,4] (channels >= split[1] zero); input_grad_a also
        writes d(loss)/d(xa) into self.dreal.  The last conv's bias gradient (sum of dlogits) is
        produced by whoever wrote dlogits (gap_bce_logits_const_f32 / gap_sum_f32).  final_hook(offset, stream): called
        when this pass has enqueued the last contribution to every gradient from `offset` to the end of the flat buffer
        (the buffer is in forward order, backward finalises it from the tail): the data-parallel reducer starts reducing
        that tail while the rest of the pass runs."""
        C = self.C
        last = self.n_conv - 1
        g = self.store.g
        self._join_wgrad()
        lb = self.bn[last - 1]
        if wgrad:
            wseg = self.store.seg(g, self.k_conv[last] + ".weight")
            if self.H[last - 1] is None:
                self._fork_wgrad(lambda: ops.cout1_conv_wgrad(self.dlogits, self.y[last - 1], wseg,
                                                              pre=(lb.scale, lb.shift, 0.2)))
            else:
                self._fork_wgrad(lambda: ops.cout1_conv_wgrad(self.dlogits, self.H[last - 1], wseg))
        inst = self.norm == "instance"
        if inst:        # plain input gradient of H; the InstanceNorm backward below applies the LeakyReLU backward
            ops.cout1_conv_dgrad(self.dlogits, self.w_fwd[last].view(-1), self.gH[last - 1])
        else:
            # the Cout = 1 dgrad kernel applies the LeakyReLU backward of the last BatchNorm layer and accumulates its sums
            ops.cout1_conv_dgrad(self.dlogits, self.w_fwd[last].view(-1), self.gH[last - 1],
                                 bwd=dict(y=self.y[last - 1], scale=lb.scale, shift=lb.shift, slope=0.2, sums=lb.sums))
        for k in range(last - 1, 0, -1):
            if inst:
                self._in_backward(self.bn[k], self.y[k], self.gH[k], None, 0.2, self.dy[k])
            else:
                self._bn_backward_fused(self.bn[k], self.y[k], self.gH[k], self.dy[k], param_grads=wgrad)
            s = self.stride(k)
            if wgrad:
                self._fork_wgrad(lambda k=k, s=s: ops.conv_wgrad(
                    self.dy[k], self.H[k - 1], self.store.seg(g, self.k_conv[k] + ".weight"), (4, 4), s, (-1, -1),
                    16 * C[k - 1], C[k - 1]))
                if final_hook is not None:
                    final_hook(self.store.off(self.k_conv[k] + ".weight"), self._wgrad_stream if self._wgrad_used else None)
            geom = ops.geom_phase_k4s2p1() if s == 2 else ops.geom_conv_dgrad_s1(4, 1)
            grid = (self.hs[k], self.ws[k]) if s == 2 else (self.hs[k - 1], self.ws[k - 1])
            # algorithmic FLOPs of a dgrad = those of the layer's forward (the stride-1 dgrad runs its GEMM over the
            # 32x32 input grid with zero-padded borders: 6.6 % more MMA work than the 31x31 forward, not counted)
            fl = 2.0 * self.dy[k].shape[0] * self.hs[k] * self.ws[k] * C[k] * C[k - 1] * 16
            if k - 1 >= 1 and inst:
                ops.conv_gemm([self.dy[k]], self.w_dg[k], geom, self.gH[k - 1], C[k - 1], grid, flops=fl)
            elif k - 1 >= 1:
                nb = self.bn[k - 1]
                ops.conv_gemm([self.dy[k]], self.w_dg[k], geom, self.gH[k - 1], C[k - 1], grid, stats=nb.sums,
                              bwd=self._bwd_epilogue(nb, self.y[k - 1], 0.2), flops=fl)
            else:   # H[0] = LeakyReLU(conv + bias): the epilogue writes dy[0] directly
                ops.conv_gemm([self.dy[k]], self.w_dg[k], geom, self.dy[0], C[0], grid,
                              bwd=self._bwd_epilogue(None, self.H[0], 0.2), flops=fl)
        if wgrad:
            self._fork_wgrad(lambda: ops.thin_conv_wgrad(self.dy[0], self._xa, self._xb,
                                                         self.store.seg(g, self.k_conv[0] + ".weight"), 128,
                                                         dbias=self.grad(self.k_conv[0] + ".bias"), c0=self.split[0],
                                                         c1=self.split[1]))
        if input_grad:
            ops.thin_convT_fwd(self.dy[0], self.w_T2, None, ACT_NONE, None, self.dfake, co=self.split[1])
            if input_grad_a:
                self.dreal = torch.zeros_like(self.dfake)
                ops.thin_convT_fwd(self.dy[0], self.w_T2a, None, ACT_NONE, None, self.dreal, co=self.split[0])
            return self.dfake
        return None


# ================================================================================================
# One GAN training iteration
# ================================================================================================
class Pix2PixTrainer:
    """train_gan_one_epoch's loop body (train_gan.py:52-74) on one GPU; `world` > 1 adds the
    data-parallel gradient all-reduce (see parallel.py)."""

    overlap_g_fwd = True     # generator forward on its own stream while D processes the real pair (see train_step)

    def __init__(self, device, lr_g: float = 1e-4, lr_d: float = 1e-4, beta1: float = 0.5, num_downs: int = 7,
                 ngf: int = 64, ndf: int = 64, n_layers: int = 3, allreduce=None, world: int = 1,
                 bucket_elems: int = 8 << 20, use_dropout: bool = False, norm: str = "batch", input_nc: int = 3,
                 output_nc: int = 3) -> None:
        """norm: "batch" (nn.BatchNorm2d, the reference default) or "instance" (nn.InstanceNorm2d, pix2pix's
        `--norm instance`) in both networks.  input_nc / output_nc (1..4): channels of real_A and of real_B / fake_B;
        the discriminator sees cat(A, B) with A as its first input_nc channels."""
        self.dev = torch.device(device)
        self.norm = norm
        self.input_nc = check_image_channels("input_nc", input_nc)
        self.output_nc = check_image_channels("output_nc", output_nc)
        # construction order G then D fixes the seeded weights (train_gan.py:138-139)
        self.G = GeneratorEngine(self.dev, input_nc, output_nc, num_downs, ngf, use_dropout=use_dropout, norm=norm)
        self.D = DiscriminatorEngine(self.dev, input_nc + output_nc, ndf, n_layers, norm=norm,
                                     split=(input_nc, output_nc))
        self.lr_g, self.lr_d, self.betas = lr_g, lr_d, (beta1, 0.999)
        self.loss_acc = torch.zeros(4, device=self.dev, dtype=torch.float64)  # d_real, d_fake, g_gan, l1 (re-zeroed by
        self.loss_out = torch.zeros(2, device=self.dev, dtype=torch.float64)  # gap_gan_losses at the end of each step)
        self.allreduce = allreduce
        self.world = world
        self.a_nhwc = None
        # data parallel: bucketed all-reduce of the flat gradient buffers; the generator's buckets are reduced
        # on a side stream while its backward pass is still running (buffer order = completion order)
        self.g_reducer = self.d_reducer = None
        self._graph = None
        self._graph_sig = None
        self._g_stream = None
        if world > 1 and allreduce is None:
            import os
            from .parallel import GradBucketReducer
            bucket_elems = int(os.environ.get("GAP_BUCKET_ELEMS", bucket_elems))      # bring-up sweeps
            from .parallel import TailReducer
            # generator: buckets in backward-completion order; the LAST bucket (reduced after the pass, i.e. exposed)
            # holds only the trailing small segments.  discriminator: its buffer is in forward order, so it is reduced
            # from the tail (the 2.1 M-parameter conv right after the head's gradients, under the rest of the pass).
            self.g_reducer = GradBucketReducer(self.G.store.g, self.G.grad_segments(), bucket_elems=bucket_elems,
                                               tail_elems=int(os.environ.get("GAP_TAIL_ELEMS", 1 << 20)))
            self.d_reducer = TailReducer(self.D.store.g, min_elems=1 << 20, comm_stream=self.g_reducer.comm_stream)
            self.G.grad_hook = self.g_reducer.mark_ready
        if world > 1:
            self.sync_replicas()

    def sync_replicas(self, src: int = 0) -> None:
        """Data parallel: every replica adopts rank `src`'s parameters, Adam state and BatchNorm buffers (like
        DistributedDataParallel at construction).  Call again after loading a checkpoint on one rank only."""
        from .parallel import broadcast_replica_state
        broadcast_replica_state([self.G, self.D], src)

    def _graph_key(self, real_A: torch.Tensor) -> tuple:
        """Everything a captured iteration bakes in: input shape / dtype, the activation sets (raw device pointers and
        TMA tensor maps of the engines' buffers) and the optimizer hyper-parameters (kernel arguments)."""
        return (tuple(real_A.shape), real_A.dtype, self.G.alloc_gen, self.D.alloc_gen, self.lr_g, self.lr_d, self.betas)

    @_on_device
    def train_step_graphed(self, real_A: torch.Tensor, real_B: torch.Tensor) -> torch.Tensor:
        """train_step through a CUDA graph: the first call (and any call after the input shape, the engines' activation
        buffers or lr / betas changed — e.g. an eager train_step at another batch size re-allocated them) runs the
        iteration eagerly and captures its launches; later calls copy the batch into the static input buffers and
        replay.  Same results as train_step (a fresh tensor per call); single-GPU only."""
        if self.world > 1 or self.G.use_dropout:      # dropout draws host-numbered masks per forward: no replay
            return self.train_step(real_A, real_B)
        if self._graph is None or self._graph_sig != self._graph_key(real_A):
            self._graph = None
            self._g_in = (torch.empty_like(real_A), torch.empty_like(real_B))
            self._g_in[0].copy_(real_A)
            self._g_in[1].copy_(real_B)
            side = torch.cuda.Stream(self.dev)
            side.wait_stream(torch.cuda.current_stream(self.dev))
            with torch.cuda.stream(side):
                first = self.train_step(*self._g_in)  # this call's iteration, eagerly (also sizes every buffer)
            torch.cuda.current_stream(self.dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):             # capture only: nothing executes here
                self._g_out = self.train_step(*self._g_in)
            self._graph, self._graph_sig = graph, self._graph_key(real_A)
            return first
        self._g_in[0].copy_(real_A, non_blocking=True)
        self._g_in[1].copy_(real_B, non_blocking=True)
        self._graph.replay()
        self.G.store.step += 1                        # host mirrors of the device-side Adam step counters
        self.D.store.step += 1
        return self._g_out.clone()

    @_on_device
    def train_step(self, real_A: torch.Tensor, real_B: torch.Tensor,
                   loss_host: Optional[torch.Tensor] = None) -> torch.Tensor:
        """real_A / real_B: fp32 NCHW in [-1, 1] on the device (what the reference's DataLoader yields), or BOTH as raw
        uint8 [n, h, w, input_nc] / [n, h, w, output_nc] images: the ToTensor + JointNormalize of dataset.py:28-29,155-159 then runs on the device
        inside the first kernels (4x less host->device traffic).  Returns a device tensor [loss_d, loss_g] (fp64); no
        host synchronisation happens here.  loss_host: a PINNED host fp64[2] tensor — the step's last kernel then stores
        the two losses straight into host memory (zero-copy over PCIe; valid once the stream has passed that kernel) and
        that tensor is returned: the per-step `.item()` of train_gan.py:72-74 without a memcpy node in the stream."""
        G, D = self.G, self.D
        u8 = real_A.dtype == torch.uint8
        if u8 != (real_B.dtype == torch.uint8):
            raise ValueError("real_A and real_B must both be fp32 NCHW or both uint8 NHWC")
        if u8:
            n, h, w, _ = real_A.shape
            cb = real_B.shape[-1]
        else:
            n, _, h, w = real_A.shape
            cb = real_B.shape[1]
        if cb != self.output_nc:
            raise ValueError(f"real_B has {cb} channels, expected output_nc = {self.output_nc}")
        if self.a_nhwc is None or self.a_nhwc.shape[:3] != (n, h, w):
            self.a_nhwc = torch.zeros(n, h, w, 4, device=self.dev, dtype=torch.bfloat16)
            self.b_nhwc = torch.zeros_like(self.a_nhwc)
        G.training = D.training = True
        if u8:
            ops.u8_hwc_to_nhwc_bf16(real_B, self.b_nhwc)
        else:
            ops.nchw_to_nhwc_bf16(real_B, self.b_nhwc)
        # ---- D step (train_gan.py:55-63)
        D.zero_grad()
        # :56 and :65 are the same forward (done once, BatchNorm buffers updated twice) unless dropout draws new masks
        a_nhwc = G.prepare_input(real_A)
        cur = torch.cuda.current_stream(self.dev)
        fork = self.overlap_g_fwd
        if fork:
            # The discriminator's pass over the REAL pair (:57-58 and its backward) does not depend on the generator:
            # run the generator forward on its own stream meanwhile, so its under-filled 8x8 .. 1x1 bottleneck layers
            # share the GPU with the discriminator's large layers.  Joined before D sees fake_B.
            if self._g_stream is None:
                self._g_stream = torch.cuda.Stream(self.dev)
            self._g_stream.wait_stream(cur)
            with torch.cuda.stream(self._g_stream):
                G.forward(real_A, bn_repeat=1 if G.use_dropout else 2, x_ready=True)
        else:
            G.forward(real_A, bn_repeat=1 if G.use_dropout else 2, x_ready=True)
        logits = D.forward(a_nhwc, self.b_nhwc)            # :57
        cnt = logits.numel()
        d_bias_last = D.grad(D.k_conv[-1] + ".bias")
        ops.bce_logits_const_f32(logits, 1.0, 0.5 / cnt, D.dlogits, self.loss_acc[0:1], d_bias_last)   # :58,61
        D.backward(wgrad=True, input_grad=False)
        if fork:
            cur.wait_stream(self._g_stream)
        logits = D.forward(a_nhwc, G.fake_bf)              # :59
        ops.bce_logits_const_f32(logits, 0.0, 0.5 / cnt, D.dlogits, self.loss_acc[1:2], d_bias_last)   # :60,61
        if self.d_reducer is not None:
            self.d_reducer.begin()
            D.backward(wgrad=True, input_grad=False,       # :62 — this pass completes the D gradients
                       final_hook=lambda off, st: self.d_reducer.ready_from(off, (st,)))
        else:
            D.backward(wgrad=True, input_grad=False)       # :62
        D._join_wgrad()
        if self.d_reducer is not None:
            self.d_reducer.finish()
        elif self.allreduce is not None:
            self.allreduce(D.store.g)
        D.adam_step(self.lr_d, self.betas, grad_scale=1.0 / self.world)   # :63
        # ---- G step (train_gan.py:64-71)
        G.zero_grad()
        if G.use_dropout:
            G.forward(real_A, bn_repeat=1)                 # :65 with fresh dropout masks
        logits = D.forward(a_nhwc, G.fake_bf)              # :66 (updated D)
        ops.bce_logits_const_f32(logits, 1.0, 1.0 / cnt, D.dlogits, self.loss_acc[2:3])   # :67
        dfake = D.backward(wgrad=False, input_grad=True)
        numel = n * self.output_nc * h * w
        ops.gen_out_bwd(G.fake_f32, real_B, dfake, LAMBDA_L1 / numel, G.dpre, self.loss_acc[3:4])  # :68-70
        if self.g_reducer is not None:
            self.g_reducer.begin()
        G.backward()
        if self.g_reducer is not None:
            G._join_wgrad()
            self.g_reducer.finish()
        elif self.allreduce is not None:
            self.allreduce(G.store.g)
        G.adam_step(self.lr_g, self.betas, grad_scale=1.0 / self.world)   # :71
        if loss_host is not None:
            if not loss_host.is_pinned() or loss_host.dtype != torch.float64 or loss_host.numel() < 2:
                raise ValueError("loss_host must be a pinned fp64 host tensor with 2 elements")
            ops.gan_losses(self.loss_acc, cnt, LAMBDA_L1, numel, loss_host)      # :61, :68-69, written over PCIe
            return loss_host
        ops.gan_losses(self.loss_acc, cnt, LAMBDA_L1, numel, self.loss_out)      # :61, :68-69
        return self.loss_out.clone()     # (callers may keep the result across steps)
