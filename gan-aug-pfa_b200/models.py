"""Drop-in replacement for the reference's ``models.py`` GAN classes.

Same names, constructor arguments, ``forward`` signatures, parameter/buffer registration order (hence
the same seeded initial weights) and ``state_dict()`` layout as the reference (models.py:149-247,
SURVEY.md §8b / App. C), so ``train_gan.py`` and ``generate_synthetic_data.py`` run unchanged with
``from models import UNetGenerator, NLayerDiscriminator`` pointing here.  The modules hold ordinary
torch Parameters / buffers; ``forward`` hands them to the native engine (libgap_b200.so through the C
ABI) and plugs the result into torch autograd with one custom Function per network, so
``loss.backward()`` and ``torch.optim.Adam`` work as in the reference.

The native kernels exist only for CUDA tensors: calling ``forward`` on CPU tensors raises (there is
no CPU fallback).  The fastest path is not this module but ``pix2pix.Pix2PixTrainer``, which keeps
the whole iteration on the device without autograd bookkeeping.
"""
from __future__ import annotations

import functools
from typing import Optional

import torch
import torch.nn as nn

from . import ops
from .pix2pix import DiscriminatorEngine, GeneratorEngine, check_image_channels, discriminator_split


# ------------------------------------------------------------------------------------------------
# module skeletons: identical structure to the reference so that keys and RNG consumption match
# ------------------------------------------------------------------------------------------------
# the keyword defaults of the two normalisations the reference handles (models.py:173-176); a norm_layer is accepted only
# in these configurations, given as the class or as functools.partial(class, <some of these keywords>)
_NORM_DEFAULTS = {
    nn.BatchNorm2d: ("batch", dict(eps=1e-5, momentum=0.1, affine=True, track_running_stats=True)),
    nn.InstanceNorm2d: ("instance", dict(eps=1e-5, momentum=0.1, affine=False, track_running_stats=False)),
}
_SUPPORTED_NORMS = ("nn.BatchNorm2d, functools.partial(nn.BatchNorm2d, affine=True, track_running_stats=True), "
                    "nn.InstanceNorm2d or functools.partial(nn.InstanceNorm2d, affine=False, track_running_stats=False)")


def norm_kind(norm_layer, use_dropout: bool = False) -> str:
    """"batch" or "instance" for a norm_layer argument the native engines implement; NotImplementedError otherwise."""
    func, args, kw = norm_layer, (), {}
    if isinstance(norm_layer, functools.partial):
        func, args, kw = norm_layer.func, norm_layer.args, norm_layer.keywords
    kind, defaults = _NORM_DEFAULTS.get(func, (None, {}))
    if kind is None or args or any(k not in defaults or v != defaults[k] for k, v in kw.items()):
        raise NotImplementedError(f"norm_layer={norm_layer!r} is not implemented natively; supported: {_SUPPORTED_NORMS}")
    if kind == "instance" and use_dropout:
        raise NotImplementedError("norm_layer=nn.InstanceNorm2d together with use_dropout=True is not implemented natively")
    return kind


def _is_dense_permutation(t: torch.Tensor) -> bool:
    """True when the tensor's elements tile a contiguous block of memory exactly once in SOME dimension order (what
    torch calls non-overlapping and dense): foreach optimizers keep their fast path for such parameters."""
    dims = sorted((st, sz) for st, sz in zip(t.stride(), t.shape) if sz > 1)
    expect = 1
    for st, sz in dims:
        if st != expect:
            return False
        expect *= sz
    return True


class _NativeModule(nn.Module):
    """Shared engine management.  The first CUDA forward builds the native engine and re-homes the module's state in
    it: every Parameter whose GEMM-native master layout is a dense permutation of the torch layout becomes a strided
    VIEW of the engine's flat fp32 master buffer (same shape, same values, `state_dict()` unchanged), so
    `torch.optim.*.step()` updates the masters in place and the only per-step synchronisation left is the one-launch
    bf16 operand re-pack; the BatchNorm buffers are aliased the other way round (the engine updates the module's
    tensors).  The three zero-padded thin-layer weights stay ordinary Parameters and are copied (three tiny launches).

    Staleness is detected through `Parameter._version` (bumped by every in-place op, i.e. by optimizers and
    `load_state_dict`).  Writes through `p.data` do not bump it: call `module.sync()` after such edits."""

    _engine_obj = None
    _engine_key = None
    _versions = None
    _copied = ()

    def _make_engine(self, device):
        raise NotImplementedError

    def _adopt_parameters(self, eng) -> None:
        copied = []
        with torch.no_grad():
            for name, q in self.named_parameters():
                view = eng.param(name)
                view.copy_(q)
                if _is_dense_permutation(view):
                    q.data = view              # same Parameter object (optimizers keep working), engine-owned storage
                else:
                    copied.append((name, q))
        object.__setattr__(self, "_copied", tuple(copied))

    def sync(self) -> None:
        """Force the engine to re-read the parameters (needed only after edits through `.data`)."""
        object.__setattr__(self, "_versions", None)

    def _engine(self):
        p = next(self.parameters())
        if not p.is_cuda:
            raise RuntimeError(f"{type(self).__name__}: the native kernels need CUDA tensors; there is no CPU "
                               "fallback (move the module with .to('cuda'))")
        key = (p.device, tuple(id(b) for b in self.buffers()))
        eng = self._engine_obj
        if eng is not None and self._engine_key == key:
            # a .to() / .float() / manual re-assignment replaced parameter storage: adopt again
            for name, q in self.named_parameters():
                if q.data_ptr() != eng.param(name).data_ptr() and not any(q is c for _, c in self._copied):
                    eng = None
                    break
        if eng is None or self._engine_key != key:
            eng = self._make_engine(p.device)
            sd = dict(self.named_buffers())
            for prefix, bn in eng.bns.items():          # alias: running stats are updated in place
                bn.running_mean = sd[prefix + ".running_mean"]
                bn.running_var = sd[prefix + ".running_var"]
                bn.nbt = sd[prefix + ".num_batches_tracked"]
            self._adopt_parameters(eng)
            object.__setattr__(self, "_engine_obj", eng)
            object.__setattr__(self, "_engine_key", key)
            object.__setattr__(self, "_versions", None)
        versions = tuple(q._version for q in self.parameters())
        if versions != self._versions:
            with torch.no_grad():
                for name, q in self._copied:
                    eng.param(name).copy_(q)
            eng.repack()
            object.__setattr__(self, "_versions", versions)
        eng.training = self.training
        return eng

    def _grads_for_autograd(self, eng, names):
        """Parameter gradients for autograd: ONE copy of the flat gradient buffer, handed out as strided views with the
        parameters' own strides (so AccumulateGrad adopts them without another copy, and later backward passes, which
        overwrite the engine's buffer, cannot disturb `p.grad`)."""
        eng._join_wgrad()
        flat = eng.store.g.clone()
        return [eng.view(flat, name) for name in names]


class _BlockFn(torch.autograd.Function):
    """A stand-alone UnetSkipConnectionBlock through the native engine (forward, input gradient, parameter gradients)."""

    @staticmethod
    def forward(ctx, module, x, grad_mode, *params):
        eng = module._engine()
        eng.forward(x.detach().contiguous().float())
        out = eng.output_nchw()
        need = grad_mode and (x.requires_grad or any(p.requires_grad for p in params))
        ctx.module = module
        ctx.x_grad = x.requires_grad
        ctx.snap = eng.detach_buffers() if need else None
        return out

    @staticmethod
    def backward(ctx, gout):
        module = ctx.module
        eng = module._engine_obj
        eng.attach_buffers(ctx.snap)
        eng.zero_grad()
        names = [name for name, _ in module.named_parameters()]
        gx = None
        if eng.virtual0:
            n, c2, h, w = gout.shape
            ops.nchw_to_nhwc_bf16(gout.contiguous().float(), eng.gR[0])      # gradient of cat([x, model(x)], 1)
            eng.backward()
            if ctx.x_grad:
                gx = torch.empty(n, c2 // 2, h, w, device=gout.device)
                ops.nhwc_to_nchw_f32(eng.dyd[0], gx, c2 // 2)
        else:
            if ctx.x_grad:
                raise NotImplementedError("gradient w.r.t. the image input of the outermost block is not provided")
            ops.tanh_bwd(gout.contiguous().float(), eng.fake_f32, eng.dpre)
            eng.backward()
        grads = module._grads_for_autograd(eng, names)
        return (None, gx, None, *grads)


class UnetSkipConnectionBlock(_NativeModule):
    """One U-Net level (models.py:167-208).  Kept as a container of the reference's layers; the
    computation happens in UNetGenerator.forward through the native engine."""

    def __init__(self, outer_nc, inner_nc, input_nc=None, submodule=None, outermost=False, innermost=False,
                 norm_layer=nn.BatchNorm2d, use_dropout=False):
        super().__init__()
        self.outermost = outermost
        # structure record for the native engine of a direct call on this block (object.__setattr__: the nested block is
        # registered once, as part of self.model, like in the reference)
        object.__setattr__(self, "_sub", submodule)
        object.__setattr__(self, "_shape", (outer_nc, inner_nc, outer_nc if input_nc is None else input_nc,
                                            bool(outermost), bool(innermost)))
        object.__setattr__(self, "_has_dropout", bool(use_dropout) or
                           (submodule is not None and getattr(submodule, "_has_dropout", False)))
        object.__setattr__(self, "_norm", norm_kind(norm_layer, use_dropout))
        if type(norm_layer) == functools.partial:
            use_bias = norm_layer.func == nn.InstanceNorm2d
        else:
            use_bias = norm_layer == nn.InstanceNorm2d
        if input_nc is None:
            input_nc = outer_nc
        downconv = nn.Conv2d(input_nc, inner_nc, kernel_size=4, stride=2, padding=1, bias=use_bias)
        downrelu = nn.LeakyReLU(0.2, True)
        downnorm = norm_layer(inner_nc)
        uprelu = nn.ReLU(True)
        upnorm = norm_layer(outer_nc)
        if outermost:
            upconv = nn.ConvTranspose2d(inner_nc * 2, outer_nc, kernel_size=4, stride=2, padding=1)
            layers = [downconv, submodule, uprelu, upconv, nn.Tanh()]
        elif innermost:
            upconv = nn.ConvTranspose2d(inner_nc, outer_nc, kernel_size=4, stride=2, padding=1, bias=use_bias)
            layers = [downrelu, downconv, uprelu, upconv, upnorm]
        else:
            upconv = nn.ConvTranspose2d(inner_nc * 2, outer_nc, kernel_size=4, stride=2, padding=1, bias=use_bias)
            layers = [downrelu, downconv, downnorm, submodule, uprelu, upconv, upnorm]
            if use_dropout:
                layers.append(nn.Dropout(0.5))
        self.model = nn.Sequential(*layers)

    def _chain(self):
        """(outer_nc, inner_nc, input_nc, outermost, innermost) of this block and the blocks nested in it."""
        out, blk = [], self
        while blk is not None:
            if not isinstance(blk, UnetSkipConnectionBlock):
                raise NotImplementedError("the native path needs UnetSkipConnectionBlock sub-modules")
            if blk._norm != self._norm:
                raise NotImplementedError("nested blocks must all use the same norm_layer")
            out.append(blk._shape)
            blk = blk._sub
        return out

    def _make_engine(self, device):
        from .spec import GeneratorSpec
        if self._has_dropout:
            raise NotImplementedError("stand-alone blocks with use_dropout=True are not implemented natively "
                                      "(UNetGenerator(use_dropout=True) is)")
        return GeneratorEngine(device, init=False, spec=GeneratorSpec.for_block_chain(self._chain(), norm=self._norm))

    def forward(self, x):
        """models.py:204-208: `self.model(x)` for the outermost block, else `torch.cat([x, self.model(x)], 1)` — where x
        has already been through the block's in-place LeakyReLU, so the skip half is LeakyReLU(x) (and, like the
        reference, the caller's tensor is modified in place to match).  Inside a UNetGenerator the generator's fused
        engine runs the whole stack; this entry point serves direct calls on a block."""
        out = _BlockFn.apply(self, x, torch.is_grad_enabled(), *self.parameters())
        if not self.outermost and not (torch.is_grad_enabled() and x.requires_grad):
            with torch.no_grad():
                x.copy_(out[:, :x.shape[1]])          # nn.LeakyReLU(0.2, True) mutated the caller's tensor (models.py:178)
        return out


class _GeneratorFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, x, grad_mode, *params):
        eng = module._engine()
        if x.requires_grad:
            raise NotImplementedError("gradient w.r.t. the generator input is not provided (the reference never needs it)")
        eng.forward(x.detach().contiguous().float())
        out = eng.output_nchw()
        ctx.module = module
        # under no_grad / for frozen parameters nothing is kept: the next forward reuses the activation buffers
        # (grad_mode is sampled by the caller: inside Function.forward autograd is always off)
        need = grad_mode and any(p.requires_grad for p in params)
        ctx.snap = eng.detach_buffers() if need else None
        return out

    @staticmethod
    def backward(ctx, gout):
        module = ctx.module
        eng = module._engine_obj
        eng.attach_buffers(ctx.snap)
        eng.zero_grad()
        ops.tanh_bwd(gout.contiguous().float(), eng.fake_f32, eng.dpre)
        eng.backward()
        grads = module._grads_for_autograd(eng, [name for name, _ in module.named_parameters()])
        return (None, None, None, *grads)


class UNetGenerator(_NativeModule):
    """U-Net generator (models.py:149-164) executing on the native sm_100a kernels."""

    def __init__(self, input_nc, output_nc, num_downs=7, ngf=64, norm_layer=nn.BatchNorm2d, use_dropout=False):
        super().__init__()
        self._norm = norm_kind(norm_layer, use_dropout)
        check_image_channels("input_nc", input_nc)
        check_image_channels("output_nc", output_nc)
        self._cfg = (input_nc, output_nc, num_downs, ngf)
        self._use_dropout = bool(use_dropout)
        blk = UnetSkipConnectionBlock(ngf * 8, ngf * 8, input_nc=None, submodule=None, norm_layer=norm_layer,
                                      innermost=True)
        for _ in range(num_downs - 5):
            blk = UnetSkipConnectionBlock(ngf * 8, ngf * 8, input_nc=None, submodule=blk, norm_layer=norm_layer,
                                          use_dropout=use_dropout)
        blk = UnetSkipConnectionBlock(ngf * 4, ngf * 8, input_nc=None, submodule=blk, norm_layer=norm_layer)
        blk = UnetSkipConnectionBlock(ngf * 2, ngf * 4, input_nc=None, submodule=blk, norm_layer=norm_layer)
        blk = UnetSkipConnectionBlock(ngf, ngf * 2, input_nc=None, submodule=blk, norm_layer=norm_layer)
        self.model = UnetSkipConnectionBlock(output_nc, ngf, input_nc=input_nc, submodule=blk, outermost=True,
                                             norm_layer=norm_layer)

    def _make_engine(self, device):
        i, o, n, f = self._cfg
        return GeneratorEngine(device, i, o, n, f, init=False, use_dropout=self._use_dropout, norm=self._norm)

    def forward(self, input):
        return _GeneratorFn.apply(self, input, torch.is_grad_enabled(), *self.parameters())

    def translate_scene(self, img, tile=256, overlap=64, batch=32, return_float=False):
        """Sliding-window image of a whole scene at its own resolution (GeneratorEngine.translate_scene): always in eval
        mode, whatever mode the module is in; no autograd.  Returns a pix2pix.SceneImage(image, values)."""
        return self._engine().translate_scene(img, tile=tile, overlap=overlap, batch=batch, return_float=return_float)


class _DiscriminatorFn(torch.autograd.Function):
    """The input cat(A, B) is split by discriminator_split: A = the first ceil(input_nc / 2) channels, B = the rest."""

    @staticmethod
    def forward(ctx, module, x, grad_mode, *params):
        eng = module._engine()
        n, c, h, w = x.shape
        if c != sum(eng.split):
            raise ValueError(f"discriminator input has {c} channels, expected input_nc = {sum(eng.split)}")
        ca = eng.split[0]
        xd = x.detach().contiguous().float()
        xa = torch.zeros(n, h, w, 4, device=x.device, dtype=torch.bfloat16)
        xb = torch.zeros_like(xa)
        ops.nchw_to_nhwc_bf16(xd[:, :ca].contiguous(), xa)
        ops.nchw_to_nhwc_bf16(xd[:, ca:].contiguous(), xb)
        logits = eng.forward(xa, xb)
        out = logits.permute(0, 3, 1, 2).clone()
        ctx.module = module
        ctx.shape = (n, h, w)
        need = grad_mode and (x.requires_grad or any(p.requires_grad for p in params))
        ctx.snap = eng.detach_buffers() if need else None
        ctx.x_grad = x.requires_grad
        return out

    @staticmethod
    def backward(ctx, gout):
        module = ctx.module
        eng = module._engine_obj
        eng.attach_buffers(ctx.snap)
        eng.zero_grad()
        n, h, w = ctx.shape
        eng.dlogits.copy_(gout.reshape(eng.dlogits.shape))
        wgrad = any(p.requires_grad for p in module.parameters())
        if wgrad:
            ops.sum_f32(eng.dlogits, eng.grad(eng.k_conv[-1] + ".bias"))
        eng.backward(wgrad=wgrad, input_grad=ctx.x_grad, input_grad_a=ctx.x_grad)
        eng._join_wgrad()
        gx = None
        if ctx.x_grad:
            ca, cb = eng.split
            gx = torch.empty(n, ca + cb, h, w, device=gout.device)
            ops.nhwc_to_nchw_f32(eng.dreal, gx, ca, ca + cb, 0)
            ops.nhwc_to_nchw_f32(eng.dfake, gx, cb, ca + cb, ca)
        names = [name for name, _ in module.named_parameters()]
        grads = module._grads_for_autograd(eng, names) if wgrad else [None] * len(names)
        return (None, gx, None, *grads)


class NLayerDiscriminator(_NativeModule):
    """PatchGAN discriminator (models.py:212-247) executing on the native sm_100a kernels.  input_nc = 2..8: the input
    is read as cat(A, B) with A = its first ceil(input_nc / 2) channels (pix2pix.discriminator_split)."""

    def __init__(self, input_nc, ndf=64, n_layers=3, norm_layer=nn.BatchNorm2d):
        super().__init__()
        self._norm = norm_kind(norm_layer)
        discriminator_split(input_nc)
        self._cfg = (input_nc, ndf, n_layers)
        use_bias = False
        kw, padw = 4, 1
        sequence = [nn.Conv2d(input_nc, ndf, kernel_size=kw, stride=2, padding=padw), nn.LeakyReLU(0.2, True)]
        nf_mult = 1
        for n in range(1, n_layers):
            nf_prev, nf_mult = nf_mult, min(2 ** n, 8)
            sequence += [nn.Conv2d(ndf * nf_prev, ndf * nf_mult, kernel_size=kw, stride=2, padding=padw, bias=use_bias),
                         norm_layer(ndf * nf_mult), nn.LeakyReLU(0.2, True)]
        nf_prev, nf_mult = nf_mult, min(2 ** n_layers, 8)
        sequence += [nn.Conv2d(ndf * nf_prev, ndf * nf_mult, kernel_size=kw, stride=1, padding=padw, bias=use_bias),
                     norm_layer(ndf * nf_mult), nn.LeakyReLU(0.2, True)]
        sequence += [nn.Conv2d(ndf * nf_mult, 1, kernel_size=kw, stride=1, padding=padw)]
        self.model = nn.Sequential(*sequence)

    def _make_engine(self, device):
        i, d, n = self._cfg
        return DiscriminatorEngine(device, i, d, n, init=False, norm=self._norm)

    def forward(self, input):
        return _DiscriminatorFn.apply(self, input, torch.is_grad_enabled(), *self.parameters())


# ================================================================================================
# Siamese U-Net (models.py:7-145): same module structure / keys / RNG order, native execution
# ================================================================================================
def double_conv(in_channels, out_channels):
    """(Conv3x3 no-bias -> BatchNorm -> ReLU) x 2 (models.py:7-15).  A plain container: SiameseUNet.forward runs it
    through the native engine."""
    return nn.Sequential(
        nn.Conv2d(in_channels, out_channels, kernel_size=3, padding=1, bias=False),
        nn.BatchNorm2d(out_channels),
        nn.ReLU(inplace=True),
        nn.Conv2d(out_channels, out_channels, kernel_size=3, padding=1, bias=False),
        nn.BatchNorm2d(out_channels),
        nn.ReLU(inplace=True),
    )


class _GateFn(torch.autograd.Function):
    """A stand-alone AttentionGate through siamese.GateEngine (forward, both input gradients, parameter gradients).
    The engine keeps the activations of its most recent forward: backward must follow its forward."""

    @staticmethod
    def forward(ctx, module, g, x, *params):
        eng = module._engine()
        out = eng.forward(g.detach(), x.detach())
        n, h, w, fl = out.shape
        res = torch.empty(n, fl, h, w, device=out.device)
        ops.nhwc_to_nchw_f32(out, res, fl)
        ctx.module = module
        ctx.needs = (g.requires_grad, x.requires_grad)
        return res

    @staticmethod
    def backward(ctx, gout):
        module = ctx.module
        eng = module._engine_obj
        eng.zero_grad()
        ops.nchw_to_nhwc_bf16(gout.contiguous().float(), eng.gout)
        eng.backward()
        grads_in = []
        for need, buf in zip(ctx.needs, (eng.gg, eng.gxs)):
            if need:
                n, h, w, c = buf.shape
                t = torch.empty(n, c, h, w, device=gout.device)
                ops.nhwc_to_nchw_f32(buf, t, c)
                grads_in.append(t)
            else:
                grads_in.append(None)
        grads = module._grads_for_autograd(eng, [name for name, _ in module.named_parameters()])
        return (None, *grads_in, *grads)


class AttentionGate(_NativeModule):
    """Attention gate (models.py:18-44).  Inside SiameseUNet the network's fused engine executes it; a direct call runs
    the same kernels through a stand-alone siamese.GateEngine."""

    def __init__(self, F_g, F_l, F_int):
        super().__init__()
        self._cfg = (F_g, F_l, F_int)
        self.W_g = nn.Sequential(nn.Conv2d(F_g, F_int, kernel_size=1, stride=1, padding=0, bias=True), nn.BatchNorm2d(F_int))
        self.W_x = nn.Sequential(nn.Conv2d(F_l, F_int, kernel_size=1, stride=1, padding=0, bias=True), nn.BatchNorm2d(F_int))
        self.psi = nn.Sequential(nn.Conv2d(F_int, 1, kernel_size=1, stride=1, padding=0, bias=True), nn.BatchNorm2d(1),
                                 nn.Sigmoid())
        self.relu = nn.ReLU(inplace=True)

    def _make_engine(self, device):
        from .siamese import GateEngine
        return GateEngine(device, *self._cfg)

    def forward(self, g, x):
        """x * Sigmoid(BN(psi(ReLU(BN(W_g g) + BN(W_x x)))))   (models.py:39-44)"""
        return _GateFn.apply(self, g, x, *self.parameters())


class _EncoderFn(torch.autograd.Function):
    """SiameseUNet.forward_encoder on its own: one pass of the shared encoder through the network's engine."""

    @staticmethod
    def forward(ctx, module, x, *params):
        eng = module._engine()
        if x.requires_grad:
            raise NotImplementedError("gradients w.r.t. the input images are not provided (the reference never needs them)")
        feats = eng.forward_encoder(x.detach())
        outs = []
        for f in feats:
            n, h, w, c = f.shape
            t = torch.empty(n, c, h, w, device=f.device)
            ops.nhwc_to_nchw_f32(f, t, c)
            outs.append(t)
        ctx.module = module
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        module = ctx.module
        eng = module._engine_obj
        eng.zero_grad()
        for lvl, g in enumerate(gouts):
            c = g.shape[1] if g is not None else eng.gS[lvl].shape[-1] // 2
            slot = eng.gS[lvl][..., :c]
            if g is None:
                slot.zero_()
            else:
                ops.nchw_to_nhwc_bf16(g.contiguous().float(), slot)
        eng.backward_encoder()
        grads = module._grads_for_autograd(eng, [name for name, _ in module.named_parameters()])
        return (None, None, *grads)


class _SiameseFn(torch.autograd.Function):
    """One forward/backward of the whole Siamese U-Net through SiameseEngine.  The engine keeps the activations of
    the most recent forward, so backward must follow its forward (train.py:141-143 does exactly that)."""

    @staticmethod
    def forward(ctx, module, x1, x2, *params):
        eng = module._engine()
        if x1.requires_grad or x2.requires_grad:
            raise NotImplementedError("gradients w.r.t. the input images are not provided (the reference never needs them)")
        logits = eng.forward(x1.detach(), x2.detach())
        ctx.module = module
        ctx.shape = tuple(logits.shape)
        # n_classes = 1: the [n, h, w] map as [n, 1, h, w]; n_classes > 1: the [n, K, h, w] class planes as they are
        return logits.unsqueeze(1).clone() if logits.dim() == 3 else logits.clone()

    @staticmethod
    def backward(ctx, gout):
        module = ctx.module
        eng = module._engine_obj
        eng.zero_grad()
        eng.dlogits.copy_(gout.reshape(ctx.shape))
        eng.backward()
        grads = module._grads_for_autograd(eng, [name for name, _ in module.named_parameters()])
        return (None, None, None, *grads)


class SiameseUNet(_NativeModule):
    """Siamese U-Net with attention gates (models.py:47-145) executing on the native sm_100a kernels.  n_classes = 1
    returns [n, 1, h, w] logits for the sigmoid losses; n_classes = 2..16 returns [n, K, h, w] logits for
    nn.CrossEntropyLoss / torch.argmax(dim=1)."""

    def __init__(self, n_channels, n_classes):
        from .siamese import check_n_classes
        check_n_classes(n_classes)
        super().__init__()
        self.n_channels = n_channels
        self.n_classes = n_classes
        self.dconv_down1 = double_conv(n_channels, 64)
        self.dconv_down2 = double_conv(64, 128)
        self.dconv_down3 = double_conv(128, 256)
        self.dconv_down4 = double_conv(256, 512)
        self.maxpool = nn.MaxPool2d(2)
        self.bottleneck = double_conv(512, 1024)
        self.upsample = nn.Upsample(scale_factor=2, mode="bilinear", align_corners=True)
        self.att3 = AttentionGate(F_g=2048, F_l=1024, F_int=512)
        self.att2 = AttentionGate(F_g=512, F_l=512, F_int=256)
        self.att1 = AttentionGate(F_g=256, F_l=256, F_int=128)
        self.att_last = AttentionGate(F_g=128, F_l=128, F_int=64)
        self.dconv_up3 = double_conv(2048 + 1024, 512)
        self.dconv_up2 = double_conv(512 + 512, 256)
        self.dconv_up1 = double_conv(256 + 256, 128)
        self.dconv_last = double_conv(128 + 128, 64)
        self.conv_last = nn.Conv2d(64, n_classes, 1)

    def _make_engine(self, device):
        from .siamese import SiameseEngine
        return SiameseEngine(device, self.n_channels, self.n_classes)

    def forward_encoder(self, x):
        """One pass of the shared encoder (models.py:92-102): returns (conv1, conv2, conv3, conv4, bottleneck).  forward()
        runs both passes and the decoder inside one fused engine call; this entry point serves direct calls."""
        return _EncoderFn.apply(self, x, *self.parameters())

    def forward(self, x1, x2):
        return _SiameseFn.apply(self, x1, x2, *self.parameters())

    def predict_scene(self, img1, img2, tile=256, overlap=64, batch=8, return_probs=False, labels=None,
                      ignore_index=-100, tta=None):
        """Sliding-window change map of a whole scene at its own resolution (SiameseEngine.predict_scene; tta: None,
        "flips" or "d4" test-time augmentation): always in eval mode, whatever mode the module is in; no autograd.
        Returns a siamese.SceneResult(pred, probs, confusion)."""
        return self._engine().predict_scene(img1, img2, tile=tile, overlap=overlap, batch=batch,
                                            return_probs=return_probs, labels=labels, ignore_index=ignore_index,
                                            tta=tta)


def predict_scene_ensemble(modules, img1, img2, tile=256, overlap=64, batch=8, tta=None, return_probs=False,
                           labels=None, ignore_index=-100):
    """Sliding-window change map of a whole scene averaged over several SiameseUNet modules (a checkpoint ensemble)
    and, with tta = "flips" / "d4", over flipped / rotated tiles (siamese.predict_scene_ensemble): always in eval mode,
    whatever mode each module is in; no autograd.  Returns a siamese.SceneResult(pred, probs, confusion)."""
    from .siamese import predict_scene_ensemble as ensemble
    if isinstance(modules, nn.Module) or not isinstance(modules, (list, tuple)) or not modules:
        raise ValueError(f"modules must be a non-empty list of SiameseUNet, got {modules!r}")
    if not all(isinstance(m, SiameseUNet) for m in modules):
        raise ValueError(f"modules must all be SiameseUNet, got {[type(m).__name__ for m in modules]}")
    return ensemble([m._engine() for m in modules], img1, img2, tile=tile, overlap=overlap, batch=batch, tta=tta,
                    return_probs=return_probs, labels=labels, ignore_index=ignore_index)
