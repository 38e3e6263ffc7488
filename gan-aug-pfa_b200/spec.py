"""Pure-Python description of the reference networks' parameter layout (no CUDA needed): channel
progressions, state_dict keys in the reference's order, and the default torch initialisation drawn
from the global RNG in the reference's module-construction order (SURVEY.md App. B.13, App. C)."""
from __future__ import annotations

import math
from typing import Dict, List, Optional

import torch

BN_LEAVES = ["weight", "bias", "running_mean", "running_var", "num_batches_tracked"]
NORMS = ("batch", "instance")   # nn.BatchNorm2d | nn.InstanceNorm2d(affine=False, track_running_stats=False)


def _check_norm(norm: str) -> str:
    if norm not in NORMS:
        raise ValueError(f"norm must be one of {NORMS}, got {norm!r}")
    return norm


def _kaiming_uniform_(t: torch.Tensor) -> None:
    """nn.Conv2d / nn.ConvTranspose2d.reset_parameters."""
    torch.nn.init.kaiming_uniform_(t, a=math.sqrt(5))


def _bias_uniform_(b: torch.Tensor, weight: torch.Tensor) -> None:
    fan_in = weight.size(1) * weight.size(2) * weight.size(3)
    bound = 1 / math.sqrt(fan_in)
    torch.nn.init.uniform_(b, -bound, bound)


def _bn_entries(sd: Dict[str, torch.Tensor], prefix: str, c: int) -> None:
    sd[prefix + ".weight"] = torch.ones(c)
    sd[prefix + ".bias"] = torch.zeros(c)
    sd[prefix + ".running_mean"] = torch.zeros(c)
    sd[prefix + ".running_var"] = torch.ones(c)
    sd[prefix + ".num_batches_tracked"] = torch.tensor(0, dtype=torch.long)


class GeneratorSpec:
    """UNetGenerator(input_nc, output_nc, num_downs, ngf) with BatchNorm2d or InstanceNorm2d, no dropout
    (models.py:149-208).

    Block j (0 = outermost ... L-1 = innermost) owns down conv `k_down[j]` (C[j-1] -> C[j]) and up
    conv `k_up[j]` (2*C[j] or C[j] -> C[j-1]); down norm `k_dbn[j]` exists for 1 <= j <= L-2, up norm
    `k_ubn[j]` for 1 <= j <= L-1.  norm="instance": the norms hold no state, and every conv has a bias
    (use_bias, models.py:173-176)."""

    def __init__(self, input_nc: int = 3, output_nc: int = 3, num_downs: int = 7, ngf: int = 64,
                 C: Optional[List[int]] = None, root: str = "model.model", virtual0: bool = False,
                 norm: str = "batch") -> None:
        """`C`, `root`, `virtual0` describe a stand-alone UnetSkipConnectionBlock chain (see `for_block_chain`);
        by default the layout is UNetGenerator's."""
        self.norm = _check_norm(norm)
        if C is None:
            if num_downs < 5:
                raise ValueError("UNetGenerator needs num_downs >= 5 (models.py:155-161)")
            # models.py:155-161: innermost ngf*8, (num_downs-5) x ngf*8, then ngf*8->4, 4->2, 2->1, outermost
            C = [ngf, ngf * 2, ngf * 4] + [ngf * 8] * (num_downs - 3)
        self.input_nc, self.output_nc, self.L, self.ngf = input_nc, output_nc, len(C), ngf
        self.virtual0 = virtual0
        L = self.L
        self.C: List[int] = list(C)
        # Sequential index of the sub-block inside its parent: 1 in the outermost block, 3 in a middle block
        if virtual0:      # level 0 does not exist: level 1 is the called block itself, its Sequential is `root`
            pref = [None, root]
            for j in range(2, L):
                pref.append(pref[-1] + ".3.model")
        else:
            pref = [root]
            for j in range(1, L):
                pref.append(pref[-1] + (".1.model" if j == 1 else ".3.model"))
        self.pref = pref
        first = None if virtual0 else pref[0] + ".0"
        self.k_down = [first] + [pref[j] + ".1" for j in range(1, L)]
        self.k_dbn: List[Optional[str]] = [None] + [pref[j] + ".2" for j in range(1, L - 1)] + [None]
        self.k_up = [None if virtual0 else pref[0] + ".3"] + [pref[j] + ".5" for j in range(1, L - 1)] + [pref[L - 1] + ".3"]
        self.k_ubn: List[Optional[str]] = [None] + [pref[j] + ".6" for j in range(1, L - 1)] + [pref[L - 1] + ".4"]
        if L == 1:
            raise ValueError("a U-Net needs at least one nested block")

    @classmethod
    def for_block_chain(cls, chain, norm: str = "batch") -> "GeneratorSpec":
        """Layout of a stand-alone UnetSkipConnectionBlock (models.py:167-208) and the blocks nested inside it.
        `chain` lists (outer_nc, inner_nc, input_nc, outermost, innermost) from the called block inwards."""
        outer0, inner0, in0, outermost0, _ = chain[0]
        for (o, i, inp, om, im), nxt in zip(chain, chain[1:] + [None]):
            if nxt is None:
                if not im:
                    raise NotImplementedError("the innermost nested block must be built with innermost=True")
            elif nxt[0] != i or nxt[2] != i or nxt[3]:
                raise NotImplementedError("nested blocks must chain outer_nc == input_nc == the parent's inner_nc")
        if outermost0:
            return cls(in0, outer0, C=[c[1] for c in chain], root="model", norm=norm)
        if in0 != outer0:
            raise NotImplementedError("a stand-alone inner block needs input_nc == outer_nc (the reference's default)")
        return cls(in0, outer0, C=[in0] + [c[1] for c in chain], root="model", virtual0=True, norm=norm)

    def down_shape(self, j: int):
        return (self.C[j], self.input_nc if j == 0 else self.C[j - 1], 4, 4)

    def up_shape(self, j: int):
        cin = self.C[j] if j == self.L - 1 else 2 * self.C[j]
        return (cin, self.output_nc if j == 0 else self.C[j - 1], 4, 4)

    def key_order(self) -> List[str]:
        """state_dict() order of the reference module: depth-first through the nested Sequentials."""
        L = self.L
        inst = self.norm == "instance"
        conv = lambda k, bias: [k + ".weight"] + ([k + ".bias"] if bias else [])
        norm = lambda k: [] if inst else [k + "." + l for l in BN_LEAVES]

        def block(j: int) -> List[str]:
            if j == 0:
                if self.virtual0:
                    return block(1)
                return conv(self.k_down[0], inst) + block(1) + conv(self.k_up[0], True)
            keys = conv(self.k_down[j], inst)
            if j < L - 1:
                keys += norm(self.k_dbn[j])
                keys += block(j + 1)
            keys += conv(self.k_up[j], inst)
            keys += norm(self.k_ubn[j])
            return keys

        return block(0)

    def default_state_dict(self) -> Dict[str, torch.Tensor]:
        """Default torch init consuming the global CPU RNG exactly like UNetGenerator.__init__: blocks are
        built innermost first (models.py:155-161); within a block downconv (+bias with InstanceNorm), then upconv
        (+bias).  InstanceNorm2d(affine=False) draws nothing and has no entries."""
        sd: Dict[str, torch.Tensor] = {}
        inst = self.norm == "instance"

        def conv(key: str, shape, bias: bool) -> None:
            w = torch.empty(*shape)
            _kaiming_uniform_(w)
            sd[key + ".weight"] = w
            if bias:
                b = torch.empty(shape[1] if key in self.k_up else shape[0])
                _bias_uniform_(b, w)
                sd[key + ".bias"] = b

        for j in range(self.L - 1, 0 if self.virtual0 else -1, -1):
            conv(self.k_down[j], self.down_shape(j), inst)
            conv(self.k_up[j], self.up_shape(j), inst or j == 0)
            if inst:
                continue
            if self.k_dbn[j] is not None:
                _bn_entries(sd, self.k_dbn[j], self.C[j])
            if self.k_ubn[j] is not None:
                _bn_entries(sd, self.k_ubn[j], self.C[j - 1])
        return {k: sd[k] for k in self.key_order()}


class DiscriminatorSpec:
    """NLayerDiscriminator(input_nc, ndf, n_layers) with BatchNorm2d or InstanceNorm2d (models.py:212-247).  The middle
    convs have no bias with either norm (use_bias = False, models.py:221)."""

    def __init__(self, input_nc: int = 6, ndf: int = 64, n_layers: int = 3, norm: str = "batch") -> None:
        self.input_nc, self.ndf, self.nl = input_nc, ndf, n_layers
        self.norm = _check_norm(norm)
        self.C = [ndf * min(2 ** k, 8) for k in range(n_layers + 1)]
        idx = [0] + [2 + 3 * (k - 1) for k in range(1, n_layers + 2)]
        self.n_conv = n_layers + 2
        self.k_conv = [f"model.{i}" for i in idx]
        self.k_bn: List[Optional[str]] = [None] + [f"model.{i + 1}" for i in idx[1:-1]] + [None]

    def conv_shape(self, k: int):
        cin = self.input_nc if k == 0 else self.C[k - 1]
        cout = 1 if k == self.n_conv - 1 else self.C[k]
        return (cout, cin, 4, 4)

    def stride(self, k: int) -> int:
        return 2 if k < self.nl else 1

    def has_bias(self, k: int) -> bool:
        return k == 0 or k == self.n_conv - 1

    def key_order(self) -> List[str]:
        keys: List[str] = []
        for k in range(self.n_conv):
            keys.append(self.k_conv[k] + ".weight")
            if self.has_bias(k):
                keys.append(self.k_conv[k] + ".bias")
            elif self.norm == "batch":
                keys += [self.k_bn[k] + "." + l for l in BN_LEAVES]
        return keys

    def default_state_dict(self) -> Dict[str, torch.Tensor]:
        sd: Dict[str, torch.Tensor] = {}
        for k in range(self.n_conv):
            w = torch.empty(*self.conv_shape(k))
            _kaiming_uniform_(w)
            sd[self.k_conv[k] + ".weight"] = w
            if self.has_bias(k):
                b = torch.empty(w.size(0))
                _bias_uniform_(b, w)
                sd[self.k_conv[k] + ".bias"] = b
            elif self.norm == "batch":
                _bn_entries(sd, self.k_bn[k], self.C[k])
        return {k: sd[k] for k in self.key_order()}


def default_state_dicts(num_downs: int = 7, ngf: int = 64, ndf: int = 64, n_layers: int = 3, norm: str = "batch"):
    """G then D, the construction order of train_gan.py:138-139 (defines the seeded weights)."""
    g = GeneratorSpec(3, 3, num_downs, ngf, norm=norm).default_state_dict()
    d = DiscriminatorSpec(6, ndf, n_layers, norm=norm).default_state_dict()
    return g, d


class SiameseSpec:
    """SiameseUNet(n_channels, n_classes) (models.py:47-145): module construction order = RNG order =
    state_dict order: dconv_down1..4, bottleneck, att3, att2, att1, att_last, dconv_up3, dconv_up2,
    dconv_up1, dconv_last, conv_last (maxpool / upsample have no state)."""

    def __init__(self, n_channels: int = 3, n_classes: int = 1) -> None:
        self.n_channels, self.n_classes = n_channels, n_classes
        self.double_convs = [("dconv_down1", n_channels, 64), ("dconv_down2", 64, 128), ("dconv_down3", 128, 256),
                             ("dconv_down4", 256, 512), ("bottleneck", 512, 1024)]
        # (name, F_g, F_l, F_int)  models.py:76-79
        self.atts = [("att3", 2048, 1024, 512), ("att2", 512, 512, 256), ("att1", 256, 256, 128),
                     ("att_last", 128, 128, 64)]
        self.up_convs = [("dconv_up3", 2048 + 1024, 512), ("dconv_up2", 512 + 512, 256),
                         ("dconv_up1", 256 + 256, 128), ("dconv_last", 128 + 128, 64)]

    def default_state_dict(self) -> Dict[str, torch.Tensor]:
        sd: Dict[str, torch.Tensor] = {}

        def dconv(name: str, cin: int, cout: int) -> None:
            for idx, ci in ((0, cin), (3, cout)):
                w = torch.empty(cout, ci, 3, 3)
                _kaiming_uniform_(w)
                sd[f"{name}.{idx}.weight"] = w
                _bn_entries(sd, f"{name}.{idx + 1}", cout)

        def conv1x1(prefix: str, cin: int, cout: int) -> None:
            w = torch.empty(cout, cin, 1, 1)
            _kaiming_uniform_(w)
            b = torch.empty(cout)
            _bias_uniform_(b, w)
            sd[prefix + ".weight"] = w
            sd[prefix + ".bias"] = b

        for name, ci, co in self.double_convs:
            dconv(name, ci, co)
        for name, fg, fl, fi in self.atts:
            conv1x1(f"{name}.W_g.0", fg, fi)
            _bn_entries(sd, f"{name}.W_g.1", fi)
            conv1x1(f"{name}.W_x.0", fl, fi)
            _bn_entries(sd, f"{name}.W_x.1", fi)
            conv1x1(f"{name}.psi.0", fi, 1)
            _bn_entries(sd, f"{name}.psi.1", 1)
        for name, ci, co in self.up_convs:
            dconv(name, ci, co)
        conv1x1("conv_last", 64, self.n_classes)
        return sd
