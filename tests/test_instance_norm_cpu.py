"""InstanceNorm2d support without a GPU: parameter layout and seeded weights of the modules, the construction-time
rejections, the oracle's InstanceNorm path against torch's own nn.InstanceNorm2d layers, and the argument checks of the
gap_in_* entry points."""
import ctypes
import functools
import hashlib

import pytest
import torch
import torch.nn as nn

from gan_aug_pfa_b200 import models as M
from gan_aug_pfa_b200 import spec
from in_oracle import instance_norm

IN_PARTIAL = functools.partial(nn.InstanceNorm2d, affine=False, track_running_stats=False)
IN_FORMS = [nn.InstanceNorm2d, IN_PARTIAL]


def _digest(sd):
    return [(k, tuple(v.shape), hashlib.sha256(v.detach().contiguous().numpy().tobytes()).hexdigest())
            for k, v in sd.items()]


@pytest.mark.parametrize("num_downs", [7, 8])
@pytest.mark.parametrize("norm_layer", IN_FORMS, ids=["class", "partial"])
def test_seeded_modules_match_the_spec(num_downs, norm_layer):
    torch.manual_seed(0)
    g = M.UNetGenerator(3, 3, num_downs, norm_layer=norm_layer)
    d = M.NLayerDiscriminator(6, norm_layer=norm_layer)
    torch.manual_seed(0)
    sg, sdd = spec.default_state_dicts(num_downs, norm="instance")
    assert _digest(g.state_dict()) == _digest(sg)
    assert _digest(d.state_dict()) == _digest(sdd)


def test_instance_norm_state_dicts_have_no_norm_entries_and_generator_biases():
    g = M.UNetGenerator(3, 3, 7, norm_layer=nn.InstanceNorm2d).state_dict()
    d = M.NLayerDiscriminator(6, norm_layer=nn.InstanceNorm2d).state_dict()
    for sd in (g, d):
        assert not [k for k in sd if "running" in k or "num_batches" in k]
        assert all(v.dim() in (1, 4) for v in sd.values())      # conv weights and biases only
    gs = spec.GeneratorSpec(3, 3, 7, norm="instance")
    for j in range(gs.L):
        assert gs.k_down[j] + ".bias" in g and gs.k_up[j] + ".bias" in g
    assert g["model.model.0.bias"].shape == (64,)
    # the discriminator's middle convs stay bias-free (use_bias = False in NLayerDiscriminator)
    assert [k for k in d if k.endswith(".bias")] == ["model.0.bias", "model.11.bias"]
    assert list(d) == spec.DiscriminatorSpec(norm="instance").key_order()


def test_block_chain_spec_carries_the_norm():
    torch.manual_seed(3)
    inner = M.UnetSkipConnectionBlock(512, 512, innermost=True, norm_layer=nn.InstanceNorm2d)
    blk = M.UnetSkipConnectionBlock(256, 512, submodule=inner, norm_layer=nn.InstanceNorm2d)
    sp = spec.GeneratorSpec.for_block_chain(blk._chain(), norm="instance")
    torch.manual_seed(3)
    assert _digest(blk.state_dict()) == _digest(sp.default_state_dict())


def _ref_block(blk, x):
    """UnetSkipConnectionBlock.forward of the reference (models.py:204-208) on the skeleton's real torch layers."""
    h = x
    for layer in blk.model:
        h = _ref_block(layer, h) if isinstance(layer, M.UnetSkipConnectionBlock) else layer(h)
    return h if blk.outermost else torch.cat([x, h], 1)


def _check_grads(params, ref_sd, out_mod, out_ref):
    w = torch.randn(out_ref.shape, generator=torch.Generator().manual_seed(5))
    gm = torch.autograd.grad((out_mod * w).sum(), [p for _, p in params])
    gr = torch.autograd.grad((out_ref * w).sum(), [ref_sd[k] for k, _ in params])
    for (k, _), a, b in zip(params, gm, gr):
        assert float((a - b).norm() / b.norm().clamp_min(1e-30)) < 1e-5 or float((a - b).abs().max()) < 1e-7, k


def test_oracle_instance_norm_path_matches_torch_modules():
    torch.manual_seed(0)
    g = M.UNetGenerator(3, 3, 6, norm_layer=nn.InstanceNorm2d)
    d = M.NLayerDiscriminator(6, norm_layer=nn.InstanceNorm2d)
    gen = torch.Generator().manual_seed(1)
    A = torch.rand(2, 3, 64, 64, generator=gen) * 2 - 1
    B = torch.rand(2, 3, 64, 64, generator=gen) * 2 - 1
    sd_g = {k: v.detach().clone().requires_grad_(True) for k, v in g.state_dict().items()}
    sd_d = {k: v.detach().clone().requires_grad_(True) for k, v in d.state_dict().items()}
    with instance_norm() as O:
        for train in (True, False):
            g.train(train)
            d.train(train)
            out_m = _ref_block(g.model, A.clone())
            out_o = O.unet_generator_forward(sd_g, A.clone(), train, None)
            assert float((out_m - out_o).detach().norm() / out_o.detach().norm()) < 1e-5
            x = torch.cat([A, out_m.detach()], 1)
            lm, lo = d.model(x.clone()), O.discriminator_forward(sd_d, x.clone(), train, None)
            assert float((lm - lo).detach().norm() / lo.detach().norm()) < 1e-5
        _check_grads(list(g.named_parameters()), sd_g, out_m, out_o)
        _check_grads(list(d.named_parameters()), sd_d, lm, lo)


@pytest.mark.parametrize("bad", [
    functools.partial(nn.InstanceNorm2d, affine=True),
    functools.partial(nn.InstanceNorm2d, track_running_stats=True),
    functools.partial(nn.InstanceNorm2d, eps=1e-3),
    functools.partial(nn.BatchNorm2d, affine=False),
    nn.GroupNorm,
    nn.LayerNorm,
], ids=["in_affine", "in_running", "in_eps", "bn_no_affine", "groupnorm", "layernorm"])
def test_unsupported_norm_layers_are_rejected_at_construction(bad):
    with pytest.raises(NotImplementedError, match="InstanceNorm2d"):
        M.UNetGenerator(3, 3, 7, norm_layer=bad)
    with pytest.raises(NotImplementedError, match="InstanceNorm2d"):
        M.NLayerDiscriminator(6, norm_layer=bad)
    with pytest.raises(NotImplementedError, match="InstanceNorm2d"):
        M.UnetSkipConnectionBlock(512, 512, innermost=True, norm_layer=bad)


@pytest.mark.parametrize("norm_layer", IN_FORMS, ids=["class", "partial"])
def test_instance_norm_with_dropout_is_rejected(norm_layer):
    with pytest.raises(NotImplementedError, match="use_dropout"):
        M.UNetGenerator(3, 3, 8, norm_layer=norm_layer, use_dropout=True)
    with pytest.raises(NotImplementedError, match="use_dropout"):
        M.UnetSkipConnectionBlock(512, 512, norm_layer=norm_layer, use_dropout=True,
                                  submodule=M.UnetSkipConnectionBlock(512, 512, innermost=True, norm_layer=norm_layer))


def test_batchnorm_partial_with_defaults_is_the_default_path():
    bn = functools.partial(nn.BatchNorm2d, affine=True, track_running_stats=True)
    torch.manual_seed(0)
    a = M.UNetGenerator(3, 3, 7, norm_layer=bn).state_dict()
    da = M.NLayerDiscriminator(6, norm_layer=bn).state_dict()
    torch.manual_seed(0)
    b = M.UNetGenerator(3, 3, 7).state_dict()
    db = M.NLayerDiscriminator(6).state_dict()
    assert _digest(a) == _digest(b) and _digest(da) == _digest(db)
    assert M.norm_kind(bn) == "batch" and M.norm_kind(nn.InstanceNorm2d) == "instance"


def test_unknown_norm_names_are_refused_by_the_specs():
    with pytest.raises(ValueError):
        spec.GeneratorSpec(norm="group")
    with pytest.raises(ValueError):
        spec.DiscriminatorSpec(norm="layer")


def test_in_entry_points_check_arguments_without_a_gpu(lib_path):
    from gan_aug_pfa_b200 import _lib
    h = _lib.lib()
    fake = ctypes.c_void_p(1 << 20)          # never dereferenced: validation fails first
    assert h.gap_in_stats(None, 64, 2, 16, 64, fake, None) == -1
    assert b"null" in h.gap_last_error_string()
    assert h.gap_in_stats(fake, 64, 2, 16, 60, fake, None) == -1          # C % 8 != 0
    assert b"C % 8" in h.gap_last_error_string()
    assert h.gap_in_stats(fake, 64, 2, 1, 64, fake, None) == -1           # H*W == 1
    assert h.gap_in_act(fake, 64, 2, 16, 64, None, fake, fake, 64, 1, None, 0, 0, None) == -1
    assert h.gap_in_act(fake, 64, 2, 16, 12, fake, fake, fake, 64, 1, None, 0, 0, None) == -1
    assert h.gap_in_act(fake, 64, 2, 16, 64, fake, fake, fake, 64, 3, None, 0, 0, None) == -1   # Tanh: not a norm act
    assert h.gap_in_bwd_reduce(fake, 64, None, 64, None, 0, 0.2, fake, fake, 2, 16, 64, fake, None) == -1
    assert h.gap_in_bwd_reduce(fake, 64, fake, 64, None, 0, 0.2, fake, fake, 2, 16, 20, fake, None) == -1
    assert h.gap_in_bwd_apply(fake, 64, fake, 64, None, 0, 0.2, fake, fake, 2, 16, 64, fake, None, 64, None, None) == -1
    assert h.gap_in_bwd_apply(fake, 64, fake, 64, None, 0, 0.2, fake, fake, 2, 16, 36, fake, fake, 64, None, None) == -1
    assert b"gap_in_bwd_apply" in h.gap_last_error_string()
