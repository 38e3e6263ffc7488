"""1-4-channel images without a GPU: parameter layout and seeded weights of the modules for other channel counts, the
construction-time rejections, the drop-in discriminator's split rule, and the argument checks of the channel-count
entry points."""
import ctypes
import hashlib

import pytest
import torch

from gan_aug_pfa_b200 import models as M
from gan_aug_pfa_b200 import checkpoint, pix2pix, siamese, spec


def _digest(sd):
    return [(k, tuple(v.shape), hashlib.sha256(v.detach().contiguous().numpy().tobytes()).hexdigest())
            for k, v in sd.items()]


@pytest.mark.parametrize("ic,oc", [(1, 3), (4, 4), (2, 1)])
def test_seeded_generator_matches_the_spec(ic, oc):
    torch.manual_seed(0)
    g = M.UNetGenerator(ic, oc, 7)
    torch.manual_seed(0)
    sd = spec.GeneratorSpec(ic, oc, 7).default_state_dict()
    assert _digest(g.state_dict()) == _digest(sd)
    assert sd["model.model.0.weight"].shape == (64, ic, 4, 4)
    assert sd["model.model.3.weight"].shape == (128, oc, 4, 4)
    assert sd["model.model.3.bias"].shape == (oc,)


@pytest.mark.parametrize("input_nc", [4, 8])
def test_seeded_discriminator_matches_the_spec(input_nc):
    torch.manual_seed(0)
    d = M.NLayerDiscriminator(input_nc)
    torch.manual_seed(0)
    sd = spec.DiscriminatorSpec(input_nc).default_state_dict()
    assert _digest(d.state_dict()) == _digest(sd)
    assert sd["model.0.weight"].shape == (64, input_nc, 4, 4)


@pytest.mark.parametrize("n_channels", [1, 4])
def test_seeded_siamese_matches_the_spec(n_channels):
    torch.manual_seed(0)
    s = M.SiameseUNet(n_channels, 1)
    torch.manual_seed(0)
    sd = spec.SiameseSpec(n_channels, 1).default_state_dict()
    assert _digest({k: v for k, v in s.state_dict().items()}) == _digest({k: sd[k] for k in s.state_dict()})
    assert sd["dconv_down1.0.weight"].shape == (64, n_channels, 3, 3)


@pytest.mark.parametrize("ic,oc", [(0, 3), (5, 3), (3, 0), (3, 5), (13, 3)])
def test_generator_channel_counts_outside_1_to_4_are_rejected(ic, oc):
    with pytest.raises(NotImplementedError, match="1 to 4 channels"):
        M.UNetGenerator(ic, oc, 7)
    with pytest.raises(NotImplementedError, match="1 to 4 channels"):
        pix2pix.GeneratorEngine(torch.device("cpu"), ic, oc, init=False)


@pytest.mark.parametrize("input_nc", [0, 1, 9, 13])
def test_discriminator_channel_counts_outside_2_to_8_are_rejected(input_nc):
    with pytest.raises(NotImplementedError, match="2 to 8 channels"):
        M.NLayerDiscriminator(input_nc)
    with pytest.raises(NotImplementedError, match="2 to 8 channels"):
        pix2pix.DiscriminatorEngine(torch.device("cpu"), input_nc, init=False)


@pytest.mark.parametrize("n_channels", [0, 5])
def test_siamese_channel_counts_outside_1_to_4_are_rejected(n_channels):
    with pytest.raises(NotImplementedError, match="1 to 4 channels"):
        siamese.SiameseEngine(torch.device("cpu"), n_channels, 1)


def test_checkpoints_with_other_channel_counts_are_refused_naming_them():
    from types import SimpleNamespace
    tr = SimpleNamespace(norm="batch", input_nc=3, output_nc=3)
    state = {"format": checkpoint.FORMAT, "kind": "pix2pix", "norm": "batch", "channels": {"input_nc": 1, "output_nc": 2}}
    with pytest.raises(ValueError, match="input_nc=1, output_nc=2.*input_nc=3, output_nc=3"):
        checkpoint.load_trainer_state(tr, state)
    # a checkpoint written before the channel counts were recorded is a 3 -> 3 run
    old = {"format": checkpoint.FORMAT, "kind": "pix2pix", "norm": "batch"}
    with pytest.raises(ValueError, match="input_nc=3, output_nc=3.*input_nc=1, output_nc=3"):
        checkpoint.load_trainer_state(SimpleNamespace(norm="batch", input_nc=1, output_nc=3), old)
    eng = SimpleNamespace(n_channels=4)
    with pytest.raises(ValueError, match="n_channels=3.*n_channels=4"):
        checkpoint.load_siamese_state(eng, {"format": checkpoint.FORMAT, "kind": "siamese"})


def test_trainer_rejects_channel_counts_before_touching_the_device():
    with pytest.raises(NotImplementedError, match="input_nc"):
        pix2pix.Pix2PixTrainer("cpu", input_nc=5)
    with pytest.raises(NotImplementedError, match="output_nc"):
        pix2pix.Pix2PixTrainer("cpu", output_nc=0)


@pytest.mark.parametrize("input_nc,split", [(2, (1, 1)), (3, (2, 1)), (4, (2, 2)), (5, (3, 2)), (6, (3, 3)),
                                            (7, (4, 3)), (8, (4, 4))])
def test_discriminator_split_rule(input_nc, split):
    # source A = the first ceil(input_nc / 2) channels of cat(A, B), source B = the rest; 6 -> 3 | 3 as before
    assert pix2pix.discriminator_split(input_nc) == split


def test_outermost_block_with_other_image_channels_builds_its_spec():
    torch.manual_seed(2)
    inner = M.UnetSkipConnectionBlock(128, 128, innermost=True)
    blk = M.UnetSkipConnectionBlock(2, 128, input_nc=1, outermost=True, submodule=inner)
    sp = spec.GeneratorSpec.for_block_chain(blk._chain())
    assert (sp.input_nc, sp.output_nc) == (1, 2)
    torch.manual_seed(2)
    assert _digest(blk.state_dict()) == _digest(sp.default_state_dict())


def test_channel_entry_points_check_arguments_without_a_gpu(lib_path):
    from gan_aug_pfa_b200 import _lib
    h = _lib.lib()
    fake = ctypes.c_void_p(1 << 20)          # never dereferenced: validation fails first
    for co in (0, 5):
        assert h.gap_thin_convT_fwd_c(fake, 128, 2, 8, 8, 128, co, fake, None, 0, None, 0, fake, 4, None, None) == -1
        assert b"co must be 1..4" in h.gap_last_error_string()
    assert h.gap_thin_convT_fwd_c(None, 128, 2, 8, 8, 128, 2, fake, None, 0, None, 0, fake, 4, None, None) == -1
    for c0, s1, c1 in ((0, None, 0), (5, None, 0), (3, None, 1), (3, fake, 0), (3, fake, 5)):
        assert h.gap_thin_conv_wgrad_c(fake, 64, fake, 4, c0, s1, 4, c1, 2, 16, 16, 64, fake, 64, None, None) == -1
        assert b"gap_thin_conv_wgrad_c" in h.gap_last_error_string()
    assert h.gap_thin_conv_wgrad_c(None, 64, fake, 4, 1, None, 0, 0, 2, 16, 16, 64, fake, 64, None, None) == -1
    for c in (0, 5):
        assert h.gap_u8_hwc_to_nhwc_bf16_c(fake, c, fake, 4, 16, None) == -1
        assert b"c must be 1..4" in h.gap_last_error_string()
        assert h.gap_resize_u8_to_nhwc_bf16_c(fake, c, 1, 8, 8, 4, 4, fake, 4, None, None) == -1
        assert b"c must be 1..4" in h.gap_last_error_string()
    assert h.gap_u8_hwc_to_nhwc_bf16_c(None, 2, fake, 4, 16, None) == -1
    for c in (0, 5):
        assert h.gap_im2col_k3s1p1_c(fake, 4, c, fake, 1, 8, 8, None) == -1
        assert b"c must be 1..4" in h.gap_last_error_string()
    assert h.gap_im2col_k3s1p1_c(None, 4, 2, fake, 1, 8, 8, None) == -1
    assert h.gap_resize_u8_to_nhwc_bf16_c(fake, 2, 1, 8, 8, 4, 4, None, 4, None, None) == -1


def test_ops_wrappers_check_channel_arguments_before_any_cuda_call():
    from gan_aug_pfa_b200 import ops
    x = torch.zeros(1, 4, 4, 64, dtype=torch.bfloat16)
    with pytest.raises(ValueError, match="co must be 1..4"):
        ops.thin_convT_fwd(x, torch.zeros(80, 64, dtype=torch.bfloat16), None, 0, None, None, co=5)
    with pytest.raises(ValueError, match="1..4"):
        ops.u8_hwc_to_nhwc_bf16(torch.zeros(1, 4, 4, 5, dtype=torch.uint8), x)
