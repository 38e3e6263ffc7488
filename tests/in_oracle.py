"""The CPU oracle with InstanceNorm2d layers (pix2pix's `--norm instance`).  TEST INFRASTRUCTURE ONLY.

oracle/pix2pix_oracle.py normalises through its module-level `batchnorm2d`; inside `instance_norm()` that function is
nn.InstanceNorm2d(affine=False, track_running_stats=False), i.e. F.instance_norm(x, eps=1e-5), so the oracle's
generator / discriminator forwards and `gan_train_step` compute the InstanceNorm networks (conv biases come from the
state_dict through `sd.get`).  tests/test_instance_norm_cpu.py checks this path against torch's own nn.InstanceNorm2d
modules."""
import contextlib

import torch.nn.functional as F

from oracle import pix2pix_oracle as O

IN_EPS = 1e-5


def _instance_norm(x, sd, prefix, train, new_buffers):
    return F.instance_norm(x, eps=IN_EPS)


@contextlib.contextmanager
def instance_norm():
    saved = O.batchnorm2d
    O.batchnorm2d = _instance_norm
    try:
        yield O
    finally:
        O.batchnorm2d = saved
