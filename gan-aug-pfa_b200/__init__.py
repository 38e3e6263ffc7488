"""B200-native conv hot path for GAN-AUG-PFA: hand-written sm_100a kernels behind a C ABI
(``lib/libgap_b200.so``, declared in ``include/gap_b200.h``) plus the thin Python host side that
mirrors the reference's ``models.py`` surface.  Import as ``gan_aug_pfa_b200``."""
__version__ = "0.1.0"


def __getattr__(name):
    # the multi-class Dice criteria, imported on first use (they pull in torch)
    if name in ("CEDiceLoss", "SoftmaxFocalDiceLoss"):
        from . import losses
        return getattr(losses, name)
    raise AttributeError(f"module {__name__!r} has no attribute {name!r}")
