"""fp64 torch reference of test-time augmentation and checkpoint ensembles over whole scenes
(siamese.predict_scene_ensemble): the dihedral tile transforms f_d and their inverses, and the blend of several passes
of per-tile logits in the documented pass order."""
import torch

from scene_ref import tile_origins
from gan_aug_pfa_b200.siamese import TTA_TRANSFORMS, scene_window


def f(x, d):
    """f_d(x) over the last two axes, d = 4 s + 2 v + u: transposed if s, then rows flipped if v, then columns if u."""
    if d & 4:
        x = x.transpose(-2, -1)
    if d & 2:
        x = x.flip(-2)
    if d & 1:
        x = x.flip(-1)
    return x


def f_inv(x, d):
    """f_d^-1: undo the flips, then transpose if s."""
    if d & 1:
        x = x.flip(-1)
    if d & 2:
        x = x.flip(-2)
    if d & 4:
        x = x.transpose(-2, -1)
    return x


def passes(n_members, tta):
    """[(member, d)] in the order the passes run."""
    return [(m, d) for m in range(n_members) for d in TTA_TRANSFORMS[tta]]


def blend_passes_ref(per_pass_tile_logits, h, w, tile, overlap):
    """p [K, H, W] (fp64) = sum_passes sum_tiles w * p_tile / sum_passes sum_tiles w, summed pass by pass in the given
    order and, within a pass, in ascending tile index.  per_pass_tile_logits: [(d, z)] with z [n_tiles, K, oy, ox] the
    logits of the transformed tiles f_d(tile); each is mapped back by f_d^-1.  K = 1 -> sigmoid, else softmax."""
    origins, (ey, ex) = tile_origins(h, w, tile, overlap)
    win = scene_window(ey)[:, None] * scene_window(ex)[None, :]
    k = per_pass_tile_logits[0][1].shape[1]
    acc = torch.zeros(k, h, w, dtype=torch.float64)
    ws = torch.zeros(h, w, dtype=torch.float64)
    for d, z in per_pass_tile_logits:
        z = f_inv(z.double().cpu(), d)
        assert tuple(z.shape[-2:]) == (ey, ex)
        p = torch.sigmoid(z) if k == 1 else torch.softmax(z, dim=1)
        for t, (y0, x0) in enumerate(origins):
            hh, ww = min(ey, h - y0), min(ex, w - x0)
            acc[:, y0:y0 + hh, x0:x0 + ww] += win[:hh, :ww] * p[t, :, :hh, :ww]
            ws[y0:y0 + hh, x0:x0 + ww] += win[:hh, :ww]
    return acc / ws
