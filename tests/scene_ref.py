"""fp64 torch reference of sliding-window scene inference (SiameseEngine.predict_scene): cut a scene into the tiles of
siamese.scene_axis with edge replication, and blend per-tile logits with the window of siamese.scene_window."""
import torch

from gan_aug_pfa_b200.siamese import scene_axis, scene_window


def tile_origins(h, w, tile, overlap):
    """[(y0, x0)] in tile-index order (row-major) and the tile extent (ey, ex)."""
    oy, ey = scene_axis(h, tile, overlap)
    ox, ex = scene_axis(w, tile, overlap)
    return [(y, x) for y in oy for x in ox], (ey, ex)


def cut_tiles(scene_chw, tile, overlap):
    """[n_tiles, C, ey, ex] crops of a [C, H, W] scene; rows / columns past the scene repeat its last one."""
    _, h, w = scene_chw.shape
    origins, (ey, ex) = tile_origins(h, w, tile, overlap)
    out = []
    for y0, x0 in origins:
        iy = (y0 + torch.arange(ey)).clamp(max=h - 1)
        ix = (x0 + torch.arange(ex)).clamp(max=w - 1)
        out.append(scene_chw[:, iy][:, :, ix])
    return torch.stack(out)


def blend_ref(tile_logits, h, w, tile, overlap):
    """p [K, H, W] (fp64) = sum_tiles w * p_tile / sum_tiles w; tile_logits [n_tiles, K, ey, ex], K = 1 -> sigmoid,
    K > 1 -> softmax over dim 1."""
    origins, (ey, ex) = tile_origins(h, w, tile, overlap)
    z = tile_logits.double().cpu()
    k = z.shape[1]
    p = torch.sigmoid(z) if k == 1 else torch.softmax(z, dim=1)
    win = scene_window(ey)[:, None] * scene_window(ex)[None, :]
    acc = torch.zeros(k, h, w, dtype=torch.float64)
    ws = torch.zeros(h, w, dtype=torch.float64)
    for t, (y0, x0) in enumerate(origins):
        hh, ww = min(ey, h - y0), min(ex, w - x0)
        acc[:, y0:y0 + hh, x0:x0 + ww] += win[:hh, :ww] * p[t, :, :hh, :ww]
        ws[y0:y0 + hh, x0:x0 + ww] += win[:hh, :ww]
    return acc / ws


def near_tie(p, eps):
    """[H, W] bool: pixels whose two largest values along dim 0 differ by less than eps (K = 1: |p - 0.5| < eps)."""
    if p.shape[0] == 1:
        return (p[0] - 0.5).abs() < eps
    top = p.topk(2, dim=0).values
    return (top[0] - top[1]) < eps


def pred_ref(p):
    """The class map of blended probabilities: argmax (ties to the lowest class) or, K = 1, p > 0.5."""
    return (p[0] > 0.5).to(torch.uint8) if p.shape[0] == 1 else p.argmax(0).to(torch.uint8)
