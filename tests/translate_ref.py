"""fp64 torch reference of the generator's sliding-window scene inference (GeneratorEngine.translate_scene): cut a
scene into the tiles of scene.scene_axis (with the generator's alignment) with edge replication, blend per-tile images
with the window of scene.scene_window, and convert to uint8 by the out_u8 rule."""
import torch

from gan_aug_pfa_b200.scene import scene_axis, scene_window


def tile_origins(h, w, tile, overlap, align):
    """[(y0, x0)] in tile-index order (row-major) and the tile extent (ey, ex)."""
    oy, ey = scene_axis(h, tile, overlap, align)
    ox, ex = scene_axis(w, tile, overlap, align)
    return [(y, x) for y in oy for x in ox], (ey, ex)


def cut_tiles(scene_chw, tile, overlap, align):
    """[n_tiles, C, ey, ex] crops of a [C, H, W] scene; rows / columns past the scene repeat its last one."""
    _, h, w = scene_chw.shape
    origins, (ey, ex) = tile_origins(h, w, tile, overlap, align)
    out = []
    for y0, x0 in origins:
        iy = (y0 + torch.arange(ey, device=scene_chw.device)).clamp(max=h - 1)
        ix = (x0 + torch.arange(ex, device=scene_chw.device)).clamp(max=w - 1)
        out.append(scene_chw[:, iy][:, :, ix])
    return torch.stack(out)


def blend_image_ref(tile_vals, h, w, tile, overlap, align):
    """v [C, H, W] (fp64) = sum_tiles w * v_tile / sum_tiles w of tile_vals [n_tiles, C, ey, ex] (no activation)."""
    origins, (ey, ex) = tile_origins(h, w, tile, overlap, align)
    v = tile_vals.double().cpu()
    c = v.shape[1]
    win = scene_window(ey)[:, None] * scene_window(ex)[None, :]
    acc = torch.zeros(c, h, w, dtype=torch.float64)
    ws = torch.zeros(h, w, dtype=torch.float64)
    for t, (y0, x0) in enumerate(origins):
        hh, ww = min(ey, h - y0), min(ex, w - x0)
        acc[:, y0:y0 + hh, x0:x0 + ww] += win[:hh, :ww] * v[t, :, :hh, :ww]
        ws[y0:y0 + hh, x0:x0 + ww] += win[:hh, :ww]
    return acc / ws


def u8_ref(v):
    """uint8 [..] of fp64 values in [-1, 1]: floor(clamp((v * 0.5 + 0.5) * 255, 0, 255)), the out_u8 rule."""
    return ((v.double() * 0.5 + 0.5) * 255).clamp(0, 255).floor().to(torch.uint8)


def near_integer(v, eps=1e-3):
    """bool mask: (v * 0.5 + 0.5) * 255 lies within eps of an integer, where fp32 rounding may pick either side."""
    s = (v.double() * 0.5 + 0.5) * 255
    return (s - s.round()).abs() < eps
