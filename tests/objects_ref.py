"""scipy reference of objects.change_objects: per-class scipy.ndimage.label, objects renumbered by their first pixel in
raster order over (n, y, x), minimum-area filtering, the object table, the pixel confusion of the filtered map and the
object counts.  Tests import it; the product never does."""
import numpy as np
from scipy import ndimage


def components(cls, kk, connectivity):
    """int64 [N, H, W]: 0 for pixels whose class is outside 1..kk-1, else the id of their `connectivity`-connected
    component of one class inside one sample, numbered 1..m by first pixel in raster order."""
    struct = ndimage.generate_binary_structure(2, 1 if connectivity == 4 else 2)
    comp = np.zeros(cls.shape, np.int64)
    nxt = 0
    for s in range(cls.shape[0]):
        for c in range(1, kk):
            lab, m = ndimage.label(cls[s] == c, structure=struct)
            comp[s][lab > 0] = lab[lab > 0] + nxt
            nxt += m
    flat = comp.ravel()
    nz = np.flatnonzero(flat)
    keys, first = np.unique(flat[nz], return_index=True)
    order = np.argsort(nz[first], kind="stable")
    remap = np.zeros(nxt + 1, np.int64)
    remap[keys[order]] = np.arange(1, len(keys) + 1)
    return remap[comp]


def needed(area, min_overlap):
    """max(1, ceil(min_overlap * area)) in fp64, elementwise over an int array of areas."""
    return np.maximum(1, np.ceil(min_overlap * np.asarray(area, np.float64))).astype(np.int64)


def change_objects_ref(pred, n_classes, labels=None, min_area=0, connectivity=8, min_overlap=0.0, ignore_index=-100):
    """dict(pred, ids, objects, confusion, object_counts) as numpy arrays, in change_objects' formats."""
    pred = np.asarray(pred)
    shape = pred.shape
    p3 = pred.reshape((1,) + shape if pred.ndim == 2 else shape).astype(np.int64)
    k, kk = n_classes, max(n_classes, 2)
    comp = components(p3, kk, connectivity)
    area = np.bincount(comp.ravel(), minlength=int(comp.max()) + 1)
    keep = area >= min_area
    keep[0] = False
    newid = np.cumsum(keep) * keep
    ids = newid[comp]
    fpred = np.where(ids > 0, p3, 0)
    n_obj = int(keep.sum())
    objects = np.zeros((n_obj, 7), np.int64)
    if n_obj:
        flat = ids.ravel()
        nz = np.flatnonzero(flat)
        keys, first = np.unique(flat[nz], return_index=True)
        objects[keys - 1, 1] = p3.ravel()[nz[first]]
        objects[:, 2] = np.bincount(flat, minlength=n_obj + 1)[1:]
        sl = np.array([[d.start, d.stop - 1] for o in ndimage.find_objects(ids) for d in o]).reshape(n_obj, 3, 2)
        objects[:, 0] = sl[:, 0, 0]
        objects[:, 3], objects[:, 5] = sl[:, 1, 0], sl[:, 1, 1]
        objects[:, 4], objects[:, 6] = sl[:, 2, 0], sl[:, 2, 1]
    out = {"pred": fpred.reshape(shape).astype(np.uint8), "ids": ids.reshape(shape).astype(np.int32),
           "objects": objects, "confusion": None, "object_counts": None}
    if labels is None:
        return out
    y = np.asarray(labels).reshape(p3.shape)
    valid = (y != ignore_index) & (y >= 0) & (y < kk)
    if k == 1:
        t, q = y[valid], fpred[valid]
        conf = np.array([np.sum((t == 1) & (q == 1)), np.sum((t == 0) & (q == 1)), np.sum((t == 1) & (q == 0)),
                         np.sum((t == 0) & (q == 0))], np.int64)
    else:
        conf = np.bincount(y[valid] * k + fpred[valid], minlength=k * k).reshape(k, k).astype(np.int64)
    lcls = np.where(valid, y, 0)
    rcomp = components(lcls, kk, connectivity)
    hit = (fpred == lcls) & (fpred != 0)
    counts = np.zeros((kk, 4), np.int64)
    m = int(rcomp.max())
    r_area = np.bincount(rcomp.ravel(), minlength=m + 1)
    r_ov = np.bincount(rcomp[hit], minlength=m + 1)
    r_cls = np.zeros(m + 1, np.int64)
    r_cls[rcomp.ravel()] = lcls.ravel()
    detected = r_ov >= needed(r_area, min_overlap)
    counts[:, 0] = np.bincount(r_cls[1:], minlength=kk)
    counts[:, 1] = np.bincount(r_cls[1:], weights=detected[1:], minlength=kk).astype(np.int64)
    p_ov = np.bincount(ids[hit], minlength=n_obj + 1)[1:]
    matched = p_ov >= needed(objects[:, 2], min_overlap)
    counts[:, 2] = np.bincount(objects[:, 1], minlength=kk)
    counts[:, 3] = np.bincount(objects[:, 1], weights=matched, minlength=kk).astype(np.int64)
    out["confusion"] = conf
    out["object_counts"] = counts
    return out
