"""Float64 reference of the surface-distance metrics (include/liftreg_b200.h, lr_surface_distances; metrics.surface_distance):
surfaces with scipy's binary_erosion, directed distances with distance_transform_edt, percentiles with np.percentile."""
import numpy as np
from scipy import ndimage as ndi

_FACES = ndi.generate_binary_structure(3, 1)


def surface(mask):
    """voxels of a boolean (D,H,W) mask with a face neighbour outside the volume or outside the mask"""
    mask = np.asarray(mask, bool)
    return mask & ~ndi.binary_erosion(mask, _FACES, border_value=0)


def directed(s_from, s_to, spacing):
    """distances (unsorted, in C order of s_from) from every voxel of s_from to the nearest voxel of s_to"""
    return ndi.distance_transform_edt(~s_to, sampling=spacing)[s_from]


def surface_distance(pred, target, spacing=(1.0, 1.0, 1.0), num_labels=None):
    """the dict metrics.surface_distance returns, for (B,D,H,W) integer-valued numpy maps, plus "directed":
    {(b, l, k): sorted distances} with k = 0 for pred -> target and 1 for target -> pred"""
    pred, target = np.asarray(pred), np.asarray(target)
    B = pred.shape[0]
    L = int(max(pred.max(), target.max())) + 1 if num_labels is None else int(num_labels)
    res = {k: np.full((B, L), np.nan) for k in ("hd", "hd95", "assd")}
    res["surface_count"] = np.zeros((B, 2, L), np.int64)
    res["directed"] = {}
    for b in range(B):
        for l in range(L):
            sp_, st_ = surface(pred[b] == l), surface(target[b] == l)
            res["surface_count"][b, :, l] = sp_.sum(), st_.sum()
            if l == 0 or not sp_.any() or not st_.any():
                continue
            d = [np.sort(directed(sp_, st_, spacing)), np.sort(directed(st_, sp_, spacing))]
            res["directed"][(b, l, 0)], res["directed"][(b, l, 1)] = d
            res["hd"][b, l] = max(d[0].max(), d[1].max())
            res["hd95"][b, l] = max(np.percentile(d[0], 95), np.percentile(d[1], 95))
            res["assd"][b, l] = (d[0].mean() + d[1].mean()) / 2
    for k in ("hd", "hd95", "assd"):
        v = res[k]
        ok = ~np.isnan(v)
        res[k + "_mean"] = np.array([v[b][ok[b]].mean() if ok[b].any() else np.nan for b in range(B)])
    return res


def brute_force(s_from, s_to, spacing):
    """all-pairs minimum of the same formula, in the same order: sqrt(((s_D d_D)^2 + (s_H d_H)^2) + (s_W d_W)^2)"""
    f = np.argwhere(s_from).astype(np.float64)
    t = np.argwhere(s_to).astype(np.float64)
    sp = np.asarray(spacing, np.float64)
    diff = (f[:, None, :] - t[None, :, :]) * sp
    sq = diff * diff
    return np.sqrt((sq[..., 0] + sq[..., 1]) + sq[..., 2]).min(axis=1)
