"""Validation metrics on the GPU: Jacobian folding statistics of a map, per-label overlap of two label maps and their
per-label surface distances (Hausdorff, HD95, average symmetric surface distance).

The reference scores each validation item on the host (networks/RegistrationNet.py:198-218 _compute_metrics): the
Jacobian determinant of phi with numpy and mermaid's finite differences (utils/utils.py:20-55, after copying the
3*D*H*W map to the host) and per-label Dice / IoU / recall / precision with Python sets (utils/metrics.py:6-121,
get_multi_metric / cal_metric).  Here jacobian_stats and label_overlap are one kernel call each (ops.jacobian_det,
ops.label_confusion) plus a readout of a few numbers per item; surface_distance is a count pass plus two distance calls
per label present in both maps.

Definitions
    Jacobian: J[c][a] = central difference of phi_c along volume axis a (the regulariser's face rules, "linear" or
        "neumann_zero") times 0.5/(2/(n_a-1)), so the identity map in [-1,1] has det 1; det is the 3x3 determinant
        expanded along the first row in fp32.  Statistics cover the voxels at least `margin` from every face:
        folding_count (#det < 0), folding_fraction (folding_count / #voxels), folding_abs_sum (sum of |det| over
        det < 0), det_min, det_max, det_mean, det_std (population) over the finite determinants, and nonfinite_count.
    Overlap: with TP = #voxels labelled l in both maps, P = #voxels labelled l in pred, T = in target,
        dice = 2 TP / (P + T), iou = TP / (P + T - TP), recall = TP / T, precision = TP / P  (float64).
        A value whose denominator is zero is NaN (dice and iou: the label is absent from both maps) and is left out of
        the means; the means are over the labels present in either map.  ignore_background drops label 0.

    Surface distance: S_M(l) is the set of voxels labelled l in map M with a face neighbour outside the volume or
        labelled otherwise (scipy's m & ~binary_erosion(m, 6-connectivity, border_value=0)).  d_PT(v), v in S_pred(l), is
        the distance in mm to the nearest voxel of S_target(l) (d_TP the same the other way), formed from the index
        offsets as scipy's distance_transform_edt forms it.  hd = max(max d_PT, max d_TP); hd95 = max(q95(d_PT),
        q95(d_TP)) with numpy's default ("linear") percentile, as MONAI's HausdorffDistanceMetric; assd = (mean d_PT +
        mean d_TP) / 2, as MONAI's symmetric SurfaceDistanceMetric and medpy's assd.  All three are NaN when either
        surface is empty; the means are over the labels present in both maps.  These are voxel-based distances, not the
        surfel-area-weighted ones of DeepMind's surface_distance package.  The reference scores no surface metric.

Parity with the reference is UNPINNED: its utils.py and metrics.py are not part of the reference tree and import
packages that are not installable, so which determinant, whether the boundary is cropped, how background is treated and
how an absent label scores there are unknown.  These are new functions, not signature-compatible replacements for
get_multi_metric or the folding helper, and dropin.install() does not rebind anything to them.
"""
import numpy as np
import torch

from . import ops


def jacobian_stats(phi, boundary="linear", margin=0, return_map=False, allow_nonfinite=False):
    """Folding statistics of maps phi (B,3,D,H,W) in [-1,1]: a dict of per-item numpy arrays (see the module docstring),
    plus "det" (the (B,D,H,W) CUDA tensor) when return_map.  Raises ValueError if a determinant is not finite unless
    allow_nonfinite (then the statistics cover the finite ones and nonfinite_count says how many were left out)."""
    stats, det = ops.jacobian_det(phi, boundary=boundary, margin=margin, want_map=return_map)
    s = stats.cpu().numpy()
    D, H, W = (int(n) for n in phi.shape[2:])
    m = int(margin)
    n_vox = (D - 2 * m) * (H - 2 * m) * (W - 2 * m)
    nonfinite = s[:, 6].astype(np.int64)
    if not allow_nonfinite and nonfinite.any():
        raise ValueError("Jacobian determinant is not finite at %s voxel(s) per item (is phi finite?)" % nonfinite.tolist())
    n_fin = (n_vox - nonfinite).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        mean = s[:, 4] / n_fin
        var = np.maximum(s[:, 5] / n_fin - mean * mean, 0.0)
    out = {
        "folding_count": s[:, 0].astype(np.int64),
        "folding_fraction": s[:, 0] / n_vox,
        "folding_abs_sum": s[:, 1],
        "det_min": s[:, 2],
        "det_max": s[:, 3],
        "det_mean": mean,
        "det_std": np.sqrt(var),
        "nonfinite_count": nonfinite,
    }
    if return_map:
        out["det"] = det
    return out


def _overlap(counts, ignore_background):
    """Per-label dice / iou / recall / precision (B,L) float64 and their means (B,) from confusion counts (B,L,L)
    (numpy int64, counts[b,p,t])."""
    c = np.asarray(counts, dtype=np.int64)
    tp = np.diagonal(c, axis1=1, axis2=2).astype(np.float64)
    n_pred = c.sum(axis=2).astype(np.float64)
    n_target = c.sum(axis=1).astype(np.float64)
    with np.errstate(invalid="ignore", divide="ignore"):
        res = {"dice": 2.0 * tp / (n_pred + n_target), "iou": tp / (n_pred + n_target - tp),
               "recall": tp / n_target, "precision": tp / n_pred}
    if ignore_background:
        for v in res.values():
            v[:, 0] = np.nan
    for k in list(res):
        v = res[k]
        ok = ~np.isnan(v)
        n = ok.sum(axis=1)
        res[k + "_mean"] = np.where(n > 0, np.where(ok, v, 0.0).sum(axis=1) / np.maximum(n, 1), np.nan)
    return res


def label_overlap(pred, target, num_labels=None, ignore_background=True):
    """Per-item, per-label overlap of label maps pred and target (B, ...) on the GPU (float32 as the nearest-mode warp
    returns them, or integer dtypes): dict of dice / iou / recall / precision (B,L) float64 and *_mean (B,) float64,
    plus the raw "counts" (B,L,L).  num_labels=None takes max+1 over both maps.  Raises ValueError if a voxel is not an
    integer label in [0, num_labels)."""
    if num_labels is None:
        hi = float(torch.maximum(pred.max(), target.max()))
        if not np.isfinite(hi) or hi < 0 or hi != int(hi) or hi >= 128:
            raise ValueError("label maps must hold integer labels in [0, 128); found a maximum of %r" % hi)
        num_labels = int(hi) + 1
    counts, invalid = ops.label_confusion(pred, target, num_labels)
    bad = invalid.cpu().numpy()
    if bad.any():
        raise ValueError("%s voxel(s) per item are not integer labels in [0, %d)" % (bad.tolist(), num_labels))
    c = counts.cpu().numpy()
    res = _overlap(c, ignore_background)
    res["counts"] = c
    return res


def _sorted_segments(dist, sizes):
    """dist (n,) with item b's values at [off[b], off[b+1]) -> each segment sorted ascending, on the device: a sort of
    the values, then a stable sort by segment."""
    B = len(sizes)
    vals, perm = torch.sort(dist)
    seg = torch.repeat_interleave(torch.arange(B, device=dist.device), torch.as_tensor(sizes, device=dist.device),
                                  output_size=dist.numel())
    _, order = torch.sort(seg[perm], stable=True)
    return vals[order]


def _q95_index(n):
    """numpy's "linear" percentile 95 of n sorted values: the indices of the two order statistics and the weight"""
    vi = (n - 1) * (95 / 100)
    lo = np.floor(vi)
    return lo.astype(np.int64), np.minimum(lo.astype(np.int64) + 1, n - 1), vi - lo


def _lerp(a, b, t):
    """numpy's lerp of two order statistics (numpy.lib._function_base_impl._lerp)"""
    diff = b - a
    return np.where(t >= 0.5, b - diff * (1 - t), a + diff * t)


def surface_distance(pred, target, spacing=(1.0, 1.0, 1.0), num_labels=None):
    """Per-item, per-label surface distances of label maps pred and target ((B,1,D,H,W) or (B,D,H,W), float32 as the
    nearest-mode warp returns them, or an integer dtype) on the GPU, with voxel spacing (s_D, s_H, s_W) in mm: dict of
    hd / hd95 / assd (B,L) float64 (label 0 is not scored and stays NaN), their *_mean (B,) over the labels present in
    both maps (NaN if none), and surface_count (B,2,L) int64 = [|S_pred(l)|, |S_target(l)|] (see the module docstring).
    num_labels=None takes max+1 over both maps.  Raises ValueError if a voxel is not an integer label in
    [0, num_labels).

    One count pass (ops.label_surface_counts) is read back; then each label present in both maps takes two
    ops.surface_distances calls, whose distances are sorted per segment on the device; only a few numbers per item and
    label are read back."""
    sp = tuple(float(s) for s in spacing)
    pred, target = ops._label_volumes(pred, target)
    if num_labels is None:
        hi = float(torch.maximum(pred.max(), target.max()))
        if not np.isfinite(hi) or hi < 0 or hi != int(hi) or hi >= 128:
            raise ValueError("label maps must hold integer labels in [0, 128); found a maximum of %r" % hi)
        num_labels = int(hi) + 1
    L = int(num_labels)
    counts, invalid = ops.label_surface_counts(pred, target, L)
    bad = invalid.cpu().numpy()
    if bad.any():
        raise ValueError("%s voxel(s) per item are not integer labels in [0, %d)" % (bad.tolist(), L))
    sc = counts.cpu().numpy()
    B = sc.shape[0]
    both = (sc[:, 0] > 0) & (sc[:, 1] > 0)
    both[:, 0] = False
    labels = [l for l in range(1, L) if both[:, l].any()]
    pieces = []                 # per label and direction: (B,5) = [count, sum, max, order statistic lo, hi]
    for l in labels:
        for k, (a, b) in enumerate(((pred, target), (target, pred))):
            n = sc[:, k, l]
            dist, seg_offset, stats = ops.surface_distances(a, b, l, sp, sizes=n)
            srt = _sorted_segments(dist, n)
            lo, hi, _ = _q95_index(np.maximum(n, 1))
            start = np.concatenate([[0], np.cumsum(n)[:-1]])
            idx = np.minimum(np.stack([start + lo, start + hi], 1), max(dist.numel() - 1, 0))
            pieces.append(torch.cat([stats, srt[torch.from_numpy(idx).to(srt.device)]], 1))
    hd, hd95, assd = (np.full((B, L), np.nan) for _ in range(3))
    if pieces:
        got = torch.stack(pieces).cpu().numpy().reshape(len(labels), 2, B, 5)
        for j, l in enumerate(labels):
            ok = both[:, l]
            _, _, t = _q95_index(np.maximum(sc[:, :, l], 1))            # (B,2)
            g = got[j]                                                    # (2,B,5)
            with np.errstate(invalid="ignore", divide="ignore"):
                mean = g[:, :, 1] / g[:, :, 0]
            q = _lerp(g[:, :, 3], g[:, :, 4], t.T)
            hd[ok, l] = np.maximum(g[0, ok, 2], g[1, ok, 2])
            hd95[ok, l] = np.maximum(q[0, ok], q[1, ok])
            assd[ok, l] = (mean[0, ok] + mean[1, ok]) / 2
    res = {"hd": hd, "hd95": hd95, "assd": assd}
    for k in list(res):
        v = res[k]
        ok = ~np.isnan(v)
        n = ok.sum(axis=1)
        res[k + "_mean"] = np.where(n > 0, np.where(ok, v, 0.0).sum(axis=1) / np.maximum(n, 1), np.nan)
    res["surface_count"] = sc
    return res
