"""Validation metrics on the GPU: Jacobian folding statistics of a map and per-label overlap of two label maps.

The reference scores each validation item on the host (networks/RegistrationNet.py:198-218 _compute_metrics): the
Jacobian determinant of phi with numpy and mermaid's finite differences (utils/utils.py:20-55, after copying the
3*D*H*W map to the host) and per-label Dice / IoU / recall / precision with Python sets (utils/metrics.py:6-121,
get_multi_metric / cal_metric).  Here each function is one kernel call (ops.jacobian_det, ops.label_confusion) plus a
readout of a few numbers per item.

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
