"""CPU references of the validation metrics (test infrastructure, imported by test_metrics_host / test_metrics_gpu).

jacobian_det restates lr_jacobian_det on the regulariser's torch restatement of mermaid's central differences
(oracle/torch_port._fd_central) in the kernel's op order; overlap_by_sets scores label maps with Python sets of voxel
indices, the way the reference's metrics.py counts.  PARITY UNPINNED against the reference's utils.py:20-55 and
metrics.py:6-121 (not part of the reference tree)."""
import numpy as np

from oracle.torch_port import _fd_central


def jacobian_det(phi, boundary="linear"):
    """Jacobian determinant (B,D,H,W) of a map phi (B,3,D,H,W) in [-1,1]: J[c][a] = _fd_central(phi_c, axis a,
    2/(n_a-1)), expanded along the first row with every product and difference a separate tensor op.  In float32 it is
    the bit-exact reference of lr_jacobian_det; in float64 the value reference."""
    sp = 1. / (np.array(phi.shape[2:]) - 1) * 2
    J = [[_fd_central(phi[:, c, ...], a + 1, sp[a], boundary) for a in range(3)] for c in range(3)]
    a = J[0][0] * (J[1][1] * J[2][2] - J[1][2] * J[2][1])
    b = J[0][1] * (J[1][0] * J[2][2] - J[1][2] * J[2][0])
    c = J[0][2] * (J[1][0] * J[2][1] - J[1][1] * J[2][0])
    return a - b + c


def overlap_by_sets(p, t, L):
    """Per-label Dice / IoU / recall / precision (float64, NaN where the denominator is zero) from Python sets."""
    out = {k: np.full(L, np.nan) for k in ("dice", "iou", "recall", "precision")}
    for l in range(L):
        P = set(np.flatnonzero(p == l).tolist())
        T = set(np.flatnonzero(t == l).tolist())
        tp = len(P & T)
        if P or T:
            out["dice"][l] = 2.0 * tp / (len(P) + len(T))
            out["iou"][l] = tp / len(P | T)
        if T:
            out["recall"][l] = tp / len(T)
        if P:
            out["precision"][l] = tp / len(P)
    return out
