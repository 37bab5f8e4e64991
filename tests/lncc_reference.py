"""Float64 reference of the local (windowed) NCC loss and its gradient (numpy only; definition in
include/liftreg_b200.h, lr_local_ncc_sum).

Box sums come from zero-padded integral volumes, built one axis at a time (a prefix sum along each axis in extended
precision, then the difference of two entries w apart), so a window sum carries no drift from the volume's extent.
`local_ncc` returns cc per voxel, the loss, the gradient by the alpha / beta / gamma formula and a per-element
abs-scale of the gradient: the same sums taken over absolute terms,
    scale_v = |g| / (B*D*H*W) * (|y_v| * sum |alpha| + |x_v| * sum |beta| + sum |gamma|).
"""
import numpy as np


def box_sum(a, w):
    """zero-padded sum over the w x w x w cube centred on each voxel of a (B,D,H,W) array"""
    r = w // 2
    out = np.asarray(a, np.longdouble)
    for ax in (1, 2, 3):
        n = out.shape[ax]
        pad = [(0, 0)] * 4
        pad[ax] = (r + 1, r)                        # a leading 0 for the prefix sum, then the r-voxel zero padding
        c = np.cumsum(np.pad(out, pad), axis=ax)
        out = np.take(c, np.arange(w, w + n), axis=ax) - np.take(c, np.arange(n), axis=ax)
    return out.astype(np.float64)


def _squeeze(a):
    a = np.asarray(a, np.float64)
    return a[:, 0] if a.ndim == 5 else a


def moments(x, y, w):
    """the five window sums Sx, Sy, Sxx, Syy, Sxy of (B,D,H,W) arrays"""
    return [box_sum(t, w) for t in (x, y, x * x, y * y, x * y)]


def local_ncc(x, y, w=9, eps=1e-5, grad_loss=1.0):
    """x, y (B,1,D,H,W) or (B,D,H,W).  Returns (cc (B,D,H,W), loss, grad (shape of x), scale (shape of x))."""
    shape = np.shape(x)
    x, y = _squeeze(x), _squeeze(y)
    n = float(w) ** 3
    Sx, Sy, Sxx, Syy, Sxy = moments(x, y, w)
    cross = Sxy - Sx * Sy / n
    vx, vy = Sxx - Sx * Sx / n, Syy - Sy * Sy / n
    d = vx * vy + eps
    ok = d > 0
    dd = np.where(ok, d, 1.0)
    cc = np.where(ok, cross * cross / dd, 0.0)
    alpha = np.where(ok, 2.0 * cross / dd, 0.0)
    beta = np.where(ok, 2.0 * cross * cross * vy / (dd * dd), 0.0)
    gamma = beta * (Sx / n) - alpha * (Sy / n)
    k = grad_loss / x.size
    grad = -k * (y * box_sum(alpha, w) - x * box_sum(beta, w) + box_sum(gamma, w))
    scale = abs(k) * (np.abs(y) * box_sum(np.abs(alpha), w) + np.abs(x) * box_sum(np.abs(beta), w)
                      + box_sum(np.abs(gamma), w))
    return cc, 1.0 - cc.mean(), grad.reshape(shape), scale.reshape(shape)


def item_losses(x, y, w=9, eps=1e-5):
    """1 - mean of cc over each item (B,)"""
    cc = local_ncc(x, y, w, eps)[0]
    return 1.0 - cc.reshape(cc.shape[0], -1).mean(1)


def inside_mask(shape, reach):
    """(D,H,W) mask of the voxels at least `reach` from every face"""
    m = np.zeros(shape, bool)
    if all(n > 2 * reach for n in shape):
        m[reach:shape[0] - reach, reach:shape[1] - reach, reach:shape[2] - reach] = True
    return m


def voxelmorph_ncc_torch(x, y, w, eps):
    """VoxelMorph's NCC(win) restated in torch (conv3d with a ones kernel, padding w//2) on (B,1,D,H,W) tensors, in
    their dtype: returns (1 - mean cc, cc)."""
    import torch
    import torch.nn.functional as F
    k = torch.ones((1, 1, w, w, w), dtype=x.dtype, device=x.device)
    p = w // 2
    S = lambda t: F.conv3d(t, k, padding=p)                                             # noqa: E731
    I_sum, J_sum, I2_sum, J2_sum, IJ_sum = S(x), S(y), S(x * x), S(y * y), S(x * y)
    n = float(w) ** 3
    u_I, u_J = I_sum / n, J_sum / n
    cross = IJ_sum - u_J * I_sum - u_I * J_sum + u_I * u_J * n
    I_var = I2_sum - 2 * u_I * I_sum + u_I * u_I * n
    J_var = J2_sum - 2 * u_J * J_sum + u_J * u_J * n
    cc = cross * cross / (I_var * J_var + eps)
    return 1.0 - cc.mean(), cc
