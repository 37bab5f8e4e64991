"""Float64 reference of the soft Dice loss of the warped label map (ops.label_dice_loss, lr_label_dice_sums /
lr_label_dice_backward; definition in include/liftreg_b200.h).  Test infrastructure, imported by test_label_dice_host and
test_label_dice_gpu.

The sample coordinates, their floors and fractions are the kernels' fp32 values (adjoint_reference._axis, zeros
padding), and the tap weights the fp32 products (wx * wy) * wz; everything after that is float64.  Next to the gradient
it returns an abs-scale, the same sum with every term replaced by its absolute value, which is what a rounding-error
bound needs:  |kernel - ref| <= k * u * scale,  u = 2^-24."""
import numpy as np

from adjoint_reference import _axis

U = 2.0 ** -24


def label_index(v, L):
    """int64 label of each value, -1 where it is not an integer in [0, L) (negative, >= L, fractional, NaN)"""
    v = np.asarray(v, np.float32)
    with np.errstate(invalid="ignore"):
        ok = np.isfinite(v) & (v >= 0) & (v < L) & (np.floor(v) == v)
    return np.where(ok, np.where(ok, v, 0).astype(np.int64), -1)


def _taps(phi, src, L):
    """per tap t = tx + 2 ty + 4 tz: (tx, ty, tz, label (B,D,H,W) int64 with -1 for outside / no label), the fractions
    (w0, w1) per axis as float64 of the fp32 values, the fp32 weights (B,D,H,W) as float64 and the multipliers (S-1)/2"""
    phi = np.ascontiguousarray(phi, np.float32)
    B, _, D, H, W = phi.shape
    (z0, wz, mz), (y0, wy, my), (x0, wx, mx) = (_axis(phi[:, a], S, False) for a, S in enumerate((D, H, W)))
    lab = label_index(src, L).reshape(B, -1)
    f32 = [tuple(np.float32(w) for w in ws) for ws in (wx, wy, wz)]
    taps = []
    for t in range(8):
        tx, ty, tz = t & 1, (t >> 1) & 1, t >> 2
        xx, yy, zz = x0 + tx, y0 + ty, z0 + tz
        ok = (xx >= 0) & (xx < W) & (yy >= 0) & (yy < H) & (zz >= 0) & (zz < D)
        lin = ((np.clip(zz, 0, D - 1) * H + np.clip(yy, 0, H - 1)) * W + np.clip(xx, 0, W - 1)).reshape(B, -1)
        tl = np.where(ok, np.take_along_axis(lab, lin, 1).reshape(ok.shape), -1)
        w = ((f32[0][tx] * f32[1][ty]) * f32[2][tz]).astype(np.float64)          # fp32 products, warp_one's order
        taps.append((tx, ty, tz, tl, w))
    return taps, (wx, wy, wz), (mz, my, mx)


def dice_sums(phi, src, tgt, L):
    """(B,L,3) float64 [I, P, T]"""
    B = phi.shape[0]
    taps, _, _ = _taps(phi, src, L)
    tl = label_index(tgt, L).reshape(B, -1)
    sums = np.zeros((B, L, 3))
    for b in range(B):
        for _, _, _, lab, w in taps:
            lb, wb = lab[b].ravel(), w[b].ravel()
            ok = lb >= 0
            sums[b, :, 1] += np.bincount(lb[ok], weights=wb[ok], minlength=L)
            hit = ok & (lb == tl[b])
            sums[b, :, 0] += np.bincount(lb[hit], weights=wb[hit], minlength=L)
        sums[b, :, 2] = np.bincount(tl[b][tl[b] >= 0], minlength=L)
    return sums


def dice_loss(sums):
    """loss and the coefficients a = d loss / d P, e = d loss / d I (B,L) from the sums, float64"""
    I, P, T = sums[..., 0], sums[..., 1], sums[..., 2]
    B = sums.shape[0]
    den = P + T
    in_s = den > 0
    in_s[:, 0] = False
    n = in_s.sum(1)
    safe = np.where(in_s, den, 1.0)
    dice = np.where(n > 0, np.where(in_s, 2.0 * I / safe, 0.0).sum(1) / np.maximum(n, 1), 1.0)
    k = (2.0 / (B * np.maximum(n, 1)))[:, None]
    a = np.where(in_s, k * I / (safe * safe), 0.0)
    e = np.where(in_s, -k / safe, 0.0)
    return 1.0 - dice.mean(), a, e


def dice_reference(phi, src, tgt, L, grad_loss=1.0):
    """(sums (B,L,3), loss, grad_phi (B,3,D,H,W), scale (B,3,D,H,W)), all float64; src and tgt (B,D,H,W)"""
    B, _, D, H, W = phi.shape
    src = np.asarray(src, np.float32).reshape(B, D, H, W)
    tgt = np.asarray(tgt, np.float32).reshape(B, D, H, W)
    sums = dice_sums(phi, src, tgt, L)
    loss, a, e = dice_loss(sums)
    taps, (wx, wy, wz), (mz, my, mx) = _taps(phi, src, L)
    tl = label_index(tgt, L)
    rows = np.arange(B)[:, None, None, None]
    g = float(grad_loss)
    gi = [np.zeros((B, D, H, W)) for _ in range(3)]         # x, y, z sums before the multiplier
    si = [np.zeros((B, D, H, W)) for _ in range(3)]
    for tx, ty, tz, lab, _ in taps:
        ok = lab >= 0
        li = np.maximum(lab, 0)
        coef = np.where(ok, a[rows, li] + np.where(lab == tl, e[rows, li], 0.0), 0.0)
        cabs = np.where(ok, np.abs(a[rows, li]) + np.where(lab == tl, np.abs(e[rows, li]), 0.0), 0.0)
        dw = (wy[ty] * wz[tz], wx[tx] * wz[tz], wx[tx] * wy[ty])
        for c, (sign, d) in enumerate(zip((tx, ty, tz), dw)):
            gi[c] += (1.0 if sign else -1.0) * d * coef
            si[c] += d * cabs
    grad = g * np.stack([mz * gi[2], my * gi[1], mx * gi[0]], axis=1)
    scale = abs(g) * np.stack([mz * si[2], my * si[1], mx * si[0]], axis=1)
    return sums, loss, grad, scale


def blob_labels(B, shape, L, seed, shift=0):
    """label maps of a few overlapping balls on background, target = the moving map rolled by `shift` along axis 0"""
    rs = np.random.RandomState(seed)
    zz, yy, xx = np.meshgrid(*[np.arange(n) for n in shape], indexing="ij")
    lab = np.zeros((B,) + shape, np.float32)
    for b in range(B):
        for k in range(1, L):
            c = [rs.uniform(0, n) for n in shape]
            r = rs.uniform(0.25, 0.5) * max(shape)
            lab[b][(zz - c[0]) ** 2 + (yy - c[1]) ** 2 + (xx - c[2]) ** 2 < r * r] = k
    return lab, np.roll(lab, shift, axis=1)


def stock_dice_loss(phi, src, tgt, L):
    """The same loss from stock ops on CUDA tensors, as VoxelMorph forms it: L one-hot channels of the moving labels
    warped by ops.warp (trilinear, zeros padding, no using_scale), soft Dice from torch sums; differentiable wrt phi
    through ops.warp's adjoint.  phi (B,3,D,H,W) float32; src, tgt (B,D,H,W) float32 label maps."""
    import torch
    from liftreg_b200 import ops
    labels = torch.arange(L, device=phi.device, dtype=torch.float32).view(1, L, 1, 1, 1)
    oh = (src[:, None] == labels).float()
    tm = (tgt[:, None] == labels).double()
    warped = ops.warp(oh, phi, zero_boundary=True, using_scale=False).double()
    sums = torch.stack([(warped * tm).sum((2, 3, 4)), warped.sum((2, 3, 4)), tm.sum((2, 3, 4))], -1)
    return ops._dice_loss_from_sums(sums).float()
