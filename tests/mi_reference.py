"""float64 reference of the mutual information (MI) similarity and its gradient (test infrastructure, imported by
test_mi_host / test_mi_gpu; definition in include/liftreg_b200.h, lr_mi_hist).

u, iota, k0 and f come from the kernels' fp32 chain (numpy float32 arithmetic rounds every op, as the kernels do):
    s = float32((nb - 1) / (hi - lo)),  u = (fmin(fmax(v, lo), hi) - lo) * s,
    iota = floor(u_y + 0.5),  k0 = min(floor(u_x), nb - 2),  f = u_x - k0
Everything after them is float64: the cubic B-spline tap weights in the header's order, the histogram accumulated in
extended precision (numpy longdouble), then
    p = hist / N,  MI_b = sum_{p > 0} p (log p - log p_y - log p_x),  loss = -mean_b MI_b
    grad_v = k * sum_m w_m'(f_v) * c(iota_v, k0_v - 1 + m),  c = log(hist / P_x) (0 where hist = 0),
    k = -(g s) / (B N), zero unless lo <= x_v <= hi
with P_x the column sums of hist taken over the rows in order, as the adjoint kernel forms them.  `mi` returns the
histogram, the loss, the gradient and its per-element abs-scale
    scale_v = |k| * sum_m |w_m'(f_v)| * |c(iota_v, k0_v - 1 + m)|   (zero outside [lo, hi]).
`mi_torch` is the stock-op composition of the same definition (clamp, B-spline weights, scatter_add into the
histogram, MI) in the dtype of its inputs; autograd differentiates it."""
import numpy as np
import torch


def scale_of(nb, lo, hi):
    lo32, hi32 = np.float32(lo), np.float32(hi)
    return lo32, hi32, np.float32((nb - 1) / (np.float64(hi32) - np.float64(lo32)))


def chain(x, y, nb, lo, hi, dtype=np.float32):
    """(u_x, iota, k0, f) per element of the (B, N) arrays x, y.  dtype float32 is the kernels' chain; float64 evaluates
    it in float64 (for central differences)"""
    lo32, hi32, s = scale_of(nb, lo, hi)
    lo_, hi_, s_ = (dtype(v) for v in (lo32, hi32, s))
    if dtype is np.float64:
        s_ = (nb - 1) / (hi_ - lo_)

    def u(v):
        v = np.asarray(v, dtype)
        return (np.fmin(np.fmax(v, lo_), hi_) - lo_) * s_
    ux, uy = u(x), u(y)
    iota = np.minimum(np.floor(uy + dtype(0.5)), nb - 1).astype(np.int64)
    k0 = np.minimum(np.floor(ux), nb - 2).astype(np.int64)
    f = ux - k0.astype(dtype)
    return ux, iota, k0, f


def weights(f):
    """the four tap weights in float64 from f, in the header's order of operations"""
    F = np.asarray(f, np.float64)
    G = 1.0 - F
    F2 = F * F
    F3 = F2 * F
    r6 = 1.0 / 6.0
    return [G * G * G * r6, ((4.0 - 6.0 * F2) + 3.0 * F3) * r6, (((1.0 + 3.0 * F) + 3.0 * F2) - 3.0 * F3) * r6, F3 * r6]


def dweights(f):
    """d w_m / d f in float64 (exact for the fp32 f)"""
    F = np.asarray(f, np.float64)
    return [-(1.0 - F) ** 2 / 2, F * (3.0 * F - 4.0) / 2, (1.0 + 2.0 * F - 3.0 * F * F) / 2, F * F / 2]


def histogram(iota, k0, f, nb):
    """(B, nb, nb+2) float64 from the per-element rows, taps and fractions of (B, N) arrays, accumulated in longdouble"""
    B = iota.shape[0]
    nc = nb + 2
    base = (np.arange(B)[:, None] * nb + iota) * nc + k0
    keys = np.concatenate([(base + m).ravel() for m in range(4)])
    vals = np.concatenate([w.ravel() for w in weights(f)]).astype(np.longdouble)
    order = np.argsort(keys, kind="stable")
    keys, vals = keys[order], vals[order]
    starts = np.flatnonzero(np.r_[True, keys[1:] != keys[:-1]])
    out = np.zeros(B * nb * nc, np.longdouble)
    out[keys[starts]] = np.add.reduceat(vals, starts)
    return out.astype(np.float64).reshape(B, nb, nc)


def mi_value(hist, N):
    """-mean_b MI_b in float64"""
    p = np.asarray(hist, np.float64) / N
    py = np.broadcast_to(p.sum(2, keepdims=True), p.shape)
    px = np.broadcast_to(p.sum(1, keepdims=True), p.shape)
    pos = p > 0
    t = np.zeros(p.shape)
    t[pos] = p[pos] * (np.log(p[pos]) - np.log(py[pos]) - np.log(px[pos]))
    return -t.sum((1, 2)).mean()


def mi(x, y, num_bins=32, value_range=(-1.0, 1.0), grad_loss=1.0, hist=None, chain_dtype=np.float32):
    """x, y (B, ...) arrays of one shape.  Returns (hist (B, nb, nb+2), loss, grad (shape of x), scale (shape of x)).
    `hist` given: the gradient is taken with it (as lr_mi_backward does), the returned hist and loss are still the
    reference's own."""
    shape = np.shape(x)
    B = shape[0]
    X = np.asarray(x).reshape(B, -1)
    Y = np.asarray(y).reshape(B, -1)
    N = X.shape[1]
    nb = int(num_bins)
    lo, hi = value_range
    _, iota, k0, f = chain(X, Y, nb, lo, hi, chain_dtype)
    own = histogram(iota, k0, f, nb)
    loss = mi_value(own, N)
    H = own if hist is None else np.asarray(hist, np.float64)
    P = H[:, 0].copy()
    for r in range(1, nb):
        P = P + H[:, r]
    c = np.zeros(H.shape)
    pos = H > 0
    c[pos] = np.log(H[pos] / np.broadcast_to(P[:, None, :], H.shape)[pos])
    lo32, hi32, s = scale_of(nb, lo, hi)
    s = np.float64(s) if chain_dtype is np.float32 else (nb - 1) / (np.float64(hi32) - np.float64(lo32))
    k = -(np.float64(np.float32(grad_loss)) * s) / (float(B) * float(N))
    Xc = np.asarray(X, chain_dtype)
    inside = (Xc >= chain_dtype(lo32)) & (Xc <= chain_dtype(hi32))
    bidx = np.arange(B)[:, None]
    grad = np.zeros(X.shape)
    scale = np.zeros(X.shape)
    for m, dw in enumerate(dweights(f)):
        cm = c[bidx, iota, k0 + m]
        grad += dw * cm
        scale += np.abs(dw) * np.abs(cm)
    grad = np.where(inside, k * grad, 0.0)
    scale = np.where(inside, abs(k) * scale, 0.0)
    return own, loss, grad.reshape(shape), scale.reshape(shape)


def mi_torch(x, y, num_bins=32, value_range=(-1.0, 1.0)):
    """the stock-op composition on (B, ...) tensors, in their dtype and on their device: the loss"""
    nb = int(num_bins)
    lo32, hi32, s32 = scale_of(nb, *value_range)
    lo, hi = float(lo32), float(hi32)
    s = float(s32) if x.dtype == torch.float32 else (nb - 1) / (hi - lo)
    B = x.shape[0]
    X, Y = x.reshape(B, -1), y.reshape(B, -1)
    N = X.shape[1]
    ux = (torch.clamp(X, lo, hi) - lo) * s
    uy = (torch.clamp(Y, lo, hi) - lo) * s
    iota = torch.floor(uy + 0.5).clamp(max=nb - 1).long()
    k0 = torch.floor(ux.detach()).clamp(max=nb - 2)
    f = ux - k0
    g = 1.0 - f
    w = [g * g * g / 6.0, (4.0 - 6.0 * f * f + 3.0 * f * f * f) / 6.0, (1.0 + 3.0 * f + 3.0 * f * f - 3.0 * f * f * f) / 6.0,
         f * f * f / 6.0]
    base = iota * (nb + 2) + k0.long()
    hist = torch.zeros(B, nb * (nb + 2), dtype=x.dtype, device=x.device)
    for m in range(4):
        hist = hist.scatter_add(1, base + m, w[m])
    p = hist.reshape(B, nb, nb + 2) / N
    py = p.sum(2, keepdim=True).expand_as(p)
    px = p.sum(1, keepdim=True).expand_as(p)
    pos = p > 0
    one = torch.ones((), dtype=p.dtype, device=p.device)
    lg = lambda t: torch.log(torch.where(pos, t, one))
    return -torch.where(pos, p * (lg(p) - lg(py) - lg(px)), 0.0).sum((1, 2)).mean()
