"""float64 reference of the normalized gradient field (NGF) similarity and its gradient (test infrastructure, imported
by test_ngf_host / test_ngf_gpu; definition in include/liftreg_b200.h, lr_ngf_sum).

g and h are the kernels' fp32 differences: oracle.torch_port._fd_central on float32 tensors, which is bit for bit what
lr_jacobian_det forms for one channel (tests/metrics_reference.py).  Everything after them is float64 in the kernels'
order of operations:
    a = g.h,  p = |g|^2 + eps^2,  q = |h|^2 + eps^2,  f = a^2 / (p q),  loss = 1 - sum f / (B*D*H*W)
    c_a = (2a/(pq)) (h_a - (a/p) g_a),  grad = -(grad_loss/(B*D*H*W)) sum_a s_a D_a^T c_a
`ngf` returns the per-item sums of f, the loss, the gradient and its per-element abs-scale
    scale(v) = |grad_loss|/(B*D*H*W) * sum_a s_a * sum over the D_a^T stencil at v of |coefficient| * |c_a|.
`ngf_torch` is the stock-op composition of the same definition in the dtype of its inputs (autograd differentiates it)."""
import numpy as np
import torch

from fold_reference import fd_adjoint
from oracle.torch_port import _fd_central


def _spacing(shape):
    return 1. / (np.array(shape) - 1) * 2


def _volume(a):
    a = np.asarray(a)
    return a[:, 0] if a.ndim == 5 else a


def diffs(v, boundary, dtype=np.float32):
    """[d_0, d_1, d_2] of a (B,D,H,W) volume: the scaled central differences of _fd_central in `dtype`, as float64"""
    t = torch.from_numpy(np.ascontiguousarray(v, dtype))
    sp = _spacing(t.shape[1:])
    return [_fd_central(t, a + 1, sp[a], boundary).numpy().astype(np.float64) for a in range(3)]


def ngf(x, y, eps=1.0, boundary="linear", grad_loss=1.0, diff_dtype=np.float32):
    """x, y (B,1,D,H,W) or (B,D,H,W).  Returns (sums (B,), loss, grad (shape of x), scale (shape of x)).  diff_dtype
    float32 takes g and h as the kernels compute them; float64 computes them in float64 (for central differences)."""
    shape = np.shape(x)
    X, Y = _volume(x), _volume(y)
    B = X.shape[0]
    g, h = diffs(X, boundary, diff_dtype), diffs(Y, boundary, diff_dtype)
    e2 = float(eps) * float(eps)
    a = g[0] * h[0] + g[1] * h[1] + g[2] * h[2]
    p = g[0] * g[0] + g[1] * g[1] + g[2] * g[2] + e2
    q = h[0] * h[0] + h[1] * h[1] + h[2] * h[2] + e2
    f = a * a / (p * q)
    sums = f.reshape(B, -1).sum(1)
    N = f.size
    t, r = 2.0 * a / (p * q), a / p
    s = 0.5 / _spacing(X.shape[1:])
    grad = np.zeros(X.shape)
    scale = np.zeros(X.shape)
    for k in range(3):
        c = t * (h[k] - r * g[k])
        grad += s[k] * fd_adjoint(c, k + 1, boundary)
        scale += s[k] * fd_adjoint(np.abs(c), k + 1, boundary, absolute=True)
    grad = -(grad_loss / N) * grad
    scale = (abs(grad_loss) / N) * scale
    return sums, 1.0 - sums.sum() / N, grad.reshape(shape), scale.reshape(shape)


def ngf_torch(x, y, eps=1.0, boundary="linear"):
    """the stock-op composition on (B,1,D,H,W) or (B,D,H,W) tensors, in their dtype and on their device: the loss"""
    X = x[:, 0] if x.dim() == 5 else x
    Y = y[:, 0] if y.dim() == 5 else y
    sp = _spacing(X.shape[1:])
    g = [_fd_central(X, a + 1, sp[a], boundary) for a in range(3)]
    h = [_fd_central(Y, a + 1, sp[a], boundary) for a in range(3)]
    e2 = float(eps) * float(eps)
    a = g[0] * h[0] + g[1] * h[1] + g[2] * h[2]
    p = g[0] * g[0] + g[1] * g[1] + g[2] * g[2] + e2
    q = h[0] * h[0] + h[1] * h[1] + h[2] * h[2] + e2
    return 1.0 - (a * a / (p * q)).mean()
