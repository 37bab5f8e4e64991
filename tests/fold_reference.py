"""float64 references of the folding penalty and its gradient (test infrastructure, imported by test_fold_penalty_host /
test_fold_penalty_gpu).

    fold(phi) = 1/(B*D*H*W) * sum over voxels of max(0, -det J)          (include/liftreg_b200.h, lr_jacobian_fold_backward)

The fold set is the one the kernels use: m = (det32 finite and < 0), det32 from the fp32 restatement of lr_jacobian_det
(metrics_reference.jacobian_det), so a reference and the kernel agree on the kink.

fold_grad_autograd is float64 autograd of grad_loss/N * sum m * (-det64), det64 the same restatement on the float64 map.
fold_grad states the same gradient explicitly, -(grad_loss/N) * sum_a s_a D_a^T (m * C[c][a]) with C the cofactors, and
returns with it an abs-scale: the same expression over absolute values, |grad_loss|/N * sum_a |s_a| |D_a|^T (m * Cabs),
with Cabs[c][a] = |J J| + |J J| (the two products of the cofactor).  By default fold_grad takes J as the fp32 values the
kernel computes (exactly: the restatement is bit-identical to it), so that the comparison measures the adjoint's own
rounding; the linear face rule's 2 I[n-1] - I[n-2] is rounded in fp32 before a difference of two close values, which
alone moves J by up to ~40 u relative at 160^3 and is the forward's definition, not an error of the adjoint."""
import numpy as np
import torch

from metrics_reference import jacobian_det
from oracle.torch_port import _fd_central


def _spacing(shape):
    return 1. / (np.array(shape) - 1) * 2


def jacobian(phi, boundary):
    """J[c][a] (each (B,D,H,W)) of a torch map with the restatement's differences and scales, in phi's dtype."""
    sp = _spacing(phi.shape[2:])
    return [[_fd_central(phi[:, c, ...], a + 1, sp[a], boundary) for a in range(3)] for c in range(3)]


def fold_mask(phi32, boundary):
    det = jacobian_det(torch.from_numpy(np.ascontiguousarray(phi32, np.float32)), boundary).numpy()
    return np.isfinite(det) & (det < 0)


def fold_value(phi32, boundary):
    """float64 penalty: mean of m * (-det64) over every voxel of the batch."""
    m = torch.from_numpy(fold_mask(phi32, boundary))
    det = jacobian_det(torch.from_numpy(np.asarray(phi32, np.float64)), boundary)
    return float(-torch.where(m, det, torch.zeros_like(det)).sum() / det.numel())


def fold_grad_autograd(phi32, boundary, grad_loss=1.0, mask=None):
    """float64 autograd of grad_loss * mean(m * (-det64)) wrt phi (phi32 cast to float64; finite maps only)."""
    m = torch.from_numpy(fold_mask(phi32, boundary) if mask is None else mask)
    p = torch.from_numpy(np.asarray(phi32, np.float64)).requires_grad_(True)
    det = jacobian_det(p, boundary)
    loss = -torch.where(m, det, torch.zeros_like(det)).sum() * (grad_loss / det.numel())
    loss.backward()
    return p.grad.numpy()


def fd_adjoint(G, axis, boundary, absolute=False):
    """D^T G along `axis` for the unscaled difference operator of _fd_central (rows xp - xm): interior rows +1 at i+1,
    -1 at i-1; linear mode rows 0 / n-1 are 2 I[1] - 2 I[0] / 2 I[n-1] - 2 I[n-2]; neumann_zero rows 0 / n-1 are zero.
    absolute: the transpose of |D| instead."""
    g = np.moveaxis(np.asarray(G, np.float64), axis, -1)
    o = np.zeros_like(g)
    n = g.shape[-1]
    neg = 1.0 if absolute else -1.0
    o[..., 2:] += g[..., 1:n - 1]
    o[..., :n - 2] += neg * g[..., 1:n - 1]
    if boundary == "linear":
        o[..., 1] += 2 * g[..., 0]
        o[..., 0] += neg * 2 * g[..., 0]
        o[..., n - 1] += 2 * g[..., n - 1]
        o[..., n - 2] += neg * 2 * g[..., n - 1]
    elif boundary != "neumann_zero":
        raise ValueError(boundary)
    return np.moveaxis(o, -1, axis)


def fold_grad(phi32, boundary, grad_loss=1.0, j_dtype=np.float32):
    """(grad, scale), both (B,3,D,H,W) float64: the explicit gradient and its abs-scale (module docstring).  J is taken
    from the fp32 restatement (j_dtype=np.float32, the kernel's values) or computed in float64 (np.float64)."""
    phi32 = np.ascontiguousarray(phi32, np.float32)
    m = fold_mask(phi32, boundary)
    J = [[t.numpy().astype(np.float64) for t in row] for row in jacobian(torch.from_numpy(phi32.astype(j_dtype)), boundary)]
    s = 0.5 / _spacing(phi32.shape[2:])
    N = m.size
    grad = np.zeros(phi32.shape)
    scale = np.zeros(phi32.shape)
    with np.errstate(invalid="ignore", over="ignore"):
        for c in range(3):
            c1, c2 = (c + 1) % 3, (c + 2) % 3
            for a in range(3):
                a1, a2 = (a + 1) % 3, (a + 2) % 3
                p, q = J[c1][a1] * J[c2][a2], J[c1][a2] * J[c2][a1]
                G = np.where(m, p - q, 0.0)
                Gabs = np.where(m, np.abs(p) + np.abs(q), 0.0)
                grad[:, c] += s[a] * fd_adjoint(G, a + 1, boundary)
                scale[:, c] += s[a] * fd_adjoint(Gabs, a + 1, boundary, absolute=True)
    return -(grad_loss / N) * grad, (abs(grad_loss) / N) * scale


REFLECTED_A = np.array([[1.0, 0.25, 0.0], [0.0, 0.75, 0.125], [0.5, 0.0, 1.0]])


def reflected_affine(shape, B=1):
    """-(A x + t) on a dyadic grid (n <= 64 per axis): every difference is exact, so J is the same constant at every
    voxel in fp32 too, and det J = -det(A) * prod(scales) < 0.  (B,3,D,H,W) float32."""
    x = np.stack(np.meshgrid(*[(np.arange(n) - (n - 1) / 2) / 32 for n in shape], indexing="ij"))
    phi = np.einsum("ij,jdhw->idhw", REFLECTED_A, x) + np.array([0.125, -0.25, 0.0625]).reshape(3, 1, 1, 1)
    return np.repeat((-phi)[None], B, 0).astype(np.float32)
