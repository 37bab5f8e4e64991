"""NGF similarity without a GPU: the float64 reference (tests/ngf_reference.py) against float64 autograd of the
stock-op composition on dyadic images and against central differences; the loss class by dotted name; the ValueErrors
of ops.ngf_loss; argument validation of the C-ABI."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

from ngf_reference import ngf, ngf_torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BOUNDARIES = ["linear", "neumann_zero"]


def dyadic(rs, shape):
    """values k/8 - 1: every fp32 difference, the 2c - d face rule and the product with s = (n-1)/4 are exact"""
    return rs.randint(0, 16, shape) / 8.0 - 1.0


def autograd(x, y, eps, boundary, grad_loss):
    xt = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    loss = ngf_torch(xt, torch.tensor(y, dtype=torch.float64), eps, boundary)
    (grad_loss * loss).backward()
    return loss.item(), xt.grad.numpy()


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("eps", [1e-2, 1.0, 10.0])
@pytest.mark.parametrize("B,shape", [(1, (2, 2, 2)), (2, (5, 7, 9)), (1, (3, 11, 6)), (2, (9, 4, 13))])
def test_reference_equals_float64_autograd(B, shape, eps, boundary):
    rs = np.random.RandomState(sum(shape) + B)
    x = dyadic(rs, (B, 1) + shape)
    y = np.where(rs.uniform(size=x.shape) < 0.5, x, dyadic(rs, x.shape))         # partly aligned edges
    sums, loss, grad, scale = ngf(x, y, eps, boundary, grad_loss=0.75)
    ref_loss, ref_grad = autograd(x, y, eps, boundary, 0.75)
    assert abs(loss - ref_loss) <= 1e-14
    assert np.all((sums >= 0) & (sums <= np.prod(shape)))
    # c_a is itself a difference, h_a - (a/p) g_a, which cancels by up to |g|^2/eps^2 (~1e4 at eps = 1e-2), and the
    # scale is taken over |c_a|: float64 round-off of the two orders of evaluation reaches ~3e-11 of it there
    assert np.all(np.abs(grad - ref_grad) <= 1e-9 * scale + 1e-300)
    assert np.all(ref_grad[scale == 0] == 0)


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("shape", [(4, 5, 6), (2, 7, 3)])
def test_reference_gradient_matches_central_differences(shape, boundary):
    rs = np.random.RandomState(11)
    zz, yy, xx = np.meshgrid(*[np.linspace(-1, 1, n) for n in shape], indexing="ij")
    x = (np.sin(2 * xx + yy) * np.cos(3 * zz - xx) + 0.3 * yy * zz)[None, None]
    y = (np.sin(2.2 * xx + 0.8 * yy) * np.cos(2.5 * zz) + 0.2 * xx)[None, None] + 0.05 * rs.uniform(-1, 1, x.shape)
    _, _, grad, _ = ngf(x, y, 0.5, boundary, diff_dtype=np.float64)
    h = 1e-6
    idx = [tuple(rs.randint(0, n) for n in x.shape) for _ in range(40)] + [(0, 0, 0, 0, 0), (0, 0) + tuple(n - 1 for n in shape)]
    for i in idx:
        hi, lo = x.copy(), x.copy()
        hi[i] += h
        lo[i] -= h
        fd = (ngf(hi, y, 0.5, boundary, diff_dtype=np.float64)[1] - ngf(lo, y, 0.5, boundary, diff_dtype=np.float64)[1]) / (2 * h)
        assert abs(fd - grad[i]) <= 1e-7 * max(abs(grad[i]), 1e-3), (i, fd, grad[i])


def test_constant_image_has_zero_gradient_and_unit_loss():
    rs = np.random.RandomState(2)
    y = dyadic(rs, (1, 1, 6, 7, 8))
    sums, loss, grad, scale = ngf(np.full(y.shape, 0.375), y)
    assert np.all(sums == 0) and loss == 1.0 and np.all(grad == 0) and np.all(scale == 0)


def test_ngf_loss_resolves_by_dotted_name():
    import torch.nn as nn

    def get_class(kls):                    # the reference's lookup (utils/general.py:9-15), as tests/test_dropin.py states it
        parts = kls.split('.')
        m = __import__(".".join(parts[:-1]))
        for comp in parts[1:]:
            m = getattr(m, comp)
        return m

    sys.path.insert(0, ROOT)
    cls = get_class("liftreg_b200.losses.NGFLoss")
    m = cls()                              # losses/SubspaceLoss.py:12 instantiates sim_class with no arguments
    assert isinstance(m, nn.Module) and (m.eps, m.boundary) == (1.0, "linear")
    from liftreg_b200 import losses
    assert isinstance(losses.SubspaceLoss(sim=cls(eps=0.5, boundary="neumann_zero")).sim, cls)


def test_ngf_loss_raises_value_errors_before_any_native_call():
    """CPU tensors: a check that passed would go on to the CUDA-only path and raise a RuntimeError instead"""
    from liftreg_b200 import ops
    x = torch.zeros(2, 1, 4, 5, 6)
    cases = [
        ((x, torch.zeros(2, 1, 4, 5, 7)), {}, "same shape"),
        ((x, torch.zeros(1, 1, 4, 5, 6)), {}, "same shape"),
        ((x[:, 0], x), {}, "same shape"),
        ((torch.zeros(2, 2, 4, 5, 6), torch.zeros(2, 2, 4, 5, 6)), {}, r"\(B,1,D,H,W\)"),
        ((torch.zeros(4, 5, 6), torch.zeros(4, 5, 6)), {}, r"\(B,1,D,H,W\)"),
        ((x, "target"), {}, r"\(B,1,D,H,W\)"),
        ((torch.zeros(1, 1, 1, 5, 6),) * 2, {}, ">= 2"),
        ((torch.zeros(1, 4, 5, 1),) * 2, {}, ">= 2"),
        ((x, x), {"eps": 0.0}, "eps"), ((x, x), {"eps": -1.0}, "eps"), ((x, x), {"eps": float("nan")}, "eps"),
        ((x, x), {"eps": float("inf")}, "eps"), ((x, x), {"eps": 1e-80}, "eps"),
        ((x, x), {"boundary": "mirror"}, "boundary"),
    ]
    for args, kw, msg in cases:
        with pytest.raises(ValueError, match=msg):
            ops.ngf_loss(*args, **kw)


@pytest.fixture(scope="module")
def lib():
    from liftreg_b200 import _native, build
    build.build()
    return _native.lib()


def test_ngf_c_abi_rejects_bad_arguments_before_any_cuda_call(lib):
    fake, g, out = ctypes.c_void_p(256), ctypes.c_void_p(512), ctypes.c_void_p(1024)
    nan, inf = float("nan"), float("inf")
    cases = [                                # (B, D, H, W, boundary, eps), expected message
        ((1, 4, 4, 4, 0, 0.0), b"eps"), ((1, 4, 4, 4, 0, -1.0), b"eps"), ((1, 4, 4, 4, 1, nan), b"eps"),
        ((1, 4, 4, 4, 0, inf), b"eps"), ((1, 4, 4, 4, 0, -inf), b"eps"), ((1, 4, 4, 4, 0, 1e-80), b"eps"),
        ((0, 4, 4, 4, 0, 1.0), b">= 2"), ((1, 1, 4, 4, 0, 1.0), b">= 2"), ((1, 4, 1, 4, 0, 1.0), b">= 2"),
        ((1, 4, 4, 1, 1, 1.0), b">= 2"), ((1, 4, -3, 4, 0, 1.0), b">= 2"),
        ((1, 4, 4, 4, 2, 1.0), b"boundary"), ((1, 4, 4, 4, -1, 1.0), b"boundary"),
        ((1, 1024, 1024, 2048, 0, 1.0), b"2^31"), ((2, 1024, 1024, 1024, 1, 1.0), b"2^31"),
        ((8, 2, 512, 262144, 0, 1.0), b"2^31"),
    ]
    for (B, D, H, W, bd, eps), msg in cases:
        assert lib.lr_ngf_sum(fake, fake, B, D, H, W, bd, eps, out, None) == -1, (B, D, H, W, bd, eps)
        assert msg in lib.lr_last_error(), (msg, lib.lr_last_error())
        assert lib.lr_ngf_backward(fake, fake, B, D, H, W, bd, eps, g, out, None) == -1, (B, D, H, W, bd, eps)
        assert msg in lib.lr_last_error(), (msg, lib.lr_last_error())
    nulls = [
        lambda: lib.lr_ngf_sum(None, fake, 1, 4, 4, 4, 0, 1.0, out, None),
        lambda: lib.lr_ngf_sum(fake, None, 1, 4, 4, 4, 0, 1.0, out, None),
        lambda: lib.lr_ngf_sum(fake, fake, 1, 4, 4, 4, 0, 1.0, None, None),
        lambda: lib.lr_ngf_backward(None, fake, 1, 4, 4, 4, 0, 1.0, g, out, None),
        lambda: lib.lr_ngf_backward(fake, None, 1, 4, 4, 4, 0, 1.0, g, out, None),
        lambda: lib.lr_ngf_backward(fake, fake, 1, 4, 4, 4, 0, 1.0, None, out, None),
        lambda: lib.lr_ngf_backward(fake, fake, 1, 4, 4, 4, 0, 1.0, g, None, None),
    ]
    for call in nulls:
        assert call() == -1 and b"null" in lib.lr_last_error()
