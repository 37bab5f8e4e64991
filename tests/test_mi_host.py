"""Mutual information similarity without a GPU: the float64 reference (tests/mi_reference.py) against float64 autograd
of the stock-op composition on dyadic images and against central differences; values outside the range and exactly at
its ends; the loss class by dotted name; the ValueErrors of ops.mi_loss; argument validation of the C-ABI."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

from mi_reference import chain, mi, mi_torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def dyadic(rs, shape):
    """values k/64 - 1.25 in [-1.25, 1.25]: some outside (-1, 1), some exactly at -1 and 1.  With the range (-1, 1),
    s = (nb - 1)/2 is dyadic for every nb, so u and f are exact and the fp32 and fp64 chains coincide"""
    return rs.randint(0, 161, shape) / 64.0 - 1.25


def autograd(x, y, nb, grad_loss):
    xt = torch.tensor(x, dtype=torch.float64, requires_grad=True)
    loss = mi_torch(xt, torch.tensor(y, dtype=torch.float64), nb)
    (grad_loss * loss).backward()
    return loss.item(), xt.grad.numpy()


@pytest.mark.parametrize("nb", [4, 7, 32, 64])
@pytest.mark.parametrize("shape", [(1, 1), (1, 300), (2, 1000), (3, 4, 5, 6)])
def test_reference_equals_float64_autograd(shape, nb):
    rs = np.random.RandomState(nb + sum(shape))
    x = dyadic(rs, shape)
    y = np.where(rs.uniform(size=shape) < 0.6, np.clip(x + rs.randint(-4, 5, shape) / 64.0, -1.5, 1.5), dyadic(rs, shape))
    hist, loss, grad, scale = mi(x, y, nb, grad_loss=0.75)
    N = x.size // shape[0]
    assert hist.shape == (shape[0], nb, nb + 2)
    assert np.all(np.abs(hist.sum((1, 2)) - N) <= 1e-12 * N)             # the tap weights sum to 1 per voxel
    assert np.all(hist >= 0)
    ref_loss, ref_grad = autograd(x, y, nb, 0.75)
    assert abs(loss - ref_loss) <= 1e-13
    assert loss <= 1e-15                                                     # MI >= 0
    # autograd also carries the terms that cancel analytically (sum_m w_m' = 0, p_y): float64 round-off of those
    assert np.all(np.abs(grad - ref_grad) <= 1e-9 * scale + 1e-13 * scale.max() + 1e-14)
    outside = (x < -1) | (x > 1)
    assert (outside.any() or x.size == 1) and np.all(grad[outside] == 0) and np.all(scale[outside] == 0)
    assert np.all(ref_grad[outside] == 0)


@pytest.mark.parametrize("nb", [4, 32])
def test_reference_gradient_matches_central_differences(nb):
    rs = np.random.RandomState(5)
    x = rs.uniform(-0.95, 0.95, (2, 150))
    y = np.clip(0.7 * x + 0.2 * np.sin(4 * x) + 0.1 * rs.uniform(-1, 1, x.shape), -1, 1)
    _, _, grad, _ = mi(x, y, nb, chain_dtype=np.float64)
    h = 1e-6
    for i in [tuple(rs.randint(0, n) for n in x.shape) for _ in range(40)]:
        hi, lo = x.copy(), x.copy()
        hi[i] += h
        lo[i] -= h
        fd = (mi(hi, y, nb, chain_dtype=np.float64)[1] - mi(lo, y, nb, chain_dtype=np.float64)[1]) / (2 * h)
        assert abs(fd - grad[i]) <= 1e-6 * np.abs(grad).max(), (i, fd, grad[i])


def test_range_ends_and_nonfinite_values_map_into_the_histogram():
    nb = 32
    x = np.array([[-1.0, 1.0, -7.0, 7.0, np.nan, np.inf, -np.inf, 0.0]], np.float32)
    ux, iota, k0, f = chain(x, x, nb, -1.0, 1.0)
    assert list(iota[0]) == [0, 31, 0, 31, 0, 31, 0, 16]
    assert list(k0[0]) == [0, 30, 0, 30, 0, 30, 0, 15] and list(f[0]) == [0, 1, 0, 1, 0, 1, 0, 0.5]
    hist, loss, grad, scale = mi(x, x, nb)
    assert np.isfinite(loss) and np.all(np.isfinite(grad)) and abs(hist.sum() - x.size) <= 1e-12
    assert np.all(grad[0, 2:7] == 0)                                         # outside [lo, hi] and NaN: no gradient


def test_constant_target_has_zero_gradient_and_zero_mi():
    rs = np.random.RandomState(3)
    x = rs.uniform(-1.2, 1.2, (2, 500))
    for v in (-1.0, 0.3, 1.0):
        hist, loss, grad, scale = mi(x, np.full(x.shape, v), 32)
        assert loss == 0.0 and np.all(grad == 0) and np.all(scale == 0)


def test_non_default_range():
    """a range whose s is not dyadic: the reference still agrees with float64 autograd up to the fp32 chain"""
    rs = np.random.RandomState(8)
    x = rs.uniform(-1100, 100, (1, 2000)).astype(np.float32)
    y = np.clip(x + rs.normal(0, 30, x.shape), -1100, 100).astype(np.float32)
    _, loss, grad, scale = mi(x, y, 24, (-1000.0, 0.0))
    ref_loss = mi_torch(torch.tensor(x, dtype=torch.float64), torch.tensor(y, dtype=torch.float64), 24, (-1000.0, 0.0)).item()
    assert abs(loss - ref_loss) <= 1e-5
    assert np.all(np.isfinite(grad)) and np.all(grad[(x < -1000) | (x > 0)] == 0)


def test_mi_loss_resolves_by_dotted_name():
    import torch.nn as nn

    def get_class(kls):                    # the reference's lookup (utils/general.py:9-15), as tests/test_dropin.py states it
        parts = kls.split('.')
        m = __import__(".".join(parts[:-1]))
        for comp in parts[1:]:
            m = getattr(m, comp)
        return m

    sys.path.insert(0, ROOT)
    cls = get_class("liftreg_b200.losses.MILoss")
    m = cls()                              # losses/SubspaceLoss.py:12 instantiates sim_class with no arguments
    assert isinstance(m, nn.Module) and (m.num_bins, m.value_range) == (32, (-1.0, 1.0))
    from liftreg_b200 import losses
    assert isinstance(losses.SubspaceLoss(sim=cls(num_bins=16, value_range=(-2, 2))).sim, cls)


def test_mi_loss_raises_value_errors_before_any_native_call():
    """CPU tensors: a check that passed would go on to the CUDA-only path and raise a RuntimeError instead"""
    from liftreg_b200 import ops
    x = torch.zeros(2, 1, 4, 5, 6)
    cases = [
        ((x, torch.zeros(2, 1, 4, 5, 7)), {}, "same shape"),
        ((x, torch.zeros(1, 1, 4, 5, 6)), {}, "same shape"),
        ((x, "target"), {}, "non-empty"),
        ((torch.zeros(()), torch.zeros(())), {}, "non-empty"),
        ((torch.zeros(2, 0), torch.zeros(2, 0)), {}, "non-empty"),
        ((torch.zeros(65536, 1), torch.zeros(65536, 1)), {}, "65535"),
        ((x, x), {"num_bins": 3}, "num_bins"), ((x, x), {"num_bins": 65}, "num_bins"),
        ((x, x), {"num_bins": 32.5}, "num_bins"), ((x, x), {"num_bins": True}, "num_bins"),
        ((x, x), {"value_range": (1.0, -1.0)}, "value_range"), ((x, x), {"value_range": (1.0, 1.0)}, "value_range"),
        ((x, x), {"value_range": (float("nan"), 1.0)}, "value_range"),
        ((x, x), {"value_range": (-1.0, float("inf"))}, "value_range"),
        ((x, x), {"value_range": (-1.0, 1e39)}, "value_range"),
        ((x, x), {"value_range": (0.0, 1e-44)}, "value_range"),
        ((x, x), {"value_range": (1.0,)}, "value_range"), ((x, x), {"value_range": "ab"}, "value_range"),
    ]
    for args, kw, msg in cases:
        with pytest.raises(ValueError, match=msg):
            ops.mi_loss(*args, **kw)


@pytest.fixture(scope="module")
def lib():
    from liftreg_b200 import _native, build
    build.build()
    return _native.lib()


def test_mi_c_abi_rejects_bad_arguments_before_any_cuda_call(lib):
    fake, g, out = ctypes.c_void_p(256), ctypes.c_void_p(512), ctypes.c_void_p(1024)
    nan, inf = float("nan"), float("inf")
    cases = [                                # (B, N, nb, lo, hi), expected message
        ((0, 64, 32, -1.0, 1.0), b"bad size"), ((65536, 64, 32, -1.0, 1.0), b"bad size"), ((1, 0, 32, -1.0, 1.0), b"bad size"),
        ((1, -5, 32, -1.0, 1.0), b"bad size"), ((1, 64, 3, -1.0, 1.0), b"num_bins"), ((1, 64, 65, -1.0, 1.0), b"num_bins"),
        ((1, 64, 32, 1.0, -1.0), b"range"), ((1, 64, 32, 1.0, 1.0), b"range"), ((1, 64, 32, nan, 1.0), b"range"),
        ((1, 64, 32, -1.0, nan), b"range"), ((1, 64, 32, -inf, 1.0), b"range"), ((1, 64, 32, -1.0, inf), b"range"),
        ((1, 64, 64, 0.0, 1e-44), b"finite positive"),
    ]
    for (B, N, nb, lo, hi), msg in cases:
        assert lib.lr_mi_hist(fake, fake, B, N, nb, lo, hi, out, None) == -1, (B, N, nb, lo, hi)
        assert msg in lib.lr_last_error(), (msg, lib.lr_last_error())
        assert lib.lr_mi_backward(fake, fake, B, N, nb, lo, hi, out, g, out, None) == -1, (B, N, nb, lo, hi)
        assert msg in lib.lr_last_error(), (msg, lib.lr_last_error())
    nulls = [
        lambda: lib.lr_mi_hist(None, fake, 1, 64, 32, -1.0, 1.0, out, None),
        lambda: lib.lr_mi_hist(fake, None, 1, 64, 32, -1.0, 1.0, out, None),
        lambda: lib.lr_mi_hist(fake, fake, 1, 64, 32, -1.0, 1.0, None, None),
        lambda: lib.lr_mi_backward(None, fake, 1, 64, 32, -1.0, 1.0, out, g, out, None),
        lambda: lib.lr_mi_backward(fake, None, 1, 64, 32, -1.0, 1.0, out, g, out, None),
        lambda: lib.lr_mi_backward(fake, fake, 1, 64, 32, -1.0, 1.0, None, g, out, None),
        lambda: lib.lr_mi_backward(fake, fake, 1, 64, 32, -1.0, 1.0, out, None, out, None),
        lambda: lib.lr_mi_backward(fake, fake, 1, 64, 32, -1.0, 1.0, out, g, None, None),
    ]
    for call in nulls:
        assert call() == -1 and b"null" in lib.lr_last_error()
