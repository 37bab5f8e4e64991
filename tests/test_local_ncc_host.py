"""Local NCC without a GPU: the float64 reference (tests/lncc_reference.py) against a float64 torch restatement of
VoxelMorph's conv3d NCC (value and autograd gradient) and against central differences; windows larger than an axis;
constant images, x == y and shift invariance; argument validation of the C-ABI; the loss class by dotted name."""
import ctypes
import os
import sys

import numpy as np
import pytest
import torch

from lncc_reference import inside_mask, local_ncc, voxelmorph_ncc_torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def voxelmorph(x, y, w, eps, grad_loss=1.0):
    """float64 torch conv3d form: (loss, cc, d loss / d x)"""
    xt = torch.tensor(np.asarray(x, np.float64), requires_grad=True)
    loss, cc = voxelmorph_ncc_torch(xt, torch.tensor(np.asarray(y, np.float64)), w, eps)
    (grad_loss * loss).backward()
    return loss.item(), cc.detach().numpy()[:, 0], xt.grad.numpy()


@pytest.mark.parametrize("B,shape,w", [(2, (7, 9, 11), 5), (1, (12, 10, 14), 9), (1, (5, 40, 7), 9), (2, (1, 6, 5), 3),
                                       (1, (4, 3, 6), 15), (1, (16, 17, 18), 15)])
def test_reference_equals_voxelmorph_conv3d_form(B, shape, w):
    rs = np.random.RandomState(sum(shape) + w)
    x = rs.uniform(-1, 1, (B, 1) + shape)
    y = 0.5 * x + rs.uniform(-1, 1, x.shape)
    cc, loss, grad, scale = local_ncc(x, y, w, 1e-5, grad_loss=0.75)
    vl, vcc, vg = voxelmorph(x, y, w, 1e-5, grad_loss=0.75)
    assert abs(loss - vl) <= 1e-14
    assert np.all(np.abs(cc - vcc) <= 1e-12)
    assert np.all(np.abs(grad - vg) <= 1e-10 * scale + 1e-18)


@pytest.mark.parametrize("shape,w", [((4, 5, 6), 3), ((3, 7, 2), 5), ((6, 2, 9), 9)])
def test_reference_gradient_matches_central_differences(shape, w):
    rs = np.random.RandomState(3)
    x = rs.uniform(-1, 1, (1, 1) + shape)
    y = 0.3 * x + rs.uniform(-1, 1, x.shape)
    _, loss0, grad, _ = local_ncc(x, y, w, 1e-3)
    h = 1e-6
    for i in [tuple(rs.randint(0, n) for n in x.shape) for _ in range(40)] + [(0, 0, 0, 0, 0), (0, 0) + tuple(n - 1 for n in shape)]:
        hi, lo = x.copy(), x.copy()
        hi[i] += h
        lo[i] -= h
        fd = (local_ncc(hi, y, w, 1e-3)[1] - local_ncc(lo, y, w, 1e-3)[1]) / (2 * h)
        assert abs(fd - grad[i]) <= 1e-7 * max(abs(grad[i]), 1e-3), (i, fd, grad[i])


def test_window_larger_than_every_axis():
    """w = 9 on a 3 x 2 x 4 volume: every window holds the whole volume plus padding, n stays w^3"""
    rs = np.random.RandomState(8)
    x, y = rs.uniform(-1, 1, (1, 1, 3, 2, 4)), rs.uniform(-1, 1, (1, 1, 3, 2, 4))
    cc, loss, grad, _ = local_ncc(x, y, 9, 1e-5)
    n = 9.0 ** 3
    Sx, Sy = x.sum(), y.sum()
    cross = (x * y).sum() - Sx * Sy / n
    vx, vy = (x * x).sum() - Sx * Sx / n, (y * y).sum() - Sy * Sy / n
    assert np.allclose(cc, cross ** 2 / (vx * vy + 1e-5), rtol=1e-13, atol=0)
    vl, _, vg = voxelmorph(x, y, 9, 1e-5)
    assert abs(loss - vl) <= 1e-14 and np.allclose(grad, vg, rtol=1e-10, atol=1e-16)


def dyadic(rs, shape):
    return rs.randint(0, 16, shape) / 8.0 - 1.0


@pytest.mark.parametrize("w", [3, 5, 9])
def test_constant_image_has_zero_cc_and_exactly_zero_gradient(w):
    """x constant: cc = 0 wherever the window lies inside the volume, and the gradient is exactly 0 wherever every
    centre of N(v) does (on dyadic data every sum is exact).  x = 0 is constant in the zero padding too: cc = 0 and the
    gradient is 0 everywhere."""
    rs = np.random.RandomState(w)
    shape = (3 * w, 3 * w + 1, 3 * w + 2)
    y = dyadic(rs, (1, 1) + shape)
    for c in (0.625, -1.0):
        x = np.full(y.shape, c)
        cc, _, grad, _ = local_ncc(x, y, w, 1e-5)
        r = w // 2
        assert np.all(cc[0][inside_mask(shape, r)] == 0) and np.any(cc[0] != 0)      # the faces see the zero padding
        assert np.all(grad[0, 0][inside_mask(shape, 2 * r)] == 0) and np.any(grad != 0)
    cc, loss, grad, scale = local_ncc(np.zeros(y.shape), y, w, 1e-5)
    assert np.all(cc == 0) and loss == 1.0 and np.all(grad == 0) and np.all(scale == 0)
    cc, _, grad, _ = local_ncc(np.zeros(y.shape), y, w, 0.0)                          # zero variance and eps = 0: cc = 0
    assert np.all(cc == 0) and np.all(grad == 0)


@pytest.mark.parametrize("w", [3, 9])
def test_identical_images(w):
    rs = np.random.RandomState(4)
    x = rs.uniform(-1, 1, (2, 1, 11, 12, 13))
    eps = 1e-3
    cc, _, _, _ = local_ncc(x, x, w, eps)
    n = float(w) ** 3
    from lncc_reference import box_sum
    Sx, Sxx = box_sum(x[:, 0], w), box_sum(x[:, 0] ** 2, w)
    var = Sxx - Sx * Sx / n
    assert np.allclose(cc, var ** 2 / (var ** 2 + eps), rtol=1e-12, atol=0)
    assert np.all(cc < 1)


def test_shift_invariance_inside_but_not_at_the_faces():
    """x -> x + b leaves cc unchanged where the whole window lies inside the volume; at the faces the zero padding is
    not shifted, so cc changes"""
    rs = np.random.RandomState(6)
    shape, w = (15, 16, 17), 5
    x, y = rs.uniform(-1, 1, (1, 1) + shape), rs.uniform(-1, 1, (1, 1) + shape)
    cc0 = local_ncc(x, y, w)[0][0]
    cc1 = local_ncc(x + 0.75, y, w)[0][0]
    inside = inside_mask(shape, w // 2)
    assert np.allclose(cc1[inside], cc0[inside], rtol=1e-9, atol=1e-12)
    face = ~inside
    assert np.all(np.abs(cc1[face] - cc0[face]) > 1e-6 * np.abs(cc0[face]))
    assert np.all(np.abs(cc1[face] - cc0[face]) > 1e-9)


def test_local_ncc_loss_resolves_by_dotted_name():
    import torch.nn as nn

    def get_class(kls):                    # the reference's lookup (utils/general.py:9-15), as tests/test_dropin.py states it
        parts = kls.split('.')
        m = __import__(".".join(parts[:-1]))
        for comp in parts[1:]:
            m = getattr(m, comp)
        return m

    sys.path.insert(0, ROOT)
    cls = get_class("liftreg_b200.losses.LocalNCCLoss")
    m = cls()
    assert isinstance(m, nn.Module) and (m.window, m.eps) == (9, 1e-5)
    from liftreg_b200 import losses
    assert isinstance(losses.SubspaceLoss(sim=cls(window=5)).sim, cls)


@pytest.fixture(scope="module")
def lib():
    from liftreg_b200 import _native, build
    build.build()
    return _native.lib()


def test_local_ncc_rejects_bad_arguments_before_any_cuda_call(lib):
    fake, g, out, ws = ctypes.c_void_p(256), ctypes.c_void_p(512), ctypes.c_void_p(1024), ctypes.c_void_p(2048)
    nan, inf = float("nan"), float("inf")
    big = 12 * 64 ** 3
    cases = [                                # (B, D, H, W, win, eps), expected message
        ((1, 4, 4, 4, 8, 1e-5), b"odd"), ((1, 4, 4, 4, 1, 1e-5), b"odd"), ((1, 4, 4, 4, 17, 1e-5), b"odd"),
        ((1, 4, 4, 4, -3, 1e-5), b"odd"), ((1, 4, 4, 4, 0, 1e-5), b"odd"),
        ((1, 4, 4, 4, 9, -1e-5), b"eps"), ((1, 4, 4, 4, 9, nan), b"eps"), ((1, 4, 4, 4, 9, inf), b"eps"),
        ((0, 4, 4, 4, 9, 1e-5), b">= 1"), ((1, 0, 4, 4, 9, 1e-5), b">= 1"), ((1, 4, -2, 4, 9, 1e-5), b">= 1"),
        ((1, 4, 4, 0, 9, 1e-5), b">= 1"),
        ((1, 1024, 1024, 2048, 9, 1e-5), b"2^31"), ((2, 1024, 1024, 1024, 9, 1e-5), b"2^31"),
        ((8, 1, 512, 524288, 3, 0.0), b"2^31"),
        ((1, 1, 1, 2 ** 30 + 1, 3, 1e-5), b"2^30"), ((1, 2 ** 31 - 1, 1, 1, 3, 1e-5), b"2^30"),
    ]
    for (B, D, H, W, win, eps), msg in cases:
        assert lib.lr_local_ncc_sum(fake, fake, B, D, H, W, win, eps, out, None) == -1, (B, D, H, W, win, eps)
        assert msg in lib.lr_last_error(), (msg, lib.lr_last_error())
        assert lib.lr_local_ncc_backward(fake, fake, B, D, H, W, win, eps, g, out, ws, big, None) == -1
        assert msg in lib.lr_last_error(), (msg, lib.lr_last_error())
        if msg != b"eps":
            assert lib.lr_local_ncc_workspace_bytes(B, D, H, W, win) == 0
    assert lib.lr_local_ncc_workspace_bytes(1, 1, 2, 2 ** 30 - 1, 3) == 12 * (2 ** 31 - 2)      # near the largest volume
    assert lib.lr_local_ncc_workspace_bytes(2, 64, 64, 64, 15) == 12 * 2 * 64 ** 3
    nulls = [
        lambda: lib.lr_local_ncc_sum(None, fake, 1, 4, 4, 4, 3, 1e-5, out, None),
        lambda: lib.lr_local_ncc_sum(fake, None, 1, 4, 4, 4, 3, 1e-5, out, None),
        lambda: lib.lr_local_ncc_sum(fake, fake, 1, 4, 4, 4, 3, 1e-5, None, None),
        lambda: lib.lr_local_ncc_backward(None, fake, 1, 4, 4, 4, 3, 1e-5, g, out, ws, big, None),
        lambda: lib.lr_local_ncc_backward(fake, None, 1, 4, 4, 4, 3, 1e-5, g, out, ws, big, None),
        lambda: lib.lr_local_ncc_backward(fake, fake, 1, 4, 4, 4, 3, 1e-5, None, out, ws, big, None),
        lambda: lib.lr_local_ncc_backward(fake, fake, 1, 4, 4, 4, 3, 1e-5, g, None, ws, big, None),
        lambda: lib.lr_local_ncc_backward(fake, fake, 1, 4, 4, 4, 3, 1e-5, g, out, None, big, None),
    ]
    for call in nulls:
        assert call() == -1 and b"null" in lib.lr_last_error()
    assert lib.lr_local_ncc_backward(fake, fake, 1, 4, 4, 4, 3, 1e-5, g, out, ws, 12 * 64 - 1, None) == -1
    assert b"workspace" in lib.lr_last_error()
