"""Folding penalty without a GPU: the float64 gradient references against autograd and central differences, the
penalty on the identity, planted folds and a reflected affine map, the SubspaceLoss opt key, and argument validation of
lr_jacobian_fold_backward through the C-ABI."""
import ctypes

import numpy as np
import pytest
import torch

from fold_reference import REFLECTED_A, fold_grad, fold_grad_autograd, fold_mask, fold_value, reflected_affine
from metrics_reference import jacobian_det
from oracle import torch_port

BOUNDARIES = ["linear", "neumann_zero"]


def identity64(shape):
    return np.stack(np.meshgrid(*[np.linspace(-1.0, 1.0, n) for n in shape], indexing="ij"))


def noisy_map(B, shape, seed, amp=0.6):
    """fp32 identity + uniform noise of `amp` grid steps: a share of the voxels fold"""
    rs = np.random.RandomState(seed)
    step = (2.0 / (np.array(shape) - 1)).reshape(1, 3, 1, 1, 1)
    return (torch_port.identity_map(shape).numpy()[None] + amp * step * rs.uniform(-1, 1, (B, 3) + shape)).astype(np.float32)


def planted_folds(shape):
    """identity with the last channel following 0,2,4,6,8,7,6,5,... grid steps along the last axis: every voxel with
    x >= 5 folds (linear mode, faces included), the others have det >= 1"""
    D, H, W = shape
    phi = identity64(shape)
    phi[2] = (np.array([2.0 * i if i < 5 else 12.0 - i for i in range(W)]) * (2.0 / (W - 1))).reshape(1, 1, W)
    return phi[None].astype(np.float32)


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("B,shape", [(2, (5, 6, 7)), (1, (2, 2, 2)), (1, (9, 3, 12)), (2, (4, 7, 2))])
def test_explicit_gradient_equals_float64_autograd(B, shape, boundary):
    phi = noisy_map(B, shape, seed=sum(shape))
    if boundary == "linear" and min(shape) > 2:
        assert fold_mask(phi, boundary).any()
    auto = fold_grad_autograd(phi, boundary, grad_loss=0.75)
    grad, scale = fold_grad(phi, boundary, grad_loss=0.75, j_dtype=np.float64)
    assert np.all(np.abs(grad - auto) <= 1e-13 * scale)
    assert np.all(grad[scale == 0] == 0) and np.all(auto[scale == 0] == 0)
    # the kernel's fp32 J moves the value by a few u of the scale (the linear face extrapolation is rounded in fp32)
    g32, s32 = fold_grad(phi, boundary, grad_loss=0.75)
    assert np.array_equal(s32 == 0, scale == 0)
    assert np.all(np.abs(g32 - grad) <= 1e-4 * scale)


@pytest.mark.parametrize("boundary", BOUNDARIES)
def test_autograd_reference_matches_central_differences(boundary):
    """planted folds plus noise, on a map whose |det| stays away from 0, so no step of the differences crosses the kink"""
    rs = np.random.RandomState(17)
    shape = (5, 6, 12)
    phi = planted_folds(shape) + (0.05 * (2.0 / 11) * rs.uniform(-1, 1, (1, 3) + shape)).astype(np.float32)
    det = jacobian_det(torch.from_numpy(phi.astype(np.float64)), boundary).numpy()
    nz = det[det != 0] if boundary == "neumann_zero" else det                   # neumann_zero: det = 0 on the faces exactly
    assert np.abs(nz).min() > 0.05 and fold_mask(phi, boundary).sum() > 20
    auto = fold_grad_autograd(phi, boundary)

    def penalty(p):
        d = jacobian_det(torch.from_numpy(p), boundary).numpy()
        return float(np.where(np.isfinite(d) & (d < 0), -d, 0.0).sum() / d.size)

    p64 = phi.astype(np.float64)
    eps = 1e-6
    idx = [tuple(rs.randint(0, n) for n in p64.shape) for _ in range(60)] + [(0, 2, 0, 0, 11), (0, 2, 4, 5, 10), (0, 0, 0, 0, 0)]
    for i in idx:
        hi, lo = p64.copy(), p64.copy()
        hi[i] += eps
        lo[i] -= eps
        fd = (penalty(hi) - penalty(lo)) / (2 * eps)
        assert abs(fd - auto[i]) <= 1e-7 * max(1.0, abs(auto[i])), (i, fd, auto[i])
    assert penalty(p64) == pytest.approx(fold_value(phi, boundary), rel=1e-15)


@pytest.mark.parametrize("boundary", BOUNDARIES)
def test_identity_is_free_and_every_planted_fold_counts(boundary):
    idm = torch_port.identity_map((17, 10, 33)).numpy()[None]
    assert not fold_mask(idm, boundary).any() and fold_value(idm, boundary) == 0.0
    grad, scale = fold_grad(idm, boundary)
    assert np.all(grad == 0) and np.all(scale == 0)
    shape = (4, 5, 12)
    phi = planted_folds(shape)
    m = fold_mask(phi, boundary)
    det = jacobian_det(torch.from_numpy(phi.astype(np.float64)), boundary).numpy()
    planted = np.zeros_like(m)
    if boundary == "linear":
        planted[..., 5:] = True
    else:                                                                      # faces are never folds: det = 0 there
        planted[:, 1:-1, 1:-1, 5:-1] = True
    assert np.array_equal(m, planted)
    assert fold_value(phi, boundary) == pytest.approx(-det[planted].sum() / det.size, rel=1e-15)


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("shape", [(9, 8, 11), (6, 7, 5)])
def test_reflected_affine_map_has_gradient_only_in_the_two_outer_layers(shape, boundary):
    phi = reflected_affine(shape)
    m = fold_mask(phi, boundary)
    inner = np.zeros(shape, bool)
    inner[1:-1, 1:-1, 1:-1] = True
    assert m[0][inner].all() and (m.all() if boundary == "linear" else not m[0][~inner].any())
    grad, scale = fold_grad(phi, boundary)
    core = np.zeros(shape, bool)
    core[2:-2, 2:-2, 2:-2] = True
    assert np.all(grad[:, :, core] == 0)                      # D_a^T of a constant vanishes more than one layer from a face
    assert np.all(scale[:, :, core] > 0)
    for c in range(3):                                        # ... and is not zero on the outer layers of each axis
        for a in range(3):
            for layer in (0, 1, shape[a] - 2, shape[a] - 1):
                sl = np.take(grad[0, c], layer, axis=a)
                if abs(reflected_affine_cofactor(c, a)) > 1e-12:
                    assert np.any(sl != 0), (c, a, layer)


def reflected_affine_cofactor(c, a):
    A = -REFLECTED_A
    return np.linalg.det(A) * np.linalg.inv(A).T[c, a]


def test_subspace_loss_reads_fold_factor():
    from liftreg_b200 import losses
    assert losses.SubspaceLoss().fold_factor == 0
    assert losses.SubspaceLoss({"fold_factor": 0.5}).fold_factor == 0.5


@pytest.fixture(scope="module")
def lib():
    from liftreg_b200 import _native, build
    build.build()
    return _native.lib()


def test_fold_backward_rejects_bad_arguments_before_any_cuda_call(lib):
    fake = ctypes.c_void_p(256)          # never dereferenced: every call below fails validation first
    g = ctypes.c_void_p(512)
    out = ctypes.c_void_p(1024)
    cases = [
        ((None, 1, 4, 4, 4, 0, g, out, None), b"null"),
        ((fake, 1, 4, 4, 4, 0, None, out, None), b"null"),
        ((fake, 1, 4, 4, 4, 0, g, None, None), b"null"),
        ((fake, 0, 4, 4, 4, 0, g, out, None), b">= 2"),
        ((fake, 1, 1, 4, 4, 0, g, out, None), b">= 2"),
        ((fake, 1, 4, 4, 1, 1, g, out, None), b">= 2"),
        ((fake, 1, 4, 4, 4, 2, g, out, None), b"boundary"),
        ((fake, 1, 4, 4, 4, -1, g, out, None), b"boundary"),
        ((fake, 1, 1024, 1024, 1024, 0, g, out, None), b"2^31"),
        ((fake, 3, 512, 512, 1024, 1, g, out, None), b"2^31"),
    ]
    for args, msg in cases:
        assert lib.lr_jacobian_fold_backward(*args) == -1, args
        assert msg in lib.lr_last_error(), (args, lib.lr_last_error())


def test_diffusion_reg_rejects_bad_arguments_before_any_cuda_call(lib):
    fake = ctypes.c_void_p(256)          # never dereferenced: every call below fails validation first
    g = ctypes.c_void_p(512)
    out = ctypes.c_void_p(1024)
    cases = [
        (lib.lr_diffusion_reg_sum, (None, 1, 4, 4, 4, 0, out, None), b"null"),
        (lib.lr_diffusion_reg_sum, (fake, 1, 4, 4, 4, 0, None, None), b"null"),
        (lib.lr_diffusion_reg_backward, (None, 1, 4, 4, 4, 0, g, out, None), b"null"),
        (lib.lr_diffusion_reg_backward, (fake, 1, 4, 4, 4, 0, None, out, None), b"null"),
        (lib.lr_diffusion_reg_backward, (fake, 1, 4, 4, 4, 0, g, None, None), b"null"),
    ]
    # (B, D, H, W, boundary): the rules both entries share
    for dims, msg in [((0, 4, 4, 4, 0), b">= 2"),
                      ((1, 1, 4, 4, 0), b">= 2"),
                      ((1, 4, 4, 1, 1), b">= 2"),
                      ((1, 4, 4, 4, 2), b"boundary"),
                      ((1, 4, 4, 4, -1), b"boundary"),
                      ((1, 1024, 1024, 1024, 0), b"2^31"),
                      ((3, 512, 512, 1024, 1), b"2^31")]:
        cases.append((lib.lr_diffusion_reg_sum, (fake, *dims, out, None), msg))
        cases.append((lib.lr_diffusion_reg_backward, (fake, *dims, g, out, None), msg))
    for fn, args, msg in cases:
        assert fn(*args) == -1, (fn.__name__, args)
        assert msg in lib.lr_last_error(), (fn.__name__, args, lib.lr_last_error())
