"""Validation metrics without a GPU: the torch restatement of the Jacobian determinant (the kernel's reference), the
overlap formulas of liftreg_b200.metrics, and argument validation of the two C-ABI entries."""
import ctypes

import numpy as np
import pytest
import torch

from metrics_reference import jacobian_det, overlap_by_sets
from oracle import torch_port


def identity64(shape):
    return np.stack(np.meshgrid(*[np.linspace(-1.0, 1.0, n) for n in shape], indexing="ij"))


def det_np_gradient(phi):
    """Independent statement: np.gradient (edge_order=1, spacing 2/(n-1)) of each channel, 3x3 determinant by numpy."""
    B = phi.shape[0]
    h = [2.0 / (n - 1) for n in phi.shape[2:]]
    out = np.empty((B,) + phi.shape[2:])
    for b in range(B):
        J = np.stack([np.stack(np.gradient(phi[b, c], *h, edge_order=1)) for c in range(3)])     # (c, a, D, H, W)
        out[b] = np.linalg.det(np.moveaxis(J, (0, 1), (-2, -1)))
    return out


@pytest.mark.parametrize("shape", [(5, 6, 7), (2, 2, 2), (9, 3, 12)])
def test_port_linear_mode_matches_np_gradient_determinant(shape):
    rs = np.random.RandomState(3)
    phi = identity64(shape)[None] + 0.3 * rs.standard_normal((2, 3) + shape) * (2.0 / (np.array(shape) - 1)).reshape(1, 3, 1, 1, 1)
    got = jacobian_det(torch.from_numpy(phi), "linear").numpy()
    assert np.abs(got - det_np_gradient(phi)).max() <= 1e-12


def test_port_affine_map_has_the_matrix_determinant_everywhere():
    shape = (6, 7, 9)
    A = np.array([[1.2, 0.3, -0.1], [0.05, 0.8, 0.2], [-0.4, 0.1, 1.1]])
    x = identity64(shape)
    phi = (np.einsum("ij,jdhw->idhw", A, x) + np.array([0.1, -0.2, 0.05]).reshape(3, 1, 1, 1))[None]
    got = jacobian_det(torch.from_numpy(phi), "linear").numpy()
    assert np.abs(got - np.linalg.det(A)).max() <= 1e-12
    # neumann_zero: the interior is still det(A), every face voxel has a zero row
    nz = jacobian_det(torch.from_numpy(phi), "neumann_zero").numpy()[0]
    assert np.abs(nz[1:-1, 1:-1, 1:-1] - np.linalg.det(A)).max() <= 1e-12
    face = np.ones(shape, bool)
    face[1:-1, 1:-1, 1:-1] = False
    assert np.all(nz[face] == 0.0)


def test_port_identity_map_fp32():
    shape = (17, 10, 33)
    idm = torch_port.identity_map(shape)[None]            # float32, the reference's identity_map
    lin = jacobian_det(idm, "linear").numpy()[0]
    assert lin.dtype == np.float32 and np.abs(lin - 1.0).max() <= 1e-5
    nz = jacobian_det(idm, "neumann_zero").numpy()[0]
    assert np.abs(nz[1:-1, 1:-1, 1:-1] - 1.0).max() <= 1e-5
    assert np.all(nz[[0, -1]] == 0) and np.all(nz[:, [0, -1]] == 0) and np.all(nz[:, :, [0, -1]] == 0)


def folded_map(shape):
    """Identity with the last channel following g = 0,2,4,6,8,7,6,5,... along the last axis: the central difference
    is positive for x <= 4 and negative for x >= 5 (faces included in linear mode)."""
    D, H, W = shape
    phi = identity64(shape)
    g = np.array([2.0 * i if i < 5 else 12.0 - i for i in range(W)]) * (2.0 / (W - 1))
    phi[2] = g.reshape(1, 1, W)
    return phi[None]


def test_port_constructed_fold_has_the_expected_sign_pattern():
    shape = (4, 5, 12)
    det = jacobian_det(torch.from_numpy(folded_map(shape)), "linear").numpy()[0]
    assert np.all(det[:, :, 5:] < 0) and np.all(det[:, :, :5] > 0)
    assert int((det < 0).sum()) == 7 * 4 * 5


def test_overlap_formulas_match_python_sets_on_host_counts():
    from liftreg_b200 import metrics
    rs = np.random.RandomState(5)
    L = 6
    p = rs.randint(0, 4, size=(2, 300))          # labels 4 and 5 absent from pred; 5 absent from both
    t = rs.randint(0, 5, size=(2, 300))
    counts = np.stack([np.bincount(p[b] * L + t[b], minlength=L * L).reshape(L, L) for b in range(2)])
    for ignore_bg in (False, True):
        res = metrics._overlap(counts, ignore_bg)
        for b in range(2):
            ref = overlap_by_sets(p[b], t[b], L)
            for k, v in ref.items():
                if ignore_bg:
                    v[0] = np.nan
                assert np.array_equal(res[k][b], v, equal_nan=True), k
                assert res[k + "_mean"][b] == pytest.approx(np.nanmean(v), rel=1e-15)
        assert np.isnan(res["dice"][:, 5]).all() and (res["dice"][:, 4] == 0).all()


@pytest.fixture(scope="module")
def lib():
    from liftreg_b200 import _native, build
    build.build()
    return _native.lib()


def test_validation_metric_entries_reject_bad_arguments_before_any_cuda_call(lib):
    fake = ctypes.c_void_p(256)          # never dereferenced: every call below fails validation first
    stats = ctypes.c_void_p(512)
    cases = [
        (lib.lr_jacobian_det, (None, 1, 4, 4, 4, 0, 0, None, stats, None), b"null"),
        (lib.lr_jacobian_det, (fake, 1, 4, 4, 4, 0, 0, None, None, None), b"null"),
        (lib.lr_jacobian_det, (fake, 1, 1, 4, 4, 0, 0, None, stats, None), b">= 2"),
        (lib.lr_jacobian_det, (fake, 1, 4, 4, 4, 2, 0, None, stats, None), b"boundary"),
        (lib.lr_jacobian_det, (fake, 1, 4, 9, 9, 0, 2, None, stats, None), b"margin"),
        (lib.lr_jacobian_det, (fake, 1, 9, 9, 9, 0, -1, None, stats, None), b"margin"),
        (lib.lr_jacobian_det, (fake, 1, 1024, 1024, 1024, 0, 0, None, stats, None), b"2^31"),
        (lib.lr_jacobian_det, (fake, 1, 1024, 1024, 1024, 0, 600, None, stats, None), b"margin"),   # margin first
        (lib.lr_label_confusion, (None, fake, 1, 10, 2, stats, stats, None), b"null"),
        (lib.lr_label_confusion, (fake, fake, 1, 10, 2, None, stats, None), b"null"),
        (lib.lr_label_confusion, (fake, fake, 1, 10, 0, stats, stats, None), b"[1, 128]"),
        (lib.lr_label_confusion, (fake, fake, 1, 10, 129, stats, stats, None), b"[1, 128]"),
        (lib.lr_label_confusion, (fake, fake, 1, 0, 2, stats, stats, None), b"bad size"),
        (lib.lr_label_confusion, (fake, fake, 0, 10, 2, stats, stats, None), b"bad size"),
    ]
    for fn, args, msg in cases:
        assert fn(*args) == -1, args
        assert msg in lib.lr_last_error(), (args, lib.lr_last_error())
