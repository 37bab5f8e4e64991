"""Folding penalty on the GPU: lr_jacobian_fold_backward element by element against the float64 reference
(tests/fold_reference.py) on the row g shapes, partial tiles, size-2 axes and an unaligned view; the forward value
against the Jacobian statistics; NaN handling; autograd; and the opt-in term of SubspaceLoss."""
import ctypes

import numpy as np
import pytest
import torch

from fold_reference import fold_grad, reflected_affine
from liftreg_b200 import synthetic
from oracle import torch_port

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
BOUNDARIES = ["linear", "neumann_zero"]
# the row g shapes (tests/test_metrics_gpu.py) without 160^3, plus partial 30 x 14 tiles in every axis, odd and even W
SHAPES = [(2, (17, 33, 40)), (1, (5, 6, 7)), (1, (2, 2, 2)), (1, (3, 2, 70)), (2, (6, 5, 33)), (1, (4, 4, 4)),
          (2, (7, 9, 6)), (1, (35, 3, 2)), (2, (24, 31, 51)), (1, (37, 19, 45)), (2, (31, 29, 61)), (1, (33, 30, 64))]
MAPS = ["smooth", "noisy", "reflected", "identity"]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def make_map(kind, B, shape, seed):
    """smooth: identity + a smooth displacement that folds in a few places; noisy: the same plus uniform noise of 0.6
    grid steps (a few percent of the voxels fold); reflected: -identity (every voxel folds); identity."""
    idm = torch_port.identity_map(shape).numpy()[None]
    if kind == "identity":
        return np.repeat(idm, B, 0)
    if kind == "reflected":
        return np.repeat(-idm, B, 0)
    phi = idm + np.stack([synthetic.smooth_displacement(shape, seed=seed + b, max_disp=0.5, coarse=4) for b in range(B)])
    if kind == "noisy":
        step = (2.0 / (np.array(shape) - 1)).reshape(1, 3, 1, 1, 1)
        phi = phi + 0.6 * step * np.random.RandomState(seed).uniform(-1, 1, phi.shape)
    return phi.astype(np.float32)


def c_backward(phi, boundary, grad_loss, out=None):
    """raw C call on a CUDA tensor (any 4-byte-aligned dense view); returns grad_phi"""
    from liftreg_b200 import _native, ops
    B, _, D, H, W = phi.shape
    g = torch.tensor([grad_loss], device=phi.device, dtype=torch.float32)
    out = torch.full_like(phi, float("nan")) if out is None else out
    _native.check(_native.lib().lr_jacobian_fold_backward(ctypes.c_void_p(phi.data_ptr()), B, D, H, W, ops.FD_BOUNDARY[boundary],
                                                          ctypes.c_void_p(g.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                                          ops._stream()), "lr_jacobian_fold_backward")
    return out


def check_gradient(got, phi, boundary, grad_loss):
    ref, scale = fold_grad(phi, boundary, grad_loss=grad_loss)
    got = got.cpu().numpy().astype(np.float64)
    assert np.all(np.isfinite(got))
    err = np.abs(got - ref)
    assert np.all(err <= 16 * U * scale), "max err / (u scale) = %g" % (err / np.where(scale > 0, U * scale, np.inf)).max()
    assert np.all(got[scale == 0] == 0)
    return ref


def value_from_stats(phi_t, boundary):
    from liftreg_b200 import ops
    stats, _ = ops.jacobian_det(phi_t, boundary)
    B, _, D, H, W = phi_t.shape
    return (stats[:, 1].sum() / float(B * D * H * W)).to(torch.float32)


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("kind", MAPS)
@pytest.mark.parametrize("B,shape", SHAPES)
def test_fold_backward_matches_float64_reference(dev, B, shape, kind, boundary):
    from liftreg_b200 import ops
    phi = make_map(kind, B, shape, seed=sum(shape) + B)
    phi_t = torch.from_numpy(phi).to(dev)
    got = c_backward(phi_t, boundary, 0.75)
    check_gradient(got, phi, boundary, 0.75)
    assert torch.equal(c_backward(phi_t, boundary, 0.75), got)                 # same bits on a second call
    if kind == "identity":
        assert torch.all(got == 0)
    val = ops.fold_penalty(phi_t, boundary)
    assert val.dtype == torch.float32 and val.shape == () and torch.equal(val, value_from_stats(phi_t, boundary))
    if kind == "identity":
        assert val.item() == 0.0


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("B,shape", [(1, (37, 19, 45)), (2, (9, 8, 11)), (1, (64, 33, 62))])
def test_reflected_affine_map_gradient_vanishes_inside(dev, B, shape, boundary):
    """J is one constant wherever the map is folded, so D_a^T (m C) is exactly 0 more than one layer from every face"""
    phi = reflected_affine(shape, B)
    got = c_backward(torch.from_numpy(phi).to(dev), boundary, 1.0)
    check_gradient(got, phi, boundary, 1.0)
    got = got.cpu().numpy()
    assert np.all(got[:, :, 2:-2, 2:-2, 2:-2] == 0)
    # ... and not zero on the two outer layers (away from the edges, where neumann_zero's zero face rows meet)
    assert np.all(got[:, 0, [0, 1, -2, -1]][:, :, 2:-2, 2:-2] != 0) and np.all(got[:, 2][..., [0, 1, -2, -1]][:, 2:-2, 2:-2] != 0)


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("B", [1, 2])
def test_fold_backward_160_cubed(dev, B, boundary):
    phi = make_map("noisy", B, (160, 160, 160), seed=3)
    got = c_backward(torch.from_numpy(phi).to(dev), boundary, 1.0)
    check_gradient(got, phi, boundary, 1.0)


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("B,shape", [(1, (33, 20, 64)), (2, (9, 8, 10)), (1, (2, 2, 2)), (1, (37, 19, 45))])
def test_fold_backward_unaligned_view(dev, B, shape, boundary):
    phi = make_map("noisy", B, shape, seed=7)
    n = phi.size
    buf = torch.zeros(n + 1, device=dev)
    buf[1:] = torch.from_numpy(phi.reshape(-1)).to(dev)
    view = buf[1:].view(phi.shape)                                             # 4 bytes off an 8-byte boundary
    obuf = torch.full((n + 1,), float("nan"), device=dev)
    oview = obuf[1:].view(phi.shape)
    assert view.data_ptr() % 8 == 4 and oview.data_ptr() % 8 == 4
    c_backward(view, boundary, 0.75, out=oview)
    check_gradient(oview, phi, boundary, 0.75)
    assert torch.isnan(obuf[0])                                                 # nothing written outside grad_phi


@pytest.mark.parametrize("boundary", BOUNDARIES)
def test_nan_in_phi_leaves_value_and_gradient_finite(dev, boundary):
    from liftreg_b200 import ops
    B, shape = 2, (20, 24, 30)
    phi = make_map("noisy", B, shape, seed=13)
    phi[1, 1, 10, 12, 15] = np.nan
    phi[0, 0, 0, 0, 0] = np.nan                                                 # a corner: the face rows read it too
    phi_t = torch.from_numpy(phi).to(dev).requires_grad_(True)
    val = ops.fold_penalty(phi_t, boundary)
    assert torch.isfinite(val) and torch.equal(val.detach(), value_from_stats(phi_t.detach(), boundary))
    val.backward()
    assert torch.all(torch.isfinite(phi_t.grad))
    # away from the NaNs' stencils the gradient is the one of the map without them
    clean = make_map("noisy", B, shape, seed=13)
    ref = c_backward(torch.from_numpy(clean).to(dev), boundary, 1.0).cpu().numpy()
    got = phi_t.grad.cpu().numpy()
    far = np.ones(phi.shape[:1] + phi.shape[2:], bool)
    far[1, 6:15, 8:17, 11:20] = False
    far[0, :5, :5, :5] = False
    assert np.array_equal(got.transpose(0, 2, 3, 4, 1)[far], ref.transpose(0, 2, 3, 4, 1)[far])


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("B,shape", [(2, (17, 33, 40)), (1, (37, 19, 45))])
def test_autograd_gradient_equals_the_c_call(dev, B, shape, boundary):
    from liftreg_b200 import ops
    phi = make_map("noisy", B, shape, seed=5)
    base = torch.from_numpy(phi).to(dev)
    p = base.clone().requires_grad_(True)
    (2.5 * ops.fold_penalty(p, boundary)).backward()
    assert torch.equal(p.grad, c_backward(base, boundary, 2.5))
    with pytest.raises(ValueError, match="boundary"):
        ops.fold_penalty(base, "mirror")
    with pytest.raises(ValueError, match=r"\(B,3,D,H,W\)"):
        ops.fold_penalty(base[:, :2], boundary)
    with pytest.raises(TypeError, match="float32"):
        ops.fold_penalty(base.double(), boundary)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.fold_penalty(base.cpu(), boundary)


def loss_inputs(dev, B=2, shape=(24, 20, 28), seed=9):
    rs = np.random.RandomState(seed)
    disp = torch.from_numpy(make_map("noisy", B, shape, seed) - torch_port.identity_map(shape).numpy()[None]).to(dev)
    warped = torch.from_numpy(rs.uniform(0, 1, (B, 1) + shape).astype(np.float32)).to(dev)
    target = torch.from_numpy(rs.uniform(0, 1, (B, 1) + shape).astype(np.float32)).to(dev)
    return disp, warped, target


@pytest.mark.parametrize("opt", [None, {}, {"fold_factor": 0}])
def test_subspace_loss_without_fold_factor_is_unchanged(dev, opt):
    from liftreg_b200 import losses, ops
    disp, warped, target = loss_inputs(dev)
    params = disp.clone().requires_grad_(True)
    res = losses.SubspaceLoss(opt)({"warped": warped, "target": target, "params": params, "epoch": 12})
    assert sorted(res) == ["reg_loss", "sim_loss", "total_loss"]
    rf = losses.SubspaceLoss().get_reg_factor(12)
    sim, reg = ops.ncc_loss(warped.reshape(2, -1), target.reshape(2, -1)), ops.diffusion_reg(disp)
    assert torch.equal(res["total_loss"].detach(), 1. * sim + rf * reg)
    assert res["sim_loss"] == sim.item() and res["reg_loss"] == reg.item()


@pytest.mark.parametrize("boundary", BOUNDARIES)
def test_subspace_loss_fold_term_is_the_sum_of_its_parts(dev, boundary):
    from liftreg_b200 import losses, ops
    disp, warped, target = loss_inputs(dev)
    ff = 0.3
    loss = losses.SubspaceLoss({"fold_factor": ff}, fd_boundary=boundary)
    params = disp.clone().requires_grad_(True)
    res = loss({"warped": warped, "target": target, "params": params, "epoch": 3})
    assert sorted(res) == ["fold_loss", "reg_loss", "sim_loss", "total_loss"]
    res["total_loss"].backward()

    rf = loss.get_reg_factor(3)
    p2 = disp.clone().requires_grad_(True)
    sim = ops.ncc_loss(warped.reshape(2, -1), target.reshape(2, -1))
    reg = ops.diffusion_reg(p2, boundary)
    phi = p2 + ops.identity_map(disp.shape[2:], dev)
    fold = ops.fold_penalty(phi, boundary)
    assert fold.item() > 0 and res["fold_loss"] == fold.item()
    assert torch.equal(res["total_loss"].detach(), (1. * sim + rf * reg + ff * fold).detach())
    g_reg, = torch.autograd.grad(rf * reg, p2)
    g_fold, = torch.autograd.grad(ff * fold, p2)
    assert torch.equal(params.grad, g_reg + g_fold)
    # the fold part is the C adjoint of phi = params + identity, scaled by fold_factor
    assert torch.equal(g_fold, c_backward(phi.detach().contiguous(), boundary, ff))
