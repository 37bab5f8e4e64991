"""NGF similarity on the GPU: lr_ngf_sum and lr_ngf_backward against the float64 reference (tests/ngf_reference.py)
on size-2 axes, partial 30 x 14 tiles, B = 2, 160^3 and an unaligned view, for smooth fields, a warped CT phantom,
x == y and piecewise-constant blocks; exact scaling, batch and repeat properties; autograd; agreement with the
stock-op composition; and SubspaceLoss(sim=NGFLoss()) through the warp."""
import ctypes

import numpy as np
import pytest
import torch

from ngf_reference import ngf, ngf_torch
from liftreg_b200 import synthetic

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
BOUNDARIES = ["linear", "neumann_zero"]
SHAPES = [(1, (2, 2, 2)), (1, (3, 5, 7)), (1, (17, 33, 45)), (2, (20, 29, 61))]
KINDS = ["smooth", "phantom", "same", "blocks"]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def smooth_field(shape, seed):
    return synthetic.smooth_displacement(shape, seed=seed, max_disp=1.0, coarse=4)[0]


def blocks(shape, seed, side):
    """piecewise-constant dyadic blocks of `side`^3 voxels: the differences vanish two voxels from a block's faces, so
    with side 6 the gradient does at the block's central 2^3 voxels"""
    rs = np.random.RandomState(seed)
    coarse = rs.randint(0, 16, tuple(-(-n // side) for n in shape)) / 8.0 - 1.0
    return np.kron(coarse, np.ones((side,) * 3))[tuple(slice(0, n) for n in shape)].astype(np.float32)


def make_pair(kind, B, shape, seed, dev):
    """(x, y) as (B,1,D,H,W) float32 numpy arrays"""
    from liftreg_b200 import ops
    if kind == "smooth":
        x = np.stack([smooth_field(shape, seed + b) for b in range(B)])
        y = np.stack([smooth_field(shape, seed + 50 + b) for b in range(B)])
    elif kind in ("phantom", "same"):
        y = np.stack([synthetic.hu_to_unit(synthetic.ct_phantom(shape, seed=seed + b)) for b in range(B)])
        if kind == "same":
            x = y.copy()
        else:                              # the phantom warped by a smooth displacement
            disp = np.stack([synthetic.smooth_displacement(shape, seed=seed + 9 + b, max_disp=0.05, coarse=4) for b in range(B)])
            phi = torch.from_numpy(disp).to(dev) + ops.identity_map(shape, dev)
            x = ops.warp(torch.from_numpy(y[:, None]).to(dev), phi)[:, 0].cpu().numpy()
    else:
        x = np.stack([blocks(shape, seed + b, 6) for b in range(B)])
        y = np.stack([blocks(shape, seed + 30 + b, 3) for b in range(B)])
    return x[:, None].astype(np.float32), y[:, None].astype(np.float32)


def c_sum(x, y, boundary, eps):
    from liftreg_b200 import _native, ops
    B, D, H, W = x.shape[0], *x.shape[-3:]
    sums = torch.full((B,), float("nan"), device=x.device, dtype=torch.float64)
    _native.check(_native.lib().lr_ngf_sum(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, D, H, W,
                                           ops.FD_BOUNDARY[boundary], eps, ctypes.c_void_p(sums.data_ptr()), ops._stream()),
                  "lr_ngf_sum")
    return sums


def c_backward(x, y, boundary, eps, grad_loss, out=None):
    """raw C call on CUDA tensors (any 4-byte-aligned dense views); returns grad_x"""
    from liftreg_b200 import _native, ops
    B, D, H, W = x.shape[0], *x.shape[-3:]
    g = torch.tensor([grad_loss], device=x.device, dtype=torch.float32)
    out = torch.full_like(x, float("nan")) if out is None else out
    _native.check(_native.lib().lr_ngf_backward(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, D, H, W,
                                                ops.FD_BOUNDARY[boundary], eps, ctypes.c_void_p(g.data_ptr()),
                                                ctypes.c_void_p(out.data_ptr()), ops._stream()), "lr_ngf_backward")
    return out


def check_against_reference(x, y, boundary, eps, grad_loss, dev, want_zero_blocks=False):
    from liftreg_b200 import ops
    sums_ref, loss_ref, grad_ref, scale = ngf(x, y, eps, boundary, grad_loss=grad_loss)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    sums = c_sum(xt, yt, boundary, eps).cpu().numpy()
    assert np.all(np.abs(sums - sums_ref) <= 1e-12 * np.abs(sums_ref)), (sums, sums_ref)
    loss = ops.ngf_loss(xt, yt, eps, boundary)
    assert loss.dtype == torch.float32 and loss.shape == ()
    assert abs(loss.item() - loss_ref) <= np.spacing(np.float32(loss_ref)), (loss.item(), loss_ref)
    got = c_backward(xt, yt, boundary, eps, grad_loss)
    k = got.cpu().numpy().astype(np.float64)
    assert np.all(np.isfinite(k))
    err = np.abs(k - grad_ref)
    assert np.all(err <= 16 * U * scale), "max err / (u scale) = %g" % (err / np.where(scale > 0, U * scale, np.inf)).max()
    assert np.all(k[scale == 0] == 0)
    if want_zero_blocks:
        assert np.any(scale == 0)
    assert torch.equal(c_backward(xt, yt, boundary, eps, grad_loss), got)                  # same bits on a second call
    return got


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("B,shape", SHAPES)
def test_sums_loss_and_gradient_match_reference(dev, B, shape, kind, boundary):
    x, y = make_pair(kind, B, shape, sum(shape) + B, dev)
    check_against_reference(x, y, boundary, 1.0, 0.75, dev, want_zero_blocks=kind == "blocks" and min(shape) >= 6)


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("kind", KINDS)
def test_160_cubed(dev, kind, boundary):
    x, y = make_pair(kind, 1, (160, 160, 160), 3, dev)
    check_against_reference(x, y, boundary, 1.0, 1.0, dev)


@pytest.mark.parametrize("eps", [1e-2, 10.0])
def test_other_eps(dev, eps):
    x, y = make_pair("phantom", 2, (20, 29, 61), 4, dev)
    check_against_reference(x, y, "linear", eps, 1.0, dev)


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("B,shape", [(1, (17, 33, 45)), (2, (20, 29, 61))])
def test_unaligned_views(dev, B, shape, boundary):
    x, y = make_pair("phantom", B, shape, 5, dev)
    n = x.size
    bufs = []
    for a in (x, y):
        buf = torch.zeros(n + 1, device=dev)
        buf[1:] = torch.from_numpy(a.reshape(-1)).to(dev)
        bufs.append(buf[1:].view(a.shape))                                     # 4 bytes off an 8-byte boundary
    obuf = torch.full((n + 1,), float("nan"), device=dev)
    oview = obuf[1:].view(x.shape)
    assert bufs[0].data_ptr() % 8 == 4 and oview.data_ptr() % 8 == 4
    c_backward(bufs[0], bufs[1], boundary, 1.0, 0.75, out=oview)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    assert torch.equal(oview, c_backward(xt, yt, boundary, 1.0, 0.75))
    assert torch.isnan(obuf[0])                                                 # nothing written outside grad_x
    s0, s1 = c_sum(bufs[0], bufs[1], boundary, 1.0), c_sum(xt, yt, boundary, 1.0)
    assert torch.all((s0 - s1).abs() <= 1e-12 * s1.abs())


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("kind", ["smooth", "phantom", "blocks"])
def test_scaling_by_two_halves_the_gradient_exactly(dev, kind, boundary):
    """(2x, 2y, 2 eps): every difference, a, p, q and c scale by powers of two, f is unchanged and c halves"""
    x, y = make_pair(kind, 2, (17, 33, 45), 6, dev)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    g1 = c_backward(xt, yt, boundary, 0.75, 1.0)
    g2 = c_backward(2 * xt, 2 * yt, boundary, 1.5, 1.0)
    assert torch.equal(g2, 0.5 * g1)
    s1, s2 = c_sum(xt, yt, boundary, 0.75), c_sum(2 * xt, 2 * yt, boundary, 1.5)
    assert torch.all((s1 - s2).abs() <= 1e-12 * s1.abs())


@pytest.mark.parametrize("boundary", BOUNDARIES)
@pytest.mark.parametrize("shape", [(3, 5, 7), (20, 29, 61), (33, 17, 40)])
def test_batch_items_are_independent_and_bits_repeat(dev, shape, boundary):
    from liftreg_b200 import _native
    x, y = make_pair("phantom", 2, shape, 7, dev)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    both = c_backward(xt, yt, boundary, 1.0, 2.0 * 0.625)
    for b in range(2):
        one = c_backward(xt[b:b + 1].contiguous(), yt[b:b + 1].contiguous(), boundary, 1.0, 0.625)
        assert torch.equal(both[b:b + 1], one)
    prev = _native.set_numerics("exact")
    try:
        exact = c_backward(xt, yt, boundary, 1.0, 1.25)
        _native.set_numerics("fast")
        fast = c_backward(xt, yt, boundary, 1.0, 1.25)
    finally:
        _native.set_numerics(prev)
    assert torch.equal(exact, both) and torch.equal(fast, both)


@pytest.mark.parametrize("five_d", [True, False])
def test_autograd_equals_the_c_calls(dev, five_d):
    from liftreg_b200 import ops
    x, y = make_pair("phantom", 2, (17, 33, 45), 8, dev)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    if not five_d:
        xt, yt = xt[:, 0], yt[:, 0]
    p = xt.clone().requires_grad_(True)
    loss = ops.ngf_loss(p, yt, 0.5, "neumann_zero")
    (2.5 * loss).backward()
    assert p.grad.shape == xt.shape
    assert torch.equal(p.grad, c_backward(xt.contiguous(), yt.contiguous(), "neumann_zero", 0.5, 2.5))
    sums = c_sum(xt, yt, "neumann_zero", 0.5)
    assert abs(loss.item() - (1.0 - sums.sum().item() / xt.numel())) <= 1e-7
    with pytest.raises(TypeError, match="float32"):
        ops.ngf_loss(xt.double(), yt.double())
    m = __import__("liftreg_b200.losses", fromlist=["NGFLoss"]).NGFLoss()
    assert torch.equal(m(xt, yt), ops.ngf_loss(xt, yt, 1.0, "linear"))


@pytest.mark.parametrize("boundary", BOUNDARIES)
def test_agrees_with_the_stock_op_composition(dev, boundary):
    from liftreg_b200 import ops
    x, y = make_pair("phantom", 2, (48, 40, 56), 10, dev)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    results = []
    for fn in (ops.ngf_loss, ngf_torch):
        p = xt.clone().requires_grad_(True)
        loss = fn(p, yt, 1.0, boundary)
        loss.backward()
        results.append((loss.item(), p.grad.double()))
    (lk, gk), (lt, gt) = results
    assert abs(lk - lt) <= 1e-6
    assert float((gk - gt).norm() / gt.norm()) <= 2e-5


def test_subspace_loss_with_ngf_backpropagates_through_the_warp(dev):
    """SubspaceLoss(sim=NGFLoss()) on a warped phantom: the total is the sum of its parts and the gradient reaching the
    displacement is finite and equals the one built from ops.ngf_loss directly"""
    from liftreg_b200 import losses, ops
    B, shape = 2, (40, 36, 44)
    target = torch.from_numpy(np.stack([synthetic.hu_to_unit(synthetic.ct_phantom(shape, seed=b))
                                        for b in range(B)])[:, None]).to(dev)
    moving = torch.from_numpy(np.stack([synthetic.hu_to_unit(synthetic.ct_phantom(shape, seed=b, noise_hu=20.0))
                                        for b in range(B)])[:, None]).to(dev)
    disp = torch.from_numpy(np.stack([synthetic.smooth_displacement(shape, seed=b, max_disp=0.05, coarse=4) for b in range(B)])).to(dev)
    idm = ops.identity_map(shape, dev)
    results = []
    for how in ("class", "direct"):
        params = disp.clone().requires_grad_(True)
        warped = ops.warp(moving, params + idm)
        if how == "class":
            out = losses.SubspaceLoss(sim=losses.NGFLoss())({"warped": warped, "target": target, "params": params, "epoch": 4})
            assert sorted(out) == ["reg_loss", "sim_loss", "total_loss"]
            total = out["total_loss"]
        else:
            total = 1. * ops.ngf_loss(warped, target) + losses.SubspaceLoss().get_reg_factor(4) * ops.diffusion_reg(params)
        total.backward()
        results.append((total.detach(), params.grad))
    (lk, gk), (lt, gt) = results
    assert torch.all(torch.isfinite(gk)) and gk.abs().max() > 0
    assert abs(lk.item() - lt.item()) <= 1e-6 and torch.allclose(gk, gt, rtol=1e-5, atol=1e-7 * gt.abs().max().item())
