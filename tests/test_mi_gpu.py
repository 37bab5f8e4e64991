"""Mutual information similarity on the GPU: lr_mi_hist and lr_mi_backward against the float64 reference
(tests/mi_reference.py) on ragged sizes, B = 2, 160^3, unaligned views, nb in {4, 32, 64} and a non-default range, for
smooth fields, a warped CT phantom pair and x == y; constant targets; NaN and inf inputs; exact scaling, batch and
repeat properties for a given histogram; autograd; agreement with the stock-op composition; and
SubspaceLoss(sim=MILoss()) through the warp."""
import ctypes

import numpy as np
import pytest
import torch

from mi_reference import mi, mi_torch
from liftreg_b200 import synthetic

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
SHAPES = [(1, (7,)), (1, (1001,)), (1, (17, 33, 45)), (2, (20, 29, 61))]
KINDS = ["smooth", "phantom", "same"]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def volume_shape(shape):
    """a 3-D shape for the generators: 1-D sizes become (1, 1, n)"""
    return shape if len(shape) == 3 else (1, 1) + tuple(shape)


def make_pair(kind, B, shape, seed, dev):
    """(x, y) as (B, *shape) float32 numpy arrays"""
    from liftreg_b200 import ops
    vs = volume_shape(shape)
    if kind == "smooth":                   # two smooth fields over a little more than the range
        x = np.stack([1.2 * synthetic.smooth_displacement(vs, seed=seed + b, max_disp=1.0, coarse=4)[0] for b in range(B)])
        y = np.stack([np.sin(3 * x[b]) + 0.3 * synthetic.smooth_displacement(vs, seed=seed + 50 + b, max_disp=1.0, coarse=4)[1]
                      for b in range(B)])
    else:
        y = np.stack([synthetic.hu_to_unit(synthetic.ct_phantom(vs, seed=seed + b)) for b in range(B)])
        if kind == "same":
            x = y.copy()
        elif len(shape) != 3:              # a row of the phantom: shifted, with noise
            x = np.roll(y, 3, axis=-1) + np.random.RandomState(seed).normal(0, 0.02, y.shape)
        else:                              # the phantom warped by a smooth displacement
            disp = np.stack([synthetic.smooth_displacement(vs, seed=seed + 9 + b, max_disp=0.05, coarse=4) for b in range(B)])
            phi = torch.from_numpy(disp).to(dev) + ops.identity_map(vs, dev)
            x = ops.warp(torch.from_numpy(y[:, None]).to(dev), phi)[:, 0].cpu().numpy()
    return x.reshape((B,) + tuple(shape)).astype(np.float32), y.reshape((B,) + tuple(shape)).astype(np.float32)


def c_hist(x, y, nb, rng=(-1.0, 1.0)):
    from liftreg_b200 import _native, ops
    B = x.shape[0]
    hist = torch.full((B, nb, nb + 2), float("nan"), device=x.device, dtype=torch.float64)
    _native.check(_native.lib().lr_mi_hist(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, x.numel() // B, nb,
                                           rng[0], rng[1], ctypes.c_void_p(hist.data_ptr()), ops._stream()), "lr_mi_hist")
    return hist


def c_backward(x, y, nb, rng, hist, grad_loss, out=None):
    """raw C call on CUDA tensors (any 4-byte-aligned dense views); returns grad_x"""
    from liftreg_b200 import _native, ops
    B = x.shape[0]
    g = torch.tensor([grad_loss], device=x.device, dtype=torch.float32)
    out = torch.full_like(x, float("nan")) if out is None else out
    _native.check(_native.lib().lr_mi_backward(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, x.numel() // B,
                                               nb, rng[0], rng[1], ctypes.c_void_p(hist.data_ptr()), ctypes.c_void_p(g.data_ptr()),
                                               ctypes.c_void_p(out.data_ptr()), ops._stream()), "lr_mi_backward")
    return out


def check_hist(h, ref):
    assert np.all(np.abs(h - ref) <= 1e-12 * np.abs(ref)), np.abs(h - ref).max()


def check_against_reference(x, y, nb, rng, grad_loss, dev):
    from liftreg_b200 import ops
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    hist = c_hist(xt, yt, nb, rng)
    h = hist.cpu().numpy()
    hist_ref, loss_ref, grad_ref, scale = mi(x, y, nb, rng, grad_loss=grad_loss, hist=h)
    check_hist(h, hist_ref)
    loss = ops.mi_loss(xt, yt, nb, rng)
    assert loss.dtype == torch.float32 and loss.shape == ()
    assert abs(loss.item() - loss_ref) <= max(np.spacing(np.float32(abs(loss_ref))), 1e-10), (loss.item(), loss_ref)
    got = c_backward(xt, yt, nb, rng, hist, grad_loss)
    k = got.cpu().numpy().astype(np.float64)
    assert np.all(np.isfinite(k))
    err = np.abs(k - grad_ref)
    assert np.all(err <= 16 * U * scale), "max err / (u scale) = %g" % (err / np.where(scale > 0, U * scale, np.inf)).max()
    assert np.all(k[scale == 0] == 0)
    lo, hi = np.float32(rng[0]), np.float32(rng[1])
    assert np.all(k[(x < lo) | (x > hi)] == 0)
    assert torch.equal(c_backward(xt, yt, nb, rng, hist, grad_loss), got)                  # same bits on a second call
    return hist, got


@pytest.mark.parametrize("nb", [4, 32, 64])
@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("B,shape", SHAPES)
def test_hist_loss_and_gradient_match_reference(dev, B, shape, kind, nb):
    x, y = make_pair(kind, B, shape, sum(shape) + B, dev)
    check_against_reference(x, y, nb, (-1.0, 1.0), 0.75, dev)


@pytest.mark.parametrize("nb", [32, 64])
@pytest.mark.parametrize("kind", ["phantom", "same"])
def test_160_cubed(dev, kind, nb):
    x, y = make_pair(kind, 1, (160, 160, 160), 3, dev)
    check_against_reference(x, y, nb, (-1.0, 1.0), 1.0, dev)


@pytest.mark.parametrize("rng", [(-0.8, 0.6), (-3.0, 2.5)])
def test_non_default_range(dev, rng):
    x, y = make_pair("phantom", 2, (20, 29, 61), 4, dev)
    check_against_reference(x, y, 24, rng, 1.0, dev)


@pytest.mark.parametrize("B,shape", [(1, (1001,)), (2, (20, 29, 61))])
def test_unaligned_views(dev, B, shape):
    x, y = make_pair("phantom", B, shape, 5, dev)
    n = x.size
    bufs = []
    for a in (x, y):
        buf = torch.zeros(n + 1, device=dev)
        buf[1:] = torch.from_numpy(a.reshape(-1)).to(dev)
        bufs.append(buf[1:].view(a.shape))                                     # 4 bytes off a 16-byte boundary
    obuf = torch.full((n + 1,), float("nan"), device=dev)
    oview = obuf[1:].view(x.shape)
    assert bufs[0].data_ptr() % 16 == 4 and oview.data_ptr() % 16 == 4
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    h0, h1 = c_hist(bufs[0], bufs[1], 32), c_hist(xt, yt, 32)
    check_hist(h0.cpu().numpy(), h1.cpu().numpy())
    c_backward(bufs[0], bufs[1], 32, (-1.0, 1.0), h1, 0.75, out=oview)
    assert torch.equal(oview, c_backward(xt, yt, 32, (-1.0, 1.0), h1, 0.75))
    assert torch.isnan(obuf[0])                                                 # nothing written outside grad_x


@pytest.mark.parametrize("v", [-1.0, 0.25, 1.0])
def test_constant_target_gives_zero_gradient_and_zero_mi(dev, v):
    from liftreg_b200 import ops
    x, _ = make_pair("phantom", 2, (20, 29, 61), 6, dev)
    xt = torch.from_numpy(x).to(dev)
    yt = torch.full_like(xt, v)
    hist = c_hist(xt, yt, 32)
    assert torch.equal(c_backward(xt, yt, 32, (-1.0, 1.0), hist, 1.0), torch.zeros_like(xt))
    assert abs(ops.mi_loss(xt, yt).item()) <= 1e-12


def test_nonfinite_inputs_count_as_range_ends(dev):
    x, y = make_pair("smooth", 1, (1001,), 7, dev)
    x[0, :6] = [np.nan, np.inf, -np.inf, 5.0, -5.0, np.nan]
    y[0, 3:9] = [np.nan, np.inf, -np.inf, np.nan, 7.0, -7.0]
    _, got = check_against_reference(x, y, 32, (-1.0, 1.0), 1.0, dev)
    assert torch.all(got[0, :6] == 0)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    assert abs(c_hist(xt, yt, 32).sum().item() - x.size) <= 1e-9


@pytest.mark.parametrize("kind", ["smooth", "phantom"])
def test_scaling_by_two_halves_the_gradient_exactly(dev, kind):
    """(2x, 2lo, 2hi): s halves exactly, so u is bit-identical; the same hist gives exactly half the gradient"""
    x, y = make_pair(kind, 2, (17, 33, 45), 8, dev)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    rng, rng2 = (-0.75, 0.875), (-1.5, 1.75)
    hist = c_hist(xt, yt, 32, rng)
    check_hist(c_hist(2 * xt, 2 * yt, 32, rng2).cpu().numpy(), hist.cpu().numpy())
    g1 = c_backward(xt, yt, 32, rng, hist, 1.0)
    g2 = c_backward(2 * xt, 2 * yt, 32, rng2, hist, 1.0)
    assert torch.equal(g2, 0.5 * g1)


@pytest.mark.parametrize("shape", [(1001,), (20, 29, 61)])
def test_batch_items_are_independent_and_bits_repeat(dev, shape):
    x, y = make_pair("phantom", 2, shape, 9, dev)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    hist = c_hist(xt, yt, 32)
    both = c_backward(xt, yt, 32, (-1.0, 1.0), hist, 2.0 * 0.625)
    for b in range(2):
        one = c_backward(xt[b:b + 1].contiguous(), yt[b:b + 1].contiguous(), 32, (-1.0, 1.0), hist[b:b + 1].contiguous(), 0.625)
        assert torch.equal(both[b:b + 1], one)
        check_hist(c_hist(xt[b:b + 1].contiguous(), yt[b:b + 1].contiguous(), 32).cpu().numpy(), hist[b:b + 1].cpu().numpy())
    assert torch.equal(c_backward(xt, yt, 32, (-1.0, 1.0), hist, 1.25), c_backward(xt, yt, 32, (-1.0, 1.0), hist, 1.25))


@pytest.mark.parametrize("five_d", [True, False])
def test_autograd_and_the_loss_class(dev, five_d):
    from liftreg_b200 import losses, ops
    x, y = make_pair("phantom", 2, (17, 33, 45), 10, dev)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    if five_d:
        xt, yt = xt[:, None], yt[:, None]
    p = xt.clone().requires_grad_(True)
    loss = ops.mi_loss(p, yt, 16)
    (2.5 * loss).backward()
    assert p.grad.shape == xt.shape
    hist = c_hist(xt, yt, 16)
    ref = c_backward(xt, yt, 16, (-1.0, 1.0), hist, 2.5)
    assert torch.allclose(p.grad, ref, rtol=1e-5, atol=1e-6 * ref.abs().max().item())
    with pytest.raises(TypeError, match="float32"):
        ops.mi_loss(xt.double(), yt.double())
    m = losses.MILoss()
    assert torch.allclose(m(xt, yt), ops.mi_loss(xt.reshape(2, -1), yt.reshape(2, -1)), rtol=0, atol=1e-7)


@pytest.mark.parametrize("nb", [8, 32])
def test_agrees_with_the_stock_op_composition(dev, nb):
    from liftreg_b200 import ops
    x, y = make_pair("phantom", 2, (48, 40, 56), 11, dev)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    results = []
    for fn, dt in ((ops.mi_loss, torch.float32), (mi_torch, torch.float64)):
        p = xt.to(dt).clone().requires_grad_(True)
        loss = fn(p, yt.to(dt), nb)
        loss.backward()
        results.append((loss.item(), p.grad.double()))
    (lk, gk), (lt, gt) = results
    assert abs(lk - lt) <= 1e-6
    assert float((gk - gt).norm() / gt.norm()) <= 2e-5


def test_subspace_loss_with_mi_backpropagates_through_the_warp(dev):
    """SubspaceLoss(sim=MILoss()) on a warped phantom: the total is the sum of its parts and the gradient reaching the
    displacement is finite and equals the one built from ops.mi_loss directly"""
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
            out = losses.SubspaceLoss(sim=losses.MILoss())({"warped": warped, "target": target, "params": params, "epoch": 4})
            assert sorted(out) == ["reg_loss", "sim_loss", "total_loss"]
            total = out["total_loss"]
        else:
            total = 1. * ops.mi_loss(warped.reshape(B, -1), target.reshape(B, -1)) \
                + losses.SubspaceLoss().get_reg_factor(4) * ops.diffusion_reg(params)
        total.backward()
        results.append((total.detach(), params.grad))
    (lk, gk), (lt, gt) = results
    assert torch.all(torch.isfinite(gk)) and gk.abs().max() > 0
    assert abs(lk.item() - lt.item()) <= 1e-6 and torch.allclose(gk, gt, rtol=1e-5, atol=1e-6 * gt.abs().max().item())
