"""Local NCC on the GPU: lr_local_ncc_sum / lr_local_ncc_backward through the C-ABI and through ops, against the
float64 reference (tests/lncc_reference.py): the loss per item within 1e-5, the gradient element by element within
4 u x abs-scale and exactly 0 where the reference is 0 by structure; repeatable bits, batch independence, unaligned
views, and SubspaceLoss(sim=LocalNCCLoss()) against the stock-torch formulation."""
import ctypes

import numpy as np
import pytest
import torch
from scipy.ndimage import maximum_filter, minimum_filter

from lncc_reference import inside_mask, item_losses, local_ncc, voxelmorph_ncc_torch
from liftreg_b200 import synthetic

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
C = 4                         # gradient bar in u x abs-scale (DESIGN.md section 3)
EPS = 1e-5
W_MAX = 15
IMAGES = ["ct", "noise", "blocks", "same", "impulse"]
# (B, (D, H, W), window): 64^3 at B = 2, ragged, axes smaller than the window, size-1 axes, every window class
CASES = [(2, (64, 64, 64), 9), (1, (37, 45, 29), 9), (1, (37, 45, 29), 3), (2, (37, 45, 29), 5), (1, (37, 45, 29), W_MAX),
         (1, (5, 40, 7), 9), (1, (1, 30, 33), 5), (2, (20, 1, 17), 9), (1, (9, 11, 1), 3), (1, (12, 17, 40), W_MAX)]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def dyadic(rs, shape, levels=16):
    """uniform values k/8 - 1: every window sum of these and of their products is exact in fp64"""
    return (rs.randint(0, levels, shape) / 8.0 - 1.0).astype(np.float32)


def make_pair(kind, B, shape, seed, w=9):
    """(x, y) float32 (B,1,D,H,W)"""
    rs = np.random.RandomState(seed)
    full = (B, 1) + tuple(shape)
    if kind == "ct":            # chest phantom in [-1, 1], air exactly -1; the target is a second phantom
        x = np.stack([synthetic.hu_to_unit(synthetic.ct_phantom(shape, seed=seed + b)) for b in range(B)])[:, None]
        y = np.stack([synthetic.hu_to_unit(synthetic.ct_phantom(shape, seed=seed + 7 + b)) for b in range(B)])[:, None]
        return x.astype(np.float32), y.astype(np.float32)
    if kind == "noise":
        return rs.uniform(-1, 1, full).astype(np.float32), rs.uniform(-1, 1, full).astype(np.float32)
    if kind == "same":
        x = rs.uniform(-1, 1, full).astype(np.float32)
        return x, x.copy()
    if kind == "blocks":        # exactly constant (2w+2)^3 blocks of dyadic values in x; dyadic noise in y
        s = 2 * w + 2
        coarse = dyadic(rs, (B, 1) + tuple((n + s - 1) // s for n in shape))
        x = coarse.repeat(s, 2).repeat(s, 3).repeat(s, 4)[:, :, :shape[0], :shape[1], :shape[2]]
        return np.ascontiguousarray(x), dyadic(rs, full)
    if kind == "impulse":       # one voxel of x set on a zero background, any y
        x = np.zeros(full, np.float32)
        x[:, 0, shape[0] // 3, shape[1] // 2, (2 * shape[2]) // 3] = 1.0
        return x, rs.uniform(-1, 1, full).astype(np.float32)
    raise ValueError(kind)


def structural_zeros(kind, x, w):
    """voxels where the gradient is 0 by structure: every centre of N(v) sees a constant x window inside the volume
    (blocks) or a window without the impulse (impulse)"""
    if kind == "impulse":
        return maximum_filter(np.abs(x[:, 0]), size=(1,) + (2 * w - 1,) * 3, mode="constant") == 0
    if kind == "blocks":
        xs = x[:, 0]
        size = (1,) + (2 * w - 1,) * 3
        const = maximum_filter(xs, size=size, mode="nearest") == minimum_filter(xs, size=size, mode="nearest")
        return const & inside_mask(xs.shape[1:], w - 1)[None]
    return None


def c_sum(x, y, w, eps=EPS):
    from liftreg_b200 import _native, ops
    B, D, H, W = x.shape[0], *x.shape[-3:]
    s = torch.full((B,), float("nan"), device=x.device, dtype=torch.float64)
    _native.check(_native.lib().lr_local_ncc_sum(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, D, H, W, w,
                                                 eps, ctypes.c_void_p(s.data_ptr()), ops._stream()), "lr_local_ncc_sum")
    return s


def c_backward(x, y, w, grad_loss, eps=EPS, out=None):
    from liftreg_b200 import _native, ops
    B, D, H, W = x.shape[0], *x.shape[-3:]
    lib = _native.lib()
    nbytes = lib.lr_local_ncc_workspace_bytes(B, D, H, W, w)
    assert nbytes == 12 * B * D * H * W
    ws = torch.full((nbytes // 4,), float("nan"), device=x.device)
    g = torch.tensor([grad_loss], device=x.device, dtype=torch.float32)
    out = torch.full_like(x, float("nan")) if out is None else out
    _native.check(lib.lr_local_ncc_backward(ctypes.c_void_p(x.data_ptr()), ctypes.c_void_p(y.data_ptr()), B, D, H, W, w, eps,
                                            ctypes.c_void_p(g.data_ptr()), ctypes.c_void_p(out.data_ptr()),
                                            ctypes.c_void_p(ws.data_ptr()), nbytes, ops._stream()), "lr_local_ncc_backward")
    return out


def check(x, y, w, got_sum, got_grad, grad_loss, kind=None):
    cc, _, ref, scale = local_ncc(x, y, w, EPS, grad_loss)
    D, H, W = x.shape[-3:]
    got_loss = 1.0 - got_sum.cpu().numpy() / (D * H * W)
    ref_loss = 1.0 - cc.reshape(cc.shape[0], -1).mean(1)
    assert np.all(np.abs(got_loss - ref_loss) <= 1e-5), (got_loss, ref_loss)
    got = got_grad.cpu().numpy().astype(np.float64)
    assert np.all(np.isfinite(got))
    err = np.abs(got - ref)
    assert np.all(err <= C * U * scale), "max err / (u scale) = %g" % (err / np.where(scale > 0, U * scale, np.inf)).max()
    assert np.all(got[scale == 0] == 0)
    if kind is not None:
        zero = structural_zeros(kind, x, w)
        if zero is not None:
            assert zero.any() or min(x.shape[-3:]) < 4 * w
            assert np.all(ref[:, 0][zero] == 0) and np.all(got[:, 0][zero] == 0)
    return ref


@pytest.mark.parametrize("kind", IMAGES)
@pytest.mark.parametrize("B,shape,w", CASES)
def test_local_ncc_matches_float64_reference(dev, B, shape, w, kind):
    x, y = make_pair(kind, B, shape, seed=sum(shape) + w, w=w)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    s = c_sum(xt, yt, w)
    g = c_backward(xt, yt, w, 0.75)
    check(x, y, w, s, g, 0.75, kind)
    assert torch.equal(c_backward(xt, yt, w, 0.75), g)                  # same bits on a second call
    assert torch.allclose(c_sum(xt, yt, w), s, rtol=1e-13, atol=0)     # fp64 atomics: order-dependent last bits only


@pytest.mark.parametrize("kind", ["ct", "noise"])
def test_local_ncc_160_cubed(dev, kind):
    x, y = make_pair(kind, 1, (160, 160, 160), seed=3)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    check(x, y, 9, c_sum(xt, yt, 9), c_backward(xt, yt, 9, 1.0), 1.0)


@pytest.mark.parametrize("kind", ["ct", "noise", "impulse"])
@pytest.mark.parametrize("shape,w", [((64, 64, 64), 9), ((37, 45, 29), 5), ((20, 1, 17), 9)])
def test_batch_items_are_independent(dev, shape, w, kind):
    """each item of a B = 2 call (grad_loss 2g) equals, bit for bit, a single-item call with g"""
    x, y = make_pair(kind, 2, shape, seed=11)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    g2 = c_backward(xt, yt, w, 1.5)
    s2 = c_sum(xt, yt, w)
    for b in range(2):
        g1 = c_backward(xt[b:b + 1].contiguous(), yt[b:b + 1].contiguous(), w, 0.75)
        assert torch.equal(g2[b:b + 1], g1)
        assert torch.allclose(c_sum(xt[b:b + 1].contiguous(), yt[b:b + 1].contiguous(), w), s2[b:b + 1], rtol=1e-13, atol=0)


@pytest.mark.parametrize("B,shape,w", [(1, (33, 20, 64), 9), (2, (9, 8, 10), 3), (1, (37, 45, 29), W_MAX)])
def test_unaligned_view(dev, B, shape, w):
    x, y = make_pair("noise", B, shape, seed=5)
    n = x.size
    bufs = [torch.zeros(n + 1, device=dev) for _ in range(2)]
    bufs[0][1:] = torch.from_numpy(x.reshape(-1)).to(dev)
    bufs[1][1:] = torch.from_numpy(y.reshape(-1)).to(dev)
    xv, yv = (b[1:].view(x.shape) for b in bufs)
    assert xv.storage_offset() == 1 and xv.data_ptr() % 8 == 4
    obuf = torch.full((n + 1,), float("nan"), device=dev)
    ov = obuf[1:].view(x.shape)
    c_backward(xv, yv, w, 0.75, out=ov)
    check(x, y, w, c_sum(xv, yv, w), ov, 0.75)
    assert torch.isnan(obuf[0])                                         # nothing written outside grad_x
    from liftreg_b200 import ops
    p = xv.clone().requires_grad_(True)                                 # aligned copy
    assert torch.equal(ops.local_ncc_loss(xv, yv, w), ops.local_ncc_loss(p, yv.clone(), w).detach())


@pytest.mark.parametrize("five_d", [True, False])
def test_autograd_equals_the_c_calls(dev, five_d):
    from liftreg_b200 import ops
    x, y = make_pair("ct", 2, (24, 30, 36), seed=9)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    if not five_d:
        xt, yt = xt[:, 0], yt[:, 0]
    p = xt.clone().requires_grad_(True)
    q = yt.clone().requires_grad_(True)
    loss = ops.local_ncc_loss(p, q, window=7, eps=1e-4)
    assert loss.dtype == torch.float32 and loss.shape == ()
    s = c_sum(xt, yt, 7, 1e-4)
    assert loss.item() == pytest.approx(1.0 - s.sum().item() / (2 * 24 * 30 * 36), abs=1e-7)
    (2.5 * loss).backward()
    assert q.grad is None and p.grad.shape == p.shape
    assert torch.equal(p.grad, c_backward(xt, yt, 7, 2.5, eps=1e-4))
    with pytest.raises(ValueError, match="shape"):
        ops.local_ncc_loss(xt, yt[:1])
    with pytest.raises(TypeError, match="float32"):
        ops.local_ncc_loss(xt.double(), yt.double())
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.local_ncc_loss(xt.cpu(), yt.cpu())
    with pytest.raises(RuntimeError, match="odd"):
        ops.local_ncc_loss(xt, yt, window=8)


def test_subspace_loss_with_local_ncc_matches_stock_torch(dev):
    """SubspaceLoss(sim=LocalNCCLoss()) on a warped image: total loss and d/d params through the warp equal the same
    loss built on VoxelMorph's conv3d formulation in fp32 torch"""
    from liftreg_b200 import losses, ops
    rs = np.random.RandomState(21)
    B, shape = 2, (40, 36, 44)
    moving = torch.from_numpy(rs.uniform(-1, 1, (B, 1) + shape).astype(np.float32)).to(dev)
    target = torch.from_numpy(rs.uniform(-1, 1, (B, 1) + shape).astype(np.float32)).to(dev)
    disp = torch.from_numpy(np.stack([synthetic.smooth_displacement(shape, seed=b, max_disp=0.05, coarse=4) for b in range(B)])).to(dev)
    idm = ops.identity_map(shape, dev)
    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False                             # full fp32 convolutions for the comparison
    try:
        results = []
        for sim in ("kernel", "torch"):
            params = disp.clone().requires_grad_(True)
            warped = ops.warp(moving, params + idm)
            if sim == "kernel":
                out = losses.SubspaceLoss(sim=losses.LocalNCCLoss())({"warped": warped, "target": target, "params": params, "epoch": 4})
                total = out["total_loss"]
            else:
                lsim = voxelmorph_ncc_torch(warped, target, 9, 1e-5)[0]
                total = 1. * lsim + losses.SubspaceLoss().get_reg_factor(4) * ops.diffusion_reg(params)
            total.backward()
            results.append((total.item(), params.grad.double()))
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    (lk, gk), (lt, gt) = results
    assert abs(lk - lt) <= 1e-5
    assert float((gk - gt).norm() / gt.norm()) <= 1e-3


def test_local_ncc_loss_class_defaults(dev):
    from liftreg_b200 import losses, ops
    x, y = make_pair("noise", 1, (20, 21, 22), seed=2)
    xt, yt = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
    m = losses.LocalNCCLoss()
    assert (m.window, m.eps) == (9, 1e-5)
    assert torch.equal(m(xt, yt), ops.local_ncc_loss(xt, yt, 9, 1e-5))
    assert abs(m(xt, yt).item() - item_losses(x, y, 9, 1e-5).mean()) <= 1e-6
