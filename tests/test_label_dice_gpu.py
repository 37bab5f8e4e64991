"""Soft Dice loss of the warped label map on the GPU: lr_label_dice_sums and lr_label_dice_backward against the float64
reference (tests/dice_reference.py) on ragged shapes, size-1 axes, partial tiles, B = 2, unaligned views and 160^3 at
L = 2, 6 and 128; the exact structure at integer sample positions; invalid labels; repeatable bits; autograd; the
stock-op composition; and the opt-in term of SubspaceLoss."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import rel_l2
from dice_reference import U, _taps, blob_labels, dice_reference, stock_dice_loss
from liftreg_b200 import synthetic
from oracle import torch_port

pytestmark = pytest.mark.gpu

K_GRAD = 16          # gradient bar in units of u * abs-scale (derived in DESIGN.md section 3)
SHAPES = [(1, (5, 6, 7)), (2, (17, 33, 40)), (1, (1, 9, 70)), (2, (6, 1, 33)), (1, (4, 5, 1)), (2, (24, 31, 51)),
          (1, (37, 19, 45)), (1, (2, 2, 2))]
MAPS = ["smooth", "noisy", "out_of_range", "identity"]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def identity(shape):
    """the library's identity map (n = 1 axes: the single voxel at -1, where the warp samples it)"""
    safe = tuple(max(n, 2) for n in shape)
    idm = torch_port.identity_map(safe).numpy()
    return np.ascontiguousarray(idm[:, :shape[0], :shape[1], :shape[2]])


def make_map(kind, B, shape, seed):
    """smooth: identity + a smooth displacement of a few voxels; noisy: plus uniform noise of 0.6 grid steps;
    out_of_range: the smooth map stretched by 1.4 about the centre, so a rim of voxels samples outside; identity"""
    idm = np.repeat(identity(shape)[None], B, 0)
    if kind == "identity":
        return idm.astype(np.float32)
    steps = np.array([2.0 / max(n - 1, 1) for n in shape]).reshape(1, 3, 1, 1, 1)
    rs = np.random.RandomState(seed)
    disp = np.stack([synthetic.smooth_displacement(tuple(max(n, 2) for n in shape), seed=seed + b, max_disp=0.5, coarse=4)
                     [:, :shape[0], :shape[1], :shape[2]] for b in range(B)])
    phi = idm + 3.0 * steps * disp / max(np.abs(disp).max(), 1e-9)
    if kind == "noisy":
        phi = phi + 0.6 * steps * rs.uniform(-1, 1, phi.shape)
    if kind == "out_of_range":
        phi = 1.4 * phi
    return phi.astype(np.float32)


def plant_invalid(src, tgt, L, seed):
    """NaN, -1, 2.5 and L in both maps at a few voxels each: no label"""
    rs = np.random.RandomState(seed)
    for m in (src, tgt):
        flat = m.reshape(-1)
        for v in (np.nan, -1.0, 2.5, float(L)):
            flat[rs.randint(0, flat.size, max(1, flat.size // 200))] = v
    return src, tgt


def labels_for(B, shape, L, seed):
    if L <= 8:
        src, tgt = blob_labels(B, shape, L, seed=seed, shift=1)
    else:                                   # many labels: blocky random regions
        rs = np.random.RandomState(seed)
        coarse = rs.randint(0, L, (B,) + tuple(max(1, n // 6 + 1) for n in shape)).astype(np.float32)
        src = coarse.repeat(6, 1).repeat(6, 2).repeat(6, 3)[:, :shape[0], :shape[1], :shape[2]]
        tgt = np.roll(src, 2, axis=1)
    return np.ascontiguousarray(src), np.ascontiguousarray(tgt)


def vp(t):
    return ctypes.c_void_p(t.data_ptr())


def c_sums(phi, src, tgt, L):
    from liftreg_b200 import _native, ops
    B, _, D, H, W = phi.shape
    sums = torch.full((B, L, 3), float("nan"), device=phi.device, dtype=torch.float64)
    _native.check(_native.lib().lr_label_dice_sums(vp(phi), vp(src), vp(tgt), B, D, H, W, L, vp(sums), ops._stream()),
                  "lr_label_dice_sums")
    return sums


def c_backward(phi, src, tgt, L, sums, grad_loss, out=None):
    from liftreg_b200 import _native, ops
    B, _, D, H, W = phi.shape
    g = torch.tensor([grad_loss], device=phi.device, dtype=torch.float32)
    out = torch.full_like(phi, float("nan")) if out is None else out
    _native.check(_native.lib().lr_label_dice_backward(vp(phi), vp(src), vp(tgt), B, D, H, W, L, vp(sums), vp(g), vp(out),
                                                       ops._stream()), "lr_label_dice_backward")
    return out


def uniform_voxels(phi, src, L):
    """(B,D,H,W) bool: the voxels whose 8 taps carry one label (or none: all outside / no label)"""
    labs = np.stack([t[3] for t in _taps(phi, src, L)[0]])
    return np.all(labs == labs[0], axis=0)


def check_all(phi, src, tgt, L, sums_t, grad_t, grad_loss):
    from liftreg_b200 import ops
    ref_sums, ref_loss, ref_grad, scale = dice_reference(phi, src, tgt, L, grad_loss)
    sums = sums_t.cpu().numpy()
    assert np.array_equal(sums[..., 2], ref_sums[..., 2])
    assert np.all(np.abs(sums[..., :2] - ref_sums[..., :2]) <= 1e-12 * np.abs(ref_sums[..., :2]))
    loss = ops._dice_loss_from_sums(sums_t).to(torch.float32).item()
    assert abs(loss - ref_loss) <= np.spacing(np.float32(ref_loss)), (loss, ref_loss)
    got = grad_t.cpu().numpy().astype(np.float64)
    assert np.all(np.isfinite(got))
    err = np.abs(got - ref_grad)
    assert np.all(err <= K_GRAD * U * scale), "max err / (u scale) = %g" % (err / np.where(scale > 0, U * scale, np.inf)).max()
    assert np.all(got[scale == 0] == 0)
    assert np.all(got.transpose(1, 0, 2, 3, 4)[:, uniform_voxels(phi, src, L)] == 0)
    return ref_loss


@pytest.mark.parametrize("L", [2, 6])
@pytest.mark.parametrize("kind", MAPS)
@pytest.mark.parametrize("B,shape", SHAPES)
def test_sums_loss_and_gradient_match_reference(dev, B, shape, kind, L):
    phi = make_map(kind, B, shape, seed=sum(shape) + B)
    src, tgt = plant_invalid(*labels_for(B, shape, L, seed=L + B), L, seed=3)
    phi_t, src_t, tgt_t = (torch.from_numpy(a).to(dev) for a in (phi, src, tgt))
    sums = c_sums(phi_t, src_t, tgt_t, L)
    grad = c_backward(phi_t, src_t, tgt_t, L, sums, 0.75)
    check_all(phi, src, tgt, L, sums, grad, 0.75)
    assert torch.equal(c_backward(phi_t, src_t, tgt_t, L, sums, 0.75), grad)          # same sums: same bits


@pytest.mark.parametrize("L", [2, 6, 128])
def test_160_cubed(dev, L):
    shape = (160, 160, 160)
    phi = make_map("noisy", 1, shape, seed=5)
    src, tgt = labels_for(1, shape, L, seed=L)
    phi_t, src_t, tgt_t = (torch.from_numpy(a).to(dev) for a in (phi, src, tgt))
    sums = c_sums(phi_t, src_t, tgt_t, L)
    check_all(phi, src, tgt, L, sums, c_backward(phi_t, src_t, tgt_t, L, sums, 1.0), 1.0)


def offset_view(a, dev):
    buf = torch.full((a.size + 1,), float("nan"), device=dev)
    buf[1:] = torch.from_numpy(np.ascontiguousarray(a).reshape(-1)).to(dev)
    return buf, buf[1:].view(a.shape)


@pytest.mark.parametrize("B,shape", [(1, (33, 20, 64)), (2, (9, 8, 10)), (1, (37, 19, 45))])
def test_unaligned_views(dev, B, shape):
    L = 6
    phi = make_map("noisy", B, shape, seed=7)
    src, tgt = labels_for(B, shape, L, seed=7)
    (_, phi_v), (_, src_v), (_, tgt_v) = (offset_view(a, dev) for a in (phi, src, tgt))
    obuf, out = offset_view(np.zeros_like(phi), dev)
    out.fill_(float("nan"))
    assert phi_v.data_ptr() % 8 == 4 and out.data_ptr() % 8 == 4
    sums = c_sums(phi_v, src_v, tgt_v, L)
    c_backward(phi_v, src_v, tgt_v, L, sums, 0.75, out=out)
    check_all(phi, src, tgt, L, sums, out, 0.75)
    assert torch.isnan(obuf[0])                                                       # nothing written outside grad_phi


@pytest.mark.parametrize("L", [2, 3, 6])
@pytest.mark.parametrize("B,shape,shift", [(1, (9, 17, 33), (0, 0, 0)), (2, (17, 9, 5), (1, -2, 3)), (1, (33, 17, 9), (-3, 0, 2)),
                                           (2, (5, 5, 5), (6, 0, 0))])
def test_integer_shifts_give_exact_sums_and_the_validation_dice(dev, B, shape, shift, L):
    """n - 1 a power of two and whole-voxel shifts: every sample position is an integer, every weight 0 or 1, so I, P, T
    are the confusion counts of the nearest-warped labels and 1 - loss is the validation Dice"""
    from liftreg_b200 import metrics, ops
    steps = np.array([2.0 / (n - 1) for n in shape])
    phi = np.repeat((identity(shape) + (np.array(shift) * steps).reshape(3, 1, 1, 1))[None], B, 0).astype(np.float32)
    src, tgt = labels_for(B, shape, L, seed=11 * L)
    phi_t, src_t, tgt_t = (torch.from_numpy(a).to(dev) for a in (phi, src, tgt))
    sums = c_sums(phi_t, src_t, tgt_t, L)
    s = sums.cpu().numpy()
    assert np.array_equal(s, np.round(s))
    nearest = ops.warp(src_t[:, None], phi_t, zero_boundary=True, using_scale=False, mode="nearest")[:, 0]
    ov = metrics.label_overlap(nearest, tgt_t, L)
    c = ov["counts"]
    assert np.array_equal(s[:, 1:, 0], np.diagonal(c, axis1=1, axis2=2)[:, 1:])
    assert np.array_equal(s[:, 1:, 1], c.sum(2)[:, 1:]) and np.array_equal(s[:, :, 2], c.sum(1))
    assert not np.isnan(ov["dice_mean"]).any()
    loss = ops.label_dice_loss(phi_t, src_t, tgt_t, L)
    assert loss.item() == np.float32(1.0 - np.mean(ov["dice_mean"]))
    assert ops._dice_loss_from_sums(sums).item() == pytest.approx(1.0 - np.mean(ov["dice_mean"]), rel=1e-15, abs=1e-16)


def test_invalid_labels_contribute_nothing(dev):
    L, B, shape = 4, 2, (12, 13, 14)
    phi = make_map("noisy", B, shape, seed=2)
    src, tgt = labels_for(B, shape, L, seed=2)
    rs = np.random.RandomState(0)
    for m in (src, tgt):
        bad = rs.uniform(size=m.shape) < 0.2
        m[bad] = rs.choice([np.nan, -1.0, 2.5, float(L), 1e9], size=int(bad.sum()))
    phi_t, src_t, tgt_t = (torch.from_numpy(a).to(dev) for a in (phi, src, tgt))
    sums = c_sums(phi_t, src_t, tgt_t, L)
    check_all(phi, src, tgt, L, sums, c_backward(phi_t, src_t, tgt_t, L, sums, 1.0), 1.0)


def test_backward_bits_repeat_across_numerics_modes_and_batch(dev):
    from liftreg_b200 import _native
    L, shape = 6, (24, 31, 51)
    phi = make_map("noisy", 2, shape, seed=4)
    src, tgt = labels_for(2, shape, L, seed=4)
    phi_t, src_t, tgt_t = (torch.from_numpy(a).to(dev) for a in (phi, src, tgt))
    sums = c_sums(phi_t, src_t, tgt_t, L)
    prev = _native.set_numerics("exact")
    try:
        exact = c_backward(phi_t, src_t, tgt_t, L, sums, 1.0)
        _native.set_numerics("fast")
        fast = c_backward(phi_t, src_t, tgt_t, L, sums, 1.0)
    finally:
        _native.set_numerics(prev)
    assert torch.equal(exact, fast)
    pair = c_backward(phi_t, src_t, tgt_t, L, sums, 2.0)
    for b in range(2):
        one = c_backward(phi_t[b:b + 1].contiguous(), src_t[b:b + 1].contiguous(), tgt_t[b:b + 1].contiguous(), L,
                         sums[b:b + 1].contiguous(), 1.0)
        assert torch.equal(pair[b:b + 1], one)


@pytest.mark.parametrize("label_shape", ["5d", "4d", "int64"])
def test_autograd_gradient_equals_the_c_call(dev, label_shape):
    from liftreg_b200 import ops
    L, B, shape = 6, 2, (17, 33, 40)
    phi = make_map("smooth", B, shape, seed=8)
    src, tgt = labels_for(B, shape, L, seed=8)
    phi_t, src_t, tgt_t = (torch.from_numpy(a).to(dev) for a in (phi, src, tgt))
    s_in, t_in = src_t, tgt_t
    if label_shape == "5d":
        s_in, t_in = src_t[:, None], tgt_t[:, None]
    elif label_shape == "int64":
        s_in, t_in = src_t.long(), tgt_t.long()
    p = phi_t.clone().requires_grad_(True)
    loss = ops.label_dice_loss(p, s_in, t_in, L)
    assert loss.dtype == torch.float32 and loss.shape == ()
    sums = loss.grad_fn.saved_tensors[3]          # the forward's sums, read before backward() frees them
    (2.5 * loss).backward()
    assert torch.equal(p.grad, c_backward(phi_t, src_t, tgt_t, L, sums, 2.5))
    check_all(phi, src, tgt, L, sums, p.grad / 2.5, 1.0)
    with pytest.raises(ValueError, match="num_labels"):
        ops.label_dice_loss(phi_t, src_t, tgt_t, 1)
    with pytest.raises(ValueError, match="source_labels"):
        ops.label_dice_loss(phi_t, src_t[:, :-1], tgt_t, L)
    with pytest.raises(ValueError, match=r"\(B,3,D,H,W\)"):
        ops.label_dice_loss(phi_t[:, :2], src_t, tgt_t, L)
    with pytest.raises(TypeError, match="float32"):
        ops.label_dice_loss(phi_t.double(), src_t, tgt_t, L)


@pytest.mark.parametrize("L", [2, 6, 14])
def test_agrees_with_the_stock_op_composition(dev, L):
    from liftreg_b200 import ops
    B, shape = 2, (40, 36, 44)
    phi = make_map("smooth", B, shape, seed=L)
    src, tgt = labels_for(B, shape, L, seed=L)
    phi_t, src_t, tgt_t = (torch.from_numpy(a).to(dev) for a in (phi, src, tgt))
    p1, p2 = phi_t.clone().requires_grad_(True), phi_t.clone().requires_grad_(True)
    fused, stock = ops.label_dice_loss(p1, src_t, tgt_t, L), stock_dice_loss(p2, src_t, tgt_t, L)
    fused.backward()
    stock.backward()
    assert abs(fused.item() - stock.item()) <= 1e-6
    assert rel_l2(p1.grad.cpu().numpy(), p2.grad.cpu().numpy()) <= 2e-5


def loss_inputs(dev, B=2, shape=(24, 20, 28), seed=9, L=2):
    rs = np.random.RandomState(seed)
    disp = torch.from_numpy(make_map("noisy", B, shape, seed) - identity(shape)[None]).to(dev)
    warped = torch.from_numpy(rs.uniform(0, 1, (B, 1) + shape).astype(np.float32)).to(dev)
    target = torch.from_numpy(rs.uniform(0, 1, (B, 1) + shape).astype(np.float32)).to(dev)
    src, tgt = labels_for(B, shape, L, seed=seed)
    return disp, warped, target, torch.from_numpy(src[:, None]).to(dev), torch.from_numpy(tgt[:, None]).to(dev)


@pytest.mark.parametrize("opt", [None, {}, {"dice_factor": 0}, {"dice_factor": 0, "dice_num_labels": 6}])
def test_subspace_loss_without_dice_factor_is_unchanged(dev, opt):
    from liftreg_b200 import losses, ops
    disp, warped, target, src, tgt = loss_inputs(dev)
    res = losses.SubspaceLoss(opt)({"warped": warped, "target": target, "params": disp.clone().requires_grad_(True),
                                    "epoch": 12, "source_label": src, "target_label": tgt})
    assert sorted(res) == ["reg_loss", "sim_loss", "total_loss"]
    rf = losses.SubspaceLoss().get_reg_factor(12)
    sim, reg = ops.ncc_loss(warped.reshape(2, -1), target.reshape(2, -1)), ops.diffusion_reg(disp)
    assert torch.equal(res["total_loss"].detach(), 1. * sim + rf * reg)


@pytest.mark.parametrize("with_fold", [False, True])
def test_subspace_loss_dice_term_is_the_sum_of_its_parts(dev, with_fold):
    from liftreg_b200 import losses, ops
    L = 3
    disp, warped, target, src, tgt = loss_inputs(dev, L=L)
    df, ff = 0.4, 0.3
    opt = {"dice_factor": df, "dice_num_labels": L}
    if with_fold:
        opt["fold_factor"] = ff
    loss = losses.SubspaceLoss(opt)
    params = disp.clone().requires_grad_(True)
    res = loss({"warped": warped, "target": target, "params": params, "epoch": 3, "source_label": src, "target_label": tgt})
    assert sorted(res) == sorted(["dice_loss", "reg_loss", "sim_loss", "total_loss"] + (["fold_loss"] if with_fold else []))
    res["total_loss"].backward()

    rf = loss.get_reg_factor(3)
    p2 = disp.clone().requires_grad_(True)
    sim = ops.ncc_loss(warped.reshape(2, -1), target.reshape(2, -1))
    reg = ops.diffusion_reg(p2)
    phi = p2 + ops.identity_map(disp.shape[2:], dev)
    dice = ops.label_dice_loss(phi, src, tgt, L)
    total = 1. * sim + rf * reg
    if with_fold:
        fold = ops.fold_penalty(phi)
        total = total + ff * fold
        assert res["fold_loss"] == fold.item()
    total = total + df * dice
    assert 0 < dice.item() < 1 and res["dice_loss"] == dice.item()
    assert torch.allclose(res["total_loss"].detach(), total.detach(), rtol=1e-6, atol=0)
    parts = [rf * reg, df * dice] + ([ff * fold] if with_fold else [])
    grads = [torch.autograd.grad(t, p2, retain_graph=True)[0] for t in parts]
    assert torch.allclose(params.grad, sum(grads), rtol=0, atol=1e-6 * float(sum(grads).abs().max()))
