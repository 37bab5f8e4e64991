"""Soft Dice loss of the warped label map without a GPU: the float64 reference (tests/dice_reference.py) against float64
autograd of stock grid_sample on one-hot channels and against central differences, the SubspaceLoss opt keys and its
missing-key error, and argument validation of lr_label_dice_sums / lr_label_dice_backward through the C-ABI."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from dice_reference import blob_labels, dice_reference, label_index


def torch_dice64(phi, src, tgt, L):
    """the stock-op composition in float64: one-hot moving labels, grid_sample (align_corners, zeros padding), soft
    Dice over the labels 1..L-1 present in either map; returns the loss and the map tensor it was computed from"""
    p = torch.from_numpy(np.asarray(phi, np.float64)).requires_grad_(True)
    grid = p.flip(1).permute(0, 2, 3, 4, 1)                     # grid_sample's x is the last axis: phi channel 2
    labels = torch.arange(L).view(1, L, 1, 1, 1)
    oh = (torch.from_numpy(label_index(src, L))[:, None] == labels).double()
    tm = (torch.from_numpy(label_index(tgt, L))[:, None] == labels).double()
    warped = F.grid_sample(oh, grid, mode="bilinear", padding_mode="zeros", align_corners=True)
    P, I, T = warped.sum((2, 3, 4)), (warped * tm).sum((2, 3, 4)), tm.sum((2, 3, 4))
    den = P + T
    in_s = den > 0
    in_s[:, 0] = False
    n = in_s.sum(1)
    dice = torch.where(in_s, 2.0 * I / torch.where(in_s, den, 1.0), 0.0).sum(1) / n.clamp(min=1)
    dice = torch.where(n > 0, dice, 1.0)
    return 1.0 - dice.mean(), p, torch.stack([I, P, T], -1)


def dyadic_map(B, shape, seed, bits=8):
    """phi = -1 + j / 2^bits, j random, a little beyond [-1, 1]: with n - 1 a power of two, every coordinate, fraction and
    weight product is exact in fp32, so fp32 and float64 sampling coincide"""
    rs = np.random.RandomState(seed)
    q = 2 ** bits
    return (-1.0 + rs.randint(-q // 16, 2 * q + q // 16 + 1, (B, 3) + shape) / q).astype(np.float32)


@pytest.mark.parametrize("L", [2, 3, 6])
@pytest.mark.parametrize("B,shape", [(1, (5, 9, 17)), (2, (3, 5, 9)), (2, (9, 2, 5)), (1, (17, 9, 3))])
def test_reference_equals_float64_autograd_of_grid_sample(B, shape, L):
    phi = dyadic_map(B, shape, seed=sum(shape) + L)
    src, tgt = blob_labels(B, shape, L, seed=L, shift=1)
    tgt[0, 0, 0, 0] = -1.0                                       # no label: counts nowhere
    src[0, -1, -1, -1] = 2.5
    sums, loss, grad, scale = dice_reference(phi, src, tgt, L, grad_loss=0.75)
    t_loss, p, t_sums = torch_dice64(phi, src, tgt, L)
    (0.75 * t_loss).backward()
    assert np.array_equal(sums[..., 2], t_sums[..., 2].detach().numpy())
    assert np.allclose(sums, t_sums.detach().numpy(), rtol=1e-14, atol=0)
    assert loss == pytest.approx(t_loss.item(), rel=1e-14, abs=1e-15)
    auto = p.grad.numpy()
    assert np.all(np.abs(grad - auto) <= 1e-12 * scale)
    assert np.all(grad[scale == 0] == 0) and np.all(auto[scale == 0] == 0)
    assert (scale > 0).mean() > 0.05


def smooth_offgrid_map(shape, seed):
    """identity shifted by half a voxel plus a smooth wobble of at most 0.25 voxel: every fraction stays in [0.2, 0.8],
    away from the integer coordinates where the derivative jumps"""
    rs = np.random.RandomState(seed)
    grids = np.meshgrid(*[np.arange(n, dtype=np.float64) for n in shape], indexing="ij")
    phi = np.empty((1, 3) + shape)
    for a, n in enumerate(shape):
        k = rs.uniform(0.5, 1.5, 3)
        wob = 0.25 * np.sin(k[0] * grids[0] + k[1] * grids[1] + k[2] * grids[2] + rs.uniform(0, 6))
        i = grids[a] + 0.5 + wob - (1.0 if a == 1 else 0.0)
        phi[0, a] = i / ((n - 1) / 2.0) - 1.0
    return phi.astype(np.float32)


@pytest.mark.parametrize("L", [2, 4])
def test_reference_matches_central_differences(L):
    shape = (6, 7, 9)
    phi = smooth_offgrid_map(shape, seed=L)
    src, tgt = blob_labels(1, shape, L, seed=10 + L, shift=2)
    _, loss, grad, _ = dice_reference(phi, src, tgt, L)
    p64 = phi.astype(np.float64)
    assert torch_dice64(p64, src, tgt, L)[0].item() == pytest.approx(loss, rel=1e-6)
    rs = np.random.RandomState(L)
    idx = [tuple(rs.randint(0, n) for n in p64.shape) for _ in range(80)]
    idx += [tuple(int(v) for v in np.unravel_index(np.argmax(np.abs(grad)), grad.shape))]
    eps = 1e-6
    top = np.abs(grad).max()
    assert top > 0
    for i in idx:
        hi, lo = p64.copy(), p64.copy()
        hi[i] += eps
        lo[i] -= eps
        fd = (torch_dice64(hi, src, tgt, L)[0].item() - torch_dice64(lo, src, tgt, L)[0].item()) / (2 * eps)
        assert abs(fd - grad[i]) <= 1e-5 * top, (i, fd, grad[i])


def test_subspace_loss_reads_dice_keys_and_names_a_missing_label_map():
    from liftreg_b200 import losses
    off = losses.SubspaceLoss()
    assert off.dice_factor == 0 and off.dice_num_labels == 2
    on = losses.SubspaceLoss({"dice_factor": 0.5, "dice_num_labels": 6})
    assert on.dice_factor == 0.5 and on.dice_num_labels == 6
    x = torch.zeros(1, 1, 4, 4, 4)
    base = {"warped": x, "target": x, "params": torch.zeros(1, 3, 4, 4, 4), "epoch": 0}
    with pytest.raises(KeyError, match="source_label"):
        on(dict(base, target_label=x))
    with pytest.raises(KeyError, match="target_label"):
        on(dict(base, source_label=x))


@pytest.fixture(scope="module")
def lib():
    from liftreg_b200 import _native, build
    build.build()
    return _native.lib()


def test_label_dice_entries_reject_bad_arguments_before_any_cuda_call(lib):
    f = ctypes.c_void_p(256)             # never dereferenced: every call below fails validation first
    s, g, o = ctypes.c_void_p(512), ctypes.c_void_p(768), ctypes.c_void_p(1024)
    shape = (1, 4, 4, 4)
    bad = [
        ((None, f, f) + shape + (2,), b"null"), ((f, None, f) + shape + (2,), b"null"), ((f, f, None) + shape + (2,), b"null"),
        ((f, f, f) + shape + (1,), b"L=1"), ((f, f, f) + shape + (129,), b"L=129"), ((f, f, f) + shape + (0,), b"L=0"),
        ((f, f, f, 0, 4, 4, 4, 2), b">= 1"), ((f, f, f, 1, 0, 4, 4, 2), b">= 1"), ((f, f, f, 1, 4, 0, 4, 2), b">= 1"),
        ((f, f, f, 1, 4, 4, 0, 2), b">= 1"), ((f, f, f, 1, 4, 4, -3, 2), b">= 1"),
        ((f, f, f, 1, 4, 4, 1 << 21, 2), b"2^21"), ((f, f, f, 3, 512, 512, 1024, 2), b"2^31"),
    ]
    for args, msg in bad:
        assert lib.lr_label_dice_sums(*args, s, None) == -1, args
        assert msg in lib.lr_last_error(), (args, lib.lr_last_error())
        assert lib.lr_label_dice_backward(*args, s, g, o, None) == -1, args
        assert msg in lib.lr_last_error(), (args, lib.lr_last_error())
    for k in range(3):                                           # the outputs and the backward's extra inputs
        bwd = [s, g, o]
        bwd[k] = None
        assert lib.lr_label_dice_backward(f, f, f, *shape, 2, *bwd, None) == -1
        assert b"null" in lib.lr_last_error()
    assert lib.lr_label_dice_sums(f, f, f, *shape, 2, None, None) == -1 and b"null" in lib.lr_last_error()
