"""The float64 adjoint references of tests/adjoint_reference.py, without a GPU: against the C oracle's adjoints, and the
warp reference against float64 autograd of stock torch's grid_sample on grids where fp32 and fp64 coordinates agree."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from adjoint_reference import U, backproject_adjoint, warp_adjoint
from oracle import c_oracle


@pytest.fixture(autouse=True)
def aten_blend():
    prev = c_oracle.set_blend("aten")
    yield
    c_oracle.set_blend(prev)


@pytest.mark.parametrize("B,C,shape", [(2, 1, (6, 5, 9)), (1, 2, (7, 4, 5)), (2, 3, (3, 8, 2))])
@pytest.mark.parametrize("zb", [False, True])
@pytest.mark.parametrize("us", [False, True])
def test_warp_reference_vs_oracle(B, C, shape, zb, us):
    rs = np.random.RandomState(5)
    img = rs.uniform(-1, 1, (B, C) + shape).astype(np.float32)
    phi = rs.uniform(-1.2, 1.2, (B, 3) + shape).astype(np.float32)
    go = rs.standard_normal((B, C) + shape).astype(np.float32)
    gi, gabs, gcnt, gp, gscale = warp_adjoint(go, img, phi, zb, us)
    ogi, ogp = c_oracle.warp_backward(go, img, phi, zb, us, "bilinear")
    assert np.all(np.abs(ogi - gi) <= 4 * U * gabs)
    assert np.all(np.abs(ogp - gp) <= 4 * U * gscale)
    assert gcnt.min() >= 0 and gcnt.max() > 0
    assert np.all(gi[gcnt == 0] == 0) and np.all(gp[gscale == 0] == 0)


def test_warp_reference_slab_and_fused_identity():
    """The slab form computes the full result's planes of d/dphi; the fused identity is the fp32 add of the map."""
    rs = np.random.RandomState(6)
    B, C, shape = 1, 2, (9, 5, 6)
    img = rs.uniform(-1, 1, (B, C) + shape).astype(np.float32)
    disp = rs.uniform(-0.3, 0.3, (B, 3) + shape).astype(np.float32)
    go = rs.standard_normal((B, C) + shape).astype(np.float32)
    full = warp_adjoint(go, img, disp + c_oracle.identity_map(shape)[None], True, True)
    fused = warp_adjoint(go, img, disp, True, True, disp_plus_identity=True)
    for a, b in zip(full, fused):
        assert np.array_equal(a, b)
    z0, z1 = 3, 7
    slab = warp_adjoint(go[:, :, z0:z1], img, disp[:, :, z0:z1], True, True, disp_plus_identity=True, z_begin=z0)
    assert np.array_equal(slab[3], full[3][:, :, z0:z1]) and np.array_equal(slab[4], full[4][:, :, z0:z1])


def _torch_warp_grads(go, img, phi, zb, us):
    """net_utils.Bilinear (reference net_utils.py:26-56) on stock torch in float64, differentiated by autograd."""
    x = torch.from_numpy(img.astype(np.float64)).requires_grad_(True)
    p = torch.from_numpy(phi.astype(np.float64)).requires_grad_(True)
    src = (x + 1) / 2 if us else x
    grid = p.permute(0, 2, 3, 4, 1)[..., [2, 1, 0]]
    out = F.grid_sample(src, grid, mode="bilinear", padding_mode="zeros" if zb else "border", align_corners=True)
    if us:
        out = out * 2 - 1
    out.backward(torch.from_numpy(go.astype(np.float64)))
    return x.grad.numpy(), p.grad.numpy()


@pytest.mark.parametrize("shape", [(17, 5, 33), (9, 17, 17)])
@pytest.mark.parametrize("zb", [False, True])
@pytest.mark.parametrize("us", [False, True])
def test_warp_reference_vs_torch_grid_sample_on_dyadic_grid(shape, zb, us):
    """Along each axis of size S with S - 1 a power of two, and with map values that are multiples of 2^-12, the
    coordinates (g + 1) (S - 1) / 2 are exact in fp32 and in fp64, so both see the same floors.  A third of the values
    sit on a face (g = +-1), on a voxel centre, or just outside, where the one-sided derivative and the border clip
    decide.  The other two axes (sizes 5 and 9) are left at g = 0 exactly, i.e. on a voxel centre."""
    rs = np.random.RandomState(7)
    B, C = 2, 2
    img = rs.uniform(-1, 1, (B, C) + shape).astype(np.float32)
    go = rs.standard_normal((B, C) + shape).astype(np.float32)
    phi = np.zeros((B, 3) + shape, np.float32)
    for a, S in enumerate(shape):
        if (S - 1) & (S - 2):
            continue
        g = np.round(rs.uniform(-1.2, 1.2, phi[:, a].shape) * 4096) / 4096
        special = np.array([-1.0, 1.0, 0.0, 2.0 / (S - 1) - 1.0, 1.0 - 2.0 / (S - 1), -1.0 - 2.0 ** -12, 1.0 + 2.0 ** -12])
        pick = rs.rand(*g.shape) < 1 / 3
        g[pick] = special[rs.randint(0, len(special), int(pick.sum()))]
        phi[:, a] = g
    gi, gabs, _, gp, gscale = warp_adjoint(go, img, phi, zb, us)
    tgi, tgp = _torch_warp_grads(go, img, phi, zb, us)
    assert np.all(np.abs(tgi - gi) <= 1e-12 * gabs)
    assert np.all(np.abs(tgp - gp) <= 1e-12 * gscale)
    assert (gscale > 0).any() and np.abs(gp).max() > 0.1


@pytest.mark.parametrize("shape,pshape,B,P", [((5, 7, 3), (9, 4), 2, 1), ((12, 6, 20), (16, 11), 1, 3),
                                              ((4, 5, 4), (2, 3), 2, 2)])
def test_backproject_reference_vs_oracle(shape, pshape, B, P):
    from liftreg_b200 import synthetic
    rs = np.random.RandomState(8)
    go = rs.standard_normal((B, P) + shape).astype(np.float32)
    poses = synthetic.wrapper_poses(60.0, P, shape[1]).astype(np.float32)
    ref, rabs, cnt = backproject_adjoint(go, poses, pshape)
    ora = c_oracle.backproject_backward(go, poses, pshape)
    assert np.all(np.abs(ora - ref) <= 4 * U * rabs)
    assert np.all(ref[cnt == 0] == 0) and cnt.max() > 0


@pytest.fixture(scope="module")
def lib():
    from liftreg_b200 import _native, build
    build.build()
    return _native.lib()


def test_fused_identity_rejects_size_one_axes_before_any_cuda_call(lib):
    """The identity map (S - 1 in a denominator) is undefined on a size-1 axis: the warp entries refuse
    disp_plus_identity there instead of computing NaN."""
    fake = ctypes.c_void_p(256)          # never dereferenced: every call below fails validation first
    for D, H, W in ((1, 6, 2), (5, 1, 7), (4, 4, 1)):
        for fn, args in ((lib.lr_warp_forward_slab, (fake, fake, 1, 1, D, H, W, 0, D, 0, 0, 1, 1, fake, None)),
                         (lib.lr_warp_backward_slab, (fake, fake, fake, 1, 1, D, H, W, 0, D, 0, 0, 1, 1, None, fake, None))):
            assert fn(*args) == -1, (fn, D, H, W)
            assert b"disp_plus_identity" in lib.lr_last_error()
