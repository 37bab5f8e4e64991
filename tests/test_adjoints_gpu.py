"""Adjoints on the GPU against the float64 references of tests/adjoint_reference.py, element by element.

Bars, with u = 2^-24:
  d/dphi (a gather)             |k - ref| <= 32 u scale   (a few roundings in the lerp tree on terms bounded by scale)
  grad_img, grad_proj (scatter) |k - ref| <= (n + 3) u abs, n = contributions (any order of the fp32 atomics)
  DRR adjoint (scatter)         rel-L2 <= 2e-5 per item and |k - ref| <= 1e-4 abs per voxel (~1600 contributions)
and exactly 0 wherever the reference's scale is 0: taps all outside (zeros padding) or a border-clipped coordinate.

The warp matrix runs padding x using_scale x disp_plus_identity x (image gradient requested or not).  For zeros padding
the last axis selects the kernel: the packed two-voxel d/dphi kernel when only the map gradient is requested (a training
step), the generic adjoint otherwise; border padding always runs the generic adjoint.
"""
import ctypes
import zlib

import numpy as np
import pytest
import torch

from adjoint_reference import U, backproject_adjoint, warp_adjoint
from conftest import rel_l2

pytestmark = pytest.mark.gpu

PHI_ULPS = 32
DRR_GRAD_TOL = 2e-5
DRR_ABS_TOL = 1e-4
ADJOINT_TOL = 1e-5


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


@pytest.fixture
def native():
    """The library module; the numerics mode a test selects is restored afterwards."""
    from liftreg_b200 import _native
    prev = _native.get_numerics()
    yield _native
    _native.set_numerics(prev)


def cu(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def assert_gather(k, ref, scale, ulps, what):
    k = np.asarray(k, np.float64)
    err, lim = np.abs(k - ref), ulps * U * scale
    bad = err > lim
    assert not bad.any(), "%s: %d of %d outside %d u scale; worst %.3g u scale at %s" % (
        what, int(bad.sum()), bad.size, ulps, float((err / np.maximum(U * scale, 1e-300))[bad].max()),
        np.unravel_index(int(np.argmax(np.where(bad, err, 0))), bad.shape))
    assert np.all(k[scale == 0] == 0), what


def assert_scatter(k, ref, aval, cnt, what):
    k = np.asarray(k, np.float64)
    err, lim = np.abs(k - ref), (cnt + 3) * U * aval
    bad = err > lim
    assert not bad.any(), "%s: %d of %d outside (n + 3) u abs; worst at %s: kernel %r, reference %r, n %d" % (
        what, int(bad.sum()), bad.size, np.unravel_index(int(np.argmax(np.where(bad, err, 0))), bad.shape),
        k[bad][0], ref[bad][0], cnt[bad][0])
    assert np.all(k[aval == 0] == 0), what


def assert_adjoint(lhs, rhs, what):
    """<A x, y> == <x, A^T y> with x, y >= 0 (no cancellation: the relative bar is a bar on the terms)."""
    assert lhs > 0 and abs(lhs - rhs) <= ADJOINT_TOL * lhs, (what, lhs, rhs)


# ------------------------------------------------------------------ warp
# id: (B, C, (D, H, W), z_begin, Dz or None for the whole volume)
WARP_CASES = {
    "13x10x33": (2, 1, (13, 10, 33), 0, None),         # H % 8 != 0; W = 33: a second tile with one live lane
    "37x21x64": (1, 2, (37, 21, 64), 0, None),         # D >= 32: tapered 8 / 4 / 2-plane blocks; C > 1
    "9x8x31": (3, 3, (9, 8, 31), 0, None),
    "5x1x7": (1, 1, (5, 1, 7), 0, None),               # size-1 axes: every voxel on the scalar path
    "1x6x2": (1, 1, (1, 6, 2), 0, None),
    "37x21x64-slab4": (1, 2, (37, 21, 64), 4, 33),     # z-slab [4, 37) of the 37-plane case
}


def _base_map(shape, z_begin, Dz):
    """Identity map planes [z_begin, z_begin+Dz): the C oracle's (bit-exact with the kernel) where it is defined."""
    from oracle import c_oracle
    if min(shape) >= 2:
        return c_oracle.identity_map(shape)[:, z_begin:z_begin + Dz]
    grid = np.stack(np.meshgrid(*[np.linspace(-1.0, 1.0, n) for n in shape], indexing="ij")).astype(np.float32)
    return grid[:, z_begin:z_begin + Dz]


def warp_inputs(case, kind, ident):
    from liftreg_b200 import synthetic
    B, C, shape, z_begin, Dz = WARP_CASES[case]
    Dz = shape[0] if Dz is None else Dz
    rs = np.random.RandomState(zlib.crc32(("%s/%s/%d" % (case, kind, ident)).encode()))
    img = rs.uniform(-1, 1, (B, C) + shape).astype(np.float32)
    go = rs.standard_normal((B, C, Dz) + shape[1:]).astype(np.float32)
    if kind == "uniform":                               # many voxels partly or fully outside
        phi = rs.uniform(-1.3, 1.3, (B, 3, Dz) + shape[1:]).astype(np.float32)
    else:
        if kind == "smooth":                            # small smooth displacement: mostly the packed path
            disp = np.stack([synthetic.smooth_displacement(shape, seed=11 + b, max_disp=0.04, coarse=4)[:, z_begin:z_begin + Dz]
                             for b in range(B)])
        else:                                           # zero displacement: integer coordinates, phi = +-1 on the faces
            disp = np.zeros((B, 3, Dz) + shape[1:], np.float32)
        phi = disp if ident else (disp + _base_map(shape, z_begin, Dz)[None]).astype(np.float32)
    return img, phi, go, z_begin


def _warp_grads(dev, img, phi, go, zb, us, ident, z_begin, want_img):
    from liftreg_b200 import ops
    ti = cu(img, dev).requires_grad_(want_img)
    tp = cu(phi, dev).requires_grad_(True)
    out = ops.warp(ti, tp, zero_boundary=zb, using_scale=us, disp_plus_identity=ident,
                   z_begin=z_begin if phi.shape[2] != img.shape[2] else None)
    out.backward(cu(go, dev))
    return (ti.grad.cpu().numpy() if want_img else None), tp.grad.cpu().numpy()


@pytest.mark.parametrize("ident", [False, True], ids=["map", "disp+id"])
@pytest.mark.parametrize("us", [False, True], ids=["noscale", "scale"])
@pytest.mark.parametrize("zb", [True, False], ids=["zeros", "border"])
@pytest.mark.parametrize("kind", ["smooth", "uniform", "identity"])
@pytest.mark.parametrize("case", list(WARP_CASES))
def test_warp_adjoint_vs_float64(dev, native, case, kind, zb, us, ident):
    shape = WARP_CASES[case][2]
    if min(shape) == 1 and (ident or kind == "identity"):
        pytest.skip("the identity map is undefined on a size-1 axis")
    img, phi, go, z_begin = warp_inputs(case, kind, ident)
    gi_ref, gabs, gcnt, gp_ref, gscale = warp_adjoint(go, img, phi, zb, us, ident, z_begin)
    assert (gscale > 0).any()

    # image gradient requested: the generic adjoint (scatter + gather in one kernel)
    gi, gp = _warp_grads(dev, img, phi, go, zb, us, ident, z_begin, want_img=True)
    assert_scatter(gi, gi_ref, gabs, gcnt, "grad_img")
    assert_gather(gp, gp_ref, gscale, PHI_ULPS, "grad_phi (with grad_img)")

    # map gradient only (zeros padding: the packed kernel), in both numerics modes and twice: a gather, so the bits
    # are the same every time
    gps = []
    for mode in ("exact", "fast", "fast"):
        native.set_numerics(mode)
        gps.append(_warp_grads(dev, img, phi, go, zb, us, ident, z_begin, want_img=False)[1])
    assert_gather(gps[0], gp_ref, gscale, PHI_ULPS, "grad_phi (map only)")
    assert np.array_equal(gps[0], gps[1]) and np.array_equal(gps[1], gps[2])


def test_warp_adjoint_full_size_training_configuration(dev):
    """The training step's d/dphi: 160^3, batch 2, one channel, zeros padding, using_scale, identity fused."""
    from liftreg_b200 import synthetic
    rs = np.random.RandomState(21)
    shape = (160, 160, 160)
    img = rs.uniform(-1, 1, (2, 1) + shape).astype(np.float32)
    disp = np.stack([synthetic.smooth_displacement(shape, seed=31 + b) for b in range(2)])
    go = rs.standard_normal((2, 1) + shape).astype(np.float32)
    _, gp = _warp_grads(dev, img, disp, go, True, True, True, 0, want_img=False)
    for b in range(2):
        _, _, _, ref, scale = warp_adjoint(go[b:b + 1], img[b:b + 1], disp[b:b + 1], True, True, True, want_img=False)
        assert_gather(gp[b:b + 1], ref, scale, PHI_ULPS, "grad_phi item %d" % b)


def test_warp_nearest_adjoint(dev, native):
    """Nearest sampling is piecewise constant: zero map gradient; an image gradient is refused (Python and C-ABI)."""
    from liftreg_b200 import ops
    rs = np.random.RandomState(22)
    img = cu(rs.uniform(-1, 1, (2, 2, 7, 9, 11)).astype(np.float32), dev)
    phi = rs.uniform(-1.1, 1.1, (2, 3, 7, 9, 11)).astype(np.float32)
    go = cu(rs.standard_normal((2, 2, 7, 9, 11)).astype(np.float32), dev)
    for zb in (False, True):
        tp = cu(phi, dev).requires_grad_(True)
        ops.warp(img, tp, zero_boundary=zb, mode="nearest").backward(go)
        assert bool((tp.grad == 0).all())
    with pytest.raises(NotImplementedError):
        ops.warp(img.clone().requires_grad_(True), cu(phi, dev), mode="nearest").backward(go)
    gimg = torch.zeros_like(img)
    gphi = torch.empty((2, 3, 7, 9, 11), device=dev)
    p = lambda t: ctypes.c_void_p(t.data_ptr())
    lib = native.lib()
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    assert lib.lr_warp_backward(p(go), p(img), p(cu(phi, dev)), 2, 2, 7, 9, 11, 0, 1, 1, 0, p(gimg), p(gphi), st) == -1
    assert b"nearest" in lib.lr_last_error()


@pytest.mark.parametrize("shape", [(5, 1, 7), (1, 6, 2), (4, 5, 1)])
def test_warp_fused_identity_rejects_size_one_axes(dev, shape):
    from liftreg_b200 import ops
    img = torch.zeros((1, 1) + shape, device=dev)
    disp = torch.zeros((1, 3) + shape, device=dev, requires_grad=True)
    with pytest.raises(RuntimeError, match="disp_plus_identity"):
        ops.warp(img, disp, disp_plus_identity=True)
    ops.warp(img, disp).sum().backward()                # the same shapes without the identity are fine
    assert bool(torch.isfinite(disp.grad).all())


# ------------------------------------------------------------------ backprojection
def bp_poses(shape, P):
    from liftreg_b200 import synthetic
    poses = synthetic.wrapper_poses(60.0, P, shape[1]).astype(np.float32)
    if P > 2:
        poses[1, 1] = shape[1] * 1.02          # an emitter close to the volume: strong magnification, rows leave the detector
    return poses


@pytest.mark.parametrize("shape,pshape,B,P", [((5, 7, 3), (9, 4), 1, 1),
                                              ((33, 6, 70), (40, 31), 3, 2),        # d > 32: several plane chunks
                                              ((40, 9, 300), (64, 350), 1, 2),      # h > 256: threads loop over columns
                                              ((2, 2, 2), (1, 1), 2, 66),           # P > 64: two view chunks
                                              ((160, 160, 160), (256, 256), 2, 4)])
def test_backproject_adjoint_vs_float64(dev, native, shape, pshape, B, P):
    from liftreg_b200 import ops
    rs = np.random.RandomState(23)
    poses = bp_poses(shape, P)
    go = rs.standard_normal((B, P) + shape).astype(np.float32)
    ref, rabs, cnt = backproject_adjoint(go, poses, pshape)
    tp = torch.zeros((B, P) + pshape, device=dev, requires_grad=True)
    ops.backproject(tp, poses, shape).backward(cu(go, dev))
    assert_scatter(tp.grad.cpu().numpy(), ref, rabs, cnt, "grad_proj")

    x = cu(rs.uniform(0, 1, (B, P) + pshape).astype(np.float32), dev)
    y = cu(rs.uniform(0, 1, (B, P) + shape).astype(np.float32), dev)
    ty = torch.zeros((B, P) + pshape, device=dev, requires_grad=True)
    ops.backproject(ty, poses, shape).backward(y)
    rhs = float((x.double() * ty.grad.double()).sum())
    for mode in ("exact", "fast"):
        native.set_numerics(mode)
        lhs = float((ops.backproject(x, poses, shape).double() * y.double()).sum())
        assert_adjoint(lhs, rhs, mode)


@pytest.mark.parametrize("shape,pshape,B,P", [((5, 7, 3), (9, 4), 2, 1), ((33, 6, 70), (40, 31), 3, 2)])
def test_backproject_adjoint_through_concat_buffer(dev, shape, pshape, B, P):
    """backproject(out=buf, channel_offset=1) writes channels 1..P of the encoder's input buffer: the projections get
    the adjoint of those channels' gradient, and the buffer's previous content gets the rest of it, channels 1..P
    zeroed (they were overwritten)."""
    from liftreg_b200 import ops
    rs = np.random.RandomState(24)
    poses = bp_poses(shape, P)
    base = torch.full((B, P + 2) + shape, 7.0, device=dev, requires_grad=True)
    buf = base.clone()
    tp = cu(rs.uniform(-1, 1, (B, P) + pshape).astype(np.float32), dev).requires_grad_(True)
    ret = ops.backproject(tp, poses, shape, out=buf, channel_offset=1)
    G = rs.standard_normal((B, P + 2) + shape).astype(np.float32)
    ret.backward(cu(G, dev))
    ref, rabs, cnt = backproject_adjoint(G[:, 1:1 + P], poses, pshape)
    assert_scatter(tp.grad.cpu().numpy(), ref, rabs, cnt, "grad_proj")
    expect = G.copy()
    expect[:, 1:1 + P] = 0
    assert np.array_equal(base.grad.cpu().numpy(), expect)


# ------------------------------------------------------------------ DRR
def _drr_case(name):
    from liftreg_b200 import synthetic
    rs = np.random.RandomState(25)
    if name == "per-item-poses":
        shape, res, B, P, ym, osc = (14, 12, 18), (20, 26), 2, 3, 0, 0.1
        poses = np.stack([synthetic.wrapper_poses(60.0, P, shape[1]), synthetic.wrapper_poses(40.0, P, shape[1], 3.0)])
        poses[1, :, 2] += 1.5
    elif name == "140-pairs":
        shape, res, B, P, ym, osc = (9, 8, 10), (12, 14), 2, 70, 0, 0.1
        poses = synthetic.wrapper_poses(80.0, P, shape[1])
    elif name == "ynorm-w":
        shape, res, B, P, ym, osc = (10, 12, 9), (16, 20), 2, 2, 1, 1.0
        poses = synthetic.wrapper_poses(60.0, P, shape[1])
    else:                                               # "1x4x1": size-1 axes
        shape, res, B, P, ym, osc = (1, 4, 1), (3, 3), 2, 2, 0, 0.1
        poses = synthetic.wrapper_poses(60.0, P, shape[1])
    go = rs.standard_normal((B, P) + res).astype(np.float32)
    return shape, res, B, P, ym, osc, poses, go


@pytest.mark.parametrize("name", ["per-item-poses", "140-pairs", "ynorm-w", "1x4x1"])
def test_drr_adjoint_vs_oracle(dev, native, name):
    from liftreg_b200 import ops
    from oracle import c_oracle
    shape, res, B, P, ym, osc, poses, go = _drr_case(name)
    sp = (2.2, 2.2, 2.2)
    v = torch.zeros((B,) + shape, device=dev, requires_grad=True)
    ops.drr_project(v, poses, res, sp, y_norm_mode=ym, out_scale=osc).backward(cu(go, dev))
    k = v.grad.cpu().numpy()
    for b in range(B):
        pb = poses[b] if poses.ndim == 3 else poses
        ref = c_oracle.drr_backward(go[b:b + 1], shape, pb, sp, ym, osc)[0]
        aval = c_oracle.drr_backward(np.abs(go[b:b + 1]), shape, pb, sp, ym, osc)[0]
        assert aval.max() > 0
        assert rel_l2(k[b], ref) <= DRR_GRAD_TOL, b
        err = np.abs(k[b].astype(np.float64) - ref)
        assert np.all(err <= DRR_ABS_TOL * aval.astype(np.float64)), (b, float((err / np.maximum(aval, 1e-30)).max()))

    rs = np.random.RandomState(26)
    x = cu(rs.uniform(0, 1, (B,) + shape).astype(np.float32), dev)
    y = cu(np.abs(go), dev)
    vy = torch.zeros((B,) + shape, device=dev, requires_grad=True)
    ops.drr_project(vy, poses, res, sp, y_norm_mode=ym, out_scale=osc).backward(y)
    rhs = float((x.double() * vy.grad.double()).sum())
    for mode in ("exact", "fast"):
        native.set_numerics(mode)
        lhs = float((ops.drr_project(x, poses, res, sp, y_norm_mode=ym, out_scale=osc).double() * y.double()).sum())
        assert_adjoint(lhs, rhs, mode)
