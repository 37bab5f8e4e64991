"""GPU parity: the CUDA path (through the C-ABI) against the CPU oracle and the reference-generated goldens.

Bars (BASELINE.json north_star): coordinates, indices and weights bit-exact; sampled outputs <= 1e-5 relative L2
per image / per volume in fp32.  Where the op order is fully reproduced (warp, backprojection, DRR with the
oracle's sequential ray sum) the comparison is exact equality.
"""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_l2

pytestmark = pytest.mark.gpu

TOL = 1e-5          # north-star tolerance, relative L2 per image / volume
GRAD_TOL = 2e-5     # gradients: fp32 atomics reorder the scatter sums
FAST_TOL = 1e-6     # LR_NUMERICS_FAST vs the reference's (ATen-order) values: blends reassociated, indices identical


@pytest.fixture(autouse=True, params=["exact", "fast"])
def numerics(request):
    """Every test runs in both numerics modes of the library (include/liftreg_b200.h).  The oracle's blend order
    follows, so comparisons against the oracle stay BIT-EXACT in both modes (in fast mode that proves the indices and
    weights are the reference's); comparisons against reference-generated goldens are exact in `exact` mode and
    <= FAST_TOL in `fast` mode (assert_ref)."""
    from liftreg_b200 import _native
    from oracle import c_oracle
    prev = _native.set_numerics(request.param)
    prev_blend = c_oracle.set_blend("fast" if request.param == "fast" else "aten")
    yield request.param
    _native.set_numerics(prev)
    c_oracle.set_blend(prev_blend)


def assert_ref(out, ref, numerics):
    """`out` against values produced by the reference itself (goldens, torch ops)."""
    out = np.asarray(out); ref = np.asarray(ref)
    if numerics == "exact":
        assert np.array_equal(out, ref)
    else:
        assert rel_l2(out, ref) <= FAST_TOL
        assert float(np.abs(out.astype(np.float64) - ref).max()) <= 4e-6 * max(1.0, float(np.abs(ref).max()))


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    from liftreg_b200 import _native
    assert _native.lib().lr_device_count() >= 1
    return torch.device("cuda:0")


def cu(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def per_image_rel_l2(a, b):
    a = a.reshape(-1, a.shape[-2], a.shape[-1]); b = b.reshape(a.shape)
    return max(rel_l2(x, y) for x, y in zip(a, b))


# ------------------------------------------------------------------ ray geometry
@pytest.mark.parametrize("name", ["ray_grid_even", "ray_grid_odd"])
def test_project_grid_bit_exact_vs_reference_golden(dev, name):
    from liftreg_b200 import sdct_projection_utils as sdct
    g = load_golden(name)
    grid, dx = sdct.project_grid_multi(g["poses"], g["resolution"], [1, 1, 1], g["obj_shape"],
                                       torch.from_numpy(g["spacing"]), dev, torch.float32)
    assert np.array_equal(grid.cpu().numpy(), g["grid"])
    assert np.array_equal(dx.cpu().numpy(), g["dx"])


def test_proj_layer_grid_bit_exact_vs_reference_golden(dev):
    from liftreg_b200 import layers
    g = load_golden("ray_grid_projlayer")
    layer = layers.proj_layer(torch.from_numpy(g["spacing"]), 1.5, 40.0, 3, tuple(g["obj_shape"]), (8, 8), dev)
    assert np.array_equal(layer.dx.cpu().numpy(), g["dx"])
    assert np.array_equal(layer.grids.cpu().numpy(), g["grid_flipped"])


def test_project_grid_vs_oracle_full_detector(dev):
    """160^3 geometry, 240^2 detector, 1 view: every one of the 9.2 M sample coordinates bit-identical."""
    from liftreg_b200 import ops, synthetic
    from oracle import c_oracle
    poses = synthetic.wrapper_poses(60.0, 4, 160)[1:2]
    grid, dx = ops.project_grid(poses, (240, 240), (160, 160, 160), (2.2, 2.2, 2.2), dev)
    og, odx = c_oracle.project_grid(poses, (240, 240), (160, 160, 160), (2.2, 2.2, 2.2))
    assert np.array_equal(dx.cpu().numpy(), odx)
    assert np.array_equal(grid.cpu().numpy(), og)


# ------------------------------------------------------------------ DRR forward
def test_drr_small_vs_golden_and_oracle(dev):
    from liftreg_b200 import sdct_projection_utils as sdct
    from oracle import c_oracle
    g = load_golden("drr_small")
    out = sdct.calculate_projection(g["vol"], g["poses"], g["resolution"], [1, 1, 1], tuple(g["spacing"]), dev)
    assert out.shape == g["proj"].shape and out.dtype == np.float32
    assert per_image_rel_l2(out, g["proj"]) <= TOL                       # reference (torch.sum cascade order)
    ora = c_oracle.drr_forward(g["vol"], g["poses"], g["resolution"], g["spacing"],
                               seg_len=c_oracle.kernel_seg_len(g["vol"].shape[1]))
    assert np.array_equal(out, ora)                                      # same fp32 ray-segment sum order: exact


def test_drr_csv_poses_and_anisotropic_spacing(dev):
    from liftreg_b200 import sdct_projection_utils as sdct
    g = load_golden("drr_small_csvposes")
    out = sdct.calculate_projection(g["vol"], g["poses"], g["resolution"], [1, 1, 1], tuple(g["spacing"]), dev)
    assert per_image_rel_l2(out, g["proj"]) <= TOL


def test_calculate_projection_wraper_with_geo_csv_file(dev, tmp_path):
    """sdct:161-177 executed end to end: emitter positions in mm from a CSV with a header line, divided by the spacing;
    default detector int(1.5 d) x int(1.5 h); numpy in, numpy out."""
    from liftreg_b200 import sdct_projection_utils as sdct
    from oracle import c_oracle
    g = load_golden("drr_small_csvposes")
    spacing = tuple(float(s) for s in g["spacing"])
    mm = g["poses"] * np.asarray(spacing)                                  # the CSV holds millimetres
    geo = tmp_path / "geo.csv"
    geo.write_text("x,y,z\n" + "\n".join(",".join(repr(float(v)) for v in row) for row in mm) + "\n")
    proj, poses = sdct.calculate_projection_wraper_with_geo_csv_file(g["vol"], spacing, str(geo), receptor_size=(30, 30))
    assert isinstance(proj, np.ndarray) and proj.dtype == np.float32 and proj.shape == g["proj"].shape
    assert np.allclose(poses, g["poses"], rtol=1e-15, atol=0)
    assert per_image_rel_l2(proj, g["proj"]) <= TOL                          # the reference's own output for these poses
    assert np.array_equal(proj, c_oracle.drr_forward(g["vol"], poses, (30, 30), spacing, seg_len=c_oracle.kernel_seg_len(g["vol"].shape[1])))
    d, _, h = g["vol"].shape                                                 # default detector: int(1.5 d) x int(1.5 h) (sdct:168-171)
    proj2, _ = sdct.calculate_projection_wraper_with_geo_csv_file(g["vol"], spacing, str(geo))
    assert proj2.shape == (poses.shape[0], int(d * 1.5), int(h * 1.5))


def test_drr_cfg1_vs_reference_golden(dev):
    """BASELINE configs[0]: 160^3, 4 views / 60 deg, 240^2 detector, against the reference's CPU output."""
    from liftreg_b200 import sdct_projection_utils as sdct, synthetic
    g = load_golden("drr_cfg1")
    mu = synthetic.hu_to_mu(synthetic.ct_phantom((160, 160, 160)))
    assert abs(mu.astype(np.float64).sum() - float(g["mu_sum64"])) <= 1e-6 * abs(float(g["mu_sum64"]))
    proj, poses = sdct.calculate_projection_wraper(mu, 60.0, 4, (2.2, 2.2, 2.2))
    assert np.array_equal(poses, g["poses"])
    assert proj.shape == (4, 240, 240)
    for p in range(4):
        assert rel_l2(proj[p, ::6, ::6], g["proj_sub"][p]) <= TOL
        assert rel_l2(proj[p, 120, :], g["proj_row"][p]) <= TOL
    norms = np.sqrt((proj.astype(np.float64) ** 2).sum(axis=(1, 2)))
    assert np.allclose(norms, g["per_view_norm"], rtol=TOL, atol=0)
    assert abs(proj.astype(np.float64).sum() - float(g["sum64"])) <= TOL * abs(float(g["sum64"]))


@pytest.mark.parametrize("shape,res,P", [((7, 9, 5), (11, 3), 1), ((33, 17, 65), (50, 97), 5), ((1, 4, 1), (3, 3), 2),
                                         ((16, 2, 16), (40, 40), 3)])
def test_drr_ragged_shapes_vs_oracle(dev, shape, res, P):
    from liftreg_b200 import ops, synthetic
    from oracle import c_oracle
    rs = np.random.RandomState(1)
    vol = rs.rand(2, *shape).astype(np.float32)
    poses = synthetic.wrapper_poses(50.0, P, shape[1])
    out = ops.drr_project(cu(vol, dev), poses, res, (2.0, 1.5, 3.0)).cpu().numpy()
    ora = c_oracle.drr_forward(vol, poses, res, (2.0, 1.5, 3.0), seg_len=c_oracle.kernel_seg_len(shape[1]))
    assert np.array_equal(out, ora)


def test_drr_rays_that_miss_the_volume_are_exactly_zero(dev):
    from liftreg_b200 import ops
    vol = torch.ones((1, 8, 8, 8), device=dev)
    poses = np.array([[0.0, 40.0, 0.0]])
    out = ops.drr_project(vol, poses, (64, 64), (1.0, 1.0, 1.0)).cpu().numpy()
    assert (out[0, 0, :8, :] == 0).all() and (out[0, 0, :, -8:] == 0).all()
    assert out[0, 0, 32, 32] > 0


def test_drr_per_item_poses_and_many_views(dev):
    """(B,P,3) pose sets and more views than one launch chunk (128)."""
    from liftreg_b200 import ops, synthetic
    from oracle import c_oracle
    rs = np.random.RandomState(4)
    vol = rs.rand(2, 6, 10, 7).astype(np.float32)
    poses = np.stack([synthetic.wrapper_poses(60.0, 70, 10), synthetic.wrapper_poses(40.0, 70, 10, 3.0)])
    out = ops.drr_project(cu(vol, dev), poses, (9, 8), (1.0, 1.0, 1.0)).cpu().numpy()
    for b in range(2):
        assert np.array_equal(out[b], c_oracle.drr_forward(vol[b], poses[b], (9, 8), (1.0, 1.0, 1.0),
                                                           seg_len=c_oracle.kernel_seg_len(10)))


def test_drr_linearity_full_size(dev):
    """Size-independent property at 160^3/240^2: DRR(a*V1 + V2) == a*DRR(V1) + DRR(V2) to fp32 round-off."""
    from liftreg_b200 import ops, synthetic
    rs = np.random.RandomState(8)
    v1 = cu(synthetic.hu_to_mu(synthetic.ct_phantom((160, 160, 160)))[None], dev)
    v2 = cu(rs.rand(1, 160, 160, 160).astype(np.float32) * 0.1, dev)
    poses = synthetic.wrapper_poses(60.0, 4, 160)
    f = lambda v: ops.drr_project(v, poses, (240, 240), (2.2, 2.2, 2.2))
    lhs = f(0.5 * v1 + v2).cpu().numpy()
    rhs = (0.5 * f(v1) + f(v2)).cpu().numpy()
    assert per_image_rel_l2(lhs, rhs) <= TOL


# ------------------------------------------------------------------ proj_layer + DRR backward
def test_proj_layer_forward_backward_vs_reference_golden(dev):
    from liftreg_b200 import layers
    g = load_golden("proj_layer")
    layer = layers.proj_layer(torch.from_numpy(g["spacing"]), float(g["resolution_scale"]), float(g["scan_range"]),
                              int(g["proj_num"]), tuple(g["in_shape"]), tuple(int(s) for s in g["out_shape"]), dev)
    x = cu(g["x"], dev).requires_grad_(True)
    y = layer(x)
    assert per_image_rel_l2(y.detach().cpu().numpy(), g["out"]) <= TOL
    y.backward(cu(g["grad_out"], dev))
    for b in range(x.shape[0]):
        assert rel_l2(x.grad[b].cpu().numpy(), g["grad_x"][b]) <= GRAD_TOL


def test_drr_peer_store_form_single_gpu(dev):
    """lr_drr_forward_peers: the kernel stores each image into several buffers, view k at k * view_stride images (what the
    view-sharded sweep uses to fill every rank's gather buffer in final view order); here both 'peers' are local."""
    from liftreg_b200 import ops, sharding, synthetic
    rs = np.random.RandomState(12)
    shape, res, P = (14, 12, 18), (21, 37), 5
    vol = cu(rs.rand(1, *shape).astype(np.float32), dev)
    poses = synthetic.wrapper_poses(60.0, P, shape[1])
    ref = ops.drr_project(vol, poses, res, (2.2, 2.2, 2.2))
    # views 1 and 3 of 5 with stride 2 into two zeroed (5,rd,rh) buffers, starting at view 1
    a, b = torch.zeros((P,) + res, device=dev), torch.zeros((P,) + res, device=dev)
    first = 4 * 1 * res[0] * res[1]
    ops.drr_project_peers(vol, poses[[1, 3]], res, (2.2, 2.2, 2.2), [a.data_ptr() + first, b.data_ptr() + first], 2)
    want = torch.zeros_like(a)
    want[1], want[3] = ref[0, 1], ref[0, 3]
    assert torch.equal(a, want) and torch.equal(b, want)
    # PeerGather on one rank: same code path as the multi-GPU sweep (IPC allocation, alternating buffers)
    pg = sharding.PeerGather(P, res[0], res[1], dev)
    for _ in range(3):
        assert torch.equal(sharding.drr_project_sharded(vol, poses, res, (2.2, 2.2, 2.2), peers=pg), ref)
    pg.close()
    with pytest.raises(Exception):
        ops.drr_project_peers(vol, poses, res, (2.2, 2.2, 2.2), [a.data_ptr()] * 9, 1)      # more than LR_MAX_PEERS


def test_drr_backward_vs_oracle_and_adjoint_identity(dev):
    from liftreg_b200 import ops, synthetic
    from oracle import c_oracle
    rs = np.random.RandomState(9)
    shape, res = (14, 12, 18), (20, 26)
    vol = rs.rand(1, *shape).astype(np.float32)
    go = rs.randn(1, 3, *res).astype(np.float32)
    poses = synthetic.wrapper_poses(60.0, 3, shape[1])
    v = cu(vol, dev).requires_grad_(True)
    y = ops.drr_project(v, poses, res, (2.2, 2.2, 2.2))
    y.backward(cu(go, dev))
    ora = c_oracle.drr_backward(go, shape, poses, (2.2, 2.2, 2.2))
    assert rel_l2(v.grad.cpu().numpy(), ora) <= GRAD_TOL
    # <DRR(v), g> == <v, DRR^T(g)>
    lhs = float((y.detach().double() * cu(go, dev).double()).sum())
    rhs = float((v.detach().double() * v.grad.double()).sum())
    assert abs(lhs - rhs) <= 1e-5 * abs(lhs)


@pytest.mark.parametrize("shape,res,P", [((10, 12, 9), (37, 70), 2),        # 8 rays per voxel: long runs of equal cells
                                         ((20, 16, 40), (33, 45), 3),       # ~1 ray per voxel: adjacent cells
                                         ((9, 8, 50), (12, 20), 2),         # rays 2.5 voxels apart: nothing to merge
                                         ((6, 5, 4), (3, 1), 1)])           # one lane alive per warp
def test_drr_backward_warp_aggregation_vs_oracle(dev, shape, res, P):
    """The warp-aggregated adjoint (runs of equal cells summed, upper-x taps handed to the neighbouring run) against the
    oracle's per-sample scatter, with zero gradients sprinkled in (rays that drop out of the merge) and detector widths
    that leave dead lanes in the last warp."""
    from liftreg_b200 import ops, synthetic
    from oracle import c_oracle
    rs = np.random.RandomState(11)
    go = rs.randn(2, P, *res).astype(np.float32)
    go[rs.rand(*go.shape) < 0.2] = 0.0
    poses = synthetic.wrapper_poses(60.0, P, shape[1])
    v = torch.zeros((2,) + shape, device=dev, requires_grad=True)
    y = ops.drr_project(v, poses, res, (2.2, 2.2, 2.2))
    y.backward(cu(go, dev))
    ora = c_oracle.drr_backward(go, shape, poses, (2.2, 2.2, 2.2))
    assert rel_l2(v.grad.cpu().numpy(), ora) <= GRAD_TOL
    w = cu(rs.rand(2, *shape).astype(np.float32), dev)                     # <DRR(w), g> == <w, DRR^T(g)>
    lhs = float((ops.drr_project(w, poses, res, (2.2, 2.2, 2.2)).double() * cu(go, dev).double()).sum())
    rhs = float((w.double() * v.grad.double()).sum())
    assert abs(lhs - rhs) <= 1e-5 * max(abs(lhs), 1e-3)


# ------------------------------------------------------------------ backprojection
def test_backproj_grid_bit_exact_vs_reference_golden(dev):
    from liftreg_b200 import sdct_projection_utils as sdct
    g = load_golden("backproj_small")
    grid = sdct.backproj_grids_with_poses(g["poses"][0:1], g["img_shape"], g["proj_shape"], device=dev)
    assert np.array_equal(grid.cpu().numpy(), g["grid"])


def test_backproject_bit_exact_vs_reference_golden_and_grad(dev, numerics):
    from liftreg_b200 import sdct_projection_utils as sdct
    g = load_golden("backproj_small")
    tp = cu(g["target_proj"], dev).requires_grad_(True)
    out = sdct.backproject(tp, g["poses"], g["img_shape"])
    assert_ref(out.detach().cpu().numpy(), g["out"], numerics)
    from oracle import c_oracle
    assert np.array_equal(out.detach().cpu().numpy(), c_oracle.backproject_forward(g["target_proj"], g["poses"][0], g["img_shape"]))
    out.backward(cu(g["grad_out"], dev))
    for b in range(tp.shape[0]):
        for p in range(tp.shape[1]):
            assert rel_l2(tp.grad[b, p].cpu().numpy(), g["grad_proj"][b, p]) <= GRAD_TOL


def test_backproject_into_concat_buffer(dev, numerics):
    """f1: write channels 1..P of the (B,1+P,d,w,h) encoder input directly (no torch.cat)."""
    from liftreg_b200 import ops
    g = load_golden("backproj_small")
    B, P = g["target_proj"].shape[:2]
    d, w, h = (int(s) for s in g["img_shape"])
    buf = torch.full((B, 1 + P, d, w, h), 7.0, device=dev)
    ret = ops.backproject(cu(g["target_proj"], dev), g["poses"], (d, w, h), out=buf, channel_offset=1)
    assert ret.data_ptr() == buf.data_ptr()
    assert (buf[:, 0] == 7.0).all()
    assert_ref(buf[:, 1:].cpu().numpy(), g["out"], numerics)


def test_backproject_cfg2_vs_reference_golden(dev):
    """BASELINE configs[1]: 4 x 256^2 -> 160^3, inputs = normalised DRRs of the phantom made by OUR DRR kernel."""
    from liftreg_b200 import ops, synthetic, sdct_projection_utils as sdct
    g = load_golden("backproj_cfg2")
    mu = synthetic.hu_to_mu(synthetic.ct_phantom((160, 160, 160)))
    poses = synthetic.wrapper_poses(60.0, 4, 160)
    proj256 = sdct.calculate_projection(mu, poses, (256, 256), [1, 1, 1], (2.2, 2.2, 2.2), dev)
    for p in range(4):
        assert rel_l2(proj256[p, ::8, ::8], g["proj256_sub"][p]) <= TOL
    tp = cu(synthetic.normalise_projection(proj256)[None], dev)
    vol = ops.backproject(tp, poses.astype(np.float32), (160, 160, 160)).cpu().numpy()
    for p in range(4):
        assert rel_l2(vol[0, p, ::10, ::10, ::10], g["out_sub"][0, p]) <= TOL
        assert rel_l2(vol[0, p, 80, 80, :], g["out_line"][p]) <= TOL
    norms = np.sqrt((vol.astype(np.float64) ** 2).sum(axis=(0, 2, 3, 4)))
    assert np.allclose(norms, g["per_view_norm"], rtol=TOL, atol=0)


@pytest.mark.parametrize("shape,pshape,B,P", [((5, 7, 3), (9, 4), 1, 1), ((33, 6, 70), (40, 31), 3, 2),
                                              ((40, 9, 300), (64, 350), 1, 2), ((2, 2, 2), (1, 1), 2, 66)])
def test_backproject_ragged_shapes_vs_oracle(dev, shape, pshape, B, P):
    from liftreg_b200 import ops, synthetic
    from oracle import c_oracle
    rs = np.random.RandomState(2)
    tp = rs.uniform(-1, 1, (B, P) + pshape).astype(np.float32)
    poses = synthetic.wrapper_poses(60.0, P, shape[1]).astype(np.float32)
    out = ops.backproject(cu(tp, dev), poses, shape).cpu().numpy()
    assert np.array_equal(out, c_oracle.backproject_forward(tp, poses, shape))


def test_backproject_constant_image_property_full_size(dev):
    """Size-independent property at 160^3: a constant detector image backprojects to that constant wherever all
    four taps are inside the detector, and to [0, c] elsewhere (zeros padding)."""
    from liftreg_b200 import ops, synthetic
    poses = synthetic.wrapper_poses(60.0, 4, 160).astype(np.float32)
    tp = torch.full((2, 4, 256, 256), 0.75, device=dev)
    vol = ops.backproject(tp, poses, (160, 160, 160))
    assert float(vol.max()) <= 0.75 + 1e-6 and float(vol.min()) >= 0.0
    assert float((vol - 0.75).abs().lt(1e-6).float().mean()) > 0.9


# ------------------------------------------------------------------ warp
@pytest.mark.parametrize("zb", [False, True])
@pytest.mark.parametrize("us", [False, True])
@pytest.mark.parametrize("mode", ["bilinear", "nearest"])
def test_warp_bit_exact_vs_reference_golden(dev, zb, us, mode, numerics):
    from liftreg_b200 import net_utils
    g = load_golden("warp_small")
    key = "zb%d_us%d_%s" % (zb, us, mode)
    img = cu(g["img"], dev).requires_grad_(mode == "bilinear")
    phi = cu(g["phi"], dev).requires_grad_(True)
    out = net_utils.Bilinear(zero_boundary=zb, using_scale=us, mode=mode)(img, phi)
    assert_ref(out.detach().cpu().numpy(), g["out_" + key], numerics if mode == "bilinear" else "exact")
    from oracle import c_oracle
    assert np.array_equal(out.detach().cpu().numpy(), c_oracle.warp_forward(g["img"], g["phi"], zb, us, mode))
    if mode == "bilinear":
        out.backward(cu(g["grad_out"], dev))
        assert rel_l2(img.grad.cpu().numpy(), g["gimg_" + key]) <= GRAD_TOL
        assert rel_l2(phi.grad.cpu().numpy(), g["gphi_" + key]) <= GRAD_TOL
    else:
        out.backward(cu(g["grad_out"], dev))
        assert float(phi.grad.abs().max()) == 0.0


def test_warp_host_tensors_are_staged_through_the_gpu(dev):
    """tools/evaluate_dir_lab.py:217-222 hands Bilinear CPU tensors."""
    from liftreg_b200 import net_utils
    g = load_golden("warp_small")
    out = net_utils.Bilinear(zero_boundary=True, using_scale=False, mode="nearest")(torch.from_numpy(g["img"]),
                                                                                  torch.from_numpy(g["phi"]))
    assert not out.is_cuda
    assert np.array_equal(out.numpy(), g["out_zb1_us0_nearest"])


def test_identity_map_bit_exact(dev):
    from liftreg_b200 import net_utils
    g = load_golden("identity_map")
    assert np.array_equal(net_utils.identity_map((7, 9, 11)).cpu().numpy(), g["id_7_9_11"])
    assert np.array_equal(net_utils.gen_identity_map([5, 6, 7], 1.0).cpu().numpy(), g["gen_5_6_7"])
    assert np.array_equal(net_utils.identity_map((160, 160, 160))[:, ::16, ::16, ::16].cpu().numpy(), g["id_160"])


def test_warp_cfg2_vs_reference_golden_and_fused_identity(dev):
    """BASELINE configs[1] warp: 160^3, Bilinear(zero_boundary=True, using_scale=True) as the model builds it."""
    from liftreg_b200 import net_utils, ops, synthetic
    g = load_golden("warp_cfg2")
    moving = cu(synthetic.hu_to_unit(synthetic.ct_phantom((160, 160, 160)))[None, None], dev)
    disp = cu(synthetic.smooth_displacement((160, 160, 160))[None], dev)
    phi = disp + net_utils.identity_map((160, 160, 160))[None]             # model :68
    assert abs(float(phi.double().sum()) - float(g["phi_sum64"])) <= 1e-6 * abs(float(g["phi_sum64"])) + 1e-3
    out = net_utils.Bilinear(zero_boundary=True, using_scale=True)(moving, phi)
    o = out[0, 0].cpu().numpy()
    assert rel_l2(o[::8, ::8, ::8], g["out_sub"]) <= TOL
    assert rel_l2(o[80, 80, :], g["out_line"]) <= TOL
    assert abs(np.sqrt((o.astype(np.float64) ** 2).sum()) - float(g["norm64"])) <= TOL * float(g["norm64"])
    fused = ops.warp(moving, disp, zero_boundary=True, using_scale=True, disp_plus_identity=True)
    assert torch.equal(fused, out)                                         # in-kernel identity == torch add


@pytest.mark.parametrize("shape,B,C", [((1, 1, 1), 1, 1), ((3, 5, 2), 2, 3), ((17, 33, 129), 1, 2), ((2, 300, 70), 1, 1)])
def test_warp_ragged_shapes_vs_oracle(dev, shape, B, C):
    from liftreg_b200 import ops
    from oracle import c_oracle
    rs = np.random.RandomState(3)
    img = rs.uniform(-1, 1, (B, C) + shape).astype(np.float32)
    phi = rs.uniform(-1.3, 1.3, (B, 3) + shape).astype(np.float32)
    for zb in (False, True):
        for mode in ("bilinear", "nearest"):
            out = ops.warp(cu(img, dev), cu(phi, dev), zero_boundary=zb, using_scale=True, mode=mode).cpu().numpy()
            assert np.array_equal(out, c_oracle.warp_forward(img, phi, zb, True, mode)), (zb, mode)


def test_warp_identity_is_idempotent_full_size(dev):
    """Size-independent property at 160^3: warping by the identity map returns the image (to 1 ulp of the rescale)."""
    from liftreg_b200 import net_utils, synthetic
    moving = cu(synthetic.hu_to_unit(synthetic.ct_phantom((160, 160, 160)))[None, None], dev)
    idm = net_utils.identity_map((160, 160, 160))[None]
    out = net_utils.Bilinear(zero_boundary=True, using_scale=True)(moving, idm)
    assert rel_l2(out.cpu().numpy(), moving.cpu().numpy()) <= TOL
    out2 = net_utils.Bilinear(zero_boundary=False, using_scale=False)(moving, idm)
    assert rel_l2(out2.cpu().numpy(), moving.cpu().numpy()) <= TOL


# ------------------------------------------------------------------ host-buffer C-ABI entry points
def test_host_entry_points_match_device_entry_points(dev, numerics):
    import ctypes
    from liftreg_b200 import _native, ops
    lib = _native.lib()
    g = load_golden("warp_small")
    img, phi = np.ascontiguousarray(g["img"]), np.ascontiguousarray(g["phi"])
    B, C, D, H, W = img.shape
    out = np.empty_like(img)
    ws = torch.empty(lib.lr_warp_forward_host_workspace_bytes(B, C, D, H, W), dtype=torch.uint8, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _native.check(lib.lr_warp_forward_host(img.ctypes.data, phi.ctypes.data, B, C, D, H, W, 0, 0, 1, 0, out.ctypes.data,
                                           ctypes.c_void_p(ws.data_ptr()), ws.numel(), st), "warp host")
    assert_ref(out, g["out_zb1_us1_bilinear"], numerics)
    # too-small workspace is reported, not crashed on
    rc = lib.lr_warp_forward_host(img.ctypes.data, phi.ctypes.data, B, C, D, H, W, 0, 0, 1, 0, out.ctypes.data,
                                  ctypes.c_void_p(ws.data_ptr()), 16, st)
    assert rc == -3 and b"workspace" in lib.lr_last_error()

    gb = load_golden("backproj_small")
    tp = np.ascontiguousarray(gb["target_proj"]); poses = np.ascontiguousarray(gb["poses"][0])
    Bp, P, pw, ph = tp.shape
    d, w, h = (int(s) for s in gb["img_shape"])
    vol = np.empty((Bp, P, d, w, h), np.float32)
    ws = torch.empty(lib.lr_backproject_forward_host_workspace_bytes(Bp, P, pw, ph, d, w, h), dtype=torch.uint8, device=dev)
    _native.check(lib.lr_backproject_forward_host(tp.ctypes.data, ops._fp(poses), Bp, P, pw, ph, d, w, h, vol.ctypes.data,
                                                  ctypes.c_void_p(ws.data_ptr()), ws.numel(), st), "backproject host")
    assert_ref(vol, gb["out"], numerics)


def test_async_host_entry_points_overlap_and_match(dev, numerics):
    """lr_*_host_async on two streams + lr_stream_synchronize (the overlapped e2e path of bench.py) against the blocking
    calls: same bits; the async calls return before their results are complete only if the caller does not sync."""
    import ctypes
    from liftreg_b200 import _native, ops
    lib = _native.lib()
    g, gb = load_golden("warp_small"), load_golden("backproj_small")
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
    img, phi = pin(g["img"]), pin(g["phi"])
    B, C, D, H, W = img.shape
    tp, poses = pin(gb["target_proj"]), np.ascontiguousarray(gb["poses"][0])
    Bp, P, pw, ph = tp.shape
    d, w, h = (int(s) for s in gb["img_shape"])
    out_w, out_b = torch.zeros(img.shape).pin_memory(), torch.zeros((Bp, P, d, w, h)).pin_memory()
    ws_w = torch.empty(lib.lr_warp_forward_host_workspace_bytes(B, C, D, H, W), dtype=torch.uint8, device=dev)
    ws_b = torch.empty(lib.lr_backproject_forward_host_workspace_bytes(Bp, P, pw, ph, d, w, h), dtype=torch.uint8, device=dev)
    sa, sb = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    _native.check(lib.lr_backproject_forward_host_async(vp(tp), ops._fp(poses), Bp, P, pw, ph, d, w, h, vp(out_b), vp(ws_b), ws_b.numel(),
                                                        ctypes.c_void_p(sa.cuda_stream)), "bp async")
    _native.check(lib.lr_warp_forward_host_async(vp(img), vp(phi), B, C, D, H, W, 0, 0, 1, 0, vp(out_w), vp(ws_w), ws_w.numel(),
                                                 ctypes.c_void_p(sb.cuda_stream)), "warp async")
    _native.check(lib.lr_stream_synchronize(ctypes.c_void_p(sa.cuda_stream)), "sync a")
    _native.check(lib.lr_stream_synchronize(ctypes.c_void_p(sb.cuda_stream)), "sync b")
    assert_ref(out_w.numpy(), g["out_zb1_us1_bilinear"], numerics)
    assert_ref(out_b.numpy(), gb["out"], numerics)
    ref_w, ref_b = np.empty_like(g["img"]), np.empty((Bp, P, d, w, h), np.float32)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _native.check(lib.lr_warp_forward_host(g["img"].ctypes.data, g["phi"].ctypes.data, B, C, D, H, W, 0, 0, 1, 0, ref_w.ctypes.data,
                                           vp(ws_w), ws_w.numel(), st), "warp host")
    _native.check(lib.lr_backproject_forward_host(gb["target_proj"].ctypes.data, ops._fp(poses), Bp, P, pw, ph, d, w, h, ref_b.ctypes.data,
                                                  vp(ws_b), ws_b.numel(), st), "bp host")
    assert np.array_equal(out_w.numpy(), ref_w) and np.array_equal(out_b.numpy(), ref_b)


def test_probe_kernels_report_plausible_peaks(dev):
    """bench.py's DRR fractions divide by these: L1-hit gather bandwidth between 5 and 40 TB/s (148 SMs x 128 B/clk x
    1.965 GHz = 37 TB/s), issue rate between 0.5 and 1.2 T warp-instructions/s (592 schedulers x 1.965 GHz = 1.16 T)."""
    import ctypes
    from liftreg_b200 import _native
    lib = _native.lib()
    sm = torch.cuda.get_device_properties(dev).multi_processor_count
    blocks, fpb, iters = sm * 8, 4096, 500
    buf, sink = torch.zeros(blocks * fpb, device=dev), torch.zeros(4, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    vp = lambda t: ctypes.c_void_p(t.data_ptr())

    def ms(fn):
        fn(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            fn()
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1) / 3

    t = ms(lambda: _native.check(lib.lr_probe_l1_gather(vp(buf), buf.numel(), blocks, fpb, iters, vp(sink), st), "probe"))
    assert 5e3 <= blocks * 256 * iters * 32 / t * 1e-6 <= 40e3
    t = ms(lambda: _native.check(lib.lr_probe_issue(blocks, 1000, vp(sink), st), "probe"))
    assert 500 <= blocks * 8 * 1000 * 8 / t * 1e-6 <= 1200
    assert lib.lr_probe_l1_gather(vp(buf), buf.numel(), blocks, 1000, iters, vp(sink), st) == -1          # not a power of two


# ------------------------------------------------------------------ error behaviour
def test_bad_arguments_are_reported_not_crashed(dev):
    import ctypes
    from liftreg_b200 import _native, ops
    lib = _native.lib()
    t = torch.zeros(8, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = ctypes.c_void_p(t.data_ptr())
    assert lib.lr_warp_forward(p, p, 0, 1, 2, 2, 2, 0, 0, 1, 0, p, st) == -1
    assert lib.lr_warp_forward(p, p, 1, 1, 2, 2, 2, 5, 0, 1, 0, p, st) == -1
    assert lib.lr_warp_forward(None, p, 1, 1, 2, 2, 2, 0, 0, 1, 0, p, st) == -1
    assert b"null" in lib.lr_last_error()
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.warp(torch.zeros(1, 1, 2, 2, 2), torch.zeros(1, 3, 2, 2, 2))
    with pytest.raises(TypeError):
        ops.warp(torch.zeros(1, 1, 2, 2, 2, device=dev, dtype=torch.float64), torch.zeros(1, 3, 2, 2, 2, device=dev))
    with pytest.raises(ValueError):
        ops.backproject(torch.zeros(1, 2, 4, 4, device=dev), np.zeros((3, 3), np.float32), (2, 2, 2))
    with pytest.raises(NotImplementedError):
        from liftreg_b200 import sdct_projection_utils as sdct
        sdct.calculate_projection(np.zeros((2, 2, 2), np.float32), np.zeros((1, 3)), (2, 2), [2, 1, 1], (1, 1, 1), dev)


# ------------------------------------------------------------------ z-slab / view sharding (single process)
def test_slab_kernels_tile_the_full_result(dev):
    """Multi-GPU building blocks: per-slab launches (any split, including 1-plane slabs) reproduce the full op."""
    from liftreg_b200 import ops, sharding, synthetic
    rs = np.random.RandomState(21)
    shape = (13, 10, 37)
    img = cu(rs.uniform(-1, 1, (2, 2) + shape).astype(np.float32), dev)
    disp = cu(rs.uniform(-0.2, 0.2, (2, 3) + shape).astype(np.float32), dev)
    tp = cu(rs.uniform(-1, 1, (2, 3, 20, 44)).astype(np.float32), dev)
    poses = synthetic.wrapper_poses(60.0, 3, shape[1]).astype(np.float32)
    full_w = ops.warp(img, disp, zero_boundary=True, using_scale=True, disp_plus_identity=True)
    full_b = ops.backproject(tp, poses, shape)
    for world in (2, 3, 13):
        parts_w, parts_b = [], []
        for r in range(world):
            z0, z1 = sharding.split_range(shape[0], world, r)
            parts_w.append(ops.warp(img, disp[:, :, z0:z1].contiguous(), zero_boundary=True, using_scale=True,
                                    disp_plus_identity=True, z_begin=z0))
            parts_b.append(ops.backproject(tp, poses, shape, slab=(z0, z1 - z0)))
        assert torch.equal(torch.cat(parts_w, dim=2), full_w)
        assert torch.equal(torch.cat(parts_b, dim=2), full_b)
    # slab warp is differentiable wrt its phi slab and matches the full gradient
    d_full = disp.clone().requires_grad_(True)
    ops.warp(img, d_full, zero_boundary=True, disp_plus_identity=True).sum().backward()
    d_slab = disp[:, :, 4:9].contiguous().requires_grad_(True)
    ops.warp(img, d_slab, zero_boundary=True, disp_plus_identity=True, z_begin=4).sum().backward()
    assert torch.equal(d_slab.grad, d_full.grad[:, :, 4:9])


def test_sharded_entry_points_world_1(dev):
    from liftreg_b200 import ops, sharding, synthetic
    rs = np.random.RandomState(22)
    vol = cu(rs.rand(2, 8, 9, 7).astype(np.float32), dev)
    poses = synthetic.wrapper_poses(60.0, 3, 9)
    a = sharding.drr_project_sharded(vol, poses, (10, 12), (1.0, 1.0, 1.0))
    assert torch.equal(a, ops.drr_project(vol, poses, (10, 12), (1.0, 1.0, 1.0)))
    tp = cu(rs.uniform(-1, 1, (1, 3, 16, 16)).astype(np.float32), dev)
    slab, zr = sharding.backproject_sharded(tp, poses.astype(np.float32), (8, 9, 7))
    assert zr == (0, 8) and torch.equal(slab, ops.backproject(tp, poses.astype(np.float32), (8, 9, 7)))


# ------------------------------------------------------------------ against stock PyTorch on the same GPU
def test_against_stock_torch_cuda_ops(dev):
    """The reference's op sequence (oracle/torch_port.py) executed by stock ATen CUDA kernels on this GPU.  ATen's
    CUDA kernels round differently from its CPU kernels (e.g. division by a scalar becomes a multiply by the
    reciprocal), so this is a tolerance check: <= 1e-5 relative L2 per image / volume."""
    from liftreg_b200 import ops, synthetic
    from oracle import torch_port
    shape, det, P = (48, 40, 56), (72, 84), 3
    hu = synthetic.ct_phantom(shape, seed=5, sigma=1.5, nodules=6, noise_hu=0.0)
    mu = synthetic.hu_to_mu(hu)
    poses = synthetic.wrapper_poses(60.0, P, shape[1])
    ref_proj = torch_port.drr(mu, poses, det, (2.2, 2.2, 2.2), device="cuda")
    our_proj = ops.drr_project(cu(mu[None], dev), poses, det, (2.2, 2.2, 2.2))[0].cpu().numpy()
    assert per_image_rel_l2(our_proj, ref_proj) <= TOL

    tp = cu(synthetic.normalise_projection(ref_proj)[None], dev)
    grids = torch_port.backproj_grid(poses[None].astype(np.float32), shape, det, device="cuda").permute(0, 1, 3, 4, 5, 2)
    ref_vol = torch_port.backproject(tp, grids)
    our_vol = ops.backproject(tp, poses.astype(np.float32), shape)
    for p in range(P):
        assert rel_l2(our_vol[0, p].cpu().numpy(), ref_vol[0, p].cpu().numpy()) <= TOL

    moving = cu(synthetic.hu_to_unit(hu)[None, None], dev)
    phi = cu((synthetic.smooth_displacement(shape, max_disp=0.08) + synthetic.identity_map_np(shape))[None], dev)
    ref_w = torch_port.warp(moving, phi, zero_boundary=True, using_scale=True)
    our_w = ops.warp(moving, phi, zero_boundary=True, using_scale=True)
    assert rel_l2(our_w.cpu().numpy(), ref_w.cpu().numpy()) <= TOL
    # gradients wrt phi against autograd through stock grid_sample
    p1 = phi.clone().requires_grad_(True); p2 = phi.clone().requires_grad_(True)
    torch_port.warp(moving, p1, zero_boundary=True, using_scale=True).square().sum().backward()
    ops.warp(moving, p2, zero_boundary=True, using_scale=True).square().sum().backward()
    assert rel_l2(p2.grad.cpu().numpy(), p1.grad.cpu().numpy()) <= GRAD_TOL


def test_model_hot_path_drop_in(dev, numerics):
    """The two drop-in sites of LiftRegDeformSubspaceBackproj (SURVEY 2 #4): lines 85-98 (backprojection + cat) via
    dropin._estimate_flow's fused buffer write, and lines 68-69 (identity add + Bilinear) via the fused warp; both
    against the reference's op sequence replayed on the CPU (oracle/torch_port.py)."""
    import types
    from liftreg_b200 import dropin, net_utils, ops, synthetic
    from oracle import torch_port
    shape, det, B, P = (20, 24, 28), (40, 36), 2, 4
    rs = np.random.RandomState(31)
    moving = rs.uniform(-1, 1, (B, 1) + shape).astype(np.float32)
    target_proj = rs.uniform(-1, 1, (B, P) + det).astype(np.float32)
    poses = np.repeat(synthetic.wrapper_poses(60.0, P, shape[1])[None], B, 0).astype(np.float32)
    disp = np.stack([synthetic.smooth_displacement(shape, seed=s, max_disp=0.1, coarse=4) for s in (1, 2)])

    # reference sequence on CPU: grids from poses[0:1], grid_sample, cat; then disp + id, Bilinear(zeros, scale)
    grids = torch_port.backproj_grid(poses[0:1], shape, det).permute(0, 1, 3, 4, 5, 2)
    ref_x = torch.cat([torch.from_numpy(moving), torch_port.backproject(torch.from_numpy(target_proj), grids)], dim=1)
    ref_phi = torch.from_numpy(disp) + torch_port.identity_map(shape)
    ref_warped = torch_port.warp(torch.from_numpy(moving), ref_phi, zero_boundary=True, using_scale=True)

    # ours: a stand-in model object exposing what _estimate_flow touches (identity encoder, zero PCA basis + mean=disp)
    captured = {}

    class Capture(torch.nn.Module):
        def forward(self, x):
            captured["x"] = x.clone()
            return x.reshape(x.shape[0], -1)[:, :3]

    nvox = int(np.prod(shape))
    fake = types.SimpleNamespace(encoders=[Capture()], pca_vectors=torch.zeros(3 * nvox, 3, device=dev),
                                 pca_mean=cu(disp[0].reshape(-1), dev))
    _, disp_field = dropin._estimate_flow(fake, cu(moving, dev), cu(target_proj, dev), torch.from_numpy(poses))
    assert_ref(captured["x"].cpu().numpy(), ref_x.numpy(), numerics)    # exact mode: bit-identical encoder input
    assert disp_field.shape == (B, 3) + shape
    id_transform = net_utils.gen_identity_map(shape, 1.0)
    phi = cu(disp, dev) + id_transform                                   # model :68
    warped = net_utils.Bilinear(zero_boundary=True, using_scale=True)(cu(moving, dev), phi)   # model :69
    assert torch.equal(phi.cpu(), ref_phi)
    assert_ref(warped.cpu().numpy(), ref_warped.numpy(), numerics)
    fused = ops.warp(cu(moving, dev), cu(disp, dev), zero_boundary=True, using_scale=True, disp_plus_identity=True)
    assert torch.equal(fused, warped)


# ------------------------------------------------------------------ maximum sizes (BASELINE configs[3] geometry)
def test_drr_cfg4_geometry_512_cubed(dev):
    """512^3 volume, 512^2 detector (the preprocessing sweep of configs[3]): two of the 64 views exactly against the
    oracle, and all 64 views through size-independent properties (finite, non-negative, view symmetry)."""
    from liftreg_b200 import ops, synthetic
    from oracle import c_oracle
    n = 512
    z = np.arange(n, dtype=np.float32)
    vol = (0.1 + 0.05 * np.sin(z / 13.0)[:, None, None] * np.cos(z / 17.0)[None, :, None]
           + 0.04 * np.sin(z / 11.0)[None, None, :]).astype(np.float32)
    poses = synthetic.wrapper_poses(60.0, 64, n)
    tv = cu(vol[None], dev)
    out = ops.drr_project(tv, poses, (512, 512), (1.0, 1.0, 1.0))
    assert out.shape == (1, 64, 512, 512)
    o = out[0].cpu().numpy()
    assert np.isfinite(o).all() and (o >= 0).all() and o.max() > 1.0
    sel = [0, 37]
    ora = c_oracle.drr_forward(vol, poses[sel], (512, 512), (1.0, 1.0, 1.0), seg_len=c_oracle.kernel_seg_len(n))
    assert np.array_equal(o[sel], ora)
    # the same volume projected with view-sharded launches (8 views per call, as 8 GPUs would) is identical
    parts = [ops.drr_project(tv, poses[i:i + 8], (512, 512), (1.0, 1.0, 1.0)) for i in range(0, 64, 8)]
    assert torch.equal(torch.cat(parts, dim=1), out)


def test_warp_and_backprojection_320_cubed_vs_oracle(dev):
    """Larger-than-benchmark volume (8x the voxels of 160^3) with batch 2: exact against the oracle."""
    from liftreg_b200 import ops, synthetic
    from oracle import c_oracle
    shape = (320, 320, 320)
    rs = np.random.RandomState(40)
    img = rs.uniform(-1, 1, (1, 1) + shape).astype(np.float32)
    disp = synthetic.smooth_displacement(shape, seed=4, max_disp=0.03, coarse=6)[None]
    phi = (disp + synthetic.identity_map_np(shape)[None]).astype(np.float32)
    out = ops.warp(cu(img, dev), cu(phi, dev), zero_boundary=True, using_scale=True).cpu().numpy()
    assert np.array_equal(out, c_oracle.warp_forward(img, phi, True, True, "bilinear"))
    tp = rs.uniform(-1, 1, (2, 2, 512, 512)).astype(np.float32)
    poses = synthetic.wrapper_poses(60.0, 2, shape[1]).astype(np.float32)
    vol = ops.backproject(cu(tp, dev), poses, shape).cpu().numpy()
    assert np.array_equal(vol, c_oracle.backproject_forward(tp, poses, shape))


def test_remaining_mirror_entry_points(dev):
    """forward_grids*, backproj_grids (old fixed geometry), calc_relative_atten_coef_cuda, DRRProjector reuse."""
    from liftreg_b200 import sdct_projection_utils as sdct, synthetic
    from oracle import c_oracle
    shp = (10, 18, 12)
    sp = torch.tensor([2.2, 1.7, 2.5])
    poses = synthetic.wrapper_poses(60.0, 3, shp[1], 3.0)
    grids, dx = sdct.forward_grids(60.0, 3, sp, shp, device=dev)
    og, odx = c_oracle.project_grid(poses, (15, 18), shp, sp.numpy())
    assert np.array_equal(grids.cpu().numpy(), og[..., ::-1]) and np.array_equal(dx.cpu().numpy(), odx)
    grids2, _ = sdct.forward_grids_with_poses(poses, sp, shp, device=dev, receptor_size=(7, 9))
    assert np.array_equal(grids2.cpu().numpy(), c_oracle.project_grid(poses, (7, 9), shp, sp.numpy())[0][..., ::-1])
    g = load_golden("backproj_grids_old")
    old = sdct.backproj_grids(float(g["scan_range"]), int(g["proj_num"]), tuple(g["img_shape"]), tuple(g["proj_shape"]), device=dev)
    assert np.abs(old.cpu().numpy() - g["grid"]).max() <= 2e-6
    a = load_golden("atten")
    t = cu(a["hu"].copy(), dev)
    mu = sdct.calc_relative_atten_coef_cuda(t)
    assert np.array_equal(mu.cpu().numpy(), a["mu"]) and float(t.min()) >= -1000.0
    # projector object reuses its buffers across calls of different sizes
    pr = sdct.DRRProjector(dev)
    d1 = load_golden("drr_small")
    for _ in range(2):
        o = pr.project_numpy(d1["vol"], d1["poses"], d1["resolution"], d1["spacing"])
        assert per_image_rel_l2(o, d1["proj"]) <= TOL
    d2 = load_golden("drr_small_csvposes")
    assert per_image_rel_l2(pr.project_numpy(d2["vol"], d2["poses"], d2["resolution"], d2["spacing"]), d2["proj"]) <= TOL


@pytest.mark.parametrize("n,offset", [(1, 0), (3, 0), (4, 0), (1027, 0), (1027, 1), (64 * 64 * 64 + 5, 0), (4099, 3)])
def test_atten_coef_vector_and_tail_paths_bit_exact(dev, n, offset):
    """HU -> attenuation (sdct:6-13): float4 groups + scalar tail, and the scalar path for a pointer that is not 16-byte
    aligned, bit for bit against the oracle; in place like the reference (the clamp is visible in the input)."""
    from liftreg_b200 import ops
    from oracle import c_oracle
    rs = np.random.RandomState(13)
    hu = rs.uniform(-1500.0, 2500.0, n + offset).astype(np.float32)
    t = cu(hu.copy(), dev)
    view = t[offset:]
    ops.atten_coef_(view)
    assert np.array_equal(view.cpu().numpy(), c_oracle.atten_coef(hu[offset:].copy()))
    assert np.array_equal(t[:offset].cpu().numpy(), hu[:offset])


# ------------------------------------------------------------------ PCA-subspace decode (row f2)
@pytest.mark.parametrize("B,K,shape", [(1, 56, (6, 5, 7)), (3, 56, (20, 24, 28)), (8, 8, (4, 4, 4)), (33, 60, (5, 6, 7)), (2, 4, (3, 3, 3)),
                                       (2, 3, (9, 8, 7)), (5, 57, (12, 10, 11)), (1, 1, (2, 2, 2)),
                                       (2, 16, (5, 6, 7)), (1, 160, (4, 5, 6))])       # K = 16, 160: the padded staging kernel
def test_pca_decode_exact_vs_oracle(dev, B, K, shape):
    from liftreg_b200 import ops
    from oracle import c_oracle
    rs = np.random.RandomState(50)
    N = 3 * int(np.prod(shape))
    basis = (rs.standard_normal((N, K)) * 1e-2).astype(np.float32)
    mean = (rs.standard_normal(N) * 1e-2).astype(np.float32)
    coefs = rs.standard_normal((B, K)).astype(np.float32)
    out = ops.pca_decode(cu(coefs, dev), cu(basis, dev), cu(mean, dev))
    assert np.array_equal(out.cpu().numpy(), c_oracle.pca_decode(coefs, basis, mean))
    phi = ops.pca_decode(cu(coefs, dev), cu(basis, dev), cu(mean, dev), img_shape=shape, add_identity=True)
    assert phi.shape == (B, 3) + shape
    assert np.array_equal(phi.reshape(B, -1).cpu().numpy(), c_oracle.pca_decode(coefs, basis, mean, img_shape=shape))
    nomean = ops.pca_decode(cu(coefs, dev), cu(basis, dev))
    assert np.array_equal(nomean.cpu().numpy(), c_oracle.pca_decode(coefs, basis))


def test_pca_decode_matches_torch_linear_and_is_differentiable(dev):
    import torch.nn.functional as F
    from liftreg_b200 import net_utils, ops
    rs = np.random.RandomState(51)
    shape = (16, 12, 20)
    N, K, B = 3 * int(np.prod(shape)), 56, 4
    basis = cu((rs.standard_normal((N, K)) * 1e-2).astype(np.float32), dev)
    mean = cu((rs.standard_normal(N) * 1e-2).astype(np.float32), dev)
    c1 = cu(rs.standard_normal((B, K)).astype(np.float32), dev).requires_grad_(True)
    c2 = c1.detach().clone().requires_grad_(True)
    ref = F.linear(c1, basis, mean).reshape(B, 3, *shape) + net_utils.gen_identity_map(shape, 1.0)    # model :102, :68
    ours = ops.pca_decode(c2, basis, mean, img_shape=shape, add_identity=True)
    assert rel_l2(ours.detach().cpu().numpy(), ref.detach().cpu().numpy()) <= TOL
    g = cu(rs.standard_normal(ref.shape).astype(np.float32), dev)
    ref.backward(g); ours.backward(g)
    assert rel_l2(c2.grad.cpu().numpy(), c1.grad.cpu().numpy()) <= GRAD_TOL


@pytest.mark.parametrize("B,K,N", [(1, 56, 3 * 11 * 13 * 7), (4, 56, 5000), (17, 8, 777), (3, 160, 2049), (2, 4, 1), (33, 60, 4097)])
def test_pca_decode_backward_vs_float64(dev, B, K, N):
    """d/dcoefs of model :102 (F.linear): grad_coefs = grad_out @ basis, the second full pass over the basis.
    fp32 partial sums in a launch-dependent order: compared with the float64 product."""
    from liftreg_b200 import _native, ops
    rs = np.random.RandomState(52)
    basis = (rs.standard_normal((N, K)) * 1e-2).astype(np.float32)
    gout = rs.standard_normal((B, N)).astype(np.float32)
    want = gout.astype(np.float64) @ basis.astype(np.float64)
    gc = torch.zeros((B, K), device=dev)
    d_gout, d_basis = cu(gout, dev), cu(basis, dev)          # keep the tensors alive across the raw-pointer call
    _native.check(_native.lib().lr_pca_decode_backward(ops._ptr(d_gout), ops._ptr(d_basis), B, K, N, ops._ptr(gc), ops._stream()),
                  "lr_pca_decode_backward")
    torch.cuda.synchronize()
    assert rel_l2(gc.cpu().numpy(), want) <= GRAD_TOL
    # through autograd, accumulating into an existing .grad
    coefs = cu(rs.standard_normal((B, K)).astype(np.float32), dev).requires_grad_(True)
    ops.pca_decode(coefs, d_basis).backward(d_gout)
    assert rel_l2(coefs.grad.cpu().numpy(), want) <= GRAD_TOL


def test_pca_decode_backward_odd_k_native_scalar_path(dev):
    """K % 4 != 0: the scalar-staging kernel (no library GEMM on the path)."""
    from liftreg_b200 import ops
    rs = np.random.RandomState(53)
    basis = cu((rs.standard_normal((300, 7)) * 1e-2).astype(np.float32), dev)
    coefs = cu(rs.standard_normal((2, 7)).astype(np.float32), dev).requires_grad_(True)
    g = cu(rs.standard_normal((2, 300)).astype(np.float32), dev)
    ops.pca_decode(coefs, basis).backward(g)
    assert rel_l2(coefs.grad.cpu().numpy(), (g.double() @ basis.double()).cpu().numpy()) <= GRAD_TOL


# ------------------------------------------------------------------ BASELINE configs[2] / configs[4] shapes
def test_cfg3_batch8_full_size_is_batch_independent(dev):
    """configs[2]: the hot-path ops of the full forward at 160^3, batch 8 (4 views, 256^2 detector).  Every batch item
    must equal the batch-1 result of the same item, bit for bit, and item 0 -- whose inputs are the phantom, its
    normalised DRRs and the smooth displacement the goldens were generated from -- must match the subsets the
    reference itself produced (tests/golden/backproj_cfg2.npz, warp_cfg2.npz)."""
    from liftreg_b200 import ops, synthetic, sdct_projection_utils as sdct
    shape, det, B, P = (160, 160, 160), (256, 256), 8, 4
    rs = np.random.RandomState(60)
    poses = synthetic.wrapper_poses(60.0, P, shape[1])
    hu = synthetic.ct_phantom(shape)
    proj0 = synthetic.normalise_projection(sdct.calculate_projection(synthetic.hu_to_mu(hu), poses, det, [1, 1, 1], (2.2, 2.2, 2.2), dev))
    proj_np = rs.uniform(-1, 1, (B, P) + det).astype(np.float32)
    proj_np[0] = proj0
    moving_np = rs.uniform(-1, 1, (B, 1) + shape).astype(np.float32)
    moving_np[0, 0] = synthetic.hu_to_unit(hu)
    poses = poses.astype(np.float32)
    proj, moving = torch.from_numpy(proj_np).to(dev), torch.from_numpy(moving_np).to(dev)
    disp = torch.stack([torch.from_numpy(synthetic.smooth_displacement(shape) if s == 0 else synthetic.smooth_displacement(shape, seed=s))
                        for s in range(B)]).to(dev)
    x = torch.empty((B, 1 + P) + shape, device=dev)                      # the encoder's concat buffer (row f1)
    x[:, :1] = moving
    ops.backproject(proj, poses, shape, out=x, channel_offset=1)
    warped = ops.warp(moving, disp, zero_boundary=True, using_scale=True, disp_plus_identity=True)
    for b in (0, 3, 7):
        assert torch.equal(x[b, 1:], ops.backproject(proj[b:b + 1], poses, shape)[0])
        assert torch.equal(warped[b:b + 1], ops.warp(moving[b:b + 1], disp[b:b + 1], zero_boundary=True, using_scale=True,
                                                     disp_plus_identity=True))
    assert torch.equal(x[:, 0], moving[:, 0])
    gb, gw = load_golden("backproj_cfg2"), load_golden("warp_cfg2")
    lifted0, warped0 = x[0, 1:].cpu().numpy(), warped[0, 0].cpu().numpy()
    for p in range(P):
        assert rel_l2(lifted0[p, ::10, ::10, ::10], gb["out_sub"][0, p]) <= TOL
        assert rel_l2(lifted0[p, 80, 80, :], gb["out_line"][p]) <= TOL
    assert rel_l2(warped0[::8, ::8, ::8], gw["out_sub"]) <= TOL and rel_l2(warped0[80, 80, :], gw["out_line"]) <= TOL


def test_cfg3_model_forward_dropin_vs_stock_cuda_ops(dev):
    """configs[2] end to end: the forward of LiftRegDeformSubspaceBackproj.model at 160^3, batch 8 -- backprojection
    grid from the first item's poses, grid_sample, torch.cat with `moving`, conv encoder, F.linear over the transposed
    (N,K) basis view (model :42), identity add and Bilinear (:68-69, :80-104) -- first as the reference's op sequence on
    stock torch CUDA ops (oracle/torch_port.py), then through dropin._estimate_flow and the B200 Bilinear, with the same
    seeded stand-in encoder and basis.  Bar of the real-model test (test_reference_model_gpu.py): <= 1e-5 relative L2
    per item for the PCA coefficients, displacement, phi and warped image."""
    import types
    import torch.nn.functional as F
    from liftreg_b200 import _native, dropin, net_utils, synthetic
    from oracle import torch_port
    shape, det, B, P, K = (160, 160, 160), (256, 256), 8, 4, 56
    N = 3 * int(np.prod(shape))
    hu = synthetic.ct_phantom(shape)
    unit = synthetic.hu_to_unit(hu)
    poses = synthetic.wrapper_poses(60.0, P, shape[1])
    tp0 = synthetic.normalise_projection(torch_port.drr(synthetic.hu_to_mu(hu), poses, det, (2.2, 2.2, 2.2), device=dev))
    moving = cu(np.stack([np.roll(unit, 3 * b, axis=b % 3) for b in range(B)])[:, None], dev)
    target_proj = cu(np.stack([np.roll(tp0, 2 * b, axis=1 + b % 2) * (1.0 - 0.05 * b) for b in range(B)]).astype(np.float32), dev)
    poses_b = torch.from_numpy(np.repeat(poses[None], B, 0).astype(np.float32))
    torch.manual_seed(2021)
    encoder = torch.nn.Sequential(torch.nn.Conv3d(1 + P, 8, 4, stride=4), torch.nn.ReLU(), torch.nn.Conv3d(8, 8, 4, stride=4),
                                  torch.nn.ReLU(), torch.nn.Flatten(), torch.nn.Linear(8 * 10 ** 3, K)).to(dev)
    gen = torch.Generator(device=dev).manual_seed(0)
    base = torch.randn((K, 65536), device=dev, generator=gen) * 1e-3
    pca_vectors = base.repeat(1, N // 65536 + 1)[:, :N].contiguous().t()                 # (N,K) view, strides (1,N)
    pca_mean = torch.randn(N, device=dev, generator=gen) * 1e-3
    del base
    prev_tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False                                              # fp32 convolutions in both runs
    try:
        with torch.no_grad():
            grids = torch_port.backproj_grid(poses_b[0:1].numpy(), shape, det, device=dev).permute(0, 1, 3, 4, 5, 2)
            x = torch.cat([moving, torch_port.backproject(target_proj, grids)], dim=1)
            del grids
            ref = {"coefs": encoder(x)}
            del x
            ref["disp"] = F.linear(ref["coefs"], pca_vectors, pca_mean).reshape((B, 3) + shape)
            ref["phi"] = ref["disp"] + torch_port.identity_map(shape).to(dev)
            ref["warped"] = torch_port.warp(moving, ref["phi"], zero_boundary=True, using_scale=True)
            ref = {k: v.cpu() for k, v in ref.items()}
            torch.cuda.empty_cache()

            model = types.SimpleNamespace(encoders=list(encoder), pca_vectors=pca_vectors, pca_mean=pca_mean)
            _native.launch_count_reset()
            coefs, disp = dropin._estimate_flow(model, moving, target_proj, poses_b)
            phi = disp + net_utils.gen_identity_map(shape, 1.0)
            warped = net_utils.Bilinear(zero_boundary=True, using_scale=True)(moving, phi)
            torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.allow_tf32 = prev_tf32
    assert _native.launch_count() >= 3                    # backprojection, PCA decode, warp ran in the native library
    assert model.pca_vectors.is_contiguous()             # the (N,K) view was made dense once
    for k, v in (("coefs", coefs), ("disp", disp), ("phi", phi), ("warped", warped)):
        out = v.cpu()
        assert out.shape == ref[k].shape, k
        for b in range(B):
            assert rel_l2(out[b].numpy(), ref[k][b].numpy()) <= TOL, (k, b)


def test_cfg5_training_step_ops_batch4_forward_backward(dev):
    """configs[4] (per-GPU share of batch 32 on 8 GPUs = 4 items): warp forward + d/dphi and the PCA decode adjoint at
    160^3; gradients against the stock torch CUDA ops on the same device."""
    import torch.nn.functional as F
    from liftreg_b200 import net_utils, ops, synthetic
    shape, B = (160, 160, 160), 4
    rs = np.random.RandomState(61)
    moving = torch.from_numpy(rs.uniform(-1, 1, (B, 1) + shape).astype(np.float32)).to(dev)
    disp0 = torch.stack([torch.from_numpy(synthetic.smooth_displacement(shape, seed=10 + s)) for s in range(B)]).to(dev)
    ident = net_utils.gen_identity_map(shape, 1.0)
    gout = torch.from_numpy(rs.standard_normal((B, 1) + shape).astype(np.float32)).to(dev)

    d1 = disp0.clone().requires_grad_(True)
    ours = ops.warp(moving, d1, zero_boundary=True, using_scale=True, disp_plus_identity=True)
    ours.backward(gout)
    d2 = disp0.clone().requires_grad_(True)
    phi = d2 + ident
    grid = torch.stack([phi[:, 2], phi[:, 1], phi[:, 0]], dim=-1)        # net_utils.py:27-30
    ref = F.grid_sample((moving + 1) / 2, grid, mode="bilinear", padding_mode="zeros", align_corners=True) * 2 - 1
    ref.backward(gout)
    for b in range(B):
        assert rel_l2(ours[b].detach().cpu().numpy(), ref[b].detach().cpu().numpy()) <= TOL
        assert rel_l2(d1.grad[b].cpu().numpy(), d2.grad[b].cpu().numpy()) <= GRAD_TOL


# ------------------------------------------------------------------ row f4: similarity loss and label warp
def test_ncc_loss_vs_reference_golden(dev):
    """NCCLoss mirror (one fused forward pass + one backward pass) against the reference's value and gradient; fp32 tolerance:
    the reference sums in torch's fp32 cascade, the kernels in fp32 partials + fp64."""
    from liftreg_b200 import losses
    g = load_golden("ncc")
    x = cu(g["warped"], dev).requires_grad_(True)
    loss = losses.NCCLoss()(x, cu(g["target"], dev))
    loss.backward()
    assert abs(loss.detach().item() - float(g["loss"])) <= 1e-6
    assert rel_l2(x.grad.cpu().numpy(), g["grad"]) <= GRAD_TOL


@pytest.mark.parametrize("B,shape", [(1, (160, 160, 160)), (4, (33, 20, 47)), (2, (1, 1, 3))])
def test_ncc_loss_vs_torch_port(dev, B, shape):
    from liftreg_b200 import ops
    from oracle import torch_port
    rs = np.random.RandomState(70)
    target = rs.uniform(-1, 1, (B, 1) + shape).astype(np.float32)
    warped = (0.6 * target + 0.4 * rs.uniform(-1, 1, (B, 1) + shape)).astype(np.float32)
    x = cu(warped, dev).requires_grad_(True)
    loss = ops.ncc_loss(x, cu(target, dev))
    (3.0 * loss).backward()
    xr = torch.from_numpy(warped).double().requires_grad_(True)            # float64 evaluation of the same formula
    ref = torch_port.ncc_loss(xr, torch.from_numpy(target).double())
    (3.0 * ref).backward()
    assert abs(loss.detach().item() - ref.detach().item()) <= 2e-6
    assert rel_l2(x.grad.cpu().numpy(), xr.grad.numpy()) <= GRAD_TOL


@pytest.mark.parametrize("boundary", ["linear", "neumann_zero"])
@pytest.mark.parametrize("B,shape", [(1, (160, 160, 160)), (2, (17, 33, 40)), (3, (5, 6, 7)), (1, (2, 2, 2)), (1, (3, 2, 70)),
                                     (2, (6, 5, 33)), (1, (4, 4, 4)), (2, (7, 9, 6)), (1, (35, 3, 2))])
def test_diffusion_regulariser_vs_torch_port(dev, B, shape, boundary):
    """SubspaceLoss.py:51-67 (mermaid central differences, both face rules): the fused kernel's value against the fp32
    torch restatement and its float64 evaluation, the gradient against autograd through the float64 one.  Even row
    lengths run the two-voxels-per-thread kernels, odd ones the scalar kernels."""
    from liftreg_b200 import ops
    from oracle import torch_port
    rs = np.random.RandomState(71)
    disp = (0.05 * rs.standard_normal((B, 3) + shape)).astype(np.float32)
    x = cu(disp, dev).requires_grad_(True)
    reg = ops.diffusion_reg(x, boundary)
    (0.7 * reg).backward()
    xr = torch.from_numpy(disp).double().requires_grad_(True)
    ref = torch_port.diffusion_reg(xr, boundary)
    (0.7 * ref).backward()
    ref32 = torch_port.diffusion_reg(torch.from_numpy(disp), boundary).item()
    assert abs(reg.item() - ref.item()) <= 2e-6 * abs(ref.item())
    assert abs(reg.item() - ref32) <= 1e-5 * abs(ref32)            # torch.mean's fp32 cascade vs fp64 accumulation here
    assert rel_l2(x.grad.cpu().numpy(), xr.grad.numpy()) <= GRAD_TOL


def test_subspace_loss_mirror(dev):
    """losses.SubspaceLoss == sim_factor * NCC + reg_factor(epoch) * regulariser (SubspaceLoss.py:20-37), through autograd."""
    from liftreg_b200 import losses
    from oracle import torch_port
    rs = np.random.RandomState(72)
    shape = (12, 14, 10)
    target = rs.uniform(-1, 1, (2, 1) + shape).astype(np.float32)
    warped = (0.5 * target + 0.5 * rs.uniform(-1, 1, (2, 1) + shape)).astype(np.float32)
    params = (0.05 * rs.standard_normal((2, 3) + shape)).astype(np.float32)
    crit = losses.loss({"initial_reg_factor": 10, "min_reg_factor": 1e-3, "reg_factor_decay_from": 10})
    w, p = cu(warped, dev).requires_grad_(True), cu(params, dev).requires_grad_(True)
    for epoch in (0, 14):
        out = crit({"warped": w, "target": cu(target, dev), "params": p, "pca_coefs": None, "epoch": epoch})
        wr, pr = torch.from_numpy(warped).double().requires_grad_(True), torch.from_numpy(params).double().requires_grad_(True)
        factor = max(losses.sigmoid_decay(epoch, static=10, k=2) * 10, 1e-3)
        ref = torch_port.ncc_loss(wr, torch.from_numpy(target).double()) + factor * torch_port.diffusion_reg(pr)
        assert abs(out["total_loss"].item() - ref.item()) <= 1e-5 * abs(ref.item())
        assert abs(out["sim_loss"] + crit.get_reg_factor(epoch) * out["reg_loss"] - out["total_loss"].item()) <= 1e-5
        w.grad = p.grad = None
        out["total_loss"].backward()
        ref.backward()
        assert rel_l2(w.grad.cpu().numpy(), wr.grad.numpy()) <= GRAD_TOL
        assert rel_l2(p.grad.cpu().numpy(), pr.grad.numpy()) <= GRAD_TOL


def test_label_warp_mirror_of_mermaid_entry_point(dev):
    """RegistrationNet.py:191-196: compute_warped_image_multiNC(labels, phi, spacing, spline_order=0, zero_boundary=True,
    use_01_input=False) == nearest-mode spatial transformer without intensity rescaling (pinned nearest arithmetic)."""
    from liftreg_b200 import mermaid_utils
    from oracle import c_oracle
    g = load_golden("warp_small")
    img, phi = g["img"], g["phi"]
    labels = (img > 0).astype(np.float32)
    out = mermaid_utils.compute_warped_image_multiNC(cu(labels, dev), cu(phi, dev), (1.0, 1.0, 1.0), spline_order=0,
                                                     zero_boundary=True, use_01_input=False)
    assert np.array_equal(out.cpu().numpy(), c_oracle.warp_forward(labels, phi, True, False, "nearest"))
    lin = mermaid_utils.compute_warped_image_multiNC(cu(img, dev), cu(phi, dev), (1.0, 1.0, 1.0), spline_order=1,
                                                     zero_boundary=False, use_01_input=False)
    assert np.array_equal(lin.cpu().numpy(), c_oracle.warp_forward(img, phi, False, False, "bilinear"))
    # use_01_input: the map is given in [0, spacing*(sz-1)] and rescaled to [-1, 1] first
    sz = np.array(phi.shape[2:], np.float64)
    spacing = 1.0 / (sz - 1)
    phi01 = ((phi.astype(np.float64) / 2 + 0.5) * (spacing * (sz - 1)).reshape(1, 3, 1, 1, 1)).astype(np.float32)
    out01 = mermaid_utils.compute_warped_image_multiNC(cu(img, dev), cu(phi01, dev), spacing, spline_order=1,
                                                       zero_boundary=False, use_01_input=True)
    assert rel_l2(out01.cpu().numpy(), lin.cpu().numpy()) <= 1e-4       # coordinates round-trip through [0, 1] in fp32


# ------------------------------------------------------------------ backprojection rows kernel
@pytest.mark.parametrize("shape,pshape,B,P", [((160, 160, 160), (256, 256), 1, 4), ((33, 6, 70), (40, 31), 3, 2),
                                              ((40, 9, 300), (64, 350), 1, 2), ((5, 7, 3), (9, 4), 2, 66), ((64, 48, 33), (20, 300), 1, 3)])
def test_backproject_rows_kernel_strided_slab_and_dense_agree(dev, shape, pshape, B, P):
    """lr_backproject_forward (the rows kernel, fast numerics) into channels 1..P of a wider buffer, into a dense
    buffer and, through lr_backproject_forward_slab, into an unaligned z-slab: bit-identical, the sentinel channels
    untouched -- and equal to the oracle's fast blend order and to ops.backproject."""
    import ctypes
    from liftreg_b200 import _native, ops, synthetic
    from oracle import c_oracle
    lib = _native.lib()
    prev = _native.set_numerics("fast")
    try:
        rs = np.random.RandomState(11)
        d, w, h = shape
        tp = cu(rs.uniform(-1, 1, (B, P) + pshape).astype(np.float32), dev)
        poses = synthetic.wrapper_poses(60.0, P, shape[1]).astype(np.float32)
        if P > 2:
            poses[1, 1] = shape[1] * 1.02          # an emitter close to the volume: strong magnification, rows leave the detector
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        vp = lambda t: ctypes.c_void_p(t.data_ptr())
        nv = d * w * h
        ref = torch.empty((B, P, d, w, h), device=dev)
        _native.check(lib.lr_backproject_forward(vp(tp), ops._fp(poses), B, P, pshape[0], pshape[1], d, w, h, vp(ref), P * nv, nv, st), "dense")
        out = torch.full((B, P + 2, d, w, h), 3.0, device=dev)            # channels 1..P of a wider buffer
        view = out[:, 1:1 + P]
        _native.check(lib.lr_backproject_forward(vp(tp), ops._fp(poses), B, P, pshape[0], pshape[1], d, w, h,
                                                 ctypes.c_void_p(view.data_ptr()), (P + 2) * nv, nv, st), "strided")
        assert torch.equal(view, ref) and bool((out[:, 0] == 3.0).all()) and bool((out[:, -1] == 3.0).all())
        if d >= 5:
            z0, nz = d // 3, max(1, d // 2 - 1)
            slab = torch.empty((B, P, nz, w, h), device=dev)
            _native.check(lib.lr_backproject_forward_slab(vp(tp), ops._fp(poses), B, P, pshape[0], pshape[1], d, w, h, z0, nz,
                                                          vp(slab), P * nz * w * h, nz * w * h, st), "slab")
            assert torch.equal(slab, ref[:, :, z0:z0 + nz])
        if nv * B * P <= 4_000_000:
            prev_blend = c_oracle.set_blend("fast")
            try:
                assert np.array_equal(ref.cpu().numpy(), c_oracle.backproject_forward(tp.cpu().numpy(), poses, shape))
            finally:
                c_oracle.set_blend(prev_blend)
        assert torch.equal(ops.backproject(tp, poses, shape), ref)
    finally:
        _native.set_numerics(prev)
