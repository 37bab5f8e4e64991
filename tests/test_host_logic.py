"""Host-side logic that needs no GPU: numerical tricks used by the kernels (emulated in numpy), the synthetic input
generators, pose synthesis, and the argument validation of the Python mirror."""
import numpy as np
import pytest
import torch

f32 = np.float32


# ---------------------------------------------------------------- kernel arithmetic, emulated bit for bit
def test_markstein_division_by_constant_is_correctly_rounded():
    """common.cuh div_const: q0 = x*rc; r = fma(-c,q0,x); q = fma(r,rc,q0) == x/c (IEEE) for the divisors the DRR
    kernel uses (d/2, (w-1)/2, w/2, h/2)."""
    rs = np.random.RandomState(0)
    xs = np.concatenate([rs.uniform(-700, 900, 2_000_000), rs.uniform(-2, 2, 500_000), rs.standard_normal(500_000) * 1e-3,
                         np.arange(-2000, 2000) / 4.0]).astype(f32)
    for c in (80.0, 79.5, 256.0, 255.5, 120.0, 64.5, 0.5, 1.5, 3.0, 13.0, 6.5, 511.5):
        c32 = f32(c)
        rc = f32(1) / c32
        q0 = (xs * rc).astype(f32)
        r = xs.astype(np.float64) - np.float64(c32) * q0.astype(np.float64)       # exact (an fma)
        assert np.all(r == r.astype(f32))
        q = (q0.astype(np.float64) + r * np.float64(rc)).astype(f32)
        assert np.array_equal(q, (xs / c32).astype(f32)), c


def test_magic_number_floor_matches_floor():
    """common.cuh floor_fi: t = x + 1.5*2^23 rounded toward -inf (FADD.RM); floor = t - 1.5*2^23; the integer floor is
    the mantissa of t.  rint_i is the round-to-nearest variant."""
    rs = np.random.RandomState(1)
    xs = np.concatenate([rs.uniform(-3, 600, 2_000_000), np.arange(-8, 600, 0.25), np.arange(-2, 3, 2.0 ** -20),
                         [-2.0, -1.0, -0.0, 0.0, 0.99999994, 1.0, 511.99997, 512.0, -4194303.5, 4194303.5]]).astype(f32)
    M = f32(12582912.0)
    exact = xs.astype(np.float64) + np.float64(M)            # exact in float64
    t = exact.astype(f32)
    t = np.where(t.astype(np.float64) > exact, np.nextafter(t, f32(-np.inf)), t)   # round toward -inf
    fl = (t - M).astype(f32)
    fi = t.view(np.int32) - np.int32(0x4B400000)
    assert np.array_equal(fl, np.floor(xs))
    assert np.array_equal(fi, np.floor(xs).astype(np.int32))
    # out-of-range and NaN inputs give indices no bounds test accepts (|i| >= 2^22)
    bad = np.array([4194304.0, 1e7, 3e9, -4194304.5, -1e7, -3e9, np.nan, np.inf, -np.inf], f32)
    with np.errstate(invalid="ignore", over="ignore"):
        tb = (bad.astype(np.float64) + np.float64(M)).astype(f32)
    ib = tb.view(np.int32).astype(np.int64) - 0x4B400000
    assert np.all((ib < 0) | (ib >= (1 << 22)))
    tn = (xs + M).astype(f32)                                  # round to nearest even
    assert np.array_equal(tn.view(np.int32) - np.int32(0x4B400000), np.rint(xs).astype(np.int32))


def test_scaling_identities_used_to_fold_constants():
    """X/d*2 == X/(d/2) and ((g+1)/2)*(S-1) == (g+1)*((S-1)/2) in fp32 (power-of-two scalings commute with rounding)."""
    rs = np.random.RandomState(2)
    x = rs.uniform(-700, 900, 1_000_000).astype(f32)
    for d in (160, 159, 512, 7, 1):
        assert np.array_equal((x / f32(d) * f32(2.0)).astype(f32), (x / f32(d / 2.0)).astype(f32))
    g = rs.uniform(-1.5, 1.5, 1_000_000).astype(f32)
    for S in (160, 159, 512, 2, 1):
        a = (((g + f32(1)) / f32(2)) * f32(S - 1)).astype(f32)
        b = ((g + f32(1)) * f32((S - 1) / 2.0)).astype(f32)
        assert np.array_equal(a, b)


# ---------------------------------------------------------------- synthetic inputs
def test_synthetic_inputs_are_deterministic_and_in_range():
    from liftreg_b200 import synthetic
    a = synthetic.ct_phantom((24, 20, 28), seed=7, sigma=1.0, nodules=6)
    b = synthetic.ct_phantom((24, 20, 28), seed=7, sigma=1.0, nodules=6)
    assert np.array_equal(a, b) and a.dtype == np.float32
    assert a.min() < -900 and a.max() > -200
    mu = synthetic.hu_to_mu(a)
    assert mu.min() >= 0 and mu.max() < 0.6
    u = synthetic.hu_to_unit(a)
    assert u.min() >= -1 and u.max() <= 1
    d = synthetic.smooth_displacement((12, 10, 14), seed=3, max_disp=0.05, coarse=4)
    assert d.shape == (3, 12, 10, 14) and abs(np.abs(d).max() - 0.05) < 1e-7
    assert np.array_equal(d, synthetic.smooth_displacement((12, 10, 14), seed=3, max_disp=0.05, coarse=4))
    p = synthetic.normalise_projection(np.array([[-1.0, 0.0, 3.0, 6.0, 9.0]], np.float32))
    assert np.allclose(p, [[-1, -1, 0, 1, 1]])


def test_pose_synthesis_matches_the_reference_formula():
    """sdct:139-144,155: x = tan(linspace(-a/2,a/2,P) deg)*3, y = 3.5, z = linspace(-.2,.2,P), all times w."""
    from liftreg_b200 import synthetic
    from liftreg_b200 import sdct_projection_utils as sdct
    from conftest import load_golden
    g = load_golden("drr_cfg1")
    assert np.array_equal(synthetic.wrapper_poses(60.0, 4, 160), g["poses"])
    assert np.array_equal(sdct._wrapper_poses_scale(60.0, 4, 3.5) * 160, g["poses"])
    p = synthetic.wrapper_poses(60.0, 4, 160)
    assert np.allclose(p[:, 1], 560.0) and np.allclose(p[[0, -1], 0], [-np.tan(np.pi / 6) * 480, np.tan(np.pi / 6) * 480])
    assert sdct._default_resolution((160, 160, 160), None) == [240, 240]
    assert sdct._default_resolution((160, 160, 160), (256, 256)) == [256, 256]


# ---------------------------------------------------------------- mirror API: validation without a GPU
def test_cpu_tensors_and_bad_arguments_raise():
    from liftreg_b200 import ops
    from liftreg_b200 import sdct_projection_utils as sdct
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.warp(torch.zeros(1, 1, 2, 2, 2), torch.zeros(1, 3, 2, 2, 2))
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.drr_project(torch.zeros(1, 2, 2, 2), np.zeros((1, 3)), (2, 2), (1, 1, 1))
    with pytest.raises(RuntimeError, match="no CPU path"):
        ops.backproject(torch.zeros(1, 1, 4, 4), np.zeros((1, 3), np.float32), (2, 2, 2))
    with pytest.raises(ValueError):
        ops.warp(torch.zeros(1, 1, 2, 2, 2), torch.zeros(1, 2, 2, 2, 2))
    with pytest.raises(ValueError):
        ops.warp(torch.zeros(1, 1, 2, 2, 2), torch.zeros(1, 3, 2, 2, 2), mode="cubic")
    with pytest.raises(ValueError):
        ops.drr_project(torch.zeros(2, 2, 2), np.zeros((1, 3)), (2, 2), (1, 1, 1))
    with pytest.raises(ValueError):
        ops.drr_project(torch.zeros(3, 2, 2, 2), np.zeros((2, 1, 3)), (2, 2), (1, 1, 1))
    with pytest.raises(ValueError):
        ops.backproject(torch.zeros(1, 2, 4, 4), np.zeros((3, 3), np.float32), (2, 2, 2))
    with pytest.raises(ValueError):
        ops.backproject(torch.zeros(1, 1, 4, 4), np.zeros((1, 3), np.float32), (4, 2, 2), slab=(3, 2))
    with pytest.raises(NotImplementedError):
        sdct.calculate_projection(np.zeros((2, 2, 2), np.float32), np.zeros((1, 3)), (2, 2), [2, 1, 1], (1, 1, 1), "cuda")
    with pytest.raises(RuntimeError, match="CUDA devices only"):
        sdct.project_grid_multi(np.zeros((1, 3)), (2, 2), [1, 1, 1], (2, 2, 2), torch.ones(3), torch.device("cpu"), torch.float32)
    with pytest.raises(NotImplementedError):
        sdct.project_grid_multi(np.zeros((1, 3)), (2, 2), [1, 1, 1], (2, 2, 2), torch.ones(3), "cuda", torch.float64)


def test_mirror_modules_expose_the_reference_surface():
    """Names and signatures of SURVEY.md 8b."""
    import inspect
    from liftreg_b200 import layers, net_utils
    from liftreg_b200 import sdct_projection_utils as sdct
    want = {
        "project_grid_multi": ["emi_pos", "resolution", "sample_rate", "obj_shape", "spacing", "device", "dtype"],
        "calculate_projection": ["img", "poses", "resolution", "sample_rate", "spacing", "device"],
        "calculate_projection_wraper": ["img_3d", "scan_range", "proj_num", "spacing", "receptor_size"],
        "calculate_projection_wraper_with_geo_csv_file": ["img_3d", "img_spacing", "geo_path", "receptor_size"],
        "backproj_grids": ["scan_range", "proj_num", "img_shape", "proj_shape", "device"],
        "forward_grids": ["scan_range", "proj_num", "spacing", "img_shape", "device", "receptor_size"],
        "backproj_grids_with_poses": ["poses", "img_shape", "proj_shape", "device"],
        "forward_grids_with_poses": ["poses", "spacing", "img_shape", "device", "receptor_size"],
        "calc_relative_atten_coef": ["img"],
        "calc_relative_atten_coef_cuda": ["img"],
    }
    for name, params in want.items():
        assert list(inspect.signature(getattr(sdct, name)).parameters) == params, name
    assert list(inspect.signature(net_utils.Bilinear.__init__).parameters) == ["self", "zero_boundary", "using_scale", "mode"]
    assert list(inspect.signature(net_utils.Bilinear.forward).parameters) == ["self", "input1", "input2"]
    assert hasattr(net_utils.Bilinear, "forward_stn")
    assert list(inspect.signature(net_utils.identity_map).parameters) == ["sz", "dtype"]
    assert list(inspect.signature(net_utils.gen_identity_map).parameters) == ["img_sz", "resize_factor", "normalized"]
    assert list(inspect.signature(layers.proj_layer.__init__).parameters) == \
        ["self", "volume_spacing", "resolution_scale", "scan_range", "proj_num", "in_shape", "out_shape", "device"]
    b = net_utils.Bilinear(zero_boundary=True)
    assert b.zero_boundary == "zeros" and b.using_scale is True and b.mode == "bilinear"
    assert net_utils.Bilinear().zero_boundary == "border"
    a = np.array([[-1500.0, -1000.0, 0.0, 1000.0]], np.float32)
    assert np.allclose(sdct.calc_relative_atten_coef(a), [[0.0, 0.0, 0.2, 0.4]])


# ------------------------------------------------------------------ launch plans (tapered block sizes) tile the work exactly
def _plan(fn, n, *args):
    import ctypes
    from liftreg_b200 import _native
    out = (ctypes.c_int * n)()
    _native.check(getattr(_native.lib(), fn)(*args, out), fn)
    return list(out)


@pytest.mark.parametrize("B", [1, 2, 8, 64])
def test_warp_forward_plan_tiles_every_plane_once(B):
    """The z-blocks of lr_warp_forward (8-, 4- and 2-plane blocks, long ones first) must cover [0, Do) exactly once for
    every slab height, whatever share the wave heuristic picks."""
    for Do in list(range(1, 70)) + [96, 159, 160, 161, 255, 256, 320, 511, 512]:
        for (H, W) in ((160, 160), (17, 33), (512, 512)):
            s0, n0, s1, n1, s2, n2 = _plan("lr_warp_forward_plan", 6, B, max(Do, 2), H, W, Do)
            assert min(s0, s1, s2) >= 1 and max(s0, s1, s2) <= 8 and min(n0, n1, n2) >= 0 and n0 + n1 + n2 >= 1
            covered, z = np.zeros(Do, np.int32), 0
            for size, n in ((s0, n0), (s1, n1), (s2, n2)):
                for _ in range(n):
                    assert z < Do, "a z-block starts beyond the slab (Do=%d B=%d H=%d W=%d)" % (Do, B, H, W)
                    covered[z:min(Do, z + size)] += 1
                    z += size
            assert (covered == 1).all(), (Do, B, H, W, (s0, n0, s1, n1, s2, n2))


@pytest.mark.parametrize("B", [1, 3, 8])
def test_backproject_forward_plan_tiles_planes_and_rows_once(B):
    """Chunks of planes x runs of rows of lr_backproject_forward: every (plane, row) belongs to exactly one block."""
    for (d, w, h) in ((160, 160, 160), (1, 4, 1), (5, 7, 3), (33, 6, 70), (64, 65, 2), (320, 320, 320), (512, 512, 512), (31, 1, 600)):
        for P in (1, 4, 64, 70):
            ichunk, isub, by, bx, n_chunks, r0, n0, r1, n1, r2, n2, grid = _plan("lr_backproject_forward_plan", 12, B, P, 256, 256, d, w, h)
            assert isub * by == ichunk and 1 <= ichunk <= 32 and isub % 4 == 0
            assert (n_chunks - 1) * ichunk < d <= n_chunks * ichunk
            # bx = column pairs per block; tiny volumes are padded up to a whole warp (warp 0 builds the row tables)
            hp = min((h + 1) // 2, 256)
            assert 1 <= bx <= 256 and bx * by <= 256 and bx == (hp if hp * by >= 32 else -(-32 // by))
            rows, j = np.zeros(w, np.int32), 0
            for run, n in ((r0, n0), (r1, n1), (r2, n2)):
                for _ in range(n):
                    assert j < w
                    rows[j:min(w, j + run)] += 1
                    j += run
            assert (rows == 1).all(), (d, w, h, P, B)
            assert grid == (n0 + n1 + n2) * n_chunks * min(P, 64) * B


def test_numerics_mode_is_settable_without_a_gpu_and_rejects_bad_values():
    """lr_set_numerics / lr_get_numerics (include/liftreg_b200.h): process-wide, no device work."""
    from liftreg_b200 import _native
    lib = _native.lib()
    prev = _native.get_numerics()
    try:
        assert _native.set_numerics("exact") == prev and _native.get_numerics() == "exact" and lib.lr_get_numerics() == 1
        assert _native.set_numerics("fast") == "exact" and lib.lr_get_numerics() == 0
        assert lib.lr_set_numerics(7) == -1 and b"mode" in lib.lr_last_error()
        assert lib.lr_get_numerics() == 0
    finally:
        _native.set_numerics(prev)

