"""Surface-distance metrics on the GPU: ops.label_surface_counts / ops.surface_distances and metrics.surface_distance
against the float64 scipy reference (tests/surface_reference.py).  Directed distances are bit-identical to scipy's at
integer spacings and within 8*2^-53*d otherwise (DESIGN.md §3)."""
import numpy as np
import pytest
import torch
from scipy import ndimage as ndi

from surface_reference import surface_distance as ref_surface_distance

pytestmark = pytest.mark.gpu

SPACINGS = [(1.0, 1.0, 1.0), (1.0, 2.0, 3.0), (2.2, 2.2, 2.2), (1.5, 0.7, 2.2)]
U = 2.0 ** -53


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def blobs(B, shape, L, seed, smooth=1.2):
    rs = np.random.RandomState(seed)
    return np.stack([np.argmax(ndi.gaussian_filter(rs.rand(L, *shape), (0,) + (smooth,) * 3), axis=0)
                     for _ in range(B)]).astype(np.int64)


def lungs(shape):
    """labels 1 and 2: the two lung ellipsoids of synthetic.ct_phantom's geometry"""
    z, y, x = np.meshgrid(*(np.linspace(-1, 1, n) for n in shape), indexing="ij")
    out = np.zeros(shape, np.int64)
    for l, cx in ((1, -0.38), (2, 0.38)):
        out[(z / 0.62) ** 2 + (y / 0.45) ** 2 + ((x - cx) / 0.30) ** 2 <= 1.0] = l
    return out


def warped_lungs(dev, shape, seeds):
    from liftreg_b200 import ops, synthetic
    t = torch.from_numpy(lungs(shape)).to(dev).float()[None, None].repeat(len(seeds), 1, 1, 1, 1)
    disp = torch.from_numpy(np.stack([synthetic.smooth_displacement(shape, seed=s, max_disp=0.08) for s in seeds])).to(dev)
    p = ops.warp(t, disp, zero_boundary=True, using_scale=False, mode="nearest", disp_plus_identity=True)
    return p[:, 0].cpu().numpy().astype(np.int64), t[:, 0].cpu().numpy().astype(np.int64)


def gpu_segments(dev, pred, target, L, spacing):
    """{(b, l, k): sorted distances} from ops.surface_distances, k = 0: pred -> target, 1: target -> pred"""
    from liftreg_b200 import ops
    p, t = torch.from_numpy(pred).to(dev), torch.from_numpy(target).to(dev)
    counts = ops.label_surface_counts(p, t, L)[0].cpu().numpy()
    out = {}
    for l in range(1, L):
        for k, (a, b) in enumerate(((p, t), (t, p))):
            n = counts[:, k, l]
            if not n.any():
                continue
            dist, off, stats = ops.surface_distances(a, b, l, spacing, sizes=n)
            d, off, st = dist.cpu().numpy(), off.cpu().numpy(), stats.cpu().numpy()
            for bb in range(len(n)):
                seg = np.sort(d[off[bb]:off[bb + 1]])
                assert st[bb, 0] == seg.size
                if seg.size:
                    assert st[bb, 2] == seg.max()
                    assert np.isclose(st[bb, 1], seg.sum(), rtol=1e-12, atol=0)     # +inf where S_to is empty
                out[(bb, l, k)] = seg
    return out


def check_against_reference(dev, pred, target, spacing, L=None):
    from liftreg_b200 import metrics
    ref = ref_surface_distance(pred, target, spacing, L)
    L = ref["hd"].shape[1]
    got = metrics.surface_distance(torch.from_numpy(pred).to(dev), torch.from_numpy(target).to(dev), spacing, L)
    assert np.array_equal(got["surface_count"], ref["surface_count"])
    segs = gpu_segments(dev, pred, target, L, spacing)
    exact = spacing in SPACINGS[:2]
    for key, r in ref["directed"].items():
        g = segs[key]
        if exact:
            assert np.array_equal(g, r), key
        else:
            assert g.shape == r.shape and np.all(np.abs(g - r) <= 8 * U * r), (key, np.max(np.abs(g - r) / np.maximum(r, 1e-300)))
    for k in ("hd", "hd95", "assd"):
        assert np.array_equal(np.isnan(got[k]), np.isnan(ref[k])), k
    ok = ~np.isnan(ref["hd"])
    if exact:
        assert np.array_equal(got["hd"][ok], ref["hd"][ok])
        h, r = got["hd95"][ok], ref["hd95"][ok]
        assert np.all(np.abs(h - r) <= 2 * np.spacing(np.maximum(r, 1e-300))), np.max(np.abs(h - r))
    else:
        assert np.all(np.abs(got["hd"][ok] - ref["hd"][ok]) <= 8 * U * ref["hd"][ok])
        assert np.allclose(got["hd95"][ok], ref["hd95"][ok], rtol=16 * U, atol=0)
    assert np.allclose(got["assd"][ok], ref["assd"][ok], rtol=1e-12, atol=0)
    for k in ("hd_mean", "hd95_mean", "assd_mean"):
        assert np.allclose(got[k], ref[k], rtol=1e-12, atol=0, equal_nan=True), k
    return got, ref


@pytest.mark.parametrize("spacing", SPACINGS)
@pytest.mark.parametrize("B,shape,L", [(2, (17, 33, 40), 4), (1, (5, 6, 7), 3), (1, (1, 7, 9), 3), (1, (9, 1, 1), 2),
                                       (1, (2, 3, 1500), 3), (2, (33, 20, 64), 5), (1, (1100, 3, 4), 2), (1, (3, 900, 5), 2)])
def test_matches_scipy_on_random_labels(dev, B, shape, L, spacing):
    pred = blobs(B, shape, L, seed=sum(shape) + L)
    target = blobs(B, shape, L, seed=sum(shape) + L + 1)
    check_against_reference(dev, pred, target, spacing)


@pytest.mark.parametrize("spacing", SPACINGS)
def test_phantom_lungs_160_cubed_two_displacements(dev, spacing):
    pred, target = warped_lungs(dev, (160, 160, 160), seeds=(3, 4))
    assert not np.array_equal(pred[0], pred[1])
    got, _ = check_against_reference(dev, pred, target, spacing, L=3)
    assert np.isfinite(got["hd"][:, 1:]).all()


@pytest.mark.parametrize("spacing", SPACINGS[:3])
def test_faces_single_voxels_and_a_filling_label(dev, spacing):
    shape = (7, 8, 9)
    t = np.zeros((3,) + shape, np.int64)
    t[0, 0], t[0, -1], t[0, :, 0], t[0, :, -1], t[0, :, :, 0], t[0, :, :, -1] = 1, 1, 1, 1, 1, 1   # every face
    t[0, 3, 4, 4] = 2                                                                            # single voxels
    t[1] = 1                                                                                     # fills the volume
    t[2, 2, 3, 3], t[2, 5, 1, 7] = 1, 2
    p = np.zeros_like(t)
    p[0, 1:, 1:, 1:] = 1
    p[0, 5, 2, 6] = 2
    p[1, 1:-1, 1:-1, 1:-1] = 1
    p[2, 6, 7, 0], p[2, 0, 0, 8] = 1, 2
    check_against_reference(dev, p, t, spacing)


def test_128_labels_of_small_blobs(dev):
    pred = blobs(1, (24, 28, 32), 128, seed=5, smooth=0.7)
    target = blobs(1, (24, 28, 32), 128, seed=6, smooth=0.7)
    assert len(np.unique(pred)) > 100
    check_against_reference(dev, pred, target, (1.0, 2.0, 3.0), L=128)


def test_float32_and_int64_maps_agree(dev):
    from liftreg_b200 import metrics
    pred, target = blobs(2, (20, 21, 22), 4, seed=7), blobs(2, (20, 21, 22), 4, seed=8)
    a = metrics.surface_distance(torch.from_numpy(pred).to(dev), torch.from_numpy(target).to(dev), (2.2,) * 3)
    b = metrics.surface_distance(torch.from_numpy(pred).float().to(dev)[:, None], torch.from_numpy(target).float().to(dev),
                                 (2.2,) * 3)
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


def test_identical_maps_give_zero_distances(dev):
    from liftreg_b200 import metrics
    m = blobs(2, (18, 19, 20), 4, seed=9)
    res = metrics.surface_distance(torch.from_numpy(m).to(dev), torch.from_numpy(m).to(dev), (1.5, 0.7, 2.2))
    for k in ("hd", "hd95", "assd"):
        v = res[k][:, 1:]
        assert (v[~np.isnan(v)] == 0).all() and (~np.isnan(v)).any()
    for key, seg in gpu_segments(dev, m, m, 4, (1.5, 0.7, 2.2)).items():
        assert (seg == 0).all(), key


def test_swapping_maps_swaps_segments_and_keeps_metrics(dev):
    from liftreg_b200 import metrics
    pred, target = blobs(2, (16, 24, 30), 4, seed=10), blobs(2, (16, 24, 30), 4, seed=11)
    sp = (2.2, 2.2, 2.2)
    ab, ba = gpu_segments(dev, pred, target, 4, sp), gpu_segments(dev, target, pred, 4, sp)
    assert set(ab) == {(b, l, 1 - k) for (b, l, k) in ba}
    for (b, l, k), seg in ab.items():
        assert np.array_equal(seg, ba[(b, l, 1 - k)])
    r1 = metrics.surface_distance(torch.from_numpy(pred).to(dev), torch.from_numpy(target).to(dev), sp)
    r2 = metrics.surface_distance(torch.from_numpy(target).to(dev), torch.from_numpy(pred).to(dev), sp)
    for k in ("hd", "hd95", "assd", "hd_mean", "hd95_mean", "assd_mean"):
        assert np.array_equal(r1[k], r2[k], equal_nan=True), k
    assert np.array_equal(r1["surface_count"], r2["surface_count"][:, ::-1])


@pytest.mark.parametrize("k_d,k_h,k_w", [(0, 0, 3), (2, 0, 0), (1, 2, 3), (0, 4, 0)])
def test_translated_box_gives_closed_form_distances(dev, k_d, k_h, k_w):
    """A box and its translate by k (less than half the box in every axis): the farthest surface voxel is a corner,
    |s*k| from the other surface in both directions, so hd = |s*k|."""
    sp = (1.0, 2.0, 3.0)
    p = np.zeros((1, 16, 17, 18), np.int64)
    t = np.zeros_like(p)
    p[0, 3:10, 2:11, 4:12] = 1
    t[0, 3 + k_d:10 + k_d, 2 + k_h:11 + k_h, 4 + k_w:12 + k_w] = 1
    got, _ = check_against_reference(dev, p, t, sp)
    want = np.sqrt(((sp[0] * k_d) ** 2 + (sp[1] * k_h) ** 2) + (sp[2] * k_w) ** 2)
    assert got["hd"][0, 1] == want
    for seg in gpu_segments(dev, p, t, 2, sp).values():
        assert seg.max() == want


def test_label_in_one_map_only_is_nan_and_leaves_the_rest(dev):
    from liftreg_b200 import metrics
    pred, target = blobs(2, (14, 15, 16), 3, seed=12), blobs(2, (14, 15, 16), 3, seed=13)
    base = metrics.surface_distance(torch.from_numpy(pred).to(dev), torch.from_numpy(target).to(dev), (1.0, 1.0, 1.0), 4)
    p2 = pred.copy()
    p2[1, :3, :3, :3] = 3                                  # label 3 in pred of item 1 only
    res = metrics.surface_distance(torch.from_numpy(p2).to(dev), torch.from_numpy(target).to(dev), (1.0, 1.0, 1.0), 4)
    assert np.isnan(res["hd"][:, 3]).all() and np.isnan(res["assd"][:, 3]).all()
    assert res["surface_count"][1, 0, 3] > 0 and res["surface_count"][1, 1, 3] == 0
    assert np.array_equal(res["hd"][0], base["hd"][0], equal_nan=True)
    assert np.array_equal(res["assd_mean"][0], base["assd_mean"][0])
    nan_mean = metrics.surface_distance(torch.from_numpy(np.where(pred == 0, 0, 1)).to(dev),
                                        torch.from_numpy(np.where(target == 0, 0, 2)).to(dev), (1.0, 1.0, 1.0))
    assert np.isnan(nan_mean["hd_mean"]).all() and np.isnan(nan_mean["hd"]).all()


def test_repeatable_and_independent_of_the_batch(dev):
    from liftreg_b200 import metrics
    pred, target = warped_lungs(dev, (64, 72, 80), seeds=(5, 6))
    sp = (1.5, 0.7, 2.2)
    a, b = gpu_segments(dev, pred, target, 3, sp), gpu_segments(dev, pred, target, 3, sp)
    one = gpu_segments(dev, pred[1:], target[1:], 3, sp)
    assert a.keys() == b.keys()
    for key in a:
        assert np.array_equal(a[key], b[key])
        if key[0] == 1:
            assert np.array_equal(a[key], one[(0,) + key[1:]])
    r1, r2 = (metrics.surface_distance(torch.from_numpy(pred).to(dev), torch.from_numpy(target).to(dev), sp) for _ in range(2))
    for k in r1:
        assert np.array_equal(r1[k], r2[k], equal_nan=True), k


@pytest.mark.parametrize("bad", [-1.0, 0.5, float("nan"), 3.0])
def test_invalid_values_raise_with_the_count(dev, bad):
    from liftreg_b200 import metrics
    pred, target = blobs(2, (6, 7, 8), 3, seed=14).astype(np.float32), blobs(2, (6, 7, 8), 3, seed=15).astype(np.float32)
    pred[1, 2, 3, 4] = bad
    pred[1, 0, 0, 0] = bad
    with pytest.raises(ValueError, match=r"\[0, 2\]"):
        metrics.surface_distance(torch.from_numpy(pred).to(dev), torch.from_numpy(target).to(dev), num_labels=3)
