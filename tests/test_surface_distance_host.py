"""Surface-distance metrics without a GPU: the float64 reference (tests/surface_reference.py) against a brute-force
all-pairs minimum and np.percentile, the percentile form metrics.surface_distance applies to its two order statistics,
and the C-ABI argument checks of the new entry points."""
import ctypes

import numpy as np
import pytest
from scipy import ndimage as ndi

from surface_reference import brute_force, directed, surface, surface_distance

SPACINGS = [(1.0, 1.0, 1.0), (1.0, 2.0, 3.0), (2.2, 2.2, 2.2), (1.5, 0.7, 2.2)]


def random_labels(shape, L, seed, smooth=1.0):
    rs = np.random.RandomState(seed)
    return np.argmax(ndi.gaussian_filter(rs.rand(L, *shape), (0,) + (smooth,) * 3), axis=0)


def test_surface_is_the_face_connected_boundary():
    m = np.zeros((5, 6, 7), bool)
    m[1:4, 1:5, 1:6] = True
    s = surface(m)
    inner = np.zeros_like(m)
    inner[2:3, 2:4, 2:5] = True
    assert np.array_equal(s, m & ~inner)
    full = np.ones((3, 4, 5), bool)               # every voxel of a volume-filling label touches a face
    assert np.array_equal(surface(full), ~np.pad(np.ones((1, 2, 3), bool), 1, constant_values=False))
    one = np.zeros((3, 3, 3), bool)
    one[1, 1, 1] = True
    assert np.array_equal(surface(one), one)


@pytest.mark.parametrize("spacing", SPACINGS)
@pytest.mark.parametrize("shape,seed", [((6, 7, 8), 0), ((5, 1, 9), 1), ((1, 1, 12), 2), ((9, 1, 1), 3), ((4, 5, 3), 4)])
def test_reference_equals_brute_force(shape, seed, spacing):
    lab = random_labels(shape, 3, seed)
    for l in range(3):
        for a, b in ((lab == l, lab != l), (lab == l, np.roll(lab == l, 1, axis=0))):
            sa, sb = surface(a), surface(b)
            if not sa.any() or not sb.any():
                continue
            ref, bf = directed(sa, sb, spacing), brute_force(sa, sb, spacing)
            if spacing in SPACINGS[:2]:
                assert np.array_equal(ref, bf)
            else:
                assert np.all(np.abs(ref - bf) <= 8 * 2.0 ** -53 * bf)


def test_reference_edge_cases_against_brute_force():
    shape = (6, 5, 7)
    faces = np.zeros(shape, bool)
    faces[0], faces[:, -1], faces[:, :, 0] = True, True, True          # a label on three faces
    single = np.zeros(shape, bool)
    single[3, 2, 4] = True
    full = np.ones(shape, bool)
    for a in (faces, single, full):
        for b in (faces, single, full):
            for sp in SPACINGS:
                ref, bf = directed(surface(a), surface(b), sp), brute_force(surface(a), surface(b), sp)
                assert np.allclose(ref, bf, rtol=8 * 2.0 ** -53, atol=0)


def test_reference_metrics_by_hand():
    """a 4-voxel cube shifted by 2 along W: every surface voxel of one map is 0 or 2 voxels from the other surface"""
    pred = np.zeros((1, 8, 8, 10), np.int64)
    target = np.zeros_like(pred)
    pred[0, 2:6, 2:6, 2:6] = 1
    target[0, 2:6, 2:6, 4:8] = 1
    res = surface_distance(pred, target, spacing=(1.0, 1.0, 2.5))
    d = res["directed"][(0, 1, 0)]
    assert res["surface_count"][0, 0, 1] == res["surface_count"][0, 1, 1] == 56
    assert d.max() == 5.0 and res["hd"][0, 1] == 5.0
    assert res["hd95"][0, 1] == np.percentile(d, 95)
    assert np.isnan(res["hd"][0, 0]) and res["hd_mean"][0] == 5.0
    assert np.array_equal(d, res["directed"][(0, 1, 1)])                 # symmetric configuration


def test_reference_absent_label_is_nan():
    pred = np.zeros((2, 4, 4, 4), np.int64)
    target = np.zeros_like(pred)
    pred[0, 1:3, 1:3, 1:3] = 1
    target[:, 0:2, 0:2, 0:2] = 1
    res = surface_distance(pred, target, num_labels=3)
    assert np.isfinite(res["hd"][0, 1]) and np.isnan(res["hd"][1, 1]) and np.isnan(res["hd"][:, 2]).all()
    assert res["surface_count"][1, 0, 1] == 0 and res["surface_count"][1, 1, 1] == 8
    assert np.isnan(res["hd_mean"][1]) and res["hd_mean"][0] == res["hd"][0, 1]


@pytest.mark.parametrize("n", [1, 2, 3, 19, 20, 21, 40, 101, 1000, 4097])
def test_percentile_from_two_order_statistics_equals_numpy(n):
    from liftreg_b200 import metrics
    rs = np.random.RandomState(n)
    for v in (np.sort(rs.rand(n) * 40), np.sort(np.sqrt(rs.randint(0, 60, n).astype(np.float64)))):
        lo, hi, t = metrics._q95_index(np.array([n]))
        assert metrics._lerp(v[lo], v[hi], t)[0] == np.percentile(v, 95)


@pytest.fixture(scope="module")
def lib():
    from liftreg_b200 import _native, build
    build.build()
    return _native.lib()


def test_surface_entries_reject_bad_arguments_before_any_cuda_call(lib):
    fake = ctypes.c_void_p(256)          # never dereferenced: every call below fails validation first
    big = 1 << 40
    cases = [
        (lib.lr_label_surface_counts, (None, fake, 1, 4, 4, 4, 2, fake, fake, None), b"null"),
        (lib.lr_label_surface_counts, (fake, fake, 1, 4, 4, 4, 2, None, fake, None), b"null"),
        (lib.lr_label_surface_counts, (fake, fake, 1, 4, 4, 4, 0, fake, fake, None), b"[1, 128]"),
        (lib.lr_label_surface_counts, (fake, fake, 1, 4, 4, 4, 129, fake, fake, None), b"[1, 128]"),
        (lib.lr_label_surface_counts, (fake, fake, 0, 4, 4, 4, 2, fake, fake, None), b"batch"),
        (lib.lr_label_surface_counts, (fake, fake, 1, 0, 4, 4, 2, fake, fake, None), b">= 1"),
        (lib.lr_label_surface_counts, (fake, fake, 2, 1024, 1024, 1024, 2, fake, fake, None), b"2^31"),
    ]
    ok = (fake, fake, 1, 4, 4, 4, 1, 1.0, 1.0, 1.0, fake, fake, fake, fake, big, None)

    def dist_case(k, v):
        a = list(ok)
        a[k] = v
        return tuple(a)
    cases += [
        (lib.lr_surface_distances, dist_case(0, None), b"null"),
        (lib.lr_surface_distances, dist_case(10, None), b"null"),
        (lib.lr_surface_distances, dist_case(11, None), b"null"),
        (lib.lr_surface_distances, dist_case(13, None), b"null"),
        (lib.lr_surface_distances, dist_case(2, 0), b"batch"),
        (lib.lr_surface_distances, dist_case(2, 65536), b"batch"),
        (lib.lr_surface_distances, dist_case(3, 0), b">= 1"),
        (lib.lr_surface_distances, dist_case(5, 0), b">= 1"),
        (lib.lr_surface_distances, dist_case(5, 65536), b"65535"),
        (lib.lr_surface_distances, dist_case(4, 70000), b"65535"),
        (lib.lr_surface_distances, (fake, fake, 1, 2048, 1024, 1024) + ok[6:], b"2^31"),
        (lib.lr_surface_distances, dist_case(6, 0), b"label"),
        (lib.lr_surface_distances, dist_case(6, 128), b"label"),
        (lib.lr_surface_distances, dist_case(7, 0.0), b"spacing"),
        (lib.lr_surface_distances, dist_case(8, -1.0), b"spacing"),
        (lib.lr_surface_distances, dist_case(9, float("nan")), b"spacing"),
        (lib.lr_surface_distances, dist_case(9, float("inf")), b"spacing"),
        (lib.lr_surface_distances, dist_case(14, 16), b"workspace"),
    ]
    for fn, args, msg in cases:
        assert fn(*args) == -1, args
        assert msg in lib.lr_last_error(), (args, lib.lr_last_error())


def test_surface_distance_workspace_query(lib):
    n = 160 ** 3
    got = lib.lr_surface_distance_workspace_bytes(1, 160, 160, 160)
    assert 16 * n <= got <= 16 * n + 6 * 256 + 24 * (160 * 160 // 128)
    assert lib.lr_surface_distance_workspace_bytes(8, 160, 160, 160) >= 8 * 16 * n
    for args in [(0, 4, 4, 4), (65536, 1, 1, 1), (1, 0, 4, 4), (1, 4, 65536, 4), (1, 4, 4, 65536), (2, 1024, 1024, 1024)]:
        assert lib.lr_surface_distance_workspace_bytes(*args) == 0, args
