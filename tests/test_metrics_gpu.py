"""Validation metrics on the GPU: the Jacobian-determinant kernel against the fp32 torch restatement (bit for bit) and its
statistics, the label confusion kernel against np.bincount (exact), and the overlap scores against Python sets."""
import numpy as np
import pytest
import torch

from metrics_reference import jacobian_det, overlap_by_sets
from oracle import torch_port

pytestmark = pytest.mark.gpu

REG_SHAPES = [(1, (160, 160, 160)), (2, (17, 33, 40)), (1, (5, 6, 7)), (1, (2, 2, 2)), (1, (3, 2, 70)),
              (2, (6, 5, 33)), (1, (4, 4, 4)), (2, (7, 9, 6)), (1, (35, 3, 2)), (2, (160, 160, 160)), (2, (24, 31, 51))]


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device("cuda:0")


def noisy_map(B, shape, seed, amp=0.4):
    """identity + per-voxel noise of `amp` grid steps: determinants spread around 1 with a share of folds."""
    rs = np.random.RandomState(seed)
    idm = torch_port.identity_map(shape).numpy()[None]
    step = (2.0 / (np.array(shape) - 1)).reshape(1, 3, 1, 1, 1)
    return (idm + amp * step * rs.standard_normal((B, 3) + shape)).astype(np.float32)


def stats_of(det, margin=0):
    """float64 statistics of a det map (B,D,H,W) over the interior box, finite values only."""
    m = margin
    d = det[:, m:det.shape[1] - m, m:det.shape[2] - m, m:det.shape[3] - m].reshape(det.shape[0], -1).astype(np.float64)
    out = []
    for v in d:
        f = v[np.isfinite(v)]
        neg = f[f < 0]
        out.append([neg.size, -neg.sum(), f.min() if f.size else np.inf, f.max() if f.size else -np.inf, f.sum(),
                    (f * f).sum(), v.size - f.size])
    return np.array(out)


def check_stats(got, ref, det):
    got = np.asarray(got)
    assert np.array_equal(got[:, [0, 6]], ref[:, [0, 6]])                     # counts exact
    assert np.array_equal(got[:, [2, 3]], ref[:, [2, 3]])                     # min / max exact
    absum = np.array([np.abs(v[np.isfinite(v)].astype(np.float64)).sum() for v in det.reshape(det.shape[0], -1)])
    assert np.all(np.abs(got[:, 1] - ref[:, 1]) <= 1e-12 * np.maximum(ref[:, 1], 1e-300))
    assert np.all(np.abs(got[:, 4] - ref[:, 4]) <= 1e-12 * np.maximum(absum, 1e-300))   # sum det: relative to sum |det|
    assert np.all(np.abs(got[:, 5] - ref[:, 5]) <= 1e-12 * ref[:, 5])


@pytest.mark.parametrize("boundary", ["linear", "neumann_zero"])
@pytest.mark.parametrize("B,shape", REG_SHAPES)
def test_jacobian_det_bit_identical_to_fp32_port(dev, B, shape, boundary):
    """Even row lengths run the two-voxels-per-thread kernel, odd ones the scalar kernel."""
    from liftreg_b200 import ops
    phi = noisy_map(B, shape, seed=sum(shape) + B)
    stats, det = ops.jacobian_det(torch.from_numpy(phi).to(dev), boundary, want_map=True)
    ref = jacobian_det(torch.from_numpy(phi), boundary).numpy()
    got = det.cpu().numpy()
    assert np.array_equal(got, ref)
    check_stats(stats.cpu().numpy(), stats_of(ref), ref)
    stats2, none = ops.jacobian_det(torch.from_numpy(phi).to(dev), boundary)         # without the map
    assert none is None
    check_stats(stats2.cpu().numpy(), stats_of(ref), ref)


@pytest.mark.parametrize("boundary", ["linear", "neumann_zero"])
@pytest.mark.parametrize("B,shape", [(1, (33, 20, 64)), (2, (9, 8, 10)), (1, (2, 2, 2))])
def test_jacobian_det_unaligned_view_takes_the_scalar_path(dev, B, shape, boundary):
    from liftreg_b200 import ops
    phi = noisy_map(B, shape, seed=7)
    n = phi.size
    buf = torch.zeros(n + 1, device=dev)
    buf[1:] = torch.from_numpy(phi.reshape(-1)).to(dev)
    view = buf[1:].view(phi.shape)                                   # 4 bytes off an 8-byte boundary
    assert view.data_ptr() % 8 == 4
    stats, det = ops.jacobian_det(view, boundary, want_map=True)
    ref = jacobian_det(torch.from_numpy(phi), boundary).numpy()
    assert np.array_equal(det.cpu().numpy(), ref)
    check_stats(stats.cpu().numpy(), stats_of(ref), ref)


@pytest.mark.parametrize("B,shape,margin", [(1, (160, 160, 160), 8), (2, (17, 33, 40), 3), (1, (7, 9, 11), 3), (2, (5, 6, 7), 1)])
def test_jacobian_stats_margin_selects_the_interior_box(dev, B, shape, margin):
    from liftreg_b200 import metrics, ops
    phi = noisy_map(B, shape, seed=11, amp=0.6)
    ref = jacobian_det(torch.from_numpy(phi), "linear").numpy()
    stats, _ = ops.jacobian_det(torch.from_numpy(phi).to(dev), "linear", margin=margin)
    check_stats(stats.cpu().numpy(), stats_of(ref, margin), ref[:, margin:shape[0] - margin, margin:shape[1] - margin, margin:shape[2] - margin])
    r = metrics.jacobian_stats(torch.from_numpy(phi).to(dev), margin=margin)
    inner = ref[:, margin:shape[0] - margin, margin:shape[1] - margin, margin:shape[2] - margin].reshape(B, -1).astype(np.float64)
    assert np.array_equal(r["folding_count"], (inner < 0).sum(1))
    assert np.allclose(r["folding_fraction"], (inner < 0).mean(1), rtol=1e-14, atol=0)
    assert np.allclose(r["det_mean"], inner.mean(1), rtol=1e-12, atol=1e-14)
    assert np.allclose(r["det_std"], inner.std(1), rtol=1e-9)
    assert np.array_equal(r["det_min"], inner.min(1)) and np.array_equal(r["det_max"], inner.max(1))


def test_nan_in_phi_shows_up_only_in_the_nonfinite_count(dev):
    from liftreg_b200 import metrics, ops
    B, shape = 2, (20, 24, 30)
    phi = noisy_map(B, shape, seed=13)
    phi[1, 1, 10, 12, 15] = np.nan
    ref = jacobian_det(torch.from_numpy(phi), "linear").numpy()
    assert np.isnan(ref[1]).sum() > 0 and np.isfinite(ref[0]).all()
    stats, _ = ops.jacobian_det(torch.from_numpy(phi).to(dev), "linear")
    got = stats.cpu().numpy()
    check_stats(got, stats_of(ref), ref)
    assert got[0, 6] == 0 and got[1, 6] == np.isnan(ref[1]).sum()
    clean = stats_of(np.where(np.isnan(ref), np.float32(1.0), ref))
    assert np.array_equal(got[:, [0, 2, 3]], clean[:, [0, 2, 3]])             # nothing else sees the NaNs
    with pytest.raises(ValueError, match="not finite"):
        metrics.jacobian_stats(torch.from_numpy(phi).to(dev))
    r = metrics.jacobian_stats(torch.from_numpy(phi).to(dev), allow_nonfinite=True)
    assert r["nonfinite_count"].tolist() == [0, int(np.isnan(ref[1]).sum())]


def test_identity_map_has_no_folds(dev):
    from liftreg_b200 import metrics, ops
    phi = ops.identity_map((160, 160, 160), dev)[None]
    r = metrics.jacobian_stats(phi, return_map=True)
    # each diagonal entry differences two fp32 coordinates near +-1 (<= 6e-8 rounding each) over a step of 2*2/159:
    # <= 5e-6 relative per entry, so det = 1 within 1.5e-5 at 160^3
    assert r["folding_count"][0] == 0 and abs(r["det_min"][0] - 1) <= 1.5e-5 and abs(r["det_max"][0] - 1) <= 1.5e-5
    assert r["det"].shape == (1, 160, 160, 160)


def bincount_ref(p, t, L):
    p = p.reshape(p.shape[0], -1).astype(np.float64)
    t = t.reshape(t.shape[0], -1).astype(np.float64)
    ok = (p >= 0) & (p < L) & (p == np.floor(p)) & (t >= 0) & (t < L) & (t == np.floor(t))
    counts = np.stack([np.bincount((p[b][ok[b]] * L + t[b][ok[b]]).astype(np.int64), minlength=L * L).reshape(L, L)
                       for b in range(p.shape[0])])
    return counts, (~ok).sum(1)


@pytest.mark.parametrize("L", [1, 2, 6, 64, 128])
@pytest.mark.parametrize("B,N,offset", [(1, 160 ** 3, 0), (3, 100003, 0), (3, 4096 * 9 + 5, 1), (1, 777, 3)])
def test_label_confusion_equals_bincount(dev, L, B, N, offset):
    from liftreg_b200 import ops
    rs = np.random.RandomState(L * 7 + N % 97)
    p = rs.randint(0, L, size=(B, N)).astype(np.float32)
    t = np.where(rs.uniform(size=(B, N)) < 0.7, p, rs.randint(0, L, size=(B, N))).astype(np.float32)
    buf = torch.zeros(2, B * N + offset, device=dev)
    buf[0, offset:] = torch.from_numpy(p.reshape(-1)).to(dev)
    buf[1, offset:] = torch.from_numpy(t.reshape(-1)).to(dev)
    counts, invalid = ops.label_confusion(buf[0, offset:].view(B, N), buf[1, offset:].view(B, N), L)
    ref_c, ref_i = bincount_ref(p, t, L)
    assert np.array_equal(counts.cpu().numpy(), ref_c) and np.array_equal(invalid.cpu().numpy(), ref_i)


def test_label_confusion_mostly_background_and_planted_invalid_values(dev):
    from liftreg_b200 import ops
    rs = np.random.RandomState(21)
    B, shape = 3, (160, 160, 160)
    for L in (2, 6):
        p = np.zeros((B,) + shape, np.float32)
        t = np.zeros((B,) + shape, np.float32)
        fg = rs.uniform(size=p.shape) < 0.001                            # 99.9 % background
        p[fg] = rs.randint(1, L, size=fg.sum()) if L > 1 else 0
        t[fg] = rs.randint(0, L, size=fg.sum())
        flat_p, flat_t = p.reshape(-1), t.reshape(-1)
        idx = rs.choice(flat_p.size, 40, replace=False)
        for k, bad in enumerate([-1.0, float(L), 0.5, np.nan]):
            flat_p[idx[k * 5:(k + 1) * 5]] = bad
            flat_t[idx[20 + k * 5:20 + (k + 1) * 5]] = bad
        counts, invalid = ops.label_confusion(torch.from_numpy(p).to(dev), torch.from_numpy(t).to(dev), L)
        ref_c, ref_i = bincount_ref(p, t, L)
        assert ref_i.sum() == 40
        assert np.array_equal(counts.cpu().numpy(), ref_c) and np.array_equal(invalid.cpu().numpy(), ref_i)
        # integer label maps are converted with .float()
        c2, i2 = ops.label_confusion(torch.from_numpy(np.nan_to_num(p, nan=-1).astype(np.int64)).to(dev),
                                     torch.from_numpy(np.nan_to_num(t, nan=-1).astype(np.int16)).to(dev), L)
        ref_c2, ref_i2 = bincount_ref(np.nan_to_num(p, nan=-1).astype(np.int64), np.nan_to_num(t, nan=-1).astype(np.int16), L)
        assert np.array_equal(c2.cpu().numpy(), ref_c2) and np.array_equal(i2.cpu().numpy(), ref_i2)


def test_label_overlap_equals_python_sets(dev):
    from liftreg_b200 import metrics
    rs = np.random.RandomState(23)
    shape = (2, 12, 10, 9)
    p = rs.randint(0, 4, size=shape).astype(np.float32)                  # label 4 only in the target
    t = np.where(rs.uniform(size=shape) < 0.6, p, rs.randint(0, 5, size=shape)).astype(np.float32)
    for ignore_bg in (True, False):
        res = metrics.label_overlap(torch.from_numpy(p).to(dev), torch.from_numpy(t).to(dev), ignore_background=ignore_bg)
        assert res["dice"].shape == (2, 5)
        for b in range(2):
            ref = overlap_by_sets(p[b].reshape(-1), t[b].reshape(-1), 5)
            for k, v in ref.items():
                if ignore_bg:
                    v[0] = np.nan
                assert np.array_equal(res[k][b], v, equal_nan=True), k
                assert res[k + "_mean"][b] == pytest.approx(np.nanmean(v), rel=1e-15)
    bad = p.copy()
    bad[0, 0, 0, 0] = 0.5
    with pytest.raises(ValueError, match="not integer labels"):
        metrics.label_overlap(torch.from_numpy(bad).to(dev), torch.from_numpy(t).to(dev))


def test_warped_labels_overlap_end_to_end(dev):
    """RegistrationNet.py:191-196 then the overlap: nearest-mode label warp through the mermaid entry point, scores on
    the GPU equal numpy's on the host copy of the warped labels."""
    from liftreg_b200 import mermaid_utils, metrics, synthetic
    rs = np.random.RandomState(29)
    shape = (64, 48, 40)
    labels = np.zeros((2, 1) + shape, np.float32)
    labels[:, :, 16:48, 10:40, 8:30] = 1
    labels[:, :, 30:40, 20:30, 12:20] = 2
    labels[1, :, 5:12, 5:12, 5:12] = 3
    phi = np.stack([synthetic.identity_map_np(shape) + synthetic.smooth_displacement(shape, seed=100 + b, coarse=4) for b in range(2)])
    warped = mermaid_utils.compute_warped_image_multiNC(torch.from_numpy(labels).to(dev), torch.from_numpy(phi.astype(np.float32)).to(dev),
                                                        (1.0, 1.0, 1.0), spline_order=0, zero_boundary=True, use_01_input=False)
    res = metrics.label_overlap(warped, torch.from_numpy(labels).to(dev), num_labels=4)
    w = warped.cpu().numpy().reshape(2, -1).astype(np.int64)
    t = labels.reshape(2, -1).astype(np.int64)
    for b in range(2):
        for l in range(1, 4):
            tp = np.sum((w[b] == l) & (t[b] == l)); npred = np.sum(w[b] == l); nt = np.sum(t[b] == l)
            if npred + nt == 0:
                assert np.isnan(res["dice"][b, l])
                continue
            assert res["dice"][b, l] == 2.0 * tp / (npred + nt)
            assert res["iou"][b, l] == tp / (npred + nt - tp)
    assert 0.5 < res["dice_mean"][0] < 1.0
