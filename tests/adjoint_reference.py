"""Float64 references of the warp and backprojection adjoints (test infrastructure, imported by
test_adjoint_reference_host / test_adjoints_gpu).

The derivative of trilinear sampling wrt the sample position jumps where a coordinate crosses an integer, so a
reference that computed the coordinates in float64 would disagree with any fp32 kernel by O(1) at those points.  Each
function therefore recomputes the sample coordinates, their floors and their fractions in float32 exactly as the
kernels do, and does everything after that in float64.  Next to each value it returns an abs-scale (the same sum over
absolute terms) and, for scatters, the number of contributions, which is what a rounding-error bound needs:

    gather  (d/dphi):  |kernel - ref| <= k * u * scale
    scatter (grad_img, grad_proj):  |kernel - ref| <= (n + 3) * u * abs     (any order of fp32 atomic adds)

with u = 2^-24.  numpy only; the C oracle supplies the identity map and the backprojection grid, both of which are
bit-exact with the kernels.
"""
import numpy as np

from oracle import c_oracle

U = 2.0 ** -24


def _axis(g, size, clip):
    """Sample coordinate of one axis as the kernels compute it: i = (g + 1) * ((S-1)/2) in fp32, clipped to [0, S-1]
    for border padding.  Returns the fp32 floor as int64, the two fp32 fractions (lower, upper tap) as float64, and
    the chain-rule multiplier (S-1)/2 of d i / d g, which is 0 where the coordinate was clipped."""
    h = np.float32(size - 1) / np.float32(2)
    i = (g + np.float32(1)) * h
    mult = np.full(i.shape, float(h))
    if clip:
        lo, hi = i <= 0, i >= np.float32(size - 1)
        i = np.where(lo, np.float32(0), np.where(hi, np.float32(size - 1), i)).astype(np.float32)
        mult[lo | hi] = 0.0
    f = np.floor(i)
    w1 = (i - f).astype(np.float64)
    w0 = ((f + np.float32(1)) - i).astype(np.float64)
    return f.astype(np.int64), (w0, w1), mult


def warp_adjoint(grad_out, img, phi, zero_boundary, using_scale, disp_plus_identity=False, z_begin=0, want_img=True):
    """Adjoint of ops.warp (linear mode) wrt the image and the map.

    grad_out (B,C,Dz,H,W), img (B,C,D,H,W), phi (B,3,Dz,H,W) holding output planes [z_begin, z_begin+Dz).
    disp_plus_identity: phi is a displacement; the map is phi + identity_map planes [z_begin, z_begin+Dz), an fp32 add.

    Returns (grad_img, img_abs, img_count, grad_phi, phi_scale):
      grad_img (B,C,D,H,W) float64, img_abs = sum of |w * g| over the same terms, img_count (B,C,D,H,W) int64 = number
      of (voxel, tap) contributions (None, None, None unless want_img);
      grad_phi (B,3,Dz,H,W) float64 and phi_scale = h_a * sum_c |g_c| * sum over in-bounds taps (|v| + 1), with h_a =
      (S_a-1)/2 of the component's axis, or 0 where border padding clipped that coordinate.
    """
    go = np.ascontiguousarray(grad_out, np.float32)
    img = np.ascontiguousarray(img, np.float32)
    phi = np.ascontiguousarray(phi, np.float32)
    B, C, D, H, W = img.shape
    Dz = phi.shape[2]
    assert phi.shape == (B, 3, Dz, H, W) and go.shape == (B, C, Dz, H, W) and 0 <= z_begin and z_begin + Dz <= D
    if disp_plus_identity:
        phi = phi + c_oracle.identity_map((D, H, W))[None, :, z_begin:z_begin + Dz]
    clip = not zero_boundary
    # phi channel a addresses volume axis a (grid_sample's x is the last axis)
    (z0, wz, mz), (y0, wy, my), (x0, wx, mx) = (_axis(phi[:, a], S, clip) for a, S in enumerate((D, H, W)))

    nv = D * H * W
    g64 = go.astype(np.float64)
    gsc = g64 * 2.0 if using_scale else g64                     # d(2 s - 1)/ds
    gi = [np.zeros_like(x0, dtype=np.float64) for _ in range(3)]   # x, y, z sums before the multiplier
    vabs = np.zeros_like(x0, dtype=np.float64)
    img_flat = img.reshape(B * C, nv)
    rows = np.arange(B)[:, None] * C
    if want_img:
        gimg = np.zeros(B * C * nv)
        gabs = np.zeros(B * C * nv)
        gcnt = np.zeros(B * C * nv, np.int64)
    for t in range(8):
        tx, ty, tz = t & 1, (t >> 1) & 1, t >> 2
        xx, yy, zz = x0 + tx, y0 + ty, z0 + tz
        ok = (xx >= 0) & (xx < W) & (yy >= 0) & (yy < H) & (zz >= 0) & (zz < D)
        lin = ((np.clip(zz, 0, D - 1) * H + np.clip(yy, 0, H - 1)) * W + np.clip(xx, 0, W - 1)).reshape(B, -1)
        okf = ok.astype(np.float64)
        for c in range(C):
            v = img_flat[rows + c, lin].reshape(ok.shape).astype(np.float64) * okf
            val = (v + 1.0) * 0.5 if using_scale else v
            gc = gsc[:, c] * okf
            gi[0] += (1.0 if tx else -1.0) * val * wy[ty] * wz[tz] * gc
            gi[1] += (1.0 if ty else -1.0) * val * wx[tx] * wz[tz] * gc
            gi[2] += (1.0 if tz else -1.0) * val * wx[tx] * wy[ty] * gc
            vabs += np.abs(g64[:, c]) * (np.abs(v) + 1.0) * okf
            if want_img:
                # d out / d img = w * g in both scalings ((img+1)/2 in, 2 s - 1 out)
                tgt = ((rows + c) * nv + lin)[ok.reshape(B, -1)]
                wg = (wx[tx] * wy[ty] * wz[tz] * g64[:, c])[ok]
                gimg += np.bincount(tgt, weights=wg, minlength=gimg.size)
                gabs += np.bincount(tgt, weights=np.abs(wg), minlength=gimg.size)
                gcnt += np.bincount(tgt, minlength=gimg.size)
    grad_phi = np.stack([mz * gi[2], my * gi[1], mx * gi[0]], axis=1)
    phi_scale = np.stack([mz * vabs, my * vabs, mx * vabs], axis=1)
    if not want_img:
        return None, None, None, grad_phi, phi_scale
    shp = (B, C, D, H, W)
    return gimg.reshape(shp), gabs.reshape(shp), gcnt.reshape(shp), grad_phi, phi_scale


def backproject_adjoint(grad_out, poses, proj_shape):
    """Adjoint of ops.backproject wrt the projections.  grad_out (B,P,d,w,h), poses (P,3) -> (grad_proj, abs, count),
    each (B,P,pw,ph): float64 value, float64 sum of |w * g|, int64 number of (voxel, tap) contributions."""
    g = np.ascontiguousarray(grad_out, np.float32)
    B, P, d, w, h = g.shape
    pw, ph = (int(s) for s in proj_shape)
    poses = np.ascontiguousarray(poses, np.float32).reshape(P, 3)
    val = np.zeros((B, P, pw * ph))
    aval = np.zeros((B, P, pw * ph))
    cnt = np.zeros((B, P, pw * ph), np.int64)
    for p in range(P):
        grid = c_oracle.backproj_grid(poses[p:p + 1], (d, w, h), (pw, ph))[0]     # (2,d,w,h): gv (axis ph), gu (axis pw)
        ix = (grid[0] + np.float32(1)) * (np.float32(ph - 1) / np.float32(2))
        iy = (grid[1] + np.float32(1)) * (np.float32(pw - 1) / np.float32(2))
        fx, fy = np.floor(ix), np.floor(iy)
        wq, n = (ix - fx).astype(np.float64).ravel(), (iy - fy).astype(np.float64).ravel()
        x0, y0 = fx.astype(np.int64).ravel(), fy.astype(np.int64).ravel()
        for ty in (0, 1):
            for tx in (0, 1):
                xx, yy = x0 + tx, y0 + ty
                ok = (xx >= 0) & (xx < ph) & (yy >= 0) & (yy < pw)
                tgt = (yy * ph + xx)[ok]
                wt = ((n if ty else 1.0 - n) * (wq if tx else 1.0 - wq))[ok]
                cnt[:, p] += np.bincount(tgt, minlength=pw * ph)[None]
                for b in range(B):
                    wg = wt * g[b, p].ravel()[ok]
                    val[b, p] += np.bincount(tgt, weights=wg, minlength=pw * ph)
                    aval[b, p] += np.bincount(tgt, weights=np.abs(wg), minlength=pw * ph)
    shp = (B, P, pw, ph)
    return val.reshape(shp), aval.reshape(shp), cnt.reshape(shp)
