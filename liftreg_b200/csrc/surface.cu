// Surface-distance validation metrics (include/liftreg_b200.h, lr_label_surface_counts / lr_surface_distances; PARITY
// UNPINNED: the reference scores no surface metric).
//
// The surface S_M(l) of label l in map M is the set of voxels with M == l that have a face neighbour outside the volume
// or != l (scipy's m & ~binary_erosion(m, 6-connectivity, border_value=0)).  It is never materialised: every kernel
// tests membership on the fly from the voxel and its 6 neighbours.
//
// lr_surface_distances is an exact separable Euclidean distance transform to S_to(label), evaluated at S_from(label):
//   pass 1 (W, contiguous)  one warp per row; warp ballots over 32-column chunks give the nearest S_to column left and
//                           right of each voxel; the nearer one (the left on a tie) is stored as an int32 column.
//   pass 2 (H)              one thread per (b, d, w) column, adjacent threads on adjacent w (coalesced): Meijster et
//                           al.'s (2000) lower envelope of the parabolas (s_H (h - h'))^2 + (s_W dw(h'))^2, stored as the
//                           packed nearest voxel (h' << 16 | w'), 0xFFFFFFFF where the plane holds no S_to voxel.
//   pass 3 (D)              the same per (b, h, w) column over the cost (s_D (d - d'))^2 + (s_H dh)^2 + (s_W dw)^2, and
//                           in the envelope's backward scan, at the voxels of S_from, the epilogue: the distance formed
//                           from the nearest voxel's offsets as scipy forms it, appended to the item's segment through a
//                           warp-aggregated counter, and count / sum / max reduced per block (no fp64 atomics at all:
//                           sm_100a turns those in shared memory into compare-and-swap loops, and global ones would make
//                           the sum's last bits depend on the order in which blocks finish).
// The envelope's stacks (parabola index s[], start t[]) live in the caller's workspace, laid out like the volume, so the
// column threads of a warp touch adjacent words.  Each envelope decision compares costs evaluated at integer positions
// (the intersection estimate is only a starting point, corrected by direct evaluation), so with integer spacings, where
// every cost is an exact integer in fp64, each column's minimum is exact whichever voxel a tie picks.
#include <cfloat>
#include <cmath>

#include "common.cuh"

namespace lr {
namespace {

constexpr int SD_ROW_WARPS = 8;          // pass 1: rows per 256-thread block
constexpr int SD_COL_THREADS = 128;      // passes 2 and 3: columns per block
constexpr int SCOUNT_THREADS = 256;
constexpr unsigned SD_NONE = 0xFFFFFFFFu;

// its label l if v is an integer in [0, L), else -1 (the test of lr_label_confusion: (v + 1.5*2^23) - 1.5*2^23 == v
// holds exactly for the integers |v| < 2^22, and the integer is then in the mantissa)
__device__ __forceinline__ int label_of(float v, float fL) {
    const float M = 12582912.0f;
    const float t = __fadd_rn(v, M);
    return v >= 0.0f && v < fL && __fsub_rn(t, M) == v ? __float_as_int(t) - 0x4B400000 : -1;
}

// m[i] (voxel (d,h,w) of one item's D x H x W block) holds fl and a face neighbour is outside or differs
__device__ __forceinline__ bool on_surface(const float *__restrict__ m, int i, int d, int h, int w, int D, int H, int W, float fl) {
    if (__ldg(m + i) != fl) return false;
    if (d == 0 || d == D - 1 || h == 0 || h == H - 1 || w == 0 || w == W - 1) return true;
    const int HW = H * W;
    return __ldg(m + i - 1) != fl || __ldg(m + i + 1) != fl || __ldg(m + i - W) != fl || __ldg(m + i + W) != fl ||
           __ldg(m + i - HW) != fl || __ldg(m + i + HW) != fl;
}

// one key per lane (key < 0: lane has nothing), called by the whole warp: equal keys are added once per warp
__device__ __forceinline__ void hist_add_warp(unsigned *__restrict__ h, int key) {
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && (threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(h + key, (unsigned)__popc(peers));
}

// counts[b][0][l] = |S_pred(l)|, counts[b][1][l] = |S_target(l)|, invalid[b] = #voxels where either value is not an
// integer in [0, L); a shared (2L+1)-bin histogram per block, merged with one 64-bit atomic per non-empty bin
__global__ void __launch_bounds__(SCOUNT_THREADS) label_surface_count_kernel(const float *__restrict__ pred,
                                                                            const float *__restrict__ target, int D, int H,
                                                                            int W, int L, unsigned long long *__restrict__ counts,
                                                                            unsigned long long *__restrict__ invalid) {
    __shared__ unsigned hist[2 * 128 + 1];
    const int nbins = 2 * L + 1, b = blockIdx.y, HW = H * W, N = D * HW;
    for (int i = threadIdx.x; i < nbins; i += SCOUNT_THREADS) hist[i] = 0u;
    __syncthreads();
    const float fL = (float)L;
    const float *pb = pred + (int64_t)b * N, *tb = target + (int64_t)b * N;
    const int stride = gridDim.x * SCOUNT_THREADS;
    // warp-uniform trip count: every lane runs every iteration (the histogram add is a warp collective)
    for (int base = blockIdx.x * SCOUNT_THREADS + (threadIdx.x & ~31); base < N; base += stride) {
        const int i = base + (threadIdx.x & 31);
        int kp = -1, kt = -1, ki = -1;
        if (i < N) {
            const int d = i / HW, r = i - d * HW, h = r / W, w = r - h * W;
            const float p = __ldg(pb + i), t = __ldg(tb + i);
            const int lp = label_of(p, fL), lt = label_of(t, fL);
            if (lp >= 0 && on_surface(pb, i, d, h, w, D, H, W, p)) kp = lp;
            if (lt >= 0 && on_surface(tb, i, d, h, w, D, H, W, t)) kt = L + lt;
            if (lp < 0 || lt < 0) ki = 2 * L;
        }
        if (__any_sync(0xffffffffu, kp >= 0)) hist_add_warp(hist, kp);
        if (__any_sync(0xffffffffu, kt >= 0)) hist_add_warp(hist, kt);
        if (__any_sync(0xffffffffu, ki >= 0)) hist_add_warp(hist, ki);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nbins; i += SCOUNT_THREADS) {
        const unsigned c = hist[i];
        if (c) atomicAdd(i < 2 * L ? counts + (int64_t)b * 2 * L + i : invalid + b, (unsigned long long)c);
    }
}

// pass 1: near[row + w] = the column of the S_to voxel nearest to w in its row (the left one on a tie), -1 if none
__global__ void __launch_bounds__(SD_ROW_WARPS * 32) sdist_row_kernel(const float *__restrict__ to, int rows, int D, int H,
                                                                     int W, float fl, int *__restrict__ near) {
    const int row = blockIdx.x * SD_ROW_WARPS + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= rows) return;                                  // whole warps leave together
    const int DH = D * H, b = row / DH, r = row - b * DH, d = r / H, h = r - d * H;
    const float *m = to + (int64_t)b * DH * W;
    const int i0 = (d * H + h) * W;
    int *out = near + (int64_t)row * W;
    int carry = -1;                                           // nearest surface column left of the chunk
    for (int c0 = 0; c0 < W; c0 += 32) {
        const int w = c0 + lane;
        const unsigned bits = __ballot_sync(0xffffffffu, w < W && on_surface(m, i0 + w, d, h, w, D, H, W, fl));
        const unsigned left = bits & (0xffffffffu >> (31 - lane));
        if (w < W) out[w] = left ? c0 + 31 - __clz(left) : carry;
        if (bits) carry = c0 + 31 - __clz(bits);
    }
    carry = -1;                                               // nearest surface column right of the chunk
    for (int c0 = (W - 1) & ~31; c0 >= 0; c0 -= 32) {
        const int w = c0 + lane;
        const unsigned bits = __ballot_sync(0xffffffffu, w < W && on_surface(m, i0 + w, d, h, w, D, H, W, fl));
        const unsigned right = bits & (0xffffffffu << lane);
        if (w < W) {
            const int lc = out[w], rc = right ? c0 + __ffs(right) - 1 : carry;
            out[w] = lc < 0 ? rc : rc < 0 ? lc : (w - lc <= rc - w ? lc : rc);
        }
        if (bits) carry = c0 + __ffs(bits) - 1;
    }
}

__device__ __forceinline__ double sq(double x) { return __dmul_rn(x, x); }

// cost of parabola i (input cost gi) at position x along an axis of spacing s
__device__ __forceinline__ double env_cost(int x, int i, double gi, double s) {
    return __dadd_rn(sq(__dmul_rn(s, (double)(x - i))), gi);
}

// entry k of one column of the volume, at p[k * st]
template <typename T>
struct Strided {
    T *p;
    int st;
    __device__ __forceinline__ T &operator[](int k) const { return p[k * st]; }
};

// Meijster's forward scan over one column of n entries (input cost g(i), +inf where the column entry has no feature),
// building the lower envelope in the stacks S/T.  Returns the stack height - 1; the top entry is (s_q, t_q, g_q).  A
// parabola u enters at the first position w > t_q where it is strictly cheaper than the top; the estimate from the
// intersection is corrected by evaluating both costs, so every decision is a comparison of costs.
template <class G, class Stk>
__device__ __forceinline__ int envelope(const G &g, int n, double s, Stk S, Stk T, int &s_q, int &t_q, double &g_q) {
    int q = 0;
    s_q = 0, t_q = 0, g_q = g(0);
    S[0] = 0, T[0] = 0;
    const double ss = __dmul_rn(s, s);
    for (int u = 1; u < n; ++u) {
        const double gu = g(u);
        if (!(gu < INFINITY)) continue;                      // never strictly cheaper than anything: never enters
        while (q >= 0 && env_cost(t_q, s_q, g_q, s) > env_cost(t_q, u, gu, s)) {
            if (--q >= 0) s_q = S[q], t_q = T[q], g_q = g(s_q);
        }
        if (q < 0) {
            q = 0, s_q = u, t_q = 0, g_q = gu;
            S[0] = u;                                         // T[0] stays 0
            continue;
        }
        const int lo = t_q + 1;
        double wd = floor(__dmul_rn(__dadd_rn(__ddiv_rn(__dsub_rn(gu, g_q), __dmul_rn(ss, (double)(u - s_q))), (double)(u + s_q)), 0.5)) + 1.0;
        if (!(wd >= (double)lo)) wd = (double)lo;            // also NaN
        if (wd > (double)n) wd = (double)n;
        int w = (int)wd;
        while (w > lo && env_cost(w - 1, u, gu, s) < env_cost(w - 1, s_q, g_q, s)) --w;
        while (w < n && !(env_cost(w, u, gu, s) < env_cost(w, s_q, g_q, s))) ++w;
        if (w < n) {
            ++q, s_q = u, t_q = w, g_q = gu;
            S[q] = u, T[q] = w;
        }
    }
    return q;
}

// pass 2 on one (b, d, w) column: out[x] = (h' << 16 | w') of the S_to voxel nearest to (x, w) within the plane
template <class In, class Stk>
__device__ __forceinline__ void col_h(In in, Stk S, Stk T, int H, int w, double s_h, double s_w, unsigned *out, int ost) {
    auto g = [&](int i) -> double {
        const int c = (int)in[i];
        return c < 0 ? INFINITY : sq(__dmul_rn(s_w, (double)(w - c)));
    };
    int s_q, t_q;
    double g_q;
    int q = envelope(g, H, s_h, S, T, s_q, t_q, g_q);
    unsigned key = g_q < INFINITY ? ((unsigned)s_q << 16) | (unsigned)in[s_q] : SD_NONE;
    for (int x = H - 1; x >= 0; --x) {
        out[x * ost] = key;
        if (x == t_q && --q >= 0) {
            s_q = S[q], t_q = T[q];
            key = ((unsigned)s_q << 16) | (unsigned)in[s_q];  // below the top, every entry is finite
        }
    }
}

// pass 2: packed[b,d,h,w] = (h' << 16 | w') of the S_to voxel nearest to (h, w) within plane (b, d), SD_NONE if none
__global__ void __launch_bounds__(SD_COL_THREADS) sdist_col_h_kernel(const int *__restrict__ near, int cols, int H, int W,
                                                                    double s_h, double s_w, int *__restrict__ S,
                                                                    int *__restrict__ T, unsigned *__restrict__ packed) {
    const int col = blockIdx.x * SD_COL_THREADS + threadIdx.x;
    if (col >= cols) return;
    const int bd = col / W, w = col - bd * W, base = bd * H * W + w;
    col_h(Strided<const int>{near + base, W}, Strided<int>{S + base, W}, Strided<int>{T + base, W}, H, w, s_h, s_w,
          packed + base, W);
}

// pass 3 on one (b, h, w) column and the epilogue at the voxels of S_from; called by whole warps (inactive lanes, with
// no column, take part in the ballots)
template <class In, class Stk>
__device__ __forceinline__ void col_d(In in, Stk S, Stk T, bool active, const float *__restrict__ m, int hw, int h, int w,
                                      int D, int H, int W, float fl, double s_d, double s_h, double s_w,
                                      unsigned long long *__restrict__ fill, int b, int64_t seg0, int64_t seg1,
                                      double *__restrict__ dist, unsigned &cnt, double &sum, double &mx) {
    const int lane = threadIdx.x & 31, HW = H * W;
    auto offs = [&](unsigned k, double &dh, double &dw) {
        dh = __dmul_rn(s_h, (double)(h - (int)(k >> 16)));
        dw = __dmul_rn(s_w, (double)(w - (int)(k & 0xFFFFu)));
    };
    auto g = [&](int i) -> double {
        const unsigned k = in[i];
        if (k == SD_NONE) return INFINITY;
        double dh, dw;
        offs(k, dh, dw);
        return __dadd_rn(sq(dh), sq(dw));
    };
    int s_q = 0, t_q = 0, q = 0;
    double g_q = INFINITY;
    if (active) q = envelope(g, D, s_d, S, T, s_q, t_q, g_q);
    unsigned key = active ? (unsigned)in[s_q] : SD_NONE;
    for (int x = D - 1; x >= 0; --x) {
        const bool hit = active && on_surface(m, x * HW + hw, x, h, w, D, H, W, fl);
        const unsigned bits = __ballot_sync(0xffffffffu, hit);
        if (bits) {
            unsigned long long at = 0;
            if (lane == __ffs(bits) - 1) at = atomicAdd(fill + b, (unsigned long long)__popc(bits));
            at = __shfl_sync(0xffffffffu, at, __ffs(bits) - 1);
            if (hit) {
                double v = INFINITY;                           // S_to(label) of this item is empty
                if (key != SD_NONE) {
                    double dh, dw;
                    offs(key, dh, dw);
                    v = __dsqrt_rn(__dadd_rn(__dadd_rn(sq(__dmul_rn(s_d, (double)(x - s_q))), sq(dh)), sq(dw)));
                }
                const int64_t pos = seg0 + (int64_t)at + __popc(bits & ((1u << lane) - 1u));
                if (pos < seg1) dist[pos] = v;
                ++cnt, sum += v, mx = fmax(mx, v);
            }
        }
        if (active && x == t_q && --q >= 0) {
            s_q = S[q], t_q = T[q];
            key = in[s_q];
        }
    }
}

// pass 3 and the epilogue; one item per blockIdx.y
__global__ void __launch_bounds__(SD_COL_THREADS) sdist_col_d_kernel(const unsigned *__restrict__ packed,
                                                                    const float *__restrict__ from, int D, int H, int W,
                                                                    float fl, double s_d, double s_h, double s_w,
                                                                    int *__restrict__ S, int *__restrict__ T,
                                                                    unsigned long long *__restrict__ fill,
                                                                    unsigned *__restrict__ done, double *__restrict__ part,
                                                                    const int64_t *__restrict__ seg_offset,
                                                                    double *__restrict__ dist, double *__restrict__ stats) {
    __shared__ double red_sum[SD_COL_THREADS / 32], red_max[SD_COL_THREADS / 32];
    __shared__ unsigned red_cnt[SD_COL_THREADS / 32];
    __shared__ bool last;
    const int HW = H * W, b = blockIdx.y, lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int hw = blockIdx.x * SD_COL_THREADS + threadIdx.x;
    const bool active = hw < HW;                             // inactive lanes still run the (uniform) scan for the ballots
    const int h = active ? hw / W : 0, w = active ? hw - h * W : 0;
    const int64_t ib = (int64_t)b * D * HW;
    const int base = (int)ib + (active ? hw : 0);
    const int64_t seg0 = seg_offset[b], seg1 = seg_offset[b + 1];
    unsigned cnt = 0;
    double sum = 0.0, mx = 0.0;
    col_d(Strided<const unsigned>{packed + base, HW}, Strided<int>{S + base, HW}, Strided<int>{T + base, HW}, active, from + ib,
          hw, h, w, D, H, W, fl, s_d, s_h, s_w, fill, b, seg0, seg1, dist, cnt, sum, mx);
    for (int o = 16; o > 0; o >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        sum += __shfl_xor_sync(0xffffffffu, sum, o);
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) red_cnt[wid] = cnt, red_sum[wid] = sum, red_max[wid] = mx;
    __syncthreads();
    // the block's partials go to part[b][blockIdx.x]; the item's last block to finish adds them in block order, so the
    // statistics do not depend on the order in which blocks finish
    const int nbx = gridDim.x;
    double *pb = part + 3 * ((int64_t)b * nbx + blockIdx.x);
    if (threadIdx.x == 0) {
        for (int k = 1; k < SD_COL_THREADS / 32; ++k) cnt += red_cnt[k], sum += red_sum[k], mx = fmax(mx, red_max[k]);
        pb[0] = (double)cnt, pb[1] = sum, pb[2] = mx;
        __threadfence();
        last = atomicAdd(done + b, 1u) == (unsigned)nbx - 1;
    }
    __syncthreads();
    if (last && threadIdx.x == 0) {
        __threadfence();
        const double *p = part + 3 * (int64_t)b * nbx;
        double c = 0.0, s = 0.0, m2 = 0.0;
        for (int k = 0; k < nbx; ++k) c += __ldcg(p + 3 * k), s += __ldcg(p + 3 * k + 1), m2 = fmax(m2, __ldcg(p + 3 * k + 2));
        stats[3 * b] = c, stats[3 * b + 1] = s, stats[3 * b + 2] = m2;
    }
}

// the argument rules the surface entries share; 0 when they hold
int surface_check(const char *who, int B, int D, int H, int W) {
    LR_REQUIRE(B >= 1 && B <= 65535, "%s: batch B=%d must be in [1, 65535]", who, B);
    LR_REQUIRE(D >= 1 && H >= 1 && W >= 1, "%s: every axis needs >= 1 entry (%dx%dx%d)", who, D, H, W);
    LR_REQUIRE((int64_t)B * D * H * W < ((int64_t)1 << 31), "%s: volume too large (B=%d, %dx%dx%d; B*D*H*W must stay below 2^31)",
               who, B, D, H, W);
    return 0;
}

// pass-3 blocks per item
unsigned sd_blocks(int H, int W) { return (unsigned)((H * W + SD_COL_THREADS - 1) / SD_COL_THREADS); }

constexpr size_t SD_ALIGN = 256;
size_t align_up(size_t n) { return (n + SD_ALIGN - 1) / SD_ALIGN * SD_ALIGN; }

}  // namespace
}  // namespace lr

using namespace lr;

extern "C" int lr_label_surface_counts(const float *pred, const float *target, int B, int D, int H, int W, int L,
                                       int64_t *counts, int64_t *invalid, lr_stream_t stream) {
    LR_REQUIRE(pred && target && counts && invalid, "label_surface_counts: null pointer");
    LR_REQUIRE(L >= 1 && L <= 128, "label_surface_counts: number of labels L=%d must be in [1, 128]", L);
    if (int e = surface_check("label_surface_counts", B, D, H, W)) return e;
    cudaStream_t st = as_stream(stream);
    if (int e = cuda_ok(cudaMemsetAsync(counts, 0, sizeof(int64_t) * (size_t)B * 2 * L, st), "label_surface_counts: memset failed")) return e;
    if (int e = cuda_ok(cudaMemsetAsync(invalid, 0, sizeof(int64_t) * (size_t)B, st), "label_surface_counts: memset failed")) return e;
    const int N = D * H * W;
    int64_t per_item = (N + SCOUNT_THREADS * 16 - 1) / (SCOUNT_THREADS * 16);      // >= 16 voxels per thread
    const int64_t cap = ((int64_t)sm_count() * 8 + B - 1) / B;
    if (per_item > cap) per_item = cap;
    const dim3 grid((unsigned)(per_item < 1 ? 1 : per_item), (unsigned)B);
    label_surface_count_kernel<<<grid, SCOUNT_THREADS, 0, st>>>(pred, target, D, H, W, L,
                                                                reinterpret_cast<unsigned long long *>(counts),
                                                                reinterpret_cast<unsigned long long *>(invalid));
    return check_launch("label_surface_count_kernel");
}

extern "C" size_t lr_surface_distance_workspace_bytes(int B, int D, int H, int W) {
    if (B < 1 || B > 65535 || D < 1 || H < 1 || W < 1 || H > 65535 || W > 65535 || (int64_t)B * D * H * W >= ((int64_t)1 << 31))
        return 0;
    const size_t n = (size_t)B * D * H * W;
    return align_up((sizeof(unsigned long long) + sizeof(unsigned)) * (size_t)B) + align_up(3 * sizeof(double) * (size_t)B * sd_blocks(H, W)) +
           4 * align_up(sizeof(int) * n);
}

extern "C" int lr_surface_distances(const float *from, const float *to, int B, int D, int H, int W, int label, double s_d,
                                    double s_h, double s_w, const int64_t *seg_offset, double *dist, double *stats,
                                    void *workspace, size_t workspace_bytes, lr_stream_t stream) {
    LR_REQUIRE(from && to && seg_offset && dist && stats && workspace, "surface_distances: null pointer");
    if (int e = surface_check("surface_distances", B, D, H, W)) return e;
    LR_REQUIRE(H <= 65535 && W <= 65535, "surface_distances: H=%d and W=%d must be <= 65535 (packed nearest-voxel coordinates)", H, W);
    LR_REQUIRE(label >= 1 && label <= 127, "surface_distances: label %d must be in [1, 128)", label);
    LR_REQUIRE(s_d > 0.0 && s_d <= DBL_MAX && s_h > 0.0 && s_h <= DBL_MAX && s_w > 0.0 && s_w <= DBL_MAX,
               "surface_distances: spacing (%g, %g, %g) must be finite and > 0", s_d, s_h, s_w);
    const size_t need = lr_surface_distance_workspace_bytes(B, D, H, W);
    LR_REQUIRE(workspace_bytes >= need, "surface_distances: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    cudaStream_t st = as_stream(stream);
    const size_t n = (size_t)B * D * H * W, vol = align_up(sizeof(int) * n);
    char *ws = static_cast<char *>(workspace);
    const unsigned nbx = sd_blocks(H, W);
    auto *fill = reinterpret_cast<unsigned long long *>(ws);
    auto *done = reinterpret_cast<unsigned *>(fill + B);
    ws += align_up((sizeof(unsigned long long) + sizeof(unsigned)) * (size_t)B);
    auto *part = reinterpret_cast<double *>(ws);
    ws += align_up(3 * sizeof(double) * (size_t)B * nbx);
    int *near = reinterpret_cast<int *>(ws), *S = reinterpret_cast<int *>(ws + vol), *T = reinterpret_cast<int *>(ws + 2 * vol);
    auto *packed = reinterpret_cast<unsigned *>(ws + 3 * vol);
    if (int e = cuda_ok(cudaMemsetAsync(fill, 0, (sizeof(unsigned long long) + sizeof(unsigned)) * (size_t)B, st), "surface_distances: memset failed"))
        return e;
    const float fl = (float)label;
    const int rows = B * D * H;
    sdist_row_kernel<<<(rows + SD_ROW_WARPS - 1) / SD_ROW_WARPS, SD_ROW_WARPS * 32, 0, st>>>(to, rows, D, H, W, fl, near);
    if (int e = check_launch("sdist_row_kernel")) return e;
    const int cols_h = B * D * W;
    sdist_col_h_kernel<<<(cols_h + SD_COL_THREADS - 1) / SD_COL_THREADS, SD_COL_THREADS, 0, st>>>(near, cols_h, H, W, s_h, s_w,
                                                                                                    S, T, packed);
    if (int e = check_launch("sdist_col_h_kernel")) return e;
    sdist_col_d_kernel<<<dim3(nbx, (unsigned)B), SD_COL_THREADS, 0, st>>>(packed, from, D, H, W, fl, s_d, s_h, s_w, S, T, fill, done,
                                                                          part, seg_offset, dist, stats);
    return check_launch("sdist_col_d_kernel");
}
