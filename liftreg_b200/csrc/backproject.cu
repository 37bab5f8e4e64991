// Backprojection: lift P detector images into a P-channel volume (per-voxel gather over views), sm_100a.
//
// Replaces reference src/liftreg/utils/sdct_projection_utils.py:227-250 (backproj_grids_with_poses, a
// 131 MB (1,P,2,d,w,h) grid) and the grid_sample block of
// src/liftreg/models/LiftRegDeformSubspaceBackproj.py:85-93.  The voxel->detector map is evaluated in
// registers with the reference's fp32 op order:
//     x_i = i - d/2,  y_j = w-1-j (reversed, sdct:232),  z_k = k - h/2
//     scale = sy / (sy - y_j)                                   (sdct:239)
//     gu = ((x_i - sx)*scale + sx) / pw * 2                     (sdct:241-242,247)   -> detector axis 0
//     gv = ((z_k - sz)*scale + sz) / ph * 2                     (sdct:248)           -> detector axis 1
// and sampled like ATen's vectorised CPU grid_sampler_2d (align_corners, zeros):
//     ix = (g+1)*((S-1)/2); w = ix-floor(ix); e = 1-w; ... out = fma(se_v,n*w, fma(sw_v,n*e, fma(ne_v,s*w, nw_v*(s*e))))
//
// Work decomposition: the v-part of the map depends on (p,j,k), the u-part on (p,i,j).  A thread owns one k
// (lanes along h: coalesced 128 B stores, near-contiguous gathers), keeps its v-part in registers and walks a
// chunk of i; the per-i u-part comes from a small shared-memory table built once per block and row j.  Batch items
// are a grid dimension.
#include "common.cuh"

namespace lr {

constexpr int BP_MAX_VIEWS = 64;   // views per launch (poses travel as kernel parameters)
#ifndef LR_BP_ICHUNK
#define LR_BP_ICHUNK 32
#endif
constexpr int BP_ICHUNK = LR_BP_ICHUNK;      // max i-planes per block (the actual chunk is balanced: ceil(d / n_chunks))

struct BpPoses {
    float s[BP_MAX_VIEWS][3];
};

struct BpDims {
    int B, P, pw, ph, d, w, h;     // d = planes of axis 0 held by the output (the whole volume, or a z-slab of it)
    int i_off;                     // absolute index of the output's first plane (0 unless slab-sharded)
    int ichunk;                    // planes per block: ceil(d / ceil(d / BP_ICHUNK)) <= BP_ICHUNK
    int isub;                      // forward: planes per sub-chunk (one blockDim.y slice); the row window restarts there
    int hp;                        // forward: ceil(h / 2), the distance between the two voxels a thread owns
    int bx, by;                    // forward: group shape (column pairs x sub-chunks)
    // forward: blocks walk runs of consecutive coronal rows j, in three sizes, longest first (blocks are dispatched in
    // index order, so the last ones to start are the short ones and the tail of the launch drains quickly):
    // nj0 runs of js0 rows, then nj1 of js1, then nj2 of js2, each for every (view, chunk)
    int js0, js1, js2, nj0, nj1, nj2;
    int n_chunks, n_vc, n_views;   // forward: chunks of planes; batch items * views * chunks; views of this launch
    int p0;                        // first view of this launch
    float half_d, half_h;          // d/2, h/2 (exact)
    ConstDiv div_pw, div_ph;       // division by (float)pw, (float)ph via Markstein (bit-identical to IEEE division)
    float hpw, hph;                // (pw-1)/2, (ph-1)/2
    int64_t proj_view_stride;      // pw*ph
    int64_t out_batch_stride, out_chan_stride;
    float zero;                    // +0.0f the compiler cannot constant-fold (see mul2_sep)
    // forward: ceil(2^32 / divisor) for the block-index decode (exact while grid * divisor < 2^32; 0 = plain division)
    unsigned m_nj0, m_nj1, m_nj2, m_chunks, m_views;
};

// x / d for 0 <= x with a precomputed magic = ceil(2^32 / d) (0: divide; d == 1 has no 32-bit magic either)
__device__ __forceinline__ int div_magic(int x, int d, unsigned magic) {
    return magic ? (int)__umulhi((unsigned)x, magic) : x / d;
}

struct AxisTap {      // one axis of the bilinear footprint
    int i0;           // floor index (may be out of range)
    float w1;         // ix - floor(ix)
};

// normalised coordinate -> (floor index, upper weight), ATen vector-kernel order
__device__ __forceinline__ AxisTap axis_tap(float centred, float s_c, float scale, ConstDiv size, float half_sm1) {
    float a = add_rn(mul_rn(sub_rn(centred, s_c), scale), s_c);   // (x - s)*scale + s
    float g = mul_rn(div_const(a, size), 2.0f);                   // / size * 2
    float ix = mul_rn(add_rn(g, 1.0f), half_sm1);                 // (g+1)*((S-1)/2)
    ix = clamp_index(ix, half_sm1 * 2.0f + 3.0f);                 // beyond [-2, S+1] no tap is in bounds
    float fl;
    AxisTap t;
    floor_fi(ix, fl, t.i0);
    t.w1 = sub_rn(ix, fl);
    return t;
}

__device__ __forceinline__ float view_scale(float sy, int w, int j) {
    float y = (float)(w - 1 - j);
    return div_rn(sy, sub_rn(sy, y));
}

// Per-plane (u-axis) entry of the block's shared table: one LDS.128 per i instead of ~25 instructions.
struct __align__(16) BpRow {
    float n, s;   // iy - floor(iy), 1 - n   (first: an aligned register pair for the packed weight products)
    int off0;     // r0 * ph: element offset of detector row r0 inside the view
    int mask;     // bit 0: row r0 inside the detector, bit 1: row r0+1 inside.  Sliding row window (relative to the
                  // previous plane of the chunk): bit 2 = moved exactly one row (reuse the upper row as the lower),
                  // bit 3 = moved further or first plane (fetch both rows), bit 4 = upper row must be fetched
};

// Compact entry for the fast path (all rows valid, so off0 >= 0): one LDS.64 instead of an LDS.128 -- a warp-wide
// broadcast LDS.128 costs ~4 L1 wavefronts, which made the table read as expensive as the gathers (ncu:
// l1tex__data_pipe_lsu_wavefronts_mem_shared = 38 % of all wavefronts).
struct __align__(8) BpRow8 {
    float n;        // iy - floor(iy); s = 1 - n is recomputed
    int packed;     // (off0 << 5) | window flags (bits 2..4 of BpRow::mask)
};

// Builds the tables; returns whether every plane this thread handled has both rows inside the detector.
__device__ __forceinline__ bool build_row_table(BpRow *rows, BpRow8 *rows8, const BpDims &g, int i_begin, int i_count,
                                                float sx, float scale, int isub, int tid, int n_thr) {
    int ok = 1;
    for (int t_idx = tid; t_idx < i_count; t_idx += n_thr) {
        AxisTap t = axis_tap((float)(g.i_off + i_begin + t_idx) - g.half_d, sx, scale, g.div_pw, g.hpw);
        BpRow r;
        r.off0 = t.i0 * g.ph;
        r.n = t.w1;
        r.s = sub_rn(1.0f, t.w1);
        r.mask = ((unsigned)t.i0 < (unsigned)g.pw ? 1 : 0) | ((unsigned)(t.i0 + 1) < (unsigned)g.pw ? 2 : 0);
        ok &= r.mask == 3;
        // consecutive planes advance the detector row by ~1..1.4 (the magnification): tell the consumer how far
        int step = 2;
        if (t_idx % isub != 0) {
            const AxisTap tp = axis_tap((float)(g.i_off + i_begin + t_idx - 1) - g.half_d, sx, scale, g.div_pw, g.hpw);
            const int dlt = t.i0 - tp.i0;
            step = (dlt == 0 || dlt == 1) ? dlt : 2;
        }
        r.mask |= step == 1 ? (4 | 16) : (step == 0 ? 0 : (8 | 16));
        rows[t_idx] = r;
        if (rows8) {
            BpRow8 c;
            c.n = r.n;
            c.packed = (int)(((unsigned)r.off0 << 5) | (unsigned)(r.mask & 28));
            rows8[t_idx] = c;
        }
    }
    return ok != 0;       // this thread's entries only: the caller reduces over the group
}

// ATen vector kernel: out = fma(se_v, n*w, fma(sw_v, n*e, fma(ne_v, s*w, nw_v * (s*e))))
__device__ __forceinline__ float bilerp(float va, float vb, float vc, float vd, float s, float n, float e, float wq) {
    const float nw = mul_rn(s, e), ne = mul_rn(s, wq), sw = mul_rn(n, e), se = mul_rn(n, wq);
    return fma_rn(vd, se, fma_rn(vc, sw, fma_rn(vb, ne, mul_rn(va, nw))));
}

// The same four taps in the separable order of the fast-numerics kernel (see backproject_forward_rows_kernel):
// the two detector rows are interpolated along the detector's second axis first, then blended along the first.
__device__ __forceinline__ float bilerp_sep(float va, float vb, float vc, float vd, float s, float n, float e, float wq) {
    const float t_lo = fma_rn(vb, wq, mul_rn(va, e)), t_up = fma_rn(vd, wq, mul_rn(vc, e));
    return fma_rn(t_up, n, mul_rn(t_lo, s));
}

// Zeros-padding path of one voxel column (k): per-tap predicates, scalar arithmetic.
template <bool SEP>
__device__ __forceinline__ void backproject_column_checked(const float *pvf, char *o, int64_t plane_bytes, const BpRow *rows,
                                                           int ii0, int ii1, int ph, bool c0, bool c1, float e, float wq) {
    for (int ii = ii0; ii < ii1; ++ii) {
        const BpRow r = rows[ii];
        const float *q0 = pvf + r.off0;
        const float *q1 = q0 + ph;
        const bool rv0 = (r.mask & 1) != 0, rv1 = (r.mask & 2) != 0;
        const float va = (rv0 && c0) ? __ldg(q0) : 0.0f, vb = (rv0 && c1) ? __ldg(q0 + 1) : 0.0f;
        const float vc = (rv1 && c0) ? __ldg(q1) : 0.0f, vd = (rv1 && c1) ? __ldg(q1 + 1) : 0.0f;
        const float res = SEP ? bilerp_sep(va, vb, vc, vd, r.s, r.n, e, wq) : bilerp(va, vb, vc, vd, r.s, r.n, e, wq);
        st_stream((float *)o, res);
        o += plane_bytes;
    }
}

// Block = (view p, chunk of planes i, group of g.jb consecutive coronal rows j); threads = (g.bx column pairs) x
// (g.by sub-chunks of g.isub planes).  A thread owns TWO voxel columns k0 = q and k1 = q + ceil(h/2) (both
// warp-contiguous, so loads and stores coalesce exactly as with one column) and evaluates them as one packed fp32x2
// stream; the per-plane table entry, flags and weights are shared by the pair.  The rows j of the group are walked
// inside the block: everything that does not depend on j (pointers, centred coordinates, plane range) is set up once
// -- with one row per block that set-up was 36 % of all executed instructions (ncu source counters).
__global__ void __launch_bounds__(256)
    backproject_forward_kernel(const float *__restrict__ proj, float *__restrict__ out, BpDims g, BpPoses poses) {
    __shared__ BpRow rows_all[2][BP_ICHUNK];
    __shared__ BpRow8 rows8_all[2][BP_ICHUNK];
    __shared__ float scale_all[2];

    const int tid = threadIdx.y * blockDim.x + threadIdx.x, n_thr = blockDim.x * blockDim.y;
    // block index -> (run of rows, chunk, view, batch item): level-major (all long runs of the whole launch first, the
    // single rows last), then (item, view, chunk), the run fastest (neighbouring blocks gather from neighbouring
    // detector patches)
    int L = blockIdx.x, nj = g.nj0, js = g.js0, j_base = 0;
    if (L >= g.nj0 * g.n_vc) {
        L -= g.nj0 * g.n_vc; nj = g.nj1; js = g.js1; j_base = g.nj0 * g.js0;
        if (L >= g.nj1 * g.n_vc) { L -= g.nj1 * g.n_vc; nj = g.nj2; js = g.js2; j_base += g.nj1 * g.js1; }
    }
    const int vc = L / nj;
    const int bv = vc / g.n_chunks;
    const int bi = bv / g.n_views;       // batch item
    const int pl = bv - bi * g.n_views;  // view inside this launch
    const int p = g.p0 + pl;
    const int i_begin = (vc - bv * g.n_chunks) * g.ichunk;
    const int i_count = min(g.ichunk, g.d - i_begin);
    const int j_begin = j_base + (L - vc * nj) * js, j_end = min(g.w, j_begin + js);
    const float sx = poses.s[pl][0], sy = poses.s[pl][1], sz = poses.s[pl][2];
    const int ii0 = threadIdx.y * g.isub, ii1 = min(i_count, ii0 + g.isub);    // this thread's planes of the chunk
    const int64_t proj_batch = (int64_t)g.P * g.proj_view_stride;
    const int64_t plane_bytes = (int64_t)g.w * g.h * 4;
    const unsigned plane = (unsigned)(g.w * g.h);
    // batch items are blocks: a batch loop inside the thread (geometry shared by the items) made the blocks B times
    // longer without adding any; at batch 8 that cost 27 us per item against 24 us for eight separate launches
    const float *pv0 = proj + bi * proj_batch + (int64_t)p * g.proj_view_stride;
    float *ob0 = out + bi * g.out_batch_stride + (int64_t)p * g.out_chan_stride + (int64_t)i_begin * g.w * g.h;

    for (int j = j_begin; j < j_end; ++j) {
        const int buf = (j - j_begin) & 1;
        BpRow *rows = rows_all[buf];
        BpRow8 *rows8 = rows8_all[buf];
        // The only true division (scale = sy / (sy - y_j), block-uniform) is done by the table-building threads and
        // broadcast through shared memory; /pw and /ph are Markstein multiplications.
        float scale = 0.0f;
        if (tid < i_count || tid == 0) {
            scale = view_scale(sy, g.w, j);
            if (tid == 0) scale_all[buf] = scale;
        }
        // double-buffered table: one barrier per row (no thread can be more than one row ahead of the slowest one)
        const bool rows_ok = __syncthreads_and(build_row_table(rows, rows8, g, i_begin, i_count, sx, scale, g.isub, tid, n_thr));
        scale = scale_all[buf];

        for (int q = threadIdx.x; q < g.hp; q += blockDim.x) {
            const int k0 = q, k1 = q + g.hp;
            const bool has1 = k1 < g.h;
            const AxisTap t0 = axis_tap((float)k0 - g.half_h, sz, scale, g.div_ph, g.hph);
            const AxisTap t1 = axis_tap((float)(has1 ? k1 : k0) - g.half_h, sz, scale, g.div_ph, g.hph);
            const float wq0 = t0.w1, e0 = sub_rn(1.0f, wq0), wq1 = t1.w1, e1 = sub_rn(1.0f, wq1);
            const bool c00 = (unsigned)t0.i0 < (unsigned)g.ph, c01 = (unsigned)(t0.i0 + 1) < (unsigned)g.ph;
            const bool c10 = (unsigned)t1.i0 < (unsigned)g.ph, c11 = (unsigned)(t1.i0 + 1) < (unsigned)g.ph;
            {
                const float *pv = pv0;
                float *ob = ob0 + (unsigned)(j * g.h);
                if (rows_ok && has1 && c00 && c01 && c10 && c11) {
                    // every tap of every plane of this chunk is inside the detector (the common case).
                    // Sliding window over detector rows: the pair's two columns of rows r0, r0+1 stay in registers;
                    // when the next plane moves one row down only the new row is fetched (2.4 loads / sample on
                    // average instead of 4).  The step (0, 1 or 2+ rows) is block-uniform; it is applied with
                    // predicated moves / loads rather than branches, which keeps the loop body straight-line.
                    const float *lo0 = opaque(pv + t0.i0), *lo1 = opaque(pv + t1.i0);         // row r0 of each column
                    const float *up0 = opaque(lo0 + g.ph), *up1 = opaque(lo1 + g.ph);         // row r0 + 1
                    float *o0 = opaque(ob + k0), *o1 = opaque(ob + k1);
                    unsigned ofs = (unsigned)ii0 * plane;
                    f32x2 va = 0, vb = 0, vc = 0, vd = 0;           // (column k0, column k1) of taps nw, ne, sw, se
                    const f32x2 e2 = pack2(e0, e1), w2 = pack2(wq0, wq1);
#pragma unroll 4
                    for (int ii = ii0; ii < ii1; ++ii) {
                        const BpRow8 r = rows8[ii];
                        const unsigned off0 = (unsigned)r.packed >> 5;
                        if (r.packed & 4) { va = vc; vb = vd; }   // moved exactly one row down: reuse the upper row
                        if (r.packed & 8) {                       // moved further (or first plane): fetch the lower row too
                            const float *q0 = lo0 + off0, *q1 = lo1 + off0;
                            va = pack2(__ldg(q0), __ldg(q1)); vb = pack2(__ldg(q0 + 1), __ldg(q1 + 1));
                        }
                        if (r.packed & 16) {
                            const float *q0 = up0 + off0, *q1 = up1 + off0;
                            vc = pack2(__ldg(q0), __ldg(q1)); vd = pack2(__ldg(q0 + 1), __ldg(q1 + 1));
                        }
                        const f32x2 n2 = splat2(r.n), s2 = splat2(sub_rn(1.0f, r.n));
                        const f32x2 nw = mul2(s2, e2), ne = mul2(s2, w2), sw = mul2(n2, e2), se = mul2(n2, w2);
                        float r0v, r1v;
                        unpack2(fma2(vd, se, fma2(vc, sw, fma2(vb, ne, mul2(va, nw)))), r0v, r1v);
                        st_stream(o0 + ofs, r0v);
                        st_stream(o1 + ofs, r1v);
                        ofs += plane;
                    }
                } else {
                    // rays leaving the detector: per-tap predicates (zeros padding)
                    backproject_column_checked<false>(pv + t0.i0, (char *)(ob + k0) + ii0 * plane_bytes, plane_bytes, rows, ii0, ii1,
                                               g.ph, c00, c01, e0, wq0);
                    if (has1)
                        backproject_column_checked<false>(pv + t1.i0, (char *)(ob + k1) + ii0 * plane_bytes, plane_bytes, rows, ii0,
                                                   ii1, g.ph, c10, c11, e1, wq1);
                }
            }
        }
    }
}

// ---- forward, fast numerics: row-driven separable form ------------------------------------------------------------
// Same decomposition, launch shape and index arithmetic as backproject_forward_kernel (floor indices and weights are
// bit-identical: the same axis_tap chain), but the bilinear blend is evaluated separably,
//     T[r][k]   = fma(P[r][c+1], wq, P[r][c] * e)             detector row r interpolated along the detector's 2nd axis
//     out[i][k] = fma(T[r0+1][k], n, T[r0][k] * s)            rows r0(i), r0(i)+1 blended along the 1st axis
// which differs from ATen's fma(se_v,n*w, fma(sw_v,n*e, fma(ne_v,s*w, nw_v*(s*e)))) by fp32 round-off only (tests: <= 1e-6
// rel-L2; the oracle restates this order too and the kernel matches it bit for bit).  A thread marches over DETECTOR ROWS
// instead of planes: consecutive planes move 1..1.4 rows down the detector (the magnification), so every row of the
// chunk's range is fetched exactly once, its T computed once (2 packed ops for the thread's two columns) and blended
// into the plane that ends at that row, if any (2 packed ops).  Per plane that is ~25 issue slots instead of ~38 for the
// plane-driven window of the exact kernel (whose predicated-off row fetches still issue).
//
// Tables, built ONCE per block for all the rows j of its run (one warp per row, in parallel, neighbours' floor rows by
// shuffle), then a single barrier; the rows are marched without any further synchronisation:
//   ev[slot]  slot = detector row - r_base.  n >= 0: the plane whose upper row this is, with row weight n; n < 0: none.
//             roff = row * ph, or -1 when the row is outside the detector (its T is exactly +0: zeros padding).
//   sub_lo/hi first (fetch only) and last slot of each sub-chunk of planes (one threadIdx.y slice).
//   rows      the per-plane table of the generic path: taken by a (block, j) whose planes do not move strictly down the
//             detector (magnification < 1, clamped far-outside coordinates) or span more than BP_EV_MAX rows.
// (Measured and dropped, profiles/README.md round 2: staging the block's output rows in shared memory and writing them
// with cp.async.bulk -- 39 us vs 23 us; a precomputed geometry plan read from global memory -- 25.6 us vs 21.4 us, DESIGN.md.)
constexpr int BP_EV_MAX = 112;
constexpr int BP_MAX_SUB = 8;
constexpr int BP_JS_MAX = 4;       // rows j per block (the longest run)
static_assert(BP_ICHUNK <= 32, "one warp builds a row's tables with one plane per lane");

struct __align__(8) BpEvent {
    float n;
    int roff;
};

// One detector row for the thread's two columns: T = fma(P[r][c+1], wq, P[r][c] * e).  ROWCHK: the row may lie outside
// the detector (roff < 0: T is exactly +0, zeros padding) -- a warp-uniform test, so a branch; COLCHK: taps of this
// thread's columns may lie outside (per-lane predicates).
template <bool ROWCHK, bool COLCHK>
__device__ __forceinline__ f32x2 bp_fetch_row(const float *lo0, const float *lo1, int roff, f32x2 e2, f32x2 w2, bool c00,
                                              bool c01, bool c10, bool c11) {
    f32x2 va, vb;
    if (COLCHK) {
        const bool rv = !ROWCHK || roff >= 0;
        const unsigned o = rv ? (unsigned)roff : 0u;
        const float *q0 = lo0 + o, *q1 = lo1 + o;
        const float a0 = (rv && c00) ? __ldg(q0) : 0.0f, b0 = (rv && c01) ? __ldg(q0 + 1) : 0.0f;
        const float a1 = (rv && c10) ? __ldg(q1) : 0.0f, b1 = (rv && c11) ? __ldg(q1 + 1) : 0.0f;
        va = pack2(a0, a1); vb = pack2(b0, b1);
    } else {
        // ROWCHK: a row outside the detector is fetched from row 0 instead and its T replaced by +0 afterwards -- two
        // selects, no branch: a branch here would keep the compiler from batching the loads of the unrolled rows
        const unsigned o = ROWCHK ? (unsigned)max(roff, 0) : (unsigned)roff;
        const float *q0 = lo0 + o, *q1 = lo1 + o;
        va = pack2(__ldg(q0), __ldg(q1)); vb = pack2(__ldg(q0 + 1), __ldg(q1 + 1));
        const f32x2 t = fma2(vb, w2, mul2(va, e2));
        return (ROWCHK && roff < 0) ? 0ull : t;
    }
    return fma2(vb, w2, mul2(va, e2));
}

#ifndef LR_BP_UNROLL
#define LR_BP_UNROLL 4
#endif
#define LR_STR2(x) #x
#define LR_STR(x) LR_STR2(x)
#define LR_BP_UNROLL_PRAGMA _Pragma(LR_STR(unroll LR_BP_UNROLL))

// One thread's two columns over one sub-chunk of planes.
template <bool ROWCHK, bool COLCHK>
__device__ __forceinline__ void bp_march_rows(const BpEvent *__restrict__ ev, int s_lo, int s_hi, const float *lo0,
                                              const float *lo1, float *o0, float *o1, unsigned ofs, unsigned step,
                                              f32x2 e2, f32x2 w2, bool c00, bool c01, bool c10, bool c11, bool has1) {
    f32x2 t_prev = bp_fetch_row<ROWCHK, COLCHK>(lo0, lo1, ev[s_lo].roff, e2, w2, c00, c01, c10, c11);
    LR_BP_UNROLL_PRAGMA
    for (int s = s_lo + 1; s <= s_hi; ++s) {
        const BpEvent e = ev[s];
        const f32x2 t = bp_fetch_row<ROWCHK, COLCHK>(lo0, lo1, e.roff, e2, w2, c00, c01, c10, c11);
        if (e.n >= 0.0f) {
            const f32x2 n2 = splat2(e.n), s2 = splat2(sub_rn(1.0f, e.n));
            float r0v, r1v;
            unpack2(fma2(t, n2, mul2(t_prev, s2)), r0v, r1v);
            st_stream(o0 + ofs, r0v);
            if (!COLCHK || has1) st_stream(o1 + ofs, r1v);
            ofs += step;
        }
        t_prev = t;
    }
}

__global__ void __launch_bounds__(256)      // ptxas settles on 64 registers (6 blocks of 160 threads per SM)
    backproject_forward_rows_kernel(const float *__restrict__ proj, float *__restrict__ out, BpDims g, BpPoses poses) {
    __shared__ BpEvent ev_all[BP_JS_MAX][BP_EV_MAX];
    __shared__ BpRow rows_all[BP_JS_MAX][BP_ICHUNK];
    __shared__ int sub_lo[BP_JS_MAX][BP_MAX_SUB], sub_hi[BP_JS_MAX][BP_MAX_SUB];
    __shared__ float scale_all[BP_JS_MAX];
    __shared__ int flags_all[BP_JS_MAX];

    const int tid = threadIdx.y * blockDim.x + threadIdx.x;
    int L = blockIdx.x, nj = g.nj0, js = g.js0, j_base = 0;      // block index -> (run of rows, chunk, view, batch item)
    unsigned m_nj = g.m_nj0;
    if (L >= g.nj0 * g.n_vc) {
        L -= g.nj0 * g.n_vc; nj = g.nj1; js = g.js1; j_base = g.nj0 * g.js0; m_nj = g.m_nj1;
        if (L >= g.nj1 * g.n_vc) { L -= g.nj1 * g.n_vc; nj = g.nj2; js = g.js2; j_base += g.nj1 * g.js1; m_nj = g.m_nj2; }
    }
    const int vc = div_magic(L, nj, m_nj);              // (three integer divisions were a third of the block prologue)
    const int bv = div_magic(vc, g.n_chunks, g.m_chunks);
    const int bi = div_magic(bv, g.n_views, g.m_views);
    const int pl = bv - bi * g.n_views;
    const int p = g.p0 + pl;
    const int i_begin = (vc - bv * g.n_chunks) * g.ichunk;
    const int i_count = min(g.ichunk, g.d - i_begin);
    const int j_begin = j_base + (L - vc * nj) * js, j_end = min(g.w, j_begin + js);
    const float sx = poses.s[pl][0], sy = poses.s[pl][1], sz = poses.s[pl][2];
    const int ii0 = threadIdx.y * g.isub, ii1 = min(i_count, ii0 + g.isub);
    const int64_t plane_bytes = (int64_t)g.w * g.h * 4;
    const unsigned plane = (unsigned)(g.w * g.h);
    const float *pv0 = proj + bi * ((int64_t)g.P * g.proj_view_stride) + (int64_t)p * g.proj_view_stride;
    float *ob0 = out + bi * g.out_batch_stride + (int64_t)p * g.out_chan_stride + (int64_t)i_begin * g.w * g.h;
    const f32x2 zero2 = splat2(g.zero);

    // ---- phase A: the tables of every row of the run, one (complete) warp per row, lane = plane of the chunk
    {
        const int warp = tid >> 5, lane = tid & 31, n_full = (int)(blockDim.x * blockDim.y) >> 5;
        if (warp < n_full) {
            for (int jr = warp; jr < j_end - j_begin; jr += n_full) {
                const int j = j_begin + jr;
                const float scale = view_scale(sy, g.w, j);
                const bool act = lane < i_count;
                const AxisTap t = axis_tap((float)(g.i_off + i_begin + (act ? lane : 0)) - g.half_d, sx, scale, g.div_pw, g.hpw);
                const int r0 = t.i0;
                const int r_prev = __shfl_up_sync(0xffffffffu, r0, 1);
                const int r_base = __shfl_sync(0xffffffffu, r0, 0);
                const int r_last = __shfl_sync(0xffffffffu, r0, i_count - 1);
                const bool mono = lane == 0 || !act || r0 > r_prev;
                const bool fast = __all_sync(0xffffffffu, mono) && (r_last + 1 - r_base < BP_EV_MAX);
                const int r_sub_last = __shfl_sync(0xffffffffu, r0, min((lane / g.isub) * g.isub + g.isub - 1, i_count - 1));
                if (act) {
                    BpRow r;
                    r.off0 = r0 * g.ph; r.n = t.w1; r.s = sub_rn(1.0f, t.w1);
                    r.mask = ((unsigned)r0 < (unsigned)g.pw ? 1 : 0) | ((unsigned)(r0 + 1) < (unsigned)g.pw ? 2 : 0);
                    rows_all[jr][lane] = r;
                    if (fast) {
                        BpEvent *ev = ev_all[jr];
                        const int slot = r0 + 1 - r_base;
                        for (int s = lane == 0 ? 0 : r_prev + 2 - r_base; s < slot; ++s) {      // rows no plane ends at
                            const int r = r_base + s;
                            BpEvent e; e.n = -1.0f; e.roff = (unsigned)r < (unsigned)g.pw ? r * g.ph : -1;
                            ev[s] = e;
                        }
                        BpEvent e; e.n = t.w1; e.roff = (unsigned)(r0 + 1) < (unsigned)g.pw ? (r0 + 1) * g.ph : -1;
                        ev[slot] = e;
                        const int sub = lane / g.isub, rem = lane - sub * g.isub;
                        // bit 30 of the first slot: every detector row of this sub-chunk lies inside the detector
                        if (rem == 0) sub_lo[jr][sub] = (slot - 1) | ((r0 >= 0 && r_sub_last + 1 < g.pw) ? (1 << 30) : 0);
                        if (rem == g.isub - 1 || lane == i_count - 1) sub_hi[jr][sub] = slot;
                    }
                }
                if (lane == 0) {
                    scale_all[jr] = scale;
                    flags_all[jr] = (fast ? 1 : 0) | ((r_base >= 0 && r_last + 1 < g.pw) ? 2 : 0);
                }
            }
        }
    }
    __syncthreads();
    if (ii0 >= ii1) return;

    // ---- phase B: march the rows, no further synchronisation
    for (int j = j_begin; j < j_end; ++j) {
        const int jr = j - j_begin;
        const int fl = flags_all[jr];
        const float scale = scale_all[jr];
        const BpRow *rows = rows_all[jr];
        for (int q = threadIdx.x; q < g.hp; q += blockDim.x) {
            const int k0 = q, k1 = q + g.hp;
            const bool has1 = k1 < g.h;
            // both column taps as one packed chain (same op sequence as axis_tap)
            const f32x2 cen = pack2((float)k0 - g.half_h, (float)(has1 ? k1 : k0) - g.half_h), sz2 = splat2(sz);
            const f32x2 a = add2(mul2_sep(sub2(cen, sz2), splat2(scale), zero2), sz2);
            const f32x2 gq = mul2(div_const2(a, g.div_ph), splat2(2.0f));
            f32x2 ix = mul2(add2(gq, splat2(1.0f)), splat2(g.hph));
            float ixa, ixb;
            unpack2(ix, ixa, ixb);
            const float hi = g.hph * 2.0f + 3.0f;
            ix = pack2(clamp_index(ixa, hi), clamp_index(ixb, hi));
            f32x2 fl2;
            int c0, c1;
            floor2_fi(ix, fl2, c0, c1);
            const f32x2 w2 = sub2(ix, fl2), e2 = sub2(splat2(1.0f), w2);
            const bool c00 = (unsigned)c0 < (unsigned)g.ph, c01 = (unsigned)(c0 + 1) < (unsigned)g.ph;
            const bool c10 = has1 && (unsigned)c1 < (unsigned)g.ph, c11 = has1 && (unsigned)(c1 + 1) < (unsigned)g.ph;
            float *ob = ob0 + (unsigned)(j * g.h);
            if (fl & 1) {
                const int s_lo_f = sub_lo[jr][threadIdx.y], s_lo = s_lo_f & ((1 << 30) - 1), s_hi = sub_hi[jr][threadIdx.y];
                // (block-uniform on purpose: a per-sub-chunk flag -- bit 30 of sub_lo -- lets more threads take the plain
                // variant but measured 23.3 us instead of 21.3: warps of one block then run different variants)
                const bool rows_in = (fl & 2) != 0;
                const float *lo0 = opaque(pv0 + c0), *lo1 = opaque(pv0 + c1);
                // all taps of the warp's columns inside the detector (a vote: the variants compute the same values)?
                const bool cols_in = __all_sync(__activemask(), has1 && c00 && c01 && c10 && c11);
                float *o0 = opaque(ob + k0), *o1 = opaque(ob + k1);
                const unsigned ofs = (unsigned)ii0 * plane;
                if (cols_in && rows_in) bp_march_rows<false, false>(ev_all[jr], s_lo, s_hi, lo0, lo1, o0, o1, ofs, plane, e2, w2, c00, c01, c10, c11, has1);
                else if (cols_in) bp_march_rows<true, false>(ev_all[jr], s_lo, s_hi, lo0, lo1, o0, o1, ofs, plane, e2, w2, c00, c01, c10, c11, has1);
                else bp_march_rows<true, true>(ev_all[jr], s_lo, s_hi, lo0, lo1, o0, o1, ofs, plane, e2, w2, c00, c01, c10, c11, has1);
            } else {
                // generic geometry: per-plane table, per-tap predicates, same separable blend
                float wq0, wq1, e0, e1;
                unpack2(w2, wq0, wq1); unpack2(e2, e0, e1);
                backproject_column_checked<true>(pv0 + c0, (char *)(ob + k0) + ii0 * plane_bytes, plane_bytes, rows, ii0, ii1, g.ph, c00, c01, e0, wq0);
                if (has1) backproject_column_checked<true>(pv0 + c1, (char *)(ob + k1) + ii0 * plane_bytes, plane_bytes, rows, ii0, ii1, g.ph, c10, c11, e1, wq1);
            }
        }
    }
}

// Adjoint wrt the projections: scatter grad_out * weight into the 4 detector taps (RED.ADD.F32).
__global__ void __launch_bounds__(256)
    backproject_backward_kernel(const float *__restrict__ gout, float *__restrict__ gproj, BpDims g, BpPoses poses) {
    __shared__ BpRow rows[BP_ICHUNK];
    const int j = blockIdx.x;
    const int i_begin = blockIdx.y * g.ichunk;
    const int pl = blockIdx.z;
    const int p = g.p0 + pl;
    const float sx = poses.s[pl][0], sy = poses.s[pl][1], sz = poses.s[pl][2];
    const float scale = view_scale(sy, g.w, j);
    const int i_count = min(g.ichunk, g.d - i_begin);
    build_row_table(rows, nullptr, g, i_begin, i_count, sx, scale, g.ichunk, threadIdx.x, blockDim.x);
    __syncthreads();
    float *pv = gproj + (int64_t)p * g.proj_view_stride;
    const int64_t proj_batch = (int64_t)g.P * g.proj_view_stride;
    const int plane = g.w * g.h;
    for (int k = threadIdx.x; k < g.h; k += blockDim.x) {
        const AxisTap tv = axis_tap((float)k - g.half_h, sz, scale, g.div_ph, g.hph);
        const float wq = tv.w1, e = sub_rn(1.0f, wq);
        const bool c0 = (unsigned)tv.i0 < (unsigned)g.ph, c1 = (unsigned)(tv.i0 + 1) < (unsigned)g.ph;
        const float *o = gout + (int64_t)p * g.out_chan_stride + ((int64_t)i_begin * g.w + j) * g.h + k;
        for (int ii = 0; ii < i_count; ++ii) {
            const BpRow r = rows[ii];
            const bool rv0 = (r.mask & 1) != 0, rv1 = (r.mask & 2) != 0;
            const float nw = mul_rn(r.s, e), ne = mul_rn(r.s, wq), sw = mul_rn(r.n, e), se = mul_rn(r.n, wq);
            float *q0 = pv + (r.off0 + tv.i0);
            float *q1 = q0 + g.ph;
            const float *ob = o;
#pragma unroll 1
            for (int b = 0; b < g.B; ++b) {
                const float go = ld_stream(ob);
                if (rv0 && c0) red_add(q0, mul_rn(nw, go));
                if (rv0 && c1) red_add(q0 + 1, mul_rn(ne, go));
                if (rv1 && c0) red_add(q1, mul_rn(sw, go));
                if (rv1 && c1) red_add(q1 + 1, mul_rn(se, go));
                q0 += proj_batch; q1 += proj_batch; ob += g.out_batch_stride;
            }
            o += plane;
        }
    }
}

// sdct:227-250 itself, for API parity: grid (P,2,d,w,h); channel 0 = gv (detector axis 1), channel 1 = gu.
__global__ void __launch_bounds__(256) backproj_grid_kernel(float *__restrict__ grid, BpDims g, BpPoses poses) {
    const int j = blockIdx.x, i = blockIdx.y, pl = blockIdx.z, p = g.p0 + pl;
    const float sx = poses.s[pl][0], sy = poses.s[pl][1], sz = poses.s[pl][2];
    const float scale = view_scale(sy, g.w, j);
    const int64_t nv = (int64_t)g.d * g.w * g.h;
    const float xi = (float)(g.i_off + i) - g.half_d;
    const float gu = mul_rn(div_const(add_rn(mul_rn(sub_rn(xi, sx), scale), sx), g.div_pw), 2.0f);
    for (int k = threadIdx.x; k < g.h; k += blockDim.x) {
        const float zk = (float)k - g.half_h;
        const float gv = mul_rn(div_const(add_rn(mul_rn(sub_rn(zk, sz), scale), sz), g.div_ph), 2.0f);
        const int64_t vox = ((int64_t)i * g.w + j) * g.h + k;
        grid[((int64_t)p * 2 + 0) * nv + vox] = gv;
        grid[((int64_t)p * 2 + 1) * nv + vox] = gu;
    }
}

static int fill_dims(BpDims &g, int B, int P, int pw, int ph, int d_total, int w, int h, int64_t obs, int64_t ocs,
                     int i_begin = 0, int i_count = -1) {
    LR_REQUIRE(B > 0 && P > 0 && pw > 0 && ph > 0 && d_total > 0 && w > 0 && h > 0,
               "backproject: non-positive dimension (B=%d P=%d pw=%d ph=%d d=%d w=%d h=%d)", B, P, pw, ph, d_total, w, h);
    const int d = i_count < 0 ? d_total : i_count;
    LR_REQUIRE(i_begin >= 0 && d > 0 && i_begin + d <= d_total, "backproject: slab [%d, %d) is not inside [0, %d)", i_begin,
               i_begin + d, d_total);
    LR_REQUIRE(d <= 65535 * (BP_ICHUNK / 2) && w < (1 << 30), "backproject: volume too large for the launch grid");
    LR_REQUIRE((int64_t)(pw + 4) * ph < (1ll << 26) && (int64_t)w * h < (1ll << 31), "backproject: detector (pw*ph must be < 2^26) / plane too large for 32-bit offsets");
    g.B = B; g.P = P; g.pw = pw; g.ph = ph; g.d = d; g.w = w; g.h = h; g.p0 = 0; g.i_off = i_begin;
    const int n_chunks = (d + BP_ICHUNK - 1) / BP_ICHUNK;
    g.ichunk = (((d + n_chunks - 1) / n_chunks + 3) / 4) * 4;      // balanced, multiple of the unroll factor
    if (g.ichunk > BP_ICHUNK) g.ichunk = BP_ICHUNK;
    g.isub = g.ichunk; g.hp = (h + 1) / 2; g.bx = g.by = 1;
    g.js0 = g.js1 = g.js2 = 1; g.nj0 = w; g.nj1 = g.nj2 = 0; g.n_chunks = g.n_vc = g.n_views = 1;
    g.half_d = (float)((double)d_total / 2.0); g.half_h = (float)((double)h / 2.0);
    g.div_pw = make_const_div((float)pw); g.div_ph = make_const_div((float)ph);
    g.hpw = (float)(pw - 1) / 2.0f; g.hph = (float)(ph - 1) / 2.0f;
    g.proj_view_stride = (int64_t)pw * ph;
    g.out_batch_stride = obs; g.out_chan_stride = ocs;
    g.zero = 0.0f;
    g.m_nj0 = g.m_nj1 = g.m_nj2 = g.m_chunks = g.m_views = 0;
    return LR_OK;
}

static int block_threads(int h) {
    int t = ((h + 31) / 32) * 32;
    return t < 32 ? 32 : (t > 256 ? 256 : t);
}

#ifndef LR_BP_ISUB
#define LR_BP_ISUB 16
#endif

#ifndef LR_BP_FWD_THREADS
#define LR_BP_FWD_THREADS 192
#endif
// Forward launch shape.  Block = (column pairs: ceil(h/2), at most 256) x (sub-chunks of the chunk's planes); each block
// walks a run of consecutive rows j.  Long runs amortise the per-block set-up, but a block of 4 rows lives ~7 us of a
// ~25 us launch, the kernel is latency-bound (throughput follows occupancy) and the grid is only a few waves, so with
// equal blocks the launch ends with every SM draining from 6 resident blocks to 0 over a whole block duration.  The
// runs therefore taper: 4 rows, then 2, then 1.
static dim3 forward_shape(BpDims &g, int n_views, unsigned &grid, int min_threads = 1) {
    g.hp = (g.h + 1) / 2;
    g.bx = g.hp > 256 ? 256 : g.hp;
    int by = LR_BP_FWD_THREADS / g.bx;
    if (by < 1) by = 1;
    int isub = LR_BP_ISUB;
    if (by * isub > BP_ICHUNK) by = BP_ICHUNK / isub;
    const int per_item = by * isub;
    const int n_chunks0 = (g.d + per_item - 1) / per_item;                    // balance the chunks over the planes
    isub = (((g.d + n_chunks0 - 1) / n_chunks0 + by - 1) / by + 3) / 4 * 4;   // multiple of the unroll factor
    if (isub > LR_BP_ISUB) isub = LR_BP_ISUB;
    if (g.bx * by < min_threads) g.bx = (min_threads + by - 1) / by;     // tiny volumes: idle lanes, but a whole warp 0
    g.by = by;
    g.isub = isub;
    g.ichunk = isub * by;
    g.n_chunks = (g.d + g.ichunk - 1) / g.ichunk;
    g.n_views = n_views;
    g.n_vc = g.n_chunks * n_views * g.B;
#ifndef LR_BP_JS0
#define LR_BP_JS0 4
#endif
    g.js0 = LR_BP_JS0; g.js1 = LR_BP_JS0 / 2; g.js2 = LR_BP_JS0 / 4 > 0 ? LR_BP_JS0 / 4 : 1;
    // share of the short runs: about 1.2 waves of work, at most half (measured: 50/30/20 % is best at batch 1 = 0.9
    // waves of 4-row blocks on 6 resident blocks per SM, 90/8/2 % at batch 8)
    const double waves = (double)((g.w + g.js0 - 1) / g.js0) * g.n_vc / (6.0 * sm_count());
    double small = 1.2 / (waves > 0.1 ? waves : 0.1);
    if (small > 0.5) small = 0.5;
    const int f0 = (int)(100.0 * (1.0 - small) + 0.5);      // percent of the rows in 4-row / 2-row runs
    const int f1 = (int)(100.0 * 0.6 * small + 0.5);
    g.nj0 = (g.w * f0 / 100) / g.js0;
    int rest = g.w - g.nj0 * g.js0;
    g.nj1 = f0 + f1 >= 100 ? (rest + g.js1 - 1) / g.js1 : (g.w * f1 / 100) / g.js1;
    if (g.nj1 * g.js1 > rest) g.nj1 = (rest + g.js1 - 1) / g.js1;
    rest -= g.nj1 * g.js1;
    g.nj2 = rest > 0 ? rest : 0;
    grid = (unsigned)((g.nj0 + g.nj1 + g.nj2) * g.n_vc);
    auto magic = [&](int dvs) -> unsigned {      // exact for every block index of this grid, else 0 (plain division)
        if (dvs <= 1 || (uint64_t)grid * (uint64_t)dvs >= (1ull << 32)) return 0u;
        return (unsigned)(((1ull << 32) + (unsigned)dvs - 1) / (unsigned)dvs);
    };
    g.m_nj0 = magic(g.nj0); g.m_nj1 = magic(g.nj1); g.m_nj2 = magic(g.nj2);
    g.m_chunks = magic(g.n_chunks); g.m_views = magic(g.n_views);
    return dim3((unsigned)g.bx, (unsigned)g.by, 1);
}

}  // namespace lr

using namespace lr;

extern "C" int lr_backproject_forward_slab(const float *proj, const float *poses, int B, int P, int pw, int ph, int d_total,
                                           int w, int h, int i_begin, int i_count, float *out,
                                           int64_t out_batch_stride, int64_t out_chan_stride, lr_stream_t stream) {
    LR_REQUIRE(proj && poses && out, "backproject_forward: null pointer");
    BpDims g;
    if (int e = fill_dims(g, B, P, pw, ph, d_total, w, h, out_batch_stride, out_chan_stride, i_begin, i_count)) return e;
    const int d = g.d;
    LR_REQUIRE(out_chan_stride >= (int64_t)d * w * h, "backproject_forward: out_chan_stride smaller than a volume");
    for (int p0 = 0; p0 < P; p0 += BP_MAX_VIEWS) {
        const int np = P - p0 < BP_MAX_VIEWS ? P - p0 : BP_MAX_VIEWS;
        BpPoses ps;
        for (int q = 0; q < np; ++q)
            for (int c = 0; c < 3; ++c) ps.s[q][c] = poses[(p0 + q) * 3 + c];
        g.p0 = p0;
        unsigned grid;
        LR_REQUIRE((int64_t)w * ((d + 3) / 4) * np * B < (1ll << 31), "backproject_forward: too many blocks for one launch");
        if (numerics_mode() == LR_NUMERICS_EXACT) {
            const dim3 block = forward_shape(g, np, grid);
            backproject_forward_kernel<<<grid, block, 0, as_stream(stream)>>>(proj, out, g, ps);
            if (int e = check_launch("backproject_forward_kernel")) return e;
            continue;
        }
        const dim3 block = forward_shape(g, np, grid, 32);
        backproject_forward_rows_kernel<<<grid, block, 0, as_stream(stream)>>>(proj, out, g, ps);
        if (int e = check_launch("backproject_forward_rows_kernel")) return e;
    }
    return LR_OK;
}

// Launch plan of the forward kernel, for host-side tests (no device work).  plan = {ichunk, isub, by, bx, n_chunks,
// run0, n0, run1, n1, run2, n2, grid}: chunks of ichunk planes (by sub-chunks of isub), bx column pairs per block;
// the w rows are walked as n0 runs of run0 rows, then n1 of run1, then n2 of run2; grid blocks in total.
extern "C" int lr_backproject_forward_plan(int B, int P, int pw, int ph, int d, int w, int h, int plan[12]) {
    LR_REQUIRE(plan, "backproject_forward_plan: null pointer");
    BpDims g;
    if (int e = fill_dims(g, B, P, pw, ph, d, w, h, 0, 0)) return e;
    unsigned grid = 0;
    const int np = P < BP_MAX_VIEWS ? P : BP_MAX_VIEWS;
    const dim3 block = forward_shape(g, np, grid, numerics_mode() == LR_NUMERICS_EXACT ? 1 : 32);
    plan[0] = g.ichunk; plan[1] = g.isub; plan[2] = (int)block.y; plan[3] = (int)block.x; plan[4] = g.n_chunks;
    plan[5] = g.js0; plan[6] = g.nj0; plan[7] = g.js1; plan[8] = g.nj1; plan[9] = g.js2; plan[10] = g.nj2; plan[11] = (int)grid;
    return LR_OK;
}

extern "C" int lr_backproject_forward(const float *proj, const float *poses, int B, int P, int pw, int ph, int d, int w,
                                      int h, float *out, int64_t out_batch_stride, int64_t out_chan_stride,
                                      lr_stream_t stream) {
    return lr_backproject_forward_slab(proj, poses, B, P, pw, ph, d, w, h, 0, d, out, out_batch_stride, out_chan_stride,
                                       stream);
}

extern "C" int lr_backproject_backward(const float *grad_out, int64_t go_batch_stride, int64_t go_chan_stride,
                                       const float *poses, int B, int P, int pw, int ph, int d, int w, int h,
                                       float *grad_proj, lr_stream_t stream) {
    LR_REQUIRE(grad_out && poses && grad_proj, "backproject_backward: null pointer");
    BpDims g;
    if (int e = fill_dims(g, B, P, pw, ph, d, w, h, go_batch_stride, go_chan_stride)) return e;
    for (int p0 = 0; p0 < P; p0 += BP_MAX_VIEWS) {
        const int np = P - p0 < BP_MAX_VIEWS ? P - p0 : BP_MAX_VIEWS;
        BpPoses ps;
        for (int q = 0; q < np; ++q)
            for (int c = 0; c < 3; ++c) ps.s[q][c] = poses[(p0 + q) * 3 + c];
        g.p0 = p0;
        dim3 grid((unsigned)w, (unsigned)((d + g.ichunk - 1) / g.ichunk), (unsigned)np);
        backproject_backward_kernel<<<grid, block_threads(h), 0, as_stream(stream)>>>(grad_out, grad_proj, g, ps);
        if (int e = check_launch("backproject_backward_kernel")) return e;
    }
    return LR_OK;
}

extern "C" int lr_backproj_grid(const float *poses, int P, int d, int w, int h, int pw, int ph, float *grid,
                                lr_stream_t stream) {
    LR_REQUIRE(poses && grid, "backproj_grid: null pointer");
    BpDims g;
    if (int e = fill_dims(g, 1, P, pw, ph, d, w, h, 0, 0)) return e;
    LR_REQUIRE(d <= 65535, "backproj_grid: d must be <= 65535");
    for (int p0 = 0; p0 < P; p0 += BP_MAX_VIEWS) {
        const int np = P - p0 < BP_MAX_VIEWS ? P - p0 : BP_MAX_VIEWS;
        BpPoses ps;
        for (int q = 0; q < np; ++q)
            for (int c = 0; c < 3; ++c) ps.s[q][c] = poses[(p0 + q) * 3 + c];
        g.p0 = p0;
        dim3 grid_dim((unsigned)w, (unsigned)d, (unsigned)np);
        backproj_grid_kernel<<<grid_dim, block_threads(h), 0, as_stream(stream)>>>(grid, g, ps);
        if (int e = check_launch("backproj_grid_kernel")) return e;
    }
    return LR_OK;
}
