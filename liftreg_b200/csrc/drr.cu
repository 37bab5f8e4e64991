// Cone-beam DRR forward projection and its adjoint (ray-marched trilinear gather), sm_100a.
//
// Replaces reference src/liftreg/utils/sdct_projection_utils.py:15-57 (project_grid_multi: a materialised
// (P,rd,rh,w,3) sample grid, 442 MB at 160^3 / 4 views / 240^2) and :59-86 (calculate_projection: flip,
// grid_sample_3d, sum over the ray, *dx, *0.1); also src/liftreg/layers/layers.py:182-236 (proj_layer,
// y normalised by w instead of w-1, no 0.1 factor).  Nothing is materialised: each thread owns one ray,
// rebuilds the sample position of every coronal plane j in registers with the reference's fp32 op order
// (so floor() indices and weights are bit-identical), gathers 8 taps through L1/L2 and accumulates in fp32
// in ray order (j ascending).  Lanes run along the detector's second axis, which maps to the volume's
// contiguous axis, so each warp-wide tap load touches one or two 128 B lines.
//
// Rays are clipped to the j-range in which they can touch the volume (a conservative superset computed from
// the closed form X(j) = lx + j*(sx-lx)/sy); samples outside contribute exactly +0 in the reference.
#include "common.cuh"

namespace lr {

constexpr int DRR_MAX_VIEWS = 128;  // (volume, pose) pairs per launch; poses travel as kernel parameters
constexpr int DRR_ROWS = 4;         // detector rows (u) per block in the one-ray-per-thread kernels (backward, grid)
#ifndef LR_DRR_PAIRS
#define LR_DRR_PAIRS 2
#endif
#ifndef LR_DRR_SEGS
#define LR_DRR_SEGS 4
#endif
constexpr int DRR_PAIRS = LR_DRR_PAIRS;        // forward: ray pairs (2 detector rows each) per block along u
static_assert(LR_DRR_SEGS >= 2, "the threads of the first two runs set up the block's rays");
constexpr int DRR_SEGS = LR_DRR_SEGS;         // forward: every ray is cut into 4 runs of ceil(w/4) coronal planes, one warp each

struct DrrView {
    float sx, sy, sz;
    int vol;  // which volume of the batch this view projects
};
struct DrrViews {
    DrrView v[DRR_MAX_VIEWS];
};

struct DrrDims {
    int d, w, h, rd, rh;
    int view0;                 // first (b,p) pair of this launch, for output addressing
    float half_rd, half_rh;    // rd/2, rh/2 (exact)
    float sp0, sp1, sp2;       // voxel spacing (mm)
    ConstDiv div_x, div_y, div_z;  // d/2, (w-1)/2 or w/2, h/2 :  X/d*2 == X/(d/2) exactly
    float hd, hw, hh;          // (d-1)/2, (w-1)/2, (h-1)/2 : ((g+1)/2)*(S-1) == (g+1)*((S-1)/2) exactly
    float lim_x, lim_z;        // clip half-widths d/2+2, h/2+2
    float out_scale;
    float zero;                // +0.0f the compiler cannot constant-fold (see mul2_sep)
    int seg_len;               // planes per ray run in the forward kernel: ceil(w / DRR_SEGS)
    int64_t nvox;
};

// Multi-GPU sweep (lr_drr_forward_peers): the kernel stores every detector pixel into the gather buffers of ALL ranks
// (peer memory over NVLink), view k of the launch at slot k * vstride, so that no collective moves the images afterwards.
struct DrrPeers {
    float *p[LR_MAX_PEERS];
    int n, vstride;
};

struct Ray {
    float sx, sy, sz, Dx, Dy, Dz, r2, dx;
    int j0, j1;  // inclusive range of coronal planes that may touch the volume
    bool clipped;  // j0..j1 came from the clip (coordinates stay within a few voxels of the volume)
};

__device__ __forceinline__ Ray ray_setup(const DrrView &vw, const DrrDims &g, int u, int v) {
    Ray r;
    r.sx = vw.sx; r.sy = vw.sy; r.sz = vw.sz;
    const float lx = (float)u - g.half_rd, lz = (float)v - g.half_rh;   // sdct:32-33 (unit-step linspace)
    const float Ix = add_rn(lx, -r.sx), Iy = add_rn(0.0f, -r.sy), Iz = add_rn(lz, -r.sz);  // sdct:35-38
    const float rc = div_rn(1.0f, Iy);                                   // sdct:39
    const float ax = mul_rn(mul_rn(Ix, rc), g.sp0), ay = mul_rn(mul_rn(Iy, rc), g.sp1), az = mul_rn(mul_rn(Iz, rc), g.sp2);
    r.dx = __fsqrt_rn(fma_rn(az, az, fma_rn(ay, ay, mul_rn(ax, ax))));   // sdct:41 (torch CPU norm order)
    const float n = __fsqrt_rn(fma_rn(Iz, Iz, fma_rn(Iy, Iy, mul_rn(Ix, Ix))));  // sdct:40
    r.Dx = div_rn(Ix, n); r.Dy = div_rn(Iy, n); r.Dz = div_rn(Iz, n);
    r.r2 = div_rn(1.0f, r.Dy);                                           // sdct:50

    // conservative clip: X(j) = lx + j*(sx-lx)/sy must lie in [-lim_x, lim_x], same for Z
    float t0 = 0.0f, t1 = (float)(g.w - 1);
    const float inv_sy = 1.0f / r.sy;
    const float bx = (r.sx - lx) * inv_sy, bz = (r.sz - lz) * inv_sy;
    if (fabsf(bx) > 1e-12f) {
        float a = (-g.lim_x - lx) / bx, b = (g.lim_x - lx) / bx;
        t0 = fmaxf(t0, fminf(a, b)); t1 = fminf(t1, fmaxf(a, b));
    } else if (fabsf(lx) > g.lim_x) t1 = -1.0f;
    if (fabsf(bz) > 1e-12f) {
        float a = (-g.lim_z - lz) / bz, b = (g.lim_z - lz) / bz;
        t0 = fmaxf(t0, fminf(a, b)); t1 = fminf(t1, fmaxf(a, b));
    } else if (fabsf(lz) > g.lim_z) t1 = -1.0f;
    r.j0 = max(0, (int)floorf(t0) - 1);
    r.j1 = min(g.w - 1, (int)ceilf(t1) + 1);
    if (!(t1 >= t0)) { r.j0 = 0; r.j1 = -1; }
    r.clipped = r.sy > (float)(g.w - 1);
    if (!r.clipped) { r.j0 = 0; r.j1 = g.w - 1; }  // emitter inside the slab: no clipping
    return r;
}

struct Sample {
    float iz, iy, ix;  // source indices along volume axes 0 (d), 1 (w), 2 (h)
};

// sdct:50-56 + flip (:76) + ATen unnormalise.  jf = (float)j is carried as a float counter (no I2F).
__device__ __forceinline__ Sample ray_point(const Ray &r, const DrrDims &g, float jf) {
    const float T = mul_rn(r.r2, sub_rn(jf, r.sy));
    const float X = add_rn(mul_rn(r.Dx, T), r.sx), Y = add_rn(mul_rn(r.Dy, T), r.sy), Z = add_rn(mul_rn(r.Dz, T), r.sz);
    const float g0 = div_const(X, g.div_x);                  // X/d*2
    const float g1 = add_rn(div_const(Y, g.div_y), -1.0f);   // Y/(w-1)*2 + -1
    const float g2 = div_const(Z, g.div_z);                  // Z/h*2
    Sample s;
    // beyond [-2, S+1] no tap is in bounds; the clamp keeps floor_fi's |x| < 2^22 precondition
    s.iz = clamp_index(mul_rn(add_rn(g0, 1.0f), g.hd), g.hd * 2.0f + 2.0f);
    s.iy = clamp_index(mul_rn(add_rn(g1, 1.0f), g.hw), g.hw * 2.0f + 2.0f);
    s.ix = clamp_index(mul_rn(add_rn(g2, 1.0f), g.hh), g.hh * 2.0f + 2.0f);
    return s;
}

struct Taps {
    float wt[8];      // ATen order: tnw tne tsw tse bnw bne bsw bse (x fastest, then y, then z)
    int base;         // voxel offset of tap (z0,y0,x0); < 2^31 (checked on the host)
    int x0, y0, z0;
    float wx1, wy1, wz1;   // fractional parts (upper-tap weights)
};

__device__ __forceinline__ Taps make_taps(const Sample &s, const DrrDims &g) {
    float fx, fy, fz;
    Taps t;
    floor_fi(s.ix, fx, t.x0);
    floor_fi(s.iy, fy, t.y0);
    floor_fi(s.iz, fz, t.z0);
    const float wx1 = sub_rn(s.ix, fx), wx0 = sub_rn(add_rn(fx, 1.0f), s.ix);
    const float wy1 = sub_rn(s.iy, fy), wy0 = sub_rn(add_rn(fy, 1.0f), s.iy);
    const float wz1 = sub_rn(s.iz, fz), wz0 = sub_rn(add_rn(fz, 1.0f), s.iz);
    const float a00 = mul_rn(wx0, wy0), a10 = mul_rn(wx1, wy0), a01 = mul_rn(wx0, wy1), a11 = mul_rn(wx1, wy1);
    t.wt[0] = mul_rn(a00, wz0); t.wt[1] = mul_rn(a10, wz0); t.wt[2] = mul_rn(a01, wz0); t.wt[3] = mul_rn(a11, wz0);
    t.wt[4] = mul_rn(a00, wz1); t.wt[5] = mul_rn(a10, wz1); t.wt[6] = mul_rn(a01, wz1); t.wt[7] = mul_rn(a11, wz1);
    t.base = (t.z0 * g.w + t.y0) * g.h + t.x0;
    t.wx1 = wx1; t.wy1 = wy1; t.wz1 = wz1;
    return t;
}

__device__ __forceinline__ bool taps_interior(const Taps &t, const DrrDims &g) {   // all 8 taps inside the volume
    return (unsigned)t.x0 < (unsigned)(g.h - 1) && (unsigned)t.y0 < (unsigned)(g.w - 1) && (unsigned)t.z0 < (unsigned)(g.d - 1);
}
__device__ __forceinline__ unsigned taps_mask(const Taps &t, const DrrDims &g) {   // bit c set <=> tap c inside
    const unsigned vx0 = (unsigned)t.x0 < (unsigned)g.h, vx1 = (unsigned)(t.x0 + 1) < (unsigned)g.h;
    const unsigned vy0 = (unsigned)t.y0 < (unsigned)g.w, vy1 = (unsigned)(t.y0 + 1) < (unsigned)g.w;
    const unsigned vz0 = (unsigned)t.z0 < (unsigned)g.d, vz1 = (unsigned)(t.z0 + 1) < (unsigned)g.d;
    const unsigned mx = vx0 | (vx1 << 1);
    const unsigned mxy = (vy0 ? mx : 0u) | ((vy1 ? mx : 0u) << 2);
    return (vz0 ? mxy : 0u) | ((vz1 ? mxy : 0u) << 4);
}

// One sample in the fast-numerics order (LR_NUMERICS_FAST): taps outside the volume enter as 0, the blend is seven fused
// lerps (x, then y, then z) over the same floor indices and fractional weights.
__device__ __forceinline__ float sample_lerp_masked(const float *__restrict__ b, unsigned m, int sy, int sz, float wx1, float wy1, float wz1) {
    float v[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        const int off = (c & 1) + ((c >> 1) & 1) * sy + (c >> 2) * sz;
        v[c] = ((m >> c) & 1u) ? __ldg(b + off) : 0.0f;
    }
    const float c00 = fma_rn(wx1, sub_rn(v[1], v[0]), v[0]), c10 = fma_rn(wx1, sub_rn(v[3], v[2]), v[2]);
    const float c01 = fma_rn(wx1, sub_rn(v[5], v[4]), v[4]), c11 = fma_rn(wx1, sub_rn(v[7], v[6]), v[6]);
    const float d0 = fma_rn(wy1, sub_rn(c10, c00), c00), d1 = fma_rn(wy1, sub_rn(c11, c01), c01);
    return fma_rn(wz1, sub_rn(d1, d0), d0);
}

// One ray, scalar, boundary-safe: the general path (also used by rays whose pair partner is missing).
template <bool FAST>
__device__ __forceinline__ float march_ray(const float *__restrict__ V, const Ray &r, const DrrDims &g, int jlo, int jhi) {
    const int sy = g.h, sz = g.w * g.h;
    float acc = 0.0f;
    const int ja = max(r.j0, jlo), jb = min(r.j1, jhi);
    float jf = (float)ja;
    for (int j = ja; j <= jb; ++j, jf += 1.0f) {
        const Sample s = ray_point(r, g, jf);
        const Taps t = make_taps(s, g);
        const unsigned m = taps_mask(t, g);
        if (m == 0u) continue;                                  // contributes exactly +0
        const float *b = V + t.base;
        float o = 0.0f;
        if (FAST) {
            o = sample_lerp_masked(b, m, sy, sz, t.wx1, t.wy1, t.wz1);
        } else {
#pragma unroll
            for (int c = 0; c < 8; ++c) {                       // ATen: out += val*w per tap, separately rounded
                const int off = (c & 1) + ((c >> 1) & 1) * sy + (c >> 2) * sz;
                if ((m >> c) & 1u) o = add_rn(o, mul_rn(__ldg(b + off), t.wt[c]));
            }
        }
        acc = add_rn(acc, o);                                   // sum over the ray (sdct:81), j ascending
    }
    return acc;
}

__device__ __forceinline__ float finish_ray(float acc, const Ray &r, const DrrDims &g) {
    float o = mul_rn(acc, r.dx);                                // * dx (sdct:81)
    if (g.out_scale != 1.0f) o = mul_rn(o, g.out_scale);        // *= 0.1 (sdct:85)
    return o;
}

// Forward kernel.  A thread owns the two rays (u, v) and (u+1, v): neighbours on detector axis 0, which have almost
// the same clip range and whose taps overlap in L1.  Both fp32 chains run as ONE packed fp32x2 stream while all 16
// taps are inside the volume; entry / exit samples take the scalar masked path.
// Ray-segment accumulation: a detector image has too few rays to fill 148 SMs (cfg 1: 3.8 k pair-warps for 9.5 k
// warp slots, ncu: 26 % warps active), so every ray is cut into DRR_SEGS runs of seg_len = ceil(w / DRR_SEGS) planes
// marched by different warps; the run sums are combined in run order.  The summation order is therefore
//     sum_{s} ( sum_{j in run s} sample_j ),  both levels ascending, fp32
// which the oracle reproduces (seg_len argument); the reference's own order is torch.sum's vectorised cascade.
#ifndef LR_DRR_MINB
#define LR_DRR_MINB 4
#endif
template <bool FAST, bool PEERS>
__global__ void __launch_bounds__(32 * DRR_PAIRS * DRR_SEGS, LR_DRR_MINB)
    drr_forward_kernel(const float *__restrict__ vol, float *__restrict__ proj, DrrDims g, DrrViews views, DrrPeers peers) {
    __shared__ float2 part[DRR_SEGS][DRR_PAIRS][32];
    __shared__ Ray rays[DRR_PAIRS][2][32];      // the block's rays, set up once (by the threads of the first two runs)
    const int v = blockIdx.x * 32 + threadIdx.x;
    const int ua = (blockIdx.y * DRR_PAIRS + threadIdx.y) * 2;
    const int seg = threadIdx.z;
    const bool live = v < g.rh && ua < g.rd;
    const bool has_b = ua + 1 < g.rd;
    float acca = 0.0f, accb = 0.0f;
    Ray ra, rb;
    // ray_setup (two square roots, seven divisions) costs as much as ~2 marched samples; the DRR_SEGS threads that march
    // the runs of one ray share one evaluation through shared memory instead of repeating it
    if (live && seg < 2) rays[threadIdx.y][seg][threadIdx.x] = ray_setup(views.v[blockIdx.z], g, (seg == 1 && has_b) ? ua + 1 : ua, v);
    __syncthreads();
    if (live) {
    const DrrView vw = views.v[blockIdx.z];
    ra = rays[threadIdx.y][0][threadIdx.x];
    rb = rays[threadIdx.y][1][threadIdx.x];
    const float *V = opaque(vol + (int64_t)vw.vol * g.nvox);
    int seg_lo = seg * g.seg_len, seg_hi = min(g.w, seg_lo + g.seg_len) - 1;         // this warp's run of planes

    if (!(ra.clipped && rb.clipped)) {          // unusual geometry (emitter inside the slab): scalar path only
        acca = march_ray<FAST>(V, ra, g, seg_lo, seg_hi);
        accb = march_ray<FAST>(V, rb, g, seg_lo, seg_hi);
    } else {
    const f32x2 zero = splat2(g.zero), one = splat2(1.0f), mone = splat2(-1.0f);
    const f32x2 Dx = pack2(ra.Dx, rb.Dx), Dy = pack2(ra.Dy, rb.Dy), Dz = pack2(ra.Dz, rb.Dz), r2 = pack2(ra.r2, rb.r2);
    const f32x2 sx = splat2(ra.sx), sy2 = splat2(ra.sy), sz2 = splat2(ra.sz);
    const unsigned sy = (unsigned)g.h, sz = (unsigned)(g.w * g.h);
    // union of the two clip ranges; outside its own range a ray has no tap in bounds and contributes exactly +0
    const int ea = ra.j1 < ra.j0, eb = rb.j1 < rb.j0;
    int j0 = ea ? rb.j0 : (eb ? ra.j0 : min(ra.j0, rb.j0));
    int j1 = ea ? rb.j1 : (eb ? ra.j1 : max(ra.j1, rb.j1));
    if (FAST) {
        // Fixed runs of ceil(w/4) planes leave the warps of a block with very different amounts of work (a ray crosses
        // the volume in a sub-range of the planes) and the finished ones wait at the block's barrier: 26 % of all warp
        // stall samples (profiles/README.md round 2).  Fast numerics cuts the pair's CLIPPED range into equal runs
        // instead; the fp32 sum is then taken in that run order (restated by the oracle: seg_len < 0).
        const int n = j1 - j0 + 1, len = n > 0 ? (n + DRR_SEGS - 1) / DRR_SEGS : 1;
        seg_lo = j0 + seg * len; seg_hi = seg_lo + len - 1;
    }
    j0 = max(j0, seg_lo); j1 = min(j1, seg_hi);

    float jf = (float)j0;
    for (int j = j0; j <= j1; ++j, jf += 1.0f) {
        // sdct:50-56 + flip (:76) + ATen unnormalise, both rays at once
        const f32x2 T = mul2(r2, splat2(sub_rn(jf, ra.sy)));
        const f32x2 X = add2(mul2_sep(Dx, T, zero), sx), Y = add2(mul2_sep(Dy, T, zero), sy2), Z = add2(mul2_sep(Dz, T, zero), sz2);
        const f32x2 g0 = div_const2(X, g.div_x);                    // X/d*2
        const f32x2 g1 = add2(div_const2(Y, g.div_y), mone);        // Y/(w-1)*2 + -1
        const f32x2 g2 = div_const2(Z, g.div_z);                    // Z/h*2
        const f32x2 iz = mul2(add2(g0, one), splat2(g.hd));
        const f32x2 iy = mul2(add2(g1, one), splat2(g.hw));
        const f32x2 ix = mul2(add2(g2, one), splat2(g.hh));
        f32x2 fx, fy, fz;
        int x0a, x0b, y0a, y0b, z0a, z0b;
        floor2_fi(ix, fx, x0a, x0b);       // clipped rays stay within a few voxels of the volume: |x| << 2^22
        floor2_fi(iy, fy, y0a, y0b);
        floor2_fi(iz, fz, z0a, z0b);
        const f32x2 wx1 = sub2(ix, fx), wy1 = sub2(iy, fy), wz1 = sub2(iz, fz);
        const bool ina = (unsigned)x0a < (unsigned)(g.h - 1) && (unsigned)y0a < (unsigned)(g.w - 1) && (unsigned)z0a < (unsigned)(g.d - 1);
        const bool inb = (unsigned)x0b < (unsigned)(g.h - 1) && (unsigned)y0b < (unsigned)(g.w - 1) && (unsigned)z0b < (unsigned)(g.d - 1);
        const int basea = (z0a * g.w + y0a) * g.h + x0a, baseb = (z0b * g.w + y0b) * g.h + x0b;
        if (ina && inb) {
            const unsigned a0 = (unsigned)basea, b0 = (unsigned)baseb;
            const float *pa0 = V + a0, *pa1 = V + (a0 + sy), *pa2 = V + (a0 + sz), *pa3 = V + (a0 + sz + sy);
            const float *pb0 = V + b0, *pb1 = V + (b0 + sy), *pb2 = V + (b0 + sz), *pb3 = V + (b0 + sz + sy);
            f32x2 val[8];
            val[0] = pack2(__ldg(pa0), __ldg(pb0)); val[1] = pack2(__ldg(pa0 + 1), __ldg(pb0 + 1));
            val[2] = pack2(__ldg(pa1), __ldg(pb1)); val[3] = pack2(__ldg(pa1 + 1), __ldg(pb1 + 1));
            val[4] = pack2(__ldg(pa2), __ldg(pb2)); val[5] = pack2(__ldg(pa2 + 1), __ldg(pb2 + 1));
            val[6] = pack2(__ldg(pa3), __ldg(pb3)); val[7] = pack2(__ldg(pa3 + 1), __ldg(pb3 + 1));
            f32x2 o;
            if (FAST) {       // seven fused lerps instead of 12 weight products + 8 products + 7 sums
                const f32x2 c00 = fma2(wx1, sub2(val[1], val[0]), val[0]), c10 = fma2(wx1, sub2(val[3], val[2]), val[2]);
                const f32x2 c01 = fma2(wx1, sub2(val[5], val[4]), val[4]), c11 = fma2(wx1, sub2(val[7], val[6]), val[6]);
                const f32x2 d0 = fma2(wy1, sub2(c10, c00), c00), d1 = fma2(wy1, sub2(c11, c01), c01);
                o = fma2(wz1, sub2(d1, d0), d0);
            } else {
                const f32x2 wx0 = sub2(add2(fx, one), ix), wy0 = sub2(add2(fy, one), iy), wz0 = sub2(add2(fz, one), iz);
                const f32x2 a00 = mul2(wx0, wy0), a10 = mul2(wx1, wy0), a01 = mul2(wx0, wy1), a11 = mul2(wx1, wy1);
                const f32x2 wt[8] = {mul2(a00, wz0), mul2(a10, wz0), mul2(a01, wz0), mul2(a11, wz0),
                                     mul2(a00, wz1), mul2(a10, wz1), mul2(a01, wz1), mul2(a11, wz1)};
                o = splat2(0.0f);
#pragma unroll
                for (int c = 0; c < 8; ++c) o = add2(o, mul2_sep(val[c], wt[c], zero));   // ATen: out += val*w, no fma
            }
            float oa, ob;
            unpack2(o, oa, ob);
            acca = add_rn(acca, oa);                                                   // sum over the ray (sdct:81)
            accb = add_rn(accb, ob);
        } else {
            const unsigned vxa0 = (unsigned)x0a < (unsigned)g.h, vxa1 = (unsigned)(x0a + 1) < (unsigned)g.h;
            const unsigned vya0 = (unsigned)y0a < (unsigned)g.w, vya1 = (unsigned)(y0a + 1) < (unsigned)g.w;
            const unsigned vza0 = (unsigned)z0a < (unsigned)g.d, vza1 = (unsigned)(z0a + 1) < (unsigned)g.d;
            const unsigned vxb0 = (unsigned)x0b < (unsigned)g.h, vxb1 = (unsigned)(x0b + 1) < (unsigned)g.h;
            const unsigned vyb0 = (unsigned)y0b < (unsigned)g.w, vyb1 = (unsigned)(y0b + 1) < (unsigned)g.w;
            const unsigned vzb0 = (unsigned)z0b < (unsigned)g.d, vzb1 = (unsigned)(z0b + 1) < (unsigned)g.d;
            const unsigned mxa = vxa0 | (vxa1 << 1), mxya = (vya0 ? mxa : 0u) | ((vya1 ? mxa : 0u) << 2);
            const unsigned mxb = vxb0 | (vxb1 << 1), mxyb = (vyb0 ? mxb : 0u) | ((vyb1 ? mxb : 0u) << 2);
            const unsigned ma = (vza0 ? mxya : 0u) | ((vza1 ? mxya : 0u) << 4);
            const unsigned mb = (vzb0 ? mxyb : 0u) | ((vzb1 ? mxyb : 0u) << 4);
            if (FAST) {
                float wxa, wxb, wya, wyb, wza, wzb;
                unpack2(wx1, wxa, wxb); unpack2(wy1, wya, wyb); unpack2(wz1, wza, wzb);
                if (ma != 0u) acca = add_rn(acca, sample_lerp_masked(V + basea, ma, (int)sy, (int)sz, wxa, wya, wza));
                if (mb != 0u) accb = add_rn(accb, sample_lerp_masked(V + baseb, mb, (int)sy, (int)sz, wxb, wyb, wzb));
            } else {
                const f32x2 wx0 = sub2(add2(fx, one), ix), wy0 = sub2(add2(fy, one), iy), wz0 = sub2(add2(fz, one), iz);
                const f32x2 a00 = mul2(wx0, wy0), a10 = mul2(wx1, wy0), a01 = mul2(wx0, wy1), a11 = mul2(wx1, wy1);
                const f32x2 wt[8] = {mul2(a00, wz0), mul2(a10, wz0), mul2(a01, wz0), mul2(a11, wz0),
                                     mul2(a00, wz1), mul2(a10, wz1), mul2(a01, wz1), mul2(a11, wz1)};
                float w_a[8], w_b[8];
#pragma unroll
                for (int c = 0; c < 8; ++c) unpack2(wt[c], w_a[c], w_b[c]);
                if (ma != 0u) {
                    float o = 0.0f;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const int off = (c & 1) + ((c >> 1) & 1) * (int)sy + (c >> 2) * (int)sz;
                        if ((ma >> c) & 1u) o = add_rn(o, mul_rn(__ldg(V + (basea + off)), w_a[c]));
                    }
                    acca = add_rn(acca, o);
                }
                if (mb != 0u) {
                    float o = 0.0f;
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        const int off = (c & 1) + ((c >> 1) & 1) * (int)sy + (c >> 2) * (int)sz;
                        if ((mb >> c) & 1u) o = add_rn(o, mul_rn(__ldg(V + (baseb + off)), w_b[c]));
                    }
                    accb = add_rn(accb, o);
                }
            }
        }
    }
    }   // packed / scalar
    }   // live
    part[seg][threadIdx.y][threadIdx.x] = make_float2(acca, accb);
    __syncthreads();
    if (seg == 0 && live) {
        float ta = part[0][threadIdx.y][threadIdx.x].x, tb = part[0][threadIdx.y][threadIdx.x].y;
#pragma unroll
        for (int s2 = 1; s2 < DRR_SEGS; ++s2) {       // run sums combined in run order
            ta = add_rn(ta, part[s2][threadIdx.y][threadIdx.x].x);
            tb = add_rn(tb, part[s2][threadIdx.y][threadIdx.x].y);
        }
        if (PEERS) {
            const int64_t off = ((int64_t)(g.view0 + blockIdx.z) * peers.vstride * g.rd + ua) * g.rh + v;
            const float oa = finish_ray(ta, ra, g), ob = finish_ray(tb, rb, g);
#pragma unroll
            for (int k = 0; k < LR_MAX_PEERS; ++k) {         // local buffer and the peers' (P2P stores over NVLink)
                if (k < peers.n) {
                    float *out = peers.p[k] + off;
                    out[0] = oa;
                    if (has_b) out[g.rh] = ob;
                }
            }
        } else {
            float *out = proj + ((int64_t)(g.view0 + blockIdx.z) * g.rd + ua) * g.rh + v;
            out[0] = finish_ray(ta, ra, g);
            if (has_b) out[g.rh] = finish_ray(tb, rb, g);
        }
    }
}

// Adjoint wrt the volume: every sample scatters (go*out_scale*dx) * w_tap into its 8 taps, warp-aggregated.  A plain
// per-sample scatter (RED.ADD.F32) is bound by the number of atomics reaching L2 (measured: half the atomics = half the
// time, profiles/README.md), and the 32 rays of a warp -- neighbours along detector axis 1, marching the same
// plane j -- hit heavily overlapping cells: consecutive lanes share their floor cell or sit one cell further along the
// volume's contiguous axis, so lane l's upper-x tap is lane l+1's lower-x tap.  Per plane the warp therefore
//   1. sums the 8 tap values of runs of consecutive lanes with the same floor cell into the run's first lane,
//   2. hands a run's four upper-x sums to the next run when that run's cell is the next one along x,
// and only then issues the atomics: ~22 cells x 4 rows instead of 32 x 8 per plane at cfg 1 (2.8x fewer).  Both steps are
// exact regroupings of the same sum (fp32 addition order differs, as it already does between runs of the atomics).
__global__ void __launch_bounds__(32 * DRR_ROWS)
    drr_backward_agg_kernel(const float *__restrict__ gproj, float *__restrict__ gvol, DrrDims g, DrrViews views) {
    const unsigned FULL = 0xffffffffu;
    const int lane = threadIdx.x;
    const int v = blockIdx.x * 32 + lane;
    const int u = blockIdx.y * DRR_ROWS + threadIdx.y;
    if (u >= g.rd) return;                                   // whole warp (u is warp-uniform)
    const DrrView vw = views.v[blockIdx.z];
    const bool live_ray = v < g.rh;
    const Ray r = ray_setup(vw, g, u, live_ray ? v : g.rh - 1);
    float *V = gvol + (int64_t)vw.vol * g.nvox;
    const int sy = g.h, sz = g.w * g.h;
    float go = live_ray ? gproj[((int64_t)(g.view0 + blockIdx.z) * g.rd + u) * g.rh + v] : 0.0f;
    if (g.out_scale != 1.0f) go = mul_rn(go, g.out_scale);
    const float gs = mul_rn(go, r.dx);
    const bool ray_on = live_ray && gs != 0.0f && r.j0 <= r.j1;
    const int jlo = __reduce_min_sync(FULL, ray_on ? r.j0 : 0x7fffffff);
    const int jhi = __reduce_max_sync(FULL, ray_on ? r.j1 : (int)0x80000000);
    float jf = (float)jlo;
    for (int j = jlo; j <= jhi; ++j, jf += 1.0f) {
        float val[8];
        unsigned m = 0u;
        int key = (int)0x80000000 + 2 * lane;                // dead lanes: unique, never equal or adjacent to a cell
        if (ray_on && j >= r.j0 && j <= r.j1) {
            const Sample s = ray_point(r, g, jf);
            const Taps t = make_taps(s, g);
            m = taps_mask(t, g);
            if (m != 0u) key = t.base;
#pragma unroll
            for (int c = 0; c < 8; ++c) val[c] = ((m >> c) & 1u) ? mul_rn(t.wt[c], gs) : 0.0f;
        } else {
#pragma unroll
            for (int c = 0; c < 8; ++c) val[c] = 0.0f;
        }
        if (__ballot_sync(FULL, m != 0u) == 0u) continue;     // no lane touches the volume on this plane
        // ---- runs of consecutive lanes with the same floor cell
        const int key_prev = __shfl_up_sync(FULL, key, 1);
        const bool follows = lane > 0 && m != 0u && key == key_prev;
        const unsigned long long E = (unsigned long long)__ballot_sync(FULL, follows);
        const bool leader = m != 0u && !follows;
        const int len = leader ? __ffsll((long long)~(E >> (lane + 1))) : 0;      // 1 + set bits of E right above this lane
        const int K = (int)__reduce_max_sync(FULL, (unsigned)(len > 0 ? len - 1 : 0));
        for (int k = 1; k <= K; ++k) {
            const bool take = leader && k < len;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float o = __shfl_down_sync(FULL, val[c], k);
                if (take) val[c] = add_rn(val[c], o);
            }
            const unsigned om = __shfl_down_sync(FULL, m, k);
            if (take) m |= om;
        }
        // ---- upper-x taps (odd c) of a run go to the next run when its cell is the next one along x
        const unsigned L = __ballot_sync(FULL, leader);
        const int nl = lane + len;                                               // first lane after this run
        const int key_next = __shfl_sync(FULL, key, nl & 31);
        const bool give = leader && nl < 32 && key_next == key + 1;
        const unsigned below = L & ((1u << lane) - 1u);
        const int p = below ? 31 - __clz((int)below) : 0;                        // leader of the previous run
        const int key_p = __shfl_sync(FULL, key, p);
        const int len_p = __shfl_sync(FULL, len, p);
        const unsigned m_p = __shfl_sync(FULL, m, p);
        const bool recv = leader && below != 0u && p + len_p == lane && key_p + 1 == key;
#pragma unroll
        for (int rrow = 0; rrow < 4; ++rrow) {
            const float o = __shfl_sync(FULL, val[2 * rrow + 1], p);
            if (recv) val[2 * rrow] = add_rn(val[2 * rrow], o);
        }
        if (recv) m |= (m_p >> 1) & 0x55u;
        if (give) m &= 0x55u;
        {   // predicated reductions, four row pointers with immediate +4 offsets (dead lanes: leader == false, any address)
            if (!leader) m = 0u;
            float *b0 = V + (leader ? key : 0), *b1 = b0 + sy, *b2 = b0 + sz, *b3 = b2 + sy;
            red_add_if(m & 1u, b0, val[0]);  red_add_if(m & 2u, b0 + 1, val[1]);
            red_add_if(m & 4u, b1, val[2]);  red_add_if(m & 8u, b1 + 1, val[3]);
            red_add_if(m & 16u, b2, val[4]); red_add_if(m & 32u, b2 + 1, val[5]);
            red_add_if(m & 64u, b3, val[6]); red_add_if(m & 128u, b3 + 1, val[7]);
        }
    }
}

// sdct:15-57 materialised, for API parity / bit-exactness checks only.
__global__ void __launch_bounds__(32 * DRR_ROWS)
    project_grid_kernel(float *__restrict__ grid, float *__restrict__ dx, DrrDims g, DrrViews views, int flip) {
    const int v = blockIdx.x * 32 + threadIdx.x;
    const int u = blockIdx.y * DRR_ROWS + threadIdx.y;
    if (v >= g.rh || u >= g.rd) return;
    const DrrView vw = views.v[blockIdx.z];
    const Ray r = ray_setup(vw, g, u, v);
    const int64_t ray = ((int64_t)(g.view0 + blockIdx.z) * g.rd + u) * g.rh + v;
    if (dx) dx[ray] = r.dx;
    if (!grid) return;
    for (int j = 0; j < g.w; ++j) {
        const float T = mul_rn(r.r2, sub_rn((float)j, r.sy));
        const float X = add_rn(mul_rn(r.Dx, T), r.sx), Y = add_rn(mul_rn(r.Dy, T), r.sy), Z = add_rn(mul_rn(r.Dz, T), r.sz);
        const float g0 = div_const(X, g.div_x), g1 = add_rn(div_const(Y, g.div_y), -1.0f), g2 = div_const(Z, g.div_z);
        float *o = grid + (ray * g.w + j) * 3;
        o[0] = flip ? g2 : g0; o[1] = g1; o[2] = flip ? g0 : g2;
    }
}

static int fill_dims(DrrDims &g, int B, int d, int w, int h, int n_pose_sets, int P, int rd, int rh,
                     const float spacing[3], int y_norm_mode, float out_scale) {
    LR_REQUIRE(B > 0 && d > 0 && w > 1 && h > 0 && P > 0 && rd > 0 && rh > 0,
               "drr: bad dimension (B=%d d=%d w=%d h=%d P=%d rd=%d rh=%d; w must be >= 2)", B, d, w, h, P, rd, rh);
    LR_REQUIRE(n_pose_sets == 1 || n_pose_sets == B, "drr: n_pose_sets must be 1 or B (got %d, B=%d)", n_pose_sets, B);
    LR_REQUIRE(y_norm_mode == LR_YNORM_WM1 || y_norm_mode == LR_YNORM_W, "drr: y_norm_mode must be 0 or 1");
    LR_REQUIRE(spacing != nullptr, "drr: spacing is null");
    LR_REQUIRE((rd + DRR_ROWS - 1) / DRR_ROWS <= 65535, "drr: detector too tall for the launch grid");
    LR_REQUIRE((int64_t)d * w * h < (1ll << 31) - 2ll * w * h - 4, "drr: d*w*h must fit 32-bit voxel offsets");
    g.d = d; g.w = w; g.h = h; g.rd = rd; g.rh = rh; g.view0 = 0;
    g.half_rd = (float)((double)rd / 2.0); g.half_rh = (float)((double)rh / 2.0);
    g.sp0 = spacing[0]; g.sp1 = spacing[1]; g.sp2 = spacing[2];
    g.div_x = make_const_div((float)((double)d / 2.0));
    g.div_y = make_const_div(y_norm_mode == LR_YNORM_WM1 ? (float)(((double)w - 1.0) / 2.0) : (float)((double)w / 2.0));
    g.div_z = make_const_div((float)((double)h / 2.0));
    g.hd = (float)(d - 1) / 2.0f; g.hw = (float)(w - 1) / 2.0f; g.hh = (float)(h - 1) / 2.0f;
    // |X| < d/2 + d/(d-1) is where a tap can be inside; +2 voxels of slack.  A single-plane axis (size 1) maps every
    // coordinate to index 0, so it is never clipped.
    g.lim_x = d > 1 ? (float)d / 2.0f + 2.0f + (float)d / (float)(d - 1) : 3.0e38f;
    g.lim_z = h > 1 ? (float)h / 2.0f + 2.0f + (float)h / (float)(h - 1) : 3.0e38f;
    g.out_scale = out_scale;
    g.zero = 0.0f;
    g.seg_len = (w + DRR_SEGS - 1) / DRR_SEGS;
    g.nvox = (int64_t)d * w * h;
    return LR_OK;
}

// Calls launch(n_views_in_chunk, DrrViews, view0) for chunks of the (b,p) list.
template <typename F>
static int for_each_view_chunk(const double *poses, int n_pose_sets, int B, int P, F launch) {
    const int total = B * P;
    for (int v0 = 0; v0 < total; v0 += DRR_MAX_VIEWS) {
        const int n = total - v0 < DRR_MAX_VIEWS ? total - v0 : DRR_MAX_VIEWS;
        DrrViews vs;
        for (int q = 0; q < n; ++q) {
            const int b = (v0 + q) / P, p = (v0 + q) % P;
            const double *ps = poses + ((size_t)(n_pose_sets == 1 ? 0 : b) * P + p) * 3;
            vs.v[q].sx = (float)ps[0]; vs.v[q].sy = (float)ps[1]; vs.v[q].sz = (float)ps[2];   // sdct:28 .type(float32)
            vs.v[q].vol = b;
        }
        if (int e = launch(n, vs, v0)) return e;
    }
    return LR_OK;
}

}  // namespace lr

using namespace lr;

extern "C" int lr_drr_forward(const float *vol, int B, int d, int w, int h, const double *poses, int n_pose_sets, int P,
                              int rd, int rh, const float spacing[3], int y_norm_mode, float out_scale, float *proj,
                              lr_stream_t stream) {
    LR_REQUIRE(vol && poses && proj, "drr_forward: null pointer");
    DrrDims g;
    if (int e = fill_dims(g, B, d, w, h, n_pose_sets, P, rd, rh, spacing, y_norm_mode, out_scale)) return e;
    return for_each_view_chunk(poses, n_pose_sets, B, P, [&](int n, const DrrViews &vs, int v0) {
        g.view0 = v0;
        dim3 grid((unsigned)((rh + 31) / 32), (unsigned)((rd + 2 * DRR_PAIRS - 1) / (2 * DRR_PAIRS)), (unsigned)n);
        const DrrPeers none = {};
        if (numerics_mode() == LR_NUMERICS_FAST) drr_forward_kernel<true, false><<<grid, dim3(32, DRR_PAIRS, DRR_SEGS), 0, as_stream(stream)>>>(vol, proj, g, vs, none);
        else drr_forward_kernel<false, false><<<grid, dim3(32, DRR_PAIRS, DRR_SEGS), 0, as_stream(stream)>>>(vol, proj, g, vs, none);
        return check_launch("drr_forward_kernel");
    });
}

extern "C" int lr_drr_forward_peers(const float *vol, int B, int d, int w, int h, const double *poses, int n_pose_sets, int P,
                                    int rd, int rh, const float spacing[3], int y_norm_mode, float out_scale,
                                    float *const *outs, int n_outs, int view_stride, lr_stream_t stream) {
    LR_REQUIRE(vol && poses && outs, "drr_forward_peers: null pointer");
    LR_REQUIRE(n_outs >= 1 && n_outs <= LR_MAX_PEERS, "drr_forward_peers: n_outs must be in [1, %d], got %d", LR_MAX_PEERS, n_outs);
    LR_REQUIRE(view_stride >= 1, "drr_forward_peers: view_stride must be >= 1, got %d", view_stride);
    DrrPeers peers = {};
    for (int k = 0; k < n_outs; ++k) {
        LR_REQUIRE(outs[k], "drr_forward_peers: outs[%d] is null", k);
        peers.p[k] = outs[k];
    }
    peers.n = n_outs; peers.vstride = view_stride;
    DrrDims g;
    if (int e = fill_dims(g, B, d, w, h, n_pose_sets, P, rd, rh, spacing, y_norm_mode, out_scale)) return e;
    return for_each_view_chunk(poses, n_pose_sets, B, P, [&](int n, const DrrViews &vs, int v0) {
        g.view0 = v0;
        dim3 grid((unsigned)((rh + 31) / 32), (unsigned)((rd + 2 * DRR_PAIRS - 1) / (2 * DRR_PAIRS)), (unsigned)n);
        if (numerics_mode() == LR_NUMERICS_FAST) drr_forward_kernel<true, true><<<grid, dim3(32, DRR_PAIRS, DRR_SEGS), 0, as_stream(stream)>>>(vol, nullptr, g, vs, peers);
        else drr_forward_kernel<false, true><<<grid, dim3(32, DRR_PAIRS, DRR_SEGS), 0, as_stream(stream)>>>(vol, nullptr, g, vs, peers);
        return check_launch("drr_forward_kernel<peers>");
    });
}

extern "C" int lr_drr_backward(const float *grad_proj, int B, int d, int w, int h, const double *poses, int n_pose_sets,
                               int P, int rd, int rh, const float spacing[3], int y_norm_mode, float out_scale,
                               float *grad_vol, lr_stream_t stream) {
    LR_REQUIRE(grad_proj && poses && grad_vol, "drr_backward: null pointer");
    DrrDims g;
    if (int e = fill_dims(g, B, d, w, h, n_pose_sets, P, rd, rh, spacing, y_norm_mode, out_scale)) return e;
    return for_each_view_chunk(poses, n_pose_sets, B, P, [&](int n, const DrrViews &vs, int v0) {
        g.view0 = v0;
        dim3 grid((unsigned)((rh + 31) / 32), (unsigned)((rd + DRR_ROWS - 1) / DRR_ROWS), (unsigned)n);
        drr_backward_agg_kernel<<<grid, dim3(32, DRR_ROWS), 0, as_stream(stream)>>>(grad_proj, grad_vol, g, vs);
        return check_launch("drr_backward_agg_kernel");
    });
}

extern "C" int lr_project_grid(const double *poses, int P, int rd, int rh, int d, int w, int h, const float spacing[3],
                               int y_norm_mode, int flip, float *grid, float *dx, lr_stream_t stream) {
    LR_REQUIRE(poses && (grid || dx), "project_grid: null pointer");
    DrrDims g;
    if (int e = fill_dims(g, 1, d, w, h, 1, P, rd, rh, spacing, y_norm_mode, 1.0f)) return e;
    return for_each_view_chunk(poses, 1, 1, P, [&](int n, const DrrViews &vs, int v0) {
        g.view0 = v0;
        dim3 grid_dim((unsigned)((rh + 31) / 32), (unsigned)((rd + DRR_ROWS - 1) / DRR_ROWS), (unsigned)n);
        project_grid_kernel<<<grid_dim, dim3(32, DRR_ROWS), 0, as_stream(stream)>>>(grid, dx, g, vs, flip);
        return check_launch("project_grid_kernel");
    });
}
