// Displacement-field warp (spatial transformer), forward and adjoint, for sm_100a.
//
// Replaces reference src/liftreg/utils/net_utils.py:26-56 (Bilinear.forward / forward_stn), i.e. the
// five-kernel sequence  (x+1)/2 -> zeros_like + 3 channel copies -> grid_sample_3d -> *2-1  (SURVEY.md §8 a9),
// plus, optionally, the `disp + identity_map` add of LiftRegDeformSubspaceBackproj.py:68.
//
// One thread per output voxel along W (coalesced phi reads / out writes, 128 B per warp); the 8 taps are a
// local gather served by L1/L2.  Arithmetic follows ATen's CPU grid_sampler_3d exactly: unnormalise
// ((g+1)/2)*(S-1), weights (x1-x)*(y1-y)*(z1-z) left to right, taps accumulated in the order
// tnw,tne,tsw,tse,bnw,bne,bsw,bse with separately rounded multiply and add.
#include "common.cuh"

// resident blocks per SM the two packed kernels are compiled for (register cap = 65536 / (32 * WARP_TY * n))
#ifndef LR_WARP_FWD_MINBLOCKS
#define LR_WARP_FWD_MINBLOCKS 8      // 64 registers
#endif
#ifndef LR_WARP_FWD_MINBLOCKS_FAST
#define LR_WARP_FWD_MINBLOCKS_FAST 10     // 51 registers: the single-channel lerp-form blend has fewer live values (8 blocks: 21.3 us, 10: 20.5)
#endif
#ifndef LR_WARP_BWD_MINBLOCKS
#define LR_WARP_BWD_MINBLOCKS 6      // 80 registers
#endif

namespace lr {

constexpr int WARP_TX = 32;   // threads along W (coalesced 128 B rows)
#ifndef LR_WARP_TY
#define LR_WARP_TY 4
#endif
constexpr int WARP_TY = LR_WARP_TY;    // thread rows per block (128-thread blocks: 23.1 us vs 23.9 us with 8 rows, 25.9 us with 16)
constexpr int WARP_VY = 2;    // forward: output rows per thread (y and y + WARP_TY), processed as packed fp32x2
constexpr int WARP_NZ = 4;    // forward: default consecutive planes per block (software-pipelined phi loads)
constexpr int WARP_NZ_MAX = 8;   // forward: planes per block of the long blocks (see forward_z_blocking)

struct WarpDims {
    int C, D, H, W;
    int nvox;            // D*H*W  (< 2^31: 32-bit voxel offsets; batch/channel offsets are 64-bit)
    int HW;              // H*W
    // Output slab (multi-GPU z-slab sharding): phi / out / grad_out / grad_phi hold planes [z_off, z_off+Do) of
    // axis 0 only, i.e. they are (B,*,Do,H,W) tensors; the image (and grad_img) is always the full (B,C,D,H,W).
    int Do, z_off, nvox_o;
    int zblocks;         // blocks along z per batch item: Do for the 1-plane kernels, ceil(Do / nz) for the forward
    // forward: z-blocks of a batch item come in three sizes, largest first (blocks are dispatched in index order, so
    // the last ones to start are the short ones and the tail of the launch drains quickly): n0 blocks of s0 planes,
    // then n1 of s1, then the rest of s2
    int zs0, zs1, zs2, zn0, zn1;
    unsigned z_magic;    // ceil(2^32 / zblocks): b = (blockIdx.z * z_magic) >> 32 for blockIdx.z < 65536
    float hx, hy, hz;    // (W-1)/2, (H-1)/2, (D-1)/2
    float mx, my, mz;    // W-1, H-1, D-1
    double sp0, sp1, sp2;  // 1/(D-1), 1/(H-1), 1/(W-1) as float64 (identity map, net_utils.py:81)
    float zero;          // +0.0f the compiler cannot constant-fold (see mul2_sep)
};

// net_utils.py:81-85 with numpy>=2 casting: fp32(float64(idx)*spacing) * 2 - 1
__device__ __forceinline__ float identity_coord(int idx, double spacing) {
    float v = __double2float_rn((double)idx * spacing);
    return sub_rn(mul_rn(v, 2.0f), 1.0f);
}

// Per-block identity-map table: the int->double conversions and fp64 multiplies are done by a few threads once
// instead of by every voxel (they run on the slow XU / fp64 pipes).
template <int ROWS>
struct IdentTable {
    float x[WARP_TX], y[ROWS], z;
};
template <int ROWS>
__device__ __forceinline__ void build_ident_table(IdentTable<ROWS> &t, const WarpDims &g, int x0, int y0, int z) {
    const int tid = threadIdx.y * WARP_TX + threadIdx.x;
    if (tid < WARP_TX) t.x[tid] = identity_coord(x0 + tid, g.sp2);
    else if (tid < WARP_TX + ROWS) t.y[tid - WARP_TX] = identity_coord(y0 + tid - WARP_TX, g.sp1);
    else if (tid == WARP_TX + ROWS) t.z = identity_coord(z, g.sp0);
    __syncthreads();
}

// One output voxel, any padding / mode, boundary-safe: the general path.
template <int PAD, int MODE, bool SCALE>
__device__ __forceinline__ void warp_one(const float *__restrict__ src, float *__restrict__ dst, const WarpDims &g,
                                         int nchan, float ix, float iy, float iz) {
    if (PAD == LR_PAD_ZEROS) {   // no tap is in bounds outside (-1, S): values there never matter; keeps |x| < 2^22
        ix = clamp_index(ix, g.mx + 2.0f); iy = clamp_index(iy, g.my + 2.0f); iz = clamp_index(iz, g.mz + 2.0f);
    }
    if (MODE == LR_MODE_NEAREST) {
        const int xn = rint_i(ix), yn = rint_i(iy), zn = rint_i(iz);  // nearbyint: half to even
        const bool ok = (unsigned)xn < (unsigned)g.W && (unsigned)yn < (unsigned)g.H && (unsigned)zn < (unsigned)g.D;
        const int off = zn * g.HW + yn * g.W + xn;
        for (int c = 0; c < nchan; ++c) {
            float v = 0.0f;
            if (ok) {
                v = __ldg(src + (int64_t)c * g.nvox + off);
                if (SCALE) v = mul_rn(add_rn(v, 1.0f), 0.5f);
            }
            if (SCALE) v = sub_rn(mul_rn(v, 2.0f), 1.0f);
            st_stream(dst + (int64_t)c * g.nvox_o, v);
        }
        return;
    }
    float fx, fy, fz;
    int x0, y0, z0;
    floor_fi(ix, fx, x0);
    floor_fi(iy, fy, y0);
    floor_fi(iz, fz, z0);
    const float wx1 = sub_rn(ix, fx), wx0 = sub_rn(add_rn(fx, 1.0f), ix);
    const float wy1 = sub_rn(iy, fy), wy0 = sub_rn(add_rn(fy, 1.0f), iy);
    const float wz1 = sub_rn(iz, fz), wz0 = sub_rn(add_rn(fz, 1.0f), iz);
    const float a00 = mul_rn(wx0, wy0), a10 = mul_rn(wx1, wy0), a01 = mul_rn(wx0, wy1), a11 = mul_rn(wx1, wy1);
    const float wt[8] = {mul_rn(a00, wz0), mul_rn(a10, wz0), mul_rn(a01, wz0), mul_rn(a11, wz0),
                         mul_rn(a00, wz1), mul_rn(a10, wz1), mul_rn(a01, wz1), mul_rn(a11, wz1)};
    const int base = z0 * g.HW + y0 * g.W + x0;
    // per-tap bounds test, out-of-bounds taps are skipped (ATen zeros padding; border mode never reads outside)
    const bool vx0 = (unsigned)x0 < (unsigned)g.W, vx1 = (unsigned)(x0 + 1) < (unsigned)g.W;
    const bool vy0 = (unsigned)y0 < (unsigned)g.H, vy1 = (unsigned)(y0 + 1) < (unsigned)g.H;
    const bool vz0 = (unsigned)z0 < (unsigned)g.D, vz1 = (unsigned)(z0 + 1) < (unsigned)g.D;
    const bool ok[8] = {vx0 && vy0 && vz0, vx1 && vy0 && vz0, vx0 && vy1 && vz0, vx1 && vy1 && vz0,
                        vx0 && vy0 && vz1, vx1 && vy0 && vz1, vx0 && vy1 && vz1, vx1 && vy1 && vz1};
    const int off[8] = {0, 1, g.W, g.W + 1, g.HW, g.HW + 1, g.HW + g.W, g.HW + g.W + 1};
#pragma unroll 1
    for (int c = 0; c < nchan; ++c) {
        const float *s = src + (int64_t)c * g.nvox + base;
        float acc = 0.0f;
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            if (ok[t]) {   // ATen: out += val * w, separately rounded, in tap order
                float val = __ldg(s + off[t]);
                if (SCALE) val = mul_rn(add_rn(val, 1.0f), 0.5f);   // net_utils.py:50 (img+1)/2, fused per tap
                acc = add_rn(acc, mul_rn(val, wt[t]));
            }
        }
        if (SCALE) acc = sub_rn(mul_rn(acc, 2.0f), 1.0f);           // net_utils.py:52
        st_stream(dst + (int64_t)c * g.nvox_o, acc);
    }
}

// Two output voxels a = (x, ya, z) and b = (x, yb, z) of one thread.  When all 16 taps are inside the volume (the
// common case) both trilinear evaluations run as ONE packed fp32x2 instruction stream; otherwise each voxel takes
// the scalar boundary-safe path.  gx/gy/gz hold the (already identity-corrected) map values of (a, b).
template <int PAD, int MODE, bool SCALE>
__device__ __forceinline__ void warp_pair(const float *__restrict__ src, float *__restrict__ dst, const WarpDims &g,
                                          int nchan, f32x2 gx, f32x2 gy, f32x2 gz, int voxa, int voxb, bool has_b) {
    // ATen unnormalise ((g+1)/2)*(S-1) == RN(RN(g+1) * ((S-1)/2)): /2 is exact and (S-1)/2 is representable
    const f32x2 one = splat2(1.0f);
    f32x2 ix = mul2(add2(gx, one), splat2(g.hx)), iy = mul2(add2(gy, one), splat2(g.hy)), iz = mul2(add2(gz, one), splat2(g.hz));
    float ixa, ixb, iya, iyb, iza, izb;
    unpack2(ix, ixa, ixb); unpack2(iy, iya, iyb); unpack2(iz, iza, izb);
    if (PAD == LR_PAD_BORDER) {   // clip_coordinates
        ixa = fminf(g.mx, fmaxf(ixa, 0.0f)); ixb = fminf(g.mx, fmaxf(ixb, 0.0f));
        iya = fminf(g.my, fmaxf(iya, 0.0f)); iyb = fminf(g.my, fmaxf(iyb, 0.0f));
        iza = fminf(g.mz, fmaxf(iza, 0.0f)); izb = fminf(g.mz, fmaxf(izb, 0.0f));
        ix = pack2(ixa, ixb); iy = pack2(iya, iyb); iz = pack2(iza, izb);
    }
    if (MODE == LR_MODE_LINEAR) {
        // Packed path: both y/z tap pairs inside (0 <= i < S-1) and at least one x tap inside (-1 < ix < W); NaN
        // fails the test and takes the safe path.  The x axis is the one that diverges inside a warp (lanes run
        // along x, so only the lanes next to a face leave the volume): its two taps are predicated instead.  A
        // masked tap loads 0, and 0 * w added to the running sum changes nothing -- exactly ATen's "skip".
        // The floors are taken first and the tests run on the integers: an out-of-range or NaN coordinate yields an
        // index far outside any volume (see floor_fi), so no float pre-test / clamp is needed on this path.
        f32x2 fx, fy, fz;
        int x0a, x0b, y0a, y0b, z0a, z0b;
        floor2_fi(ix, fx, x0a, x0b);
        floor2_fi(iy, fy, y0a, y0b);
        floor2_fi(iz, fz, z0a, z0b);
        const bool ina = (unsigned)(x0a + 1) < (unsigned)(g.W + 1) && (unsigned)y0a < (unsigned)(g.H - 1) && (unsigned)z0a < (unsigned)(g.D - 1);
        const bool inb = (unsigned)(x0b + 1) < (unsigned)(g.W + 1) && (unsigned)y0b < (unsigned)(g.H - 1) && (unsigned)z0b < (unsigned)(g.D - 1);
        if (ina && inb) {
            const f32x2 wx1 = sub2(ix, fx), wx0 = sub2(add2(fx, one), ix);
            const f32x2 wy1 = sub2(iy, fy), wy0 = sub2(add2(fy, one), iy);
            const f32x2 wz1 = sub2(iz, fz), wz0 = sub2(add2(fz, one), iz);
            const f32x2 a00 = mul2(wx0, wy0), a10 = mul2(wx1, wy0), a01 = mul2(wx0, wy1), a11 = mul2(wx1, wy1);
            // net_utils.py:50 samples (img+1)/2: the exact scaling by 1/2 commutes with every rounding below (no
            // underflow: weights are products of three fractions >= 2^-24), so it is applied once to the two z
            // weights instead of to each of the 8 tap values; the "+1" stays per tap.
            const f32x2 half = splat2(0.5f);
            const f32x2 wz0s = SCALE ? mul2(wz0, half) : wz0, wz1s = SCALE ? mul2(wz1, half) : wz1;
            const f32x2 wt[8] = {mul2(a00, wz0s), mul2(a10, wz0s), mul2(a01, wz0s), mul2(a11, wz0s),
                                 mul2(a00, wz1s), mul2(a10, wz1s), mul2(a01, wz1s), mul2(a11, wz1s)};
            const bool la = x0a >= 0, ha = x0a < g.W - 1, lb = x0b >= 0, hb = x0b < g.W - 1;   // x taps inside?
            // Only the lanes next to an x face ever mask a tap; when no lane of the warp does (a vote over whichever
            // lanes are here -- both variants compute the same values), the taps load unpredicated, straight into the
            // packed register pairs, without the preset constants and moves of the masked form.
            const bool all_in = __all_sync(__activemask(), la && ha && lb && hb);
            // signed 32-bit element offsets (x0 may be -1): each row pointer is one IMAD.WIDE off an opaque base
            const int a0 = z0a * g.HW + y0a * g.W + x0a, b0 = z0b * g.HW + y0b * g.W + x0b;
            const int a1 = a0 + g.W, a2 = a0 + g.HW, a3 = a2 + g.W;
            const int b1 = b0 + g.W, b2 = b0 + g.HW, b3 = b2 + g.W;
            const f32x2 two = splat2(2.0f), zero = splat2(g.zero);
#pragma unroll 1
            for (int c = 0; c < nchan; ++c) {
                const float *sc = opaque(src + (int64_t)c * g.nvox);
                const float *pa0 = sc + a0, *pa1 = sc + a1, *pa2 = sc + a2, *pa3 = sc + a3;
                const float *pb0 = sc + b0, *pb1 = sc + b1, *pb2 = sc + b2, *pb3 = sc + b3;
                f32x2 v[8];
                if (all_in) {
                    v[0] = pack2(__ldg(pa0), __ldg(pb0)); v[1] = pack2(__ldg(pa0 + 1), __ldg(pb0 + 1));
                    v[2] = pack2(__ldg(pa1), __ldg(pb1)); v[3] = pack2(__ldg(pa1 + 1), __ldg(pb1 + 1));
                    v[4] = pack2(__ldg(pa2), __ldg(pb2)); v[5] = pack2(__ldg(pa2 + 1), __ldg(pb2 + 1));
                    v[6] = pack2(__ldg(pa3), __ldg(pb3)); v[7] = pack2(__ldg(pa3 + 1), __ldg(pb3 + 1));
                } else {
// masked tap: a value whose (rescaled) intensity is exactly 0: -1 when sampling (img+1)/2, else 0
#define LR_TAP(p, ok) ((ok) ? __ldg(p) : (SCALE ? -1.0f : 0.0f))
                    v[0] = pack2(LR_TAP(pa0, la), LR_TAP(pb0, lb)); v[1] = pack2(LR_TAP(pa0 + 1, ha), LR_TAP(pb0 + 1, hb));
                    v[2] = pack2(LR_TAP(pa1, la), LR_TAP(pb1, lb)); v[3] = pack2(LR_TAP(pa1 + 1, ha), LR_TAP(pb1 + 1, hb));
                    v[4] = pack2(LR_TAP(pa2, la), LR_TAP(pb2, lb)); v[5] = pack2(LR_TAP(pa2 + 1, ha), LR_TAP(pb2 + 1, hb));
                    v[6] = pack2(LR_TAP(pa3, la), LR_TAP(pb3, lb)); v[7] = pack2(LR_TAP(pa3 + 1, ha), LR_TAP(pb3 + 1, hb));
#undef LR_TAP
                }
                // ATen: out += val * w per tap, product and sum rounded separately, in tap order (mul2_sep keeps ptxas
                // from contracting the pair into one FFMA2)
                f32x2 acc = splat2(0.0f);
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    f32x2 val = v[t];
                    if (SCALE) val = add2(val, one);               // net_utils.py:50 (img+1)/2; the /2 lives in wt[]
                    acc = add2(acc, mul2_sep(val, wt[t], zero));
                }
                if (SCALE) acc = sub2(mul2(acc, two), one);        // net_utils.py:52 (x2 is exact: fusing is harmless)
                float ra, rb;
                unpack2(acc, ra, rb);
                st_stream(dst + (int64_t)c * g.nvox_o + voxa, ra);
                if (has_b) st_stream(dst + (int64_t)c * g.nvox_o + voxb, rb);
            }
            return;
        }
    }
    warp_one<PAD, MODE, SCALE>(src, dst + voxa, g, nchan, ixa, iya, iza);
    if (has_b) warp_one<PAD, MODE, SCALE>(src, dst + voxb, g, nchan, ixb, iyb, izb);
}

// ---- fast numerics (lr_set_numerics(LR_NUMERICS_FAST), linear mode) ---------------------------------------------------
// Coordinates, floors and the three fractional weights are the same bit-exact chain as above; the 8-tap blend is
// evaluated as seven fused linear interpolations,
//     x:  c = fma(wx1, v(x0+1) - v(x0), v(x0))   (4x)      y:  fma(wy1, c(y0+1) - c(y0), c(y0))   (2x)      z: likewise (1x)
// instead of ATen's 8 separately rounded (value * weight) products and 7 sums over 12 weight products.  `using_scale`
// (sample (img+1)/2, return 2*out-1, net_utils.py:48-52) cancels exactly in real arithmetic because the weights sum to 1:
// the taps are blended as they are, and a tap that zeros padding skips (intensity 0 after the rescaling) enters as -1.
// 14 packed blend operations per voxel pair instead of 24 + 14 weight products + 2; <= 1e-6 rel-L2 from the exact mode.
template <int PAD, bool SCALE>
__device__ __forceinline__ void warp_one_fast(const float *__restrict__ src, float *__restrict__ dst, const WarpDims &g,
                                              int nchan, float ix, float iy, float iz) {
    if (PAD == LR_PAD_ZEROS) {
        ix = clamp_index(ix, g.mx + 2.0f); iy = clamp_index(iy, g.my + 2.0f); iz = clamp_index(iz, g.mz + 2.0f);
    }
    float fx, fy, fz;
    int x0, y0, z0;
    floor_fi(ix, fx, x0);
    floor_fi(iy, fy, y0);
    floor_fi(iz, fz, z0);
    const float wx1 = sub_rn(ix, fx), wy1 = sub_rn(iy, fy), wz1 = sub_rn(iz, fz);
    const int base = z0 * g.HW + y0 * g.W + x0;
    const bool vx0 = (unsigned)x0 < (unsigned)g.W, vx1 = (unsigned)(x0 + 1) < (unsigned)g.W;
    const bool vy0 = (unsigned)y0 < (unsigned)g.H, vy1 = (unsigned)(y0 + 1) < (unsigned)g.H;
    const bool vz0 = (unsigned)z0 < (unsigned)g.D, vz1 = (unsigned)(z0 + 1) < (unsigned)g.D;
    const bool ok[8] = {vx0 && vy0 && vz0, vx1 && vy0 && vz0, vx0 && vy1 && vz0, vx1 && vy1 && vz0,
                        vx0 && vy0 && vz1, vx1 && vy0 && vz1, vx0 && vy1 && vz1, vx1 && vy1 && vz1};
    const int off[8] = {0, 1, g.W, g.W + 1, g.HW, g.HW + 1, g.HW + g.W, g.HW + g.W + 1};
    const float masked = SCALE ? -1.0f : 0.0f;
#pragma unroll 1
    for (int c = 0; c < nchan; ++c) {
        const float *s = src + (int64_t)c * g.nvox + base;
        float v[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) v[t] = ok[t] ? __ldg(s + off[t]) : masked;
        const float c00 = fma_rn(wx1, sub_rn(v[1], v[0]), v[0]), c10 = fma_rn(wx1, sub_rn(v[3], v[2]), v[2]);
        const float c01 = fma_rn(wx1, sub_rn(v[5], v[4]), v[4]), c11 = fma_rn(wx1, sub_rn(v[7], v[6]), v[6]);
        const float d0 = fma_rn(wy1, sub_rn(c10, c00), c00), d1 = fma_rn(wy1, sub_rn(c11, c01), c01);
        st_stream(dst + (int64_t)c * g.nvox_o, fma_rn(wz1, sub_rn(d1, d0), d0));
    }
}

template <int PAD, bool SCALE>
__device__ __forceinline__ void warp_pair_fast(const float *__restrict__ src, float *__restrict__ dst, const WarpDims &g,
                                               int nchan, f32x2 gx, f32x2 gy, f32x2 gz, int voxa, int voxb, bool has_b) {
    const f32x2 one = splat2(1.0f);
    f32x2 ix = mul2(add2(gx, one), splat2(g.hx)), iy = mul2(add2(gy, one), splat2(g.hy)), iz = mul2(add2(gz, one), splat2(g.hz));
    if (PAD == LR_PAD_BORDER) {   // clip_coordinates
        float ixa, ixb, iya, iyb, iza, izb;
        unpack2(ix, ixa, ixb); unpack2(iy, iya, iyb); unpack2(iz, iza, izb);
        ixa = fminf(g.mx, fmaxf(ixa, 0.0f)); ixb = fminf(g.mx, fmaxf(ixb, 0.0f));
        iya = fminf(g.my, fmaxf(iya, 0.0f)); iyb = fminf(g.my, fmaxf(iyb, 0.0f));
        iza = fminf(g.mz, fmaxf(iza, 0.0f)); izb = fminf(g.mz, fmaxf(izb, 0.0f));
        ix = pack2(ixa, ixb); iy = pack2(iya, iyb); iz = pack2(iza, izb);
    }
    f32x2 fx, fy, fz;
    int x0a, x0b, y0a, y0b, z0a, z0b;
    floor2_fi(ix, fx, x0a, x0b);
    floor2_fi(iy, fy, y0a, y0b);
    floor2_fi(iz, fz, z0a, z0b);
    // packed path: both y/z tap pairs inside and at least one x tap inside (as warp_pair); NaN / far-out coordinates
    // floor to indices outside any volume and take the scalar path.  (Masking the y / z faces here as well, so that the
    // ~8 % of voxel pairs on the faces and the displaced rim stay on the packed path, was measured slower: forward 20.8
    // vs 20.5 us, d/dphi 33.5 vs 31.9 us -- the twelve extra predicates cost the interior pairs more than the scalar path
    // costs the rim.)
    const bool ina = (unsigned)(x0a + 1) < (unsigned)(g.W + 1) && (unsigned)y0a < (unsigned)(g.H - 1) && (unsigned)z0a < (unsigned)(g.D - 1);
    const bool inb = (unsigned)(x0b + 1) < (unsigned)(g.W + 1) && (unsigned)y0b < (unsigned)(g.H - 1) && (unsigned)z0b < (unsigned)(g.D - 1);
    if (ina && inb) {
        const f32x2 wx1 = sub2(ix, fx), wy1 = sub2(iy, fy), wz1 = sub2(iz, fz);
        const bool la = x0a >= 0, ha = x0a < g.W - 1, lb = x0b >= 0, hb = x0b < g.W - 1;   // x taps inside?
        const bool all_in = __all_sync(__activemask(), la && ha && lb && hb);
        const int a0 = z0a * g.HW + y0a * g.W + x0a, b0 = z0b * g.HW + y0b * g.W + x0b;
        const int a1 = a0 + g.W, a2 = a0 + g.HW, a3 = a2 + g.W;
        const int b1 = b0 + g.W, b2 = b0 + g.HW, b3 = b2 + g.W;
#pragma unroll 1
        for (int c = 0; c < nchan; ++c) {
            const float *sc = opaque(src + (int64_t)c * g.nvox);
            const float *pa0 = sc + a0, *pa1 = sc + a1, *pa2 = sc + a2, *pa3 = sc + a3;
            const float *pb0 = sc + b0, *pb1 = sc + b1, *pb2 = sc + b2, *pb3 = sc + b3;
            f32x2 v[8];
            if (all_in) {
                v[0] = pack2(__ldg(pa0), __ldg(pb0)); v[1] = pack2(__ldg(pa0 + 1), __ldg(pb0 + 1));
                v[2] = pack2(__ldg(pa1), __ldg(pb1)); v[3] = pack2(__ldg(pa1 + 1), __ldg(pb1 + 1));
                v[4] = pack2(__ldg(pa2), __ldg(pb2)); v[5] = pack2(__ldg(pa2 + 1), __ldg(pb2 + 1));
                v[6] = pack2(__ldg(pa3), __ldg(pb3)); v[7] = pack2(__ldg(pa3 + 1), __ldg(pb3 + 1));
            } else {
#define LR_TAP(p, ok) ((ok) ? __ldg(p) : (SCALE ? -1.0f : 0.0f))
                v[0] = pack2(LR_TAP(pa0, la), LR_TAP(pb0, lb)); v[1] = pack2(LR_TAP(pa0 + 1, ha), LR_TAP(pb0 + 1, hb));
                v[2] = pack2(LR_TAP(pa1, la), LR_TAP(pb1, lb)); v[3] = pack2(LR_TAP(pa1 + 1, ha), LR_TAP(pb1 + 1, hb));
                v[4] = pack2(LR_TAP(pa2, la), LR_TAP(pb2, lb)); v[5] = pack2(LR_TAP(pa2 + 1, ha), LR_TAP(pb2 + 1, hb));
                v[6] = pack2(LR_TAP(pa3, la), LR_TAP(pb3, lb)); v[7] = pack2(LR_TAP(pa3 + 1, ha), LR_TAP(pb3 + 1, hb));
#undef LR_TAP
            }
            const f32x2 c00 = fma2(wx1, sub2(v[1], v[0]), v[0]), c10 = fma2(wx1, sub2(v[3], v[2]), v[2]);
            const f32x2 c01 = fma2(wx1, sub2(v[5], v[4]), v[4]), c11 = fma2(wx1, sub2(v[7], v[6]), v[6]);
            const f32x2 d0 = fma2(wy1, sub2(c10, c00), c00), d1 = fma2(wy1, sub2(c11, c01), c01);
            float ra, rb;
            unpack2(fma2(wz1, sub2(d1, d0), d0), ra, rb);
            st_stream(dst + (int64_t)c * g.nvox_o + voxa, ra);
            if (has_b) st_stream(dst + (int64_t)c * g.nvox_o + voxb, rb);
        }
        return;
    }
    float ixa, ixb, iya, iyb, iza, izb;
    unpack2(ix, ixa, ixb); unpack2(iy, iya, iyb); unpack2(iz, iza, izb);
    warp_one_fast<PAD, SCALE>(src, dst + voxa, g, nchan, ixa, iya, iza);
    if (has_b) warp_one_fast<PAD, SCALE>(src, dst + voxb, g, nchan, ixb, iyb, izb);
}

// Forward kernel.  Thread (tx, ty) of block (bx, by, bz) owns output voxels (x, y, z) and (x, y + WARP_TY, z) for
// a run of consecutive planes z (8, 4 or 2: forward_z_blocking).  The map values of plane z+1 are fetched into registers before plane z is
// processed, so the HBM latency of the phi stream (the only compulsory traffic besides the store) is hidden behind a
// whole plane of arithmetic instead of being exposed once per voxel.
template <int PAD, int MODE, bool SCALE, bool IDENT, bool C1, bool FAST>
__global__ void __launch_bounds__(WARP_TX * WARP_TY, (FAST && C1 && MODE == LR_MODE_LINEAR) ? LR_WARP_FWD_MINBLOCKS_FAST : LR_WARP_FWD_MINBLOCKS)
    warp_forward_kernel(const float *__restrict__ img, const float *__restrict__ phi, float *__restrict__ out, WarpDims g) {
    __shared__ IdentTable<WARP_TY * WARP_VY> ident;
    __shared__ float ident_z[WARP_NZ_MAX];
    const int x = blockIdx.x * WARP_TX + threadIdx.x;
    const int ya = blockIdx.y * (WARP_TY * WARP_VY) + threadIdx.y;
    const int b = g.zblocks == 1 ? (int)blockIdx.z : (int)__umulhi(blockIdx.z, g.z_magic);   // 2^32/1 does not fit the magic
    const int zb = blockIdx.z - b * g.zblocks;
    int z_first, zsize;                                             // first plane (inside the output slab) of this block
    if (zb < g.zn0) { z_first = zb * g.zs0; zsize = g.zs0; }
    else if (zb < g.zn0 + g.zn1) { z_first = g.zn0 * g.zs0 + (zb - g.zn0) * g.zs1; zsize = g.zs1; }
    else { z_first = g.zn0 * g.zs0 + g.zn1 * g.zs1 + (zb - g.zn0 - g.zn1) * g.zs2; zsize = g.zs2; }
    const int nz = min(zsize, g.Do - z_first);
    if (IDENT) {
        if (threadIdx.y == 0 && threadIdx.x < nz) ident_z[threadIdx.x] = identity_coord(z_first + threadIdx.x + g.z_off, g.sp0);
        build_ident_table(ident, g, blockIdx.x * WARP_TX, blockIdx.y * (WARP_TY * WARP_VY), 0);
    }
    if (x >= g.W || ya >= g.H) return;
    const bool has_b = ya + WARP_TY < g.H;                     // second voxel exists (else: computed on row ya, not stored)
    const int yb = has_b ? ya + WARP_TY : ya;
    int voxa = z_first * g.HW + ya * g.W + x, voxb = z_first * g.HW + yb * g.W + x;

    // channel c of phi addresses volume axis c; grid_sample's x is the last axis (net_utils.py:27-30)
    const float *p0 = opaque(phi + (int64_t)b * 3 * g.nvox_o);
    const float *p1 = opaque(p0 + g.nvox_o);
    const float *p2 = opaque(p1 + g.nvox_o);
    const int nchan = C1 ? 1 : g.C;   // C == 1 (the moving CT, label maps) gets a loop-free instantiation
    const float *src = opaque(img + (int64_t)b * nchan * g.nvox);
    float *dst = opaque(out + (int64_t)b * nchan * g.nvox_o);
    f32x2 idx = 0, idy = 0;
    if (IDENT) {  // LiftRegDeformSubspaceBackproj.py:68  deform_field = disp_field + id_transform
        idx = splat2(ident.x[threadIdx.x]);
        idy = pack2(ident.y[threadIdx.y], ident.y[has_b ? threadIdx.y + WARP_TY : threadIdx.y]);
    }

    float cza = ld_stream(p0 + (unsigned)voxa), cya = ld_stream(p1 + (unsigned)voxa), cxa = ld_stream(p2 + (unsigned)voxa);
    float czb = ld_stream(p0 + (unsigned)voxb), cyb = ld_stream(p1 + (unsigned)voxb), cxb = ld_stream(p2 + (unsigned)voxb);
#pragma unroll 1
    for (int zi = 0; zi < nz; ++zi) {
        float nza = 0.f, nya = 0.f, nxa = 0.f, nzb = 0.f, nyb = 0.f, nxb = 0.f;
        if (zi + 1 < nz) {   // prefetch the next plane's map values
            const unsigned na = (unsigned)(voxa + g.HW), nb = (unsigned)(voxb + g.HW);
            nza = ld_stream(p0 + na); nya = ld_stream(p1 + na); nxa = ld_stream(p2 + na);
            nzb = ld_stream(p0 + nb); nyb = ld_stream(p1 + nb); nxb = ld_stream(p2 + nb);
        }
        f32x2 gx = pack2(cxa, cxb), gy = pack2(cya, cyb), gz = pack2(cza, czb);
        if (IDENT) {
            gz = add2(gz, splat2(ident_z[zi]));
            gy = add2(gy, idy);
            gx = add2(gx, idx);
        }
        if (FAST && MODE == LR_MODE_LINEAR) warp_pair_fast<PAD, SCALE>(src, dst, g, nchan, gx, gy, gz, voxa, voxb, has_b);
        else warp_pair<PAD, MODE, SCALE>(src, dst, g, nchan, gx, gy, gz, voxa, voxb, has_b);
        cza = nza; cya = nya; cxa = nxa; czb = nzb; cyb = nyb; cxb = nxb;
        voxa += g.HW; voxb += g.HW;
    }
}

// Adjoint.  grad_phi is a per-voxel gather (no atomics); grad_img is a scatter (RED.ADD.F32).
// Follows ATen grid_sampler_3d_backward: gix -= tnw_val*(y1-y)*(z1-z)*gOut ... ; grad_grid = (S-1)/2 * gi,
// zeroed where a border-clipped coordinate is outside (clip_coordinates_set_grad).
template <int PAD, bool SCALE, bool IDENT>
__global__ void __launch_bounds__(WARP_TX * WARP_TY)
    warp_backward_kernel(const float *__restrict__ gout, const float *__restrict__ img, const float *__restrict__ phi,
                         float *__restrict__ gimg, float *__restrict__ gphi, WarpDims g) {
    __shared__ IdentTable<WARP_TY> ident;
    const int x = blockIdx.x * WARP_TX + threadIdx.x;
    const int y = blockIdx.y * WARP_TY + threadIdx.y;
    const int b = g.zblocks == 1 ? (int)blockIdx.z : (int)__umulhi(blockIdx.z, g.z_magic);   // 2^32/1 does not fit the magic
    const int z = blockIdx.z - b * g.Do;
    if (IDENT) build_ident_table(ident, g, blockIdx.x * WARP_TX, blockIdx.y * WARP_TY, z + g.z_off);
    if (x >= g.W || y >= g.H) return;
    const int vox = z * g.HW + y * g.W + x;

    const float *phi_b = phi + (int64_t)b * 3 * g.nvox_o + vox;
    float gz = ld_stream(phi_b), gy = ld_stream(phi_b + g.nvox_o), gx = ld_stream(phi_b + 2 * (int64_t)g.nvox_o);
    if (IDENT) {
        gz = add_rn(gz, ident.z);
        gy = add_rn(gy, ident.y[threadIdx.y]);
        gx = add_rn(gx, ident.x[threadIdx.x]);
    }
    float ix = mul_rn(add_rn(gx, 1.0f), g.hx), iy = mul_rn(add_rn(gy, 1.0f), g.hy), iz = mul_rn(add_rn(gz, 1.0f), g.hz);
    float mx = g.hx, my = g.hy, mz = g.hz;
    if (PAD == LR_PAD_BORDER) {
        if (ix <= 0.0f) { ix = 0.0f; mx = 0.0f; } else if (ix >= g.mx) { ix = g.mx; mx = 0.0f; }
        if (iy <= 0.0f) { iy = 0.0f; my = 0.0f; } else if (iy >= g.my) { iy = g.my; my = 0.0f; }
        if (iz <= 0.0f) { iz = 0.0f; mz = 0.0f; } else if (iz >= g.mz) { iz = g.mz; mz = 0.0f; }
    } else {
        ix = clamp_index(ix, g.mx + 2.0f); iy = clamp_index(iy, g.my + 2.0f); iz = clamp_index(iz, g.mz + 2.0f);
    }
    float fx, fy, fz;
    int x0, y0, z0;
    floor_fi(ix, fx, x0);
    floor_fi(iy, fy, y0);
    floor_fi(iz, fz, z0);
    const float wx[2] = {sub_rn(add_rn(fx, 1.0f), ix), sub_rn(ix, fx)};
    const float wy[2] = {sub_rn(add_rn(fy, 1.0f), iy), sub_rn(iy, fy)};
    const float wz[2] = {sub_rn(add_rn(fz, 1.0f), iz), sub_rn(iz, fz)};
    const int base = z0 * g.HW + y0 * g.W + x0;

    float gix = 0.0f, giy = 0.0f, giz = 0.0f;
    for (int c = 0; c < g.C; ++c) {
        const int64_t chan = ((int64_t)b * g.C + c) * g.nvox;
        float go = ld_stream(gout + ((int64_t)b * g.C + c) * g.nvox_o + vox);
        if (SCALE) go = mul_rn(go, 2.0f);
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int tx = t & 1, ty = (t >> 1) & 1, tz = t >> 2;
            const bool ok = (unsigned)(x0 + tx) < (unsigned)g.W && (unsigned)(y0 + ty) < (unsigned)g.H &&
                            (unsigned)(z0 + tz) < (unsigned)g.D;
            if (!ok) continue;
            const int64_t o = chan + base + tx + ty * g.W + tz * g.HW;
            if (gimg) {
                float wv = mul_rn(mul_rn(mul_rn(wx[tx], wy[ty]), wz[tz]), go);
                red_add(gimg + o, SCALE ? mul_rn(wv, 0.5f) : wv);
            }
            if (gphi) {
                float val = __ldg(img + o);
                if (SCALE) val = mul_rn(add_rn(val, 1.0f), 0.5f);
                const float tx_ = mul_rn(mul_rn(mul_rn(val, wy[ty]), wz[tz]), go);
                const float ty_ = mul_rn(mul_rn(mul_rn(val, wx[tx]), wz[tz]), go);
                const float tz_ = mul_rn(mul_rn(mul_rn(val, wx[tx]), wy[ty]), go);
                gix = tx ? add_rn(gix, tx_) : sub_rn(gix, tx_);
                giy = ty ? add_rn(giy, ty_) : sub_rn(giy, ty_);
                giz = tz ? add_rn(giz, tz_) : sub_rn(giz, tz_);
            }
        }
    }
    if (gphi) {
        float *gp = gphi + (int64_t)b * 3 * g.nvox_o + vox;
        st_stream(gp, mul_rn(mz, giz));
        st_stream(gp + g.nvox_o, mul_rn(my, giy));
        st_stream(gp + 2 * (int64_t)g.nvox_o, mul_rn(mx, gix));
    }
}

// d(warp)/d(phi) only, zeros padding: what a training step needs (the moving image is data, model :69).  Same
// two-voxels-per-thread packed layout as the forward kernel.  The gradient is a gather, so it is deterministic; it is
// evaluated as a tree of fused lerps over tap differences (24 packed operations for the three components), which
// differs from ATen's expression order by fp32 round-off only (tests: <= 2e-5 rel-L2).
template <bool SCALE>
__device__ __forceinline__ void warp_bwd_phi_one(const float *__restrict__ gout_b, const float *__restrict__ img_b,
                                                 float *__restrict__ gp, const WarpDims &g, int vox, float ix, float iy,
                                                 float iz) {
    ix = clamp_index(ix, g.mx + 2.0f); iy = clamp_index(iy, g.my + 2.0f); iz = clamp_index(iz, g.mz + 2.0f);
    float fx, fy, fz;
    int x0, y0, z0;
    floor_fi(ix, fx, x0);
    floor_fi(iy, fy, y0);
    floor_fi(iz, fz, z0);
    const float wx[2] = {sub_rn(add_rn(fx, 1.0f), ix), sub_rn(ix, fx)};
    const float wy[2] = {sub_rn(add_rn(fy, 1.0f), iy), sub_rn(iy, fy)};
    const float wz[2] = {sub_rn(add_rn(fz, 1.0f), iz), sub_rn(iz, fz)};
    const int base = z0 * g.HW + y0 * g.W + x0;
    float gix = 0.0f, giy = 0.0f, giz = 0.0f;
    for (int c = 0; c < g.C; ++c) {
        float go = ld_stream(gout_b + (int64_t)c * g.nvox_o + vox);
        if (SCALE) go = mul_rn(go, 2.0f);
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int tx = t & 1, ty = (t >> 1) & 1, tz = t >> 2;
            const bool ok = (unsigned)(x0 + tx) < (unsigned)g.W && (unsigned)(y0 + ty) < (unsigned)g.H &&
                            (unsigned)(z0 + tz) < (unsigned)g.D;
            if (!ok) continue;
            float val = __ldg(img_b + (int64_t)c * g.nvox + base + tx + ty * g.W + tz * g.HW);
            if (SCALE) val = mul_rn(add_rn(val, 1.0f), 0.5f);
            const float tx_ = mul_rn(mul_rn(mul_rn(val, wy[ty]), wz[tz]), go);
            const float ty_ = mul_rn(mul_rn(mul_rn(val, wx[tx]), wz[tz]), go);
            const float tz_ = mul_rn(mul_rn(mul_rn(val, wx[tx]), wy[ty]), go);
            gix = tx ? add_rn(gix, tx_) : sub_rn(gix, tx_);
            giy = ty ? add_rn(giy, ty_) : sub_rn(giy, ty_);
            giz = tz ? add_rn(giz, tz_) : sub_rn(giz, tz_);
        }
    }
    st_stream(gp + vox, mul_rn(g.hz, giz));
    st_stream(gp + g.nvox_o + vox, mul_rn(g.hy, giy));
    st_stream(gp + 2 * (int64_t)g.nvox_o + vox, mul_rn(g.hx, gix));
}

// One plane of d/dphi for the thread's two voxels; gz/gy/gx are the (identity-corrected) map values of (a, b).
template <bool SCALE, bool C1>
__device__ __forceinline__ void warp_bwd_phi_pair(const float *__restrict__ gout_b, const float *__restrict__ img_b,
                                                  float *__restrict__ gp, const WarpDims &g, f32x2 gx, f32x2 gy, f32x2 gz,
                                                  int voxa, int voxb, bool has_b, f32x2 go_c1) {
    const f32x2 one = splat2(1.0f);
    const f32x2 ix = mul2(add2(gx, one), splat2(g.hx)), iy = mul2(add2(gy, one), splat2(g.hy)), iz = mul2(add2(gz, one), splat2(g.hz));

    f32x2 fx, fy, fz;
    int x0a, x0b, y0a, y0b, z0a, z0b;
    floor2_fi(ix, fx, x0a, x0b);
    floor2_fi(iy, fy, y0a, y0b);
    floor2_fi(iz, fz, z0a, z0b);
    // packed path: y/z tap pairs inside, at least one x tap inside (the x taps are predicated: lanes run along x, so
    // the faces x = 0 / W-1 are where a warp would otherwise diverge); a masked tap reads as intensity 0 = skipped
    const bool ina = (unsigned)(x0a + 1) < (unsigned)(g.W + 1) && (unsigned)y0a < (unsigned)(g.H - 1) && (unsigned)z0a < (unsigned)(g.D - 1);
    const bool inb = (unsigned)(x0b + 1) < (unsigned)(g.W + 1) && (unsigned)y0b < (unsigned)(g.H - 1) && (unsigned)z0b < (unsigned)(g.D - 1);
    if (!(ina && inb)) {
        float ixa, ixb, iya, iyb, iza, izb;
        unpack2(ix, ixa, ixb); unpack2(iy, iya, iyb); unpack2(iz, iza, izb);
        warp_bwd_phi_one<SCALE>(gout_b, img_b, gp, g, voxa, ixa, iya, iza);
        if (has_b) warp_bwd_phi_one<SCALE>(gout_b, img_b, gp, g, voxb, ixb, iyb, izb);
        return;
    }
    const f32x2 wx1 = sub2(ix, fx), wy1 = sub2(iy, fy), wz1 = sub2(iz, fz);
    const bool la = x0a >= 0, ha = x0a < g.W - 1, lb = x0b >= 0, hb = x0b < g.W - 1;   // x taps inside?
    const bool all_in = __all_sync(__activemask(), la && ha && lb && hb);                 // no lane masks a tap: plain loads
    const int a0 = z0a * g.HW + y0a * g.W + x0a, b0 = z0b * g.HW + y0b * g.W + x0b;      // signed: x0 may be -1
    const int a1 = a0 + g.W, a2 = a0 + g.HW, a3 = a2 + g.W;
    const int b1 = b0 + g.W, b2 = b0 + g.HW, b3 = b2 + g.W;
    f32x2 gix = splat2(0.0f), giy = splat2(0.0f), giz = splat2(0.0f);
#pragma unroll 1
    const int nchan = C1 ? 1 : g.C;
    for (int c = 0; c < nchan; ++c) {
        const float *sc = opaque(img_b + (int64_t)c * g.nvox);
        const float *goc = gout_b + (int64_t)c * g.nvox_o;
        // SCALE: d/dphi of 2*sample((img+1)/2) - 1.  The exact scalings by 2 (grad_out) and 1/2 (tap values) cancel, and
        // so does the "+1": the derivatives of the eight weights sum to zero.  The taps are used as they are; a tap that
        // zeros padding skips has rescaled intensity 0, i.e. enters as -1.
        // (single-channel images: grad_out of this plane was prefetched by the caller together with the map)
        const f32x2 go = C1 ? go_c1 : pack2(ld_stream(goc + (unsigned)voxa), ld_stream(goc + (unsigned)voxb));
        const float *pa0 = sc + a0, *pa1 = sc + a1, *pa2 = sc + a2, *pa3 = sc + a3;
        const float *pb0 = sc + b0, *pb1 = sc + b1, *pb2 = sc + b2, *pb3 = sc + b3;
        f32x2 v[8];     // tap index t = tx + 2 ty + 4 tz
        if (all_in) {
            v[0] = pack2(__ldg(pa0), __ldg(pb0)); v[1] = pack2(__ldg(pa0 + 1), __ldg(pb0 + 1));
            v[2] = pack2(__ldg(pa1), __ldg(pb1)); v[3] = pack2(__ldg(pa1 + 1), __ldg(pb1 + 1));
            v[4] = pack2(__ldg(pa2), __ldg(pb2)); v[5] = pack2(__ldg(pa2 + 1), __ldg(pb2 + 1));
            v[6] = pack2(__ldg(pa3), __ldg(pb3)); v[7] = pack2(__ldg(pa3 + 1), __ldg(pb3 + 1));
        } else {
#define LR_TAP(p, ok) ((ok) ? __ldg(p) : (SCALE ? -1.0f : 0.0f))
            v[0] = pack2(LR_TAP(pa0, la), LR_TAP(pb0, lb)); v[1] = pack2(LR_TAP(pa0 + 1, ha), LR_TAP(pb0 + 1, hb));
            v[2] = pack2(LR_TAP(pa1, la), LR_TAP(pb1, lb)); v[3] = pack2(LR_TAP(pa1 + 1, ha), LR_TAP(pb1 + 1, hb));
            v[4] = pack2(LR_TAP(pa2, la), LR_TAP(pb2, lb)); v[5] = pack2(LR_TAP(pa2 + 1, ha), LR_TAP(pb2 + 1, hb));
            v[6] = pack2(LR_TAP(pa3, la), LR_TAP(pb3, lb)); v[7] = pack2(LR_TAP(pa3 + 1, ha), LR_TAP(pb3 + 1, hb));
#undef LR_TAP
        }
        // The trilinear interpolant and its three partial derivatives as a tree of fused lerps (24 packed operations):
        //   e = x-differences of the four (y,z) rows, c = x-lerps;  d/dx = lerp_z(lerp_y(e));
        //   f = y-differences of c;  d/dy = lerp_z(f);  d/dz = lerp_y(c)(z1) - lerp_y(c)(z0)
        const f32x2 e00 = sub2(v[1], v[0]), e10 = sub2(v[3], v[2]), e01 = sub2(v[5], v[4]), e11 = sub2(v[7], v[6]);
        const f32x2 c00 = fma2(wx1, e00, v[0]), c10 = fma2(wx1, e10, v[2]), c01 = fma2(wx1, e01, v[4]), c11 = fma2(wx1, e11, v[6]);
        const f32x2 ex0 = fma2(wy1, sub2(e10, e00), e00), ex1 = fma2(wy1, sub2(e11, e01), e01);
        const f32x2 f0 = sub2(c10, c00), f1 = sub2(c11, c01);
        const f32x2 d0 = fma2(wy1, f0, c00), d1 = fma2(wy1, f1, c01);
        gix = fma2(go, fma2(wz1, sub2(ex1, ex0), ex0), gix);
        giy = fma2(go, fma2(wz1, sub2(f1, f0), f0), giy);
        giz = fma2(go, sub2(d1, d0), giz);
    }
    float ra, rb;
    unpack2(mul2(splat2(g.hz), giz), ra, rb);
    st_stream(gp + (unsigned)voxa, ra); if (has_b) st_stream(gp + (unsigned)voxb, rb);
    unpack2(mul2(splat2(g.hy), giy), ra, rb);
    st_stream(gp + g.nvox_o + voxa, ra); if (has_b) st_stream(gp + g.nvox_o + voxb, rb);
    unpack2(mul2(splat2(g.hx), gix), ra, rb);
    st_stream(gp + 2 * (int64_t)g.nvox_o + voxa, ra); if (has_b) st_stream(gp + 2 * (int64_t)g.nvox_o + voxb, rb);
}

// Same block shape and tapered z-blocking as the forward kernel: a run of consecutive planes per block, the map
// values of plane z+1 fetched into registers before plane z is evaluated.  (With one plane per block the map and
// grad_out loads sat at the head of every block with nothing to hide them: ncu long-scoreboard 7.3 warps per issue.)
template <bool SCALE, bool IDENT, bool C1>
__global__ void __launch_bounds__(WARP_TX * WARP_TY, LR_WARP_BWD_MINBLOCKS)
    warp_backward_phi_kernel(const float *__restrict__ gout, const float *__restrict__ img, const float *__restrict__ phi,
                             float *__restrict__ gphi, WarpDims g) {
    __shared__ IdentTable<WARP_TY * WARP_VY> ident;
    __shared__ float ident_z[WARP_NZ_MAX];
    const int x = blockIdx.x * WARP_TX + threadIdx.x;
    const int ya = blockIdx.y * (WARP_TY * WARP_VY) + threadIdx.y;
    const int b = g.zblocks == 1 ? (int)blockIdx.z : (int)__umulhi(blockIdx.z, g.z_magic);
    const int zb = blockIdx.z - b * g.zblocks;
    int z_first, zsize;
    if (zb < g.zn0) { z_first = zb * g.zs0; zsize = g.zs0; }
    else if (zb < g.zn0 + g.zn1) { z_first = g.zn0 * g.zs0 + (zb - g.zn0) * g.zs1; zsize = g.zs1; }
    else { z_first = g.zn0 * g.zs0 + g.zn1 * g.zs1 + (zb - g.zn0 - g.zn1) * g.zs2; zsize = g.zs2; }
    const int nz = min(zsize, g.Do - z_first);
    if (IDENT) {
        if (threadIdx.y == 0 && threadIdx.x < nz) ident_z[threadIdx.x] = identity_coord(z_first + threadIdx.x + g.z_off, g.sp0);
        build_ident_table(ident, g, blockIdx.x * WARP_TX, blockIdx.y * (WARP_TY * WARP_VY), 0);
    }
    if (x >= g.W || ya >= g.H) return;
    const bool has_b = ya + WARP_TY < g.H;
    const int yb = has_b ? ya + WARP_TY : ya;
    int voxa = z_first * g.HW + ya * g.W + x, voxb = z_first * g.HW + yb * g.W + x;

    const float *p0 = opaque(phi + (int64_t)b * 3 * g.nvox_o);
    const float *p1 = opaque(p0 + g.nvox_o);
    const float *p2 = opaque(p1 + g.nvox_o);
    const float *gout_b = opaque(gout + (int64_t)b * g.C * g.nvox_o);
    const float *img_b = opaque(img + (int64_t)b * g.C * g.nvox);
    float *gp = opaque(gphi + (int64_t)b * 3 * g.nvox_o);
    f32x2 idx = 0, idy = 0;
    if (IDENT) {
        idx = splat2(ident.x[threadIdx.x]);
        idy = pack2(ident.y[threadIdx.y], ident.y[has_b ? threadIdx.y + WARP_TY : threadIdx.y]);
    }
    float cza = ld_stream(p0 + (unsigned)voxa), cya = ld_stream(p1 + (unsigned)voxa), cxa = ld_stream(p2 + (unsigned)voxa);
    float czb = ld_stream(p0 + (unsigned)voxb), cyb = ld_stream(p1 + (unsigned)voxb), cxb = ld_stream(p2 + (unsigned)voxb);
    float cga = 0.f, cgb = 0.f;      // grad_out of the current plane (single-channel images only)
    if (C1) { cga = ld_stream(gout_b + (unsigned)voxa); cgb = ld_stream(gout_b + (unsigned)voxb); }
#pragma unroll 1
    for (int zi = 0; zi < nz; ++zi) {
        float nza = 0.f, nya = 0.f, nxa = 0.f, nzb = 0.f, nyb = 0.f, nxb = 0.f, nga = 0.f, ngb = 0.f;
        if (zi + 1 < nz) {   // prefetch the next plane's map values (and grad_out: it comes from HBM like the map)
            const unsigned na = (unsigned)(voxa + g.HW), nb = (unsigned)(voxb + g.HW);
            nza = ld_stream(p0 + na); nya = ld_stream(p1 + na); nxa = ld_stream(p2 + na);
            nzb = ld_stream(p0 + nb); nyb = ld_stream(p1 + nb); nxb = ld_stream(p2 + nb);
            if (C1) { nga = ld_stream(gout_b + na); ngb = ld_stream(gout_b + nb); }
        }
        f32x2 gx = pack2(cxa, cxb), gy = pack2(cya, cyb), gz = pack2(cza, czb);
        if (IDENT) {
            gz = add2(gz, splat2(ident_z[zi]));
            gy = add2(gy, idy);
            gx = add2(gx, idx);
        }
        warp_bwd_phi_pair<SCALE, C1>(gout_b, img_b, gp, g, gx, gy, gz, voxa, voxb, has_b, pack2(cga, cgb));
        cza = nza; cya = nya; cxa = nxa; czb = nzb; cyb = nyb; cxb = nxb; cga = nga; cgb = ngb;
        voxa += g.HW; voxb += g.HW;
    }
}

constexpr int IDENT_PLANES = 8;
__global__ void __launch_bounds__(WARP_TX * WARP_TY) identity_map_kernel(float *__restrict__ out, WarpDims g) {
    __shared__ IdentTable<WARP_TY> ident;
    const int x = blockIdx.x * WARP_TX + threadIdx.x;
    const int y = blockIdx.y * WARP_TY + threadIdx.y;
    build_ident_table(ident, g, blockIdx.x * WARP_TX, blockIdx.y * WARP_TY, 0);      // x / y tables once per block
    if (x >= g.W || y >= g.H) return;
    const float cy = ident.y[threadIdx.y], cx = ident.x[threadIdx.x];
    const int z_end = min(g.D, ((int)blockIdx.z + 1) * IDENT_PLANES);
    for (int z = blockIdx.z * IDENT_PLANES; z < z_end; ++z) {                         // a run of planes per block: 1.5 KB per block
        const int vox = z * g.HW + y * g.W + x;                                       // and plane was mostly launch overhead
        st_stream(out + vox, identity_coord(z, g.sp0));
        st_stream(out + (int64_t)g.nvox + vox, cy);
        st_stream(out + 2 * (int64_t)g.nvox + vox, cx);
    }
}

__device__ __forceinline__ float atten_one(float hu, ConstDiv k1000) {
    const float v = fmaxf(hu, -1000.0f);                                      // sdct:8
    return mul_rn(div_const(add_rn(v, 1000.0f), k1000), 0.2f);                // sdct:9 (division by a constant: bit-identical to IEEE)
}

// n4 float4 groups (16-byte-aligned pointers) + a scalar tail
__global__ void __launch_bounds__(256) atten_coef_kernel(const float *__restrict__ hu, float *__restrict__ mu, int64_t n, int64_t n4, ConstDiv k1000) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i = t; i < n4; i += stride) {
        float4 v = ld_stream4(reinterpret_cast<const float4 *>(hu) + i);
        v.x = atten_one(v.x, k1000); v.y = atten_one(v.y, k1000); v.z = atten_one(v.z, k1000); v.w = atten_one(v.w, k1000);
        st_stream4(reinterpret_cast<float4 *>(mu) + i, v);
    }
    for (int64_t i = 4 * n4 + t; i < n; i += stride) mu[i] = atten_one(hu[i], k1000);
}

static WarpDims make_dims(int C, int D, int H, int W, int z_begin = 0, int z_count = -1) {
    WarpDims g;
    g.C = C; g.D = D; g.H = H; g.W = W;
    g.nvox = D * H * W;
    g.HW = H * W;
    g.Do = z_count < 0 ? D : z_count;
    g.z_off = z_begin;
    g.nvox_o = g.Do * H * W;
    g.zblocks = g.Do;
    g.z_magic = (unsigned)(((1ull << 32) + (unsigned)g.zblocks - 1) / (unsigned)g.zblocks);
    g.hx = (float)(W - 1) / 2.0f; g.hy = (float)(H - 1) / 2.0f; g.hz = (float)(D - 1) / 2.0f;
    g.mx = (float)(W - 1); g.my = (float)(H - 1); g.mz = (float)(D - 1);
    g.sp0 = 1.0 / (double)(D - 1); g.sp1 = 1.0 / (double)(H - 1); g.sp2 = 1.0 / (double)(W - 1);
    g.zero = 0.0f;
    g.zs0 = g.zs1 = g.zs2 = 1; g.zn0 = g.zblocks; g.zn1 = 0;
    return g;
}

static int check_warp_args(int B, int C, int D, int H, int W, int padding, int mode, int disp_plus_identity = 0) {
    LR_REQUIRE(B > 0 && C > 0 && D > 0 && H > 0 && W > 0, "warp: non-positive dimension (B=%d C=%d D=%d H=%d W=%d)", B, C, D, H, W);
    // the identity map divides by S-1 (as lr_identity_map, which rejects these sizes): undefined on a size-1 axis
    LR_REQUIRE(!disp_plus_identity || (D > 1 && H > 1 && W > 1),
               "warp: disp_plus_identity needs every size >= 2 (D=%d H=%d W=%d)", D, H, W);
    LR_REQUIRE((int64_t)D * H * W < (1ll << 31) - 2 * (int64_t)H * W - 4, "warp: D*H*W must fit 32-bit voxel offsets");
    LR_REQUIRE(D < 65536 && (H + WARP_TY - 1) / WARP_TY <= 65535, "warp: D and H/8 must be < 65536 (grid limits)");
    LR_REQUIRE(W < (1 << 21) && H < (1 << 21), "warp: H and W must be < 2^21 (mantissa floor)");
    LR_REQUIRE(padding == LR_PAD_ZEROS || padding == LR_PAD_BORDER, "warp: padding must be 0 (zeros) or 1 (border)");
    LR_REQUIRE(mode == LR_MODE_LINEAR || mode == LR_MODE_NEAREST, "warp: mode must be 0 (linear) or 1 (nearest)");
    return LR_OK;
}

// grid.z = D * (batch items of this launch) must stay <= 65535: batches are launched in chunks
static int batch_chunk(int D) { return 65535 / D > 0 ? 65535 / D : 1; }
static dim3 warp_grid(int nb, int D, int H, int W, int rows_per_thread = 1) {
    const int rows = WARP_TY * rows_per_thread;
    return dim3((unsigned)((W + WARP_TX - 1) / WARP_TX), (unsigned)((H + rows - 1) / rows), (unsigned)(D * nb));
}

// z-blocking of the forward kernel.  A block is long (a plane of a 32 x 16 tile costs ~1.8 us, the block set-up about
// one plane), the kernel is latency-bound (throughput follows occupancy), and at batch 1 the grid is only a few waves:
// with equal blocks the launch ends with every SM draining from full to empty over a whole block duration
// (~15 % of the kernel at 160^3).  So the blocks taper: most planes go into 8-plane blocks (set-up amortised), the rest
// into 4- and 2-plane blocks that are dispatched last (per batch item) and fill the tail.  The short blocks' share is about 1.2 waves of
// work, at most 45 % (measured: 55/27/18 % is best at batch 1 = 1.7 waves, 100/0/0 at batch 8 = 13.5 waves).
static void forward_z_blocking(WarpDims &g, int n_batch, double resident_blocks = 4.0, double max_small = 0.45) {
    const int Do = g.Do;
    g.zs0 = WARP_NZ_MAX; g.zs1 = 4; g.zs2 = 2;
    if (Do < 32) {
        g.zs0 = g.zs1 = g.zs2 = WARP_NZ;
        g.zn0 = (Do + WARP_NZ - 1) / WARP_NZ; g.zn1 = 0;
        g.zblocks = g.zn0;
    } else {
        const double tiles = (double)((g.W + WARP_TX - 1) / WARP_TX) * ((g.H + WARP_TY * WARP_VY - 1) / (WARP_TY * WARP_VY));
        const double waves = tiles * n_batch * ((Do + g.zs0 - 1) / g.zs0) / (resident_blocks * sm_count());   // (tuned with these counts)
        double small = 1.2 / (waves > 0.1 ? waves : 0.1);
        if (small > max_small) small = max_small;
        const int f0 = (int)(100.0 * (1.0 - small) + 0.5);      // percent of the planes in 8- / 4-plane blocks
        const int f1 = (int)(100.0 * 0.6 * small + 0.5);
        g.zn0 = (Do * f0 / 100) / g.zs0;
        const int rest = Do - g.zn0 * g.zs0;
        g.zn1 = f0 + f1 >= 100 ? (rest + g.zs1 - 1) / g.zs1 : (Do * f1 / 100) / g.zs1;
        if (g.zn1 * g.zs1 > rest) g.zn1 = (rest + g.zs1 - 1) / g.zs1;
        const int rest2 = rest - g.zn1 * g.zs1 > 0 ? rest - g.zn1 * g.zs1 : 0;
        g.zblocks = g.zn0 + g.zn1 + (rest2 + g.zs2 - 1) / g.zs2;
    }
    g.z_magic = (unsigned)(((1ull << 32) + (unsigned)g.zblocks - 1) / (unsigned)g.zblocks);
}

template <int PAD, int MODE>
static void launch_fwd(bool scale, bool ident, dim3 grid, cudaStream_t st, const float *img, const float *phi, float *out,
                       const WarpDims &g) {
    const dim3 blk(WARP_TX, WARP_TY);
    const bool fast = MODE == LR_MODE_LINEAR && numerics_mode() == LR_NUMERICS_FAST;
#define LR_LAUNCH_FWD(S, I)                                                                                          \
    do {                                                                                                             \
        if (fast) {                                                                                                  \
            if (g.C == 1) warp_forward_kernel<PAD, LR_MODE_LINEAR, S, I, true, true><<<grid, blk, 0, st>>>(img, phi, out, g);   \
            else warp_forward_kernel<PAD, LR_MODE_LINEAR, S, I, false, true><<<grid, blk, 0, st>>>(img, phi, out, g);           \
        } else if (g.C == 1) warp_forward_kernel<PAD, MODE, S, I, true, false><<<grid, blk, 0, st>>>(img, phi, out, g);          \
        else warp_forward_kernel<PAD, MODE, S, I, false, false><<<grid, blk, 0, st>>>(img, phi, out, g);                         \
    } while (0)
    if (scale) {
        if (ident) LR_LAUNCH_FWD(true, true);
        else LR_LAUNCH_FWD(true, false);
    } else {
        if (ident) LR_LAUNCH_FWD(false, true);
        else LR_LAUNCH_FWD(false, false);
    }
#undef LR_LAUNCH_FWD
}

template <int PAD>
static void launch_bwd(bool scale, bool ident, dim3 grid, cudaStream_t st, const float *gout, const float *img,
                       const float *phi, float *gimg, float *gphi, const WarpDims &g) {
    const dim3 blk(WARP_TX, WARP_TY);
    if (scale) {
        if (ident) warp_backward_kernel<PAD, true, true><<<grid, blk, 0, st>>>(gout, img, phi, gimg, gphi, g);
        else warp_backward_kernel<PAD, true, false><<<grid, blk, 0, st>>>(gout, img, phi, gimg, gphi, g);
    } else {
        if (ident) warp_backward_kernel<PAD, false, true><<<grid, blk, 0, st>>>(gout, img, phi, gimg, gphi, g);
        else warp_backward_kernel<PAD, false, false><<<grid, blk, 0, st>>>(gout, img, phi, gimg, gphi, g);
    }
}

}  // namespace lr

using namespace lr;

static int check_slab(int D, int z_begin, int z_count) {
    LR_REQUIRE(z_begin >= 0 && z_count > 0 && z_begin + z_count <= D, "warp: slab [%d, %d) is not inside [0, %d)", z_begin,
               z_begin + z_count, D);
    return LR_OK;
}

extern "C" int lr_warp_forward_slab(const float *img, const float *phi, int B, int C, int D, int H, int W, int z_begin,
                                    int z_count, int padding, int mode, int using_scale, int disp_plus_identity,
                                    float *out, lr_stream_t stream) {
    LR_REQUIRE(img && phi && out, "warp_forward: null pointer");
    if (int e = check_warp_args(B, C, D, H, W, padding, mode, disp_plus_identity)) return e;
    if (int e = check_slab(D, z_begin, z_count)) return e;
    WarpDims g = make_dims(C, D, H, W, z_begin, z_count);
    cudaStream_t st = as_stream(stream);
    const bool sc = using_scale != 0, id = disp_plus_identity != 0;
    const int chunk = batch_chunk((g.Do + 1) / 2);          // upper bound of the z-blocks per item
    for (int b0 = 0; b0 < B; b0 += chunk) {
        const int nb = B - b0 < chunk ? B - b0 : chunk;
        forward_z_blocking(g, nb);
        const dim3 grid = warp_grid(nb, g.zblocks, H, W, WARP_VY);
        const float *im = img + (int64_t)b0 * C * g.nvox, *ph = phi + (int64_t)b0 * 3 * g.nvox_o;
        float *o = out + (int64_t)b0 * C * g.nvox_o;
        if (padding == LR_PAD_ZEROS) {
            if (mode == LR_MODE_LINEAR) launch_fwd<LR_PAD_ZEROS, LR_MODE_LINEAR>(sc, id, grid, st, im, ph, o, g);
            else launch_fwd<LR_PAD_ZEROS, LR_MODE_NEAREST>(sc, id, grid, st, im, ph, o, g);
        } else {
            if (mode == LR_MODE_LINEAR) launch_fwd<LR_PAD_BORDER, LR_MODE_LINEAR>(sc, id, grid, st, im, ph, o, g);
            else launch_fwd<LR_PAD_BORDER, LR_MODE_NEAREST>(sc, id, grid, st, im, ph, o, g);
        }
        if (int e = check_launch("warp_forward_kernel")) return e;
    }
    return LR_OK;
}

// Launch plan of the forward kernel, for host-side tests (no device work): how the Do planes of an item are cut into
// z-blocks.  plan = {size0, n0, size1, n1, size2, n2}: n0 blocks of size0 planes, then n1 of size1, then n2 of size2
// (the last block may be partial).
extern "C" int lr_warp_forward_plan(int B, int D, int H, int W, int z_count, int plan[6]) {
    LR_REQUIRE(plan, "warp_forward_plan: null pointer");
    if (int e = check_warp_args(B, 1, D, H, W, LR_PAD_ZEROS, LR_MODE_LINEAR)) return e;
    if (int e = check_slab(D, 0, z_count)) return e;
    WarpDims g = make_dims(1, D, H, W, 0, z_count);
    const int chunk = batch_chunk((g.Do + 1) / 2);
    forward_z_blocking(g, B < chunk ? B : chunk);
    plan[0] = g.zs0; plan[1] = g.zn0; plan[2] = g.zs1; plan[3] = g.zn1; plan[4] = g.zs2; plan[5] = g.zblocks - g.zn0 - g.zn1;
    return LR_OK;
}

extern "C" int lr_warp_forward(const float *img, const float *phi, int B, int C, int D, int H, int W, int padding,
                               int mode, int using_scale, int disp_plus_identity, float *out, lr_stream_t stream) {
    return lr_warp_forward_slab(img, phi, B, C, D, H, W, 0, D, padding, mode, using_scale, disp_plus_identity, out, stream);
}

extern "C" int lr_warp_backward_slab(const float *grad_out, const float *img, const float *phi, int B, int C, int D, int H,
                                     int W, int z_begin, int z_count, int padding, int mode, int using_scale,
                                     int disp_plus_identity, float *grad_img, float *grad_phi, lr_stream_t stream) {
    LR_REQUIRE(grad_out && img && phi, "warp_backward: null pointer");
    if (int e = check_warp_args(B, C, D, H, W, padding, mode, disp_plus_identity)) return e;
    if (int e = check_slab(D, z_begin, z_count)) return e;
    if (!grad_img && !grad_phi) return LR_OK;
    cudaStream_t st = as_stream(stream);
    WarpDims g = make_dims(C, D, H, W, z_begin, z_count);
    if (mode == LR_MODE_NEAREST) {
        // nearest sampling is piecewise constant in phi: zero grid gradient (ATen does the same); the image
        // gradient is a pure scatter, which the linear kernel cannot express -> not needed by the reference
        // (evaluate_dir_lab.py:221 warps label maps without autograd).
        LR_REQUIRE(!grad_img, "warp_backward: grad_img is not supported for nearest mode");
        return cuda_ok(cudaMemsetAsync(grad_phi, 0, sizeof(float) * 3 * (size_t)B * g.nvox_o, st), "warp_backward: memset failed");
    }
    const bool sc = using_scale != 0, id = disp_plus_identity != 0;
    const int chunk = batch_chunk(g.Do);
    for (int b0 = 0; b0 < B; b0 += chunk) {
        const int nb = B - b0 < chunk ? B - b0 : chunk;
        const dim3 grid = warp_grid(nb, g.Do, H, W);
        const int64_t io = (int64_t)b0 * C * g.nvox, oo = (int64_t)b0 * C * g.nvox_o, po = (int64_t)b0 * 3 * g.nvox_o;
        float *gi = grad_img ? grad_img + io : nullptr, *gp = grad_phi ? grad_phi + po : nullptr;
        if (padding == LR_PAD_ZEROS && !gi) {
            // training configuration: map gradient only -> packed two-voxel kernel
            WarpDims gz = g;                      // this kernel walks runs of planes (tapered z-blocks, as the forward)
            forward_z_blocking(gz, nb, 6.0, 0.5);  // 6 resident blocks per SM; measured at 160^3: 50/30/20 % -> 32.0 us, 64/21/15 % -> 33.2 us
            const dim3 grid2 = warp_grid(nb, gz.zblocks, H, W, WARP_VY);
            const dim3 blk(WARP_TX, WARP_TY);
#define LR_LAUNCH_BWD_PHI(S, I)                                                                                              \
    do {                                                                                                                     \
        if (C == 1) warp_backward_phi_kernel<S, I, true><<<grid2, blk, 0, st>>>(grad_out + oo, img + io, phi + po, gp, gz);   \
        else warp_backward_phi_kernel<S, I, false><<<grid2, blk, 0, st>>>(grad_out + oo, img + io, phi + po, gp, gz);         \
    } while (0)
            if (sc) {
                if (id) LR_LAUNCH_BWD_PHI(true, true);
                else LR_LAUNCH_BWD_PHI(true, false);
            } else {
                if (id) LR_LAUNCH_BWD_PHI(false, true);
                else LR_LAUNCH_BWD_PHI(false, false);
            }
#undef LR_LAUNCH_BWD_PHI
        } else if (padding == LR_PAD_ZEROS) launch_bwd<LR_PAD_ZEROS>(sc, id, grid, st, grad_out + oo, img + io, phi + po, gi, gp, g);
        else launch_bwd<LR_PAD_BORDER>(sc, id, grid, st, grad_out + oo, img + io, phi + po, gi, gp, g);
        if (int e = check_launch("warp_backward_kernel")) return e;
    }
    return LR_OK;
}

extern "C" int lr_warp_backward(const float *grad_out, const float *img, const float *phi, int B, int C, int D, int H,
                                int W, int padding, int mode, int using_scale, int disp_plus_identity, float *grad_img,
                                float *grad_phi, lr_stream_t stream) {
    return lr_warp_backward_slab(grad_out, img, phi, B, C, D, H, W, 0, D, padding, mode, using_scale, disp_plus_identity,
                                 grad_img, grad_phi, stream);
}

extern "C" int lr_identity_map(int D, int H, int W, float *out, lr_stream_t stream) {
    LR_REQUIRE(out, "identity_map: null pointer");
    LR_REQUIRE(D > 1 && H > 1 && W > 1 && D <= 65535, "identity_map: each size must be in [2, 65535]");
    LR_REQUIRE((int64_t)D * H * W < (1ll << 31), "identity_map: D*H*W must fit 32 bits");
    WarpDims g = make_dims(1, D, H, W);
    identity_map_kernel<<<warp_grid(1, (D + IDENT_PLANES - 1) / IDENT_PLANES, H, W), dim3(WARP_TX, WARP_TY), 0, as_stream(stream)>>>(out, g);
    return check_launch("identity_map_kernel");
}

extern "C" int lr_atten_coef(const float *hu, int64_t n, float *mu, lr_stream_t stream) {
    LR_REQUIRE(hu && mu && n >= 0, "atten_coef: bad argument");
    if (n == 0) return LR_OK;
    const bool vec = ((uintptr_t)hu % 16 == 0) && ((uintptr_t)mu % 16 == 0);
    const int64_t n4 = vec ? n / 4 : 0, work = n4 + (n - 4 * n4);
    const int64_t cap = (int64_t)sm_count() * 8;
    const int blocks = (int)((work + 255) / 256 < cap ? (work + 255) / 256 : cap);
    atten_coef_kernel<<<blocks, 256, 0, as_stream(stream)>>>(hu, mu, n, n4, make_const_div(1000.0f));
    return check_launch("atten_coef_kernel");
}
