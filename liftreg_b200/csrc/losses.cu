// Similarity loss on the warp output (SURVEY.md 8f row f4): the reference's NCCLoss, sm_100a.
//
// Replaces reference src/liftreg/layers/losses.py:14-29 (NCCLoss.forward), used as the training similarity
// (src/liftreg/losses/SubspaceLoss.py:12,27) and as the validation score (src/liftreg/networks/RegistrationNet.py:210-212):
//     a = x - mean(x) + 1e-10,  b = y - mean(y) + 1e-10                       (per batch item, over all voxels)
//     ncc = mean(a*b) / sqrt(mean(a^2) * mean(b^2)),   loss = 1 - mean_over_batch(ncc)
// The reference runs ~10 elementwise / reduction kernels over the two volumes (each re-reading 16 MB per item at 160^3);
// here the forward is ONE pass over x and y (raw moments about the item's first voxel, rewritten into the centred ones by a
// B-thread kernel) and the backward is one pass.  Per-thread partial sums are fp32 over a handful of elements, everything above that
// is accumulated in fp64 (warp shuffles, shared memory, one fp64 atomic per block), so the result does not depend on the launch shape
// beyond fp64 round-off.
#include <cfloat>

#include "common.cuh"

namespace lr {

constexpr int NCC_THREADS = 256;
constexpr int NCC_SUMS = 7;          // per item: sum x, sum y, sum a*b, sum a*a, sum b*b, sum a, sum b

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block reduction of NV per-thread values, then ONE fp64 atomic per value and block (an atomic per warp made the few
// accumulator addresses the bottleneck: 96 us instead of 17 us per 160^3 pair).
template <int NV>
__device__ __forceinline__ void block_accumulate(const float (&v)[NV], double *__restrict__ dst) {
    __shared__ double part[NCC_THREADS / 32][NV];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
        const double w = warp_sum((double)v[k]);
        if (lane == 0) part[warp][k] = w;
    }
    __syncthreads();
    if (threadIdx.x < NV) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < NCC_THREADS / 32; ++w) t += part[w][threadIdx.x];
        atomicAdd(dst + threadIdx.x, t);
    }
}

// the centred values exactly as the reference forms them in fp32 (losses.py:21-22): (x - mean) + 1e-10
__device__ __forceinline__ float centred(float v, float mean) { return add_rn(sub_rn(v, mean), 1e-10f); }

// Single-pass forward.  The centring needs the means, which is why the reference reads x and y twice; but with
// u = x - k, v = y - l for ANY constants k, l the centred moments follow from the raw moments of u and v:
//     a = x - mean + eps = u - dx  (dx = mean - k - eps)   =>   sum a*a = sum u*u - 2 dx sum u + N dx^2, etc.
// and the cancellation in these differences is mild when k, l lie within a few standard deviations of the means.  k and l are
// the item's first voxels (every thread reads them); per-thread fp32 partials over a few elements, everything above in fp64
// as before; a B-thread kernel then rewrites the five raw sums into the seven-entry layout the backward and the host use.
// What is not reproduced is the fp32 rounding of each (x - mean) + 1e-10 that the reference's op-for-op form performs
// (oracle/torch_port.ncc_loss; the 1e-10 is below half an ulp of all but the elements within 1e-3 of the mean): that
// rounding moves the loss by ~1e-8.
__global__ void __launch_bounds__(NCC_THREADS) ncc_shifted_kernel(const float *__restrict__ x, const float *__restrict__ y, int64_t N,
                                                                  double *__restrict__ sums) {
    const int b = blockIdx.y;
    const float *xb = x + (int64_t)b * N, *yb = y + (int64_t)b * N;
    const float k = __ldg(xb), l = __ldg(yb);
    float su = 0.0f, sv = 0.0f, suv = 0.0f, suu = 0.0f, svv = 0.0f;
    const int64_t t = (int64_t)blockIdx.x * NCC_THREADS + threadIdx.x, stride = (int64_t)gridDim.x * NCC_THREADS;
    // 16-byte loads where the item's rows allow it (four times the bytes in flight per thread: the scalar loop was bound by
    // memory latency at full occupancy, 2.6 TB/s), scalar tail
    const int64_t n4 = (((uintptr_t)xb | (uintptr_t)yb) % 16 == 0) ? N / 4 : 0;
    for (int64_t i = t; i < n4; i += stride) {
        const float4 a = ld_stream4(reinterpret_cast<const float4 *>(xb) + i), c = ld_stream4(reinterpret_cast<const float4 *>(yb) + i);
        const float u0 = a.x - k, u1 = a.y - k, u2 = a.z - k, u3 = a.w - k, v0 = c.x - l, v1 = c.y - l, v2 = c.z - l, v3 = c.w - l;
        su += (u0 + u1) + (u2 + u3); sv += (v0 + v1) + (v2 + v3);
        suv = fmaf(u0, v0, fmaf(u1, v1, fmaf(u2, v2, fmaf(u3, v3, suv))));
        suu = fmaf(u0, u0, fmaf(u1, u1, fmaf(u2, u2, fmaf(u3, u3, suu))));
        svv = fmaf(v0, v0, fmaf(v1, v1, fmaf(v2, v2, fmaf(v3, v3, svv))));
    }
    for (int64_t i = 4 * n4 + t; i < N; i += stride) {
        const float u = ld_stream(xb + i) - k, v = ld_stream(yb + i) - l;
        su += u; sv += v;
        suv = fmaf(u, v, suv); suu = fmaf(u, u, suu); svv = fmaf(v, v, svv);
    }
    const float vals[5] = {su, sv, suv, suu, svv};
    block_accumulate<5>(vals, sums + b * NCC_SUMS);
}

__global__ void ncc_finalize_kernel(const float *__restrict__ x, const float *__restrict__ y, int64_t N, int B, double *__restrict__ sums) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    double *s = sums + b * NCC_SUMS;
    const double n = (double)N, k = (double)x[(int64_t)b * N], l = (double)y[(int64_t)b * N];
    const double Su = s[0], Sv = s[1], Suv = s[2], Suu = s[3], Svv = s[4];
    const double Sx = Su + n * k, Sy = Sv + n * l;
    const double dx = (double)(float)(Sx / n) - k, dy = (double)(float)(Sy / n) - l;      // the means as the fp32 values the backward uses
    s[0] = Sx; s[1] = Sy;
    s[2] = Suv - dy * Su - dx * Sv + n * dx * dy;
    s[3] = Suu - 2.0 * dx * Su + n * dx * dx;
    s[4] = Svv - 2.0 * dy * Sv + n * dy * dy;
    s[5] = Su - n * dx; s[6] = Sv - n * dy;
}

// backward wrt x:  ncc = Sab / sqrt(Saa Sbb);  d ncc / d a_i = c1 b_i - c2 a_i  with c1 = 1/sqrt(Saa Sbb),
// c2 = Sab / (Saa sqrt(Saa Sbb));  a_i = x_i - mean(x) + eps  =>  d ncc / d x_j = g_j - mean(g).
// grad_x = scale * (c1 b - c2 a - c3),  c3 = c1 Sb/N - c2 Sa/N,  scale = -grad_loss / B  (loss = 1 - mean_b ncc).
__global__ void __launch_bounds__(NCC_THREADS) ncc_backward_kernel(const float *__restrict__ x, const float *__restrict__ y, int64_t N,
                                                                   const double *__restrict__ sums, const float *__restrict__ grad_loss,
                                                                   int B, float *__restrict__ gx) {
    const int b = blockIdx.y;
    const double *s = sums + b * NCC_SUMS;
    const float mx = (float)(s[0] / (double)N), my = (float)(s[1] / (double)N);
    const double root = sqrt(s[3] * s[4]);
    const double c1 = 1.0 / root, c2 = s[2] / (s[3] * root);
    const double c3 = c1 * s[6] / (double)N - c2 * s[5] / (double)N;
    const double scale = -(double)grad_loss[0] / (double)B;
    const float f1 = (float)(scale * c1), f2 = (float)(scale * c2), f3 = (float)(scale * c3);
    const float *xb = x + (int64_t)b * N, *yb = y + (int64_t)b * N;
    float *gb = gx + (int64_t)b * N;
    const int64_t t = (int64_t)blockIdx.x * NCC_THREADS + threadIdx.x, stride = (int64_t)gridDim.x * NCC_THREADS;
    const int64_t n4 = (((uintptr_t)xb | (uintptr_t)yb | (uintptr_t)gb) % 16 == 0) ? N / 4 : 0;
    for (int64_t i = t; i < n4; i += stride) {
        const float4 xv = ld_stream4(reinterpret_cast<const float4 *>(xb) + i), yv = ld_stream4(reinterpret_cast<const float4 *>(yb) + i);
        float4 o;
        o.x = fmaf(f1, centred(yv.x, my), fmaf(-f2, centred(xv.x, mx), -f3));
        o.y = fmaf(f1, centred(yv.y, my), fmaf(-f2, centred(xv.y, mx), -f3));
        o.z = fmaf(f1, centred(yv.z, my), fmaf(-f2, centred(xv.z, mx), -f3));
        o.w = fmaf(f1, centred(yv.w, my), fmaf(-f2, centred(xv.w, mx), -f3));
        st_stream4(reinterpret_cast<float4 *>(gb) + i, o);
    }
    for (int64_t i = 4 * n4 + t; i < N; i += stride) {
        const float a = centred(ld_stream(xb + i), mx), c = centred(ld_stream(yb + i), my);
        st_stream(gb + i, fmaf(f1, c, fmaf(-f2, a, -f3)));
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Displacement regulariser of the subspace loss, reference src/liftreg/losses/SubspaceLoss.py:51-67:
//     fd = mermaid.finite_differences.FD_torch(spacing*2),  spacing = 1/(shape-1)
//     reg = mean_{b,voxel} sum_{c<3} dXc(disp_c)^2 + dYc(disp_c)^2 + dZc(disp_c)^2
// dXc = (xp - xm) * (0.5/spacing[0]) is mermaid's central difference along the FIRST spatial axis (Y: second, Z: last).
// mermaid is a third-party dependency that is absent from /root/reference (requirements.txt:61 pins `mermaid==0.3.2`);
// its central difference is restated here.  What the call site fixes: interior voxels use (I[i+1] - I[i-1]) * scale.
// What only mermaid's source fixes is the boundary rule, so both of its published modes are offered:
//     LR_FD_LINEAR (0, FD_torch's default mode='linear'): the missing neighbour is extrapolated linearly,
//                  xp[n-1] = 2 I[n-1] - I[n-2], xm[0] = 2 I[0] - I[1]  (a one-sided difference at the faces)
//     LR_FD_NEUMANN_ZERO (1): the central difference is zero on the faces.
// The reference needs 9 difference kernels, 9 squares, 8 sums and a mean (each a pass over 16 MB * B at 160^3); here the
// forward is ONE pass over the displacement (12 B per voxel from HBM, neighbours from L1/L2) and the backward one more.
constexpr int REG_TX = 32, REG_TY = 8;                 // block tile: 32 voxels along the fastest axis, 8 rows
#ifndef LR_REG_PF
#define LR_REG_PF 4
#endif
#ifndef LR_REG_WAVES
#define LR_REG_WAVES 1
#endif
// A thread marches planes serially and has only three first-touch loads in flight per plane (one per channel), so the
// march is bound by DRAM latency, not bandwidth; the planes LR_REG_PF ahead are pulled into L2 while it works.
__device__ __forceinline__ void prefetch_l2(const float *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }

struct RegDims {
    int d, h, w;              // first, second, last spatial axis (the reference calls them D, W, H)
    int zchunk, n_zchunks;    // planes of the first axis marched by one block
    float sd, sh, sw;         // 0.5 / (2/(n-1)) per axis, rounded to fp32 like the Python scalar entering the tensor op
};

// unscaled (xp - xm) from the upper / lower neighbour u, d (loaded with offsets clamped at the faces) and the centre c
template <int MODE>
__device__ __forceinline__ float fd_delta(float u, float d, float c, bool lo, bool hi) {
    if (MODE != 0) return (lo || hi) ? 0.0f : sub_rn(u, d);
    const float xp = hi ? fmaf(2.0f, c, -d) : u;          // 2 I[n-1] - I[n-2]   (2c is exact, so this is sub_rn(mul_rn(2,c), d))
    const float xm = lo ? fmaf(2.0f, c, -u) : d;          // 2 I[0] - I[1]
    return sub_rn(xp, xm);
}

__device__ __forceinline__ void block_accumulate_f64(double v, double *__restrict__ dst) {
    __shared__ double part64[NCC_THREADS / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const double w = warp_sum(v);
    if (lane == 0) part64[warp] = w;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
#pragma unroll
        for (int k = 0; k < NCC_THREADS / 32; ++k) t += part64[k];
        atomicAdd(dst, t);
    }
}

// Forward: a block owns a 32 x 8 tile of (last, second) axis positions and marches a chunk of planes of the first axis
// with a three-plane register window per channel (each plane is read from HBM once; the in-plane neighbours hit L1).
template <int MODE>
__global__ void __launch_bounds__(NCC_THREADS) diffusion_reg_kernel(const float *__restrict__ disp, RegDims g, double *__restrict__ sum) {
    const int x = blockIdx.x * REG_TX + (threadIdx.x & 31), y = blockIdx.y * REG_TY + (threadIdx.x >> 5);
    const int zc = blockIdx.z % g.n_zchunks, b = blockIdx.z / g.n_zchunks;
    const int z0 = zc * g.zchunk, z1 = min(g.d, z0 + g.zchunk);
    const int64_t plane = (int64_t)g.h * g.w, cstride = plane * g.d;
    double acc = 0.0;
    if (x < g.w && y < g.h) {
        const bool xlo = x == 0, xhi = x == g.w - 1, ylo = y == 0, yhi = y == g.h - 1;
        const int oxu = xhi ? 0 : 1, oxd = xlo ? 0 : -1;
        const int oyu = yhi ? 0 : g.w, oyd = ylo ? 0 : -g.w;
        // 32-bit element indices (the host checks B*3*D*H*W < 2^31): one IMAD.WIDE per address instead of 64-bit chains
        const unsigned pl = (unsigned)plane, cs = (unsigned)cstride;
        unsigned i0 = ((unsigned)b * 3u * (unsigned)g.d + (unsigned)z0) * pl + (unsigned)y * (unsigned)g.w + (unsigned)x;
        float vm[3], vc[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            vc[c] = __ldg(disp + (i0 + c * cs));
            vm[c] = z0 > 0 ? __ldg(disp + (i0 + c * cs - pl)) : vc[c];
        }
        for (int z = z0; z < z1; ++z, i0 += pl) {
            const bool zlo = z == 0, zhi = z == g.d - 1;
            float l2 = 0.0f;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const unsigned ic = i0 + c * cs;
                const float cc = vc[c];
                const float vp = zhi ? cc : __ldg(disp + (ic + pl));      // allocating load: the next iteration's in-plane neighbours hit L1
                if (LR_REG_PF > 0 && z + LR_REG_PF <= z1) prefetch_l2(disp + (ic + LR_REG_PF * pl));
                const float yu = __ldg(disp + (ic + oyu)), yd = __ldg(disp + (ic + oyd));
                const float xu = __ldg(disp + (ic + oxu)), xd = __ldg(disp + (ic + oxd));
                const float dd = mul_rn(fd_delta<MODE>(vp, vm[c], cc, zlo, zhi), g.sd);
                const float dh = mul_rn(fd_delta<MODE>(yu, yd, cc, ylo, yhi), g.sh);
                const float dw = mul_rn(fd_delta<MODE>(xu, xd, cc, xlo, xhi), g.sw);
                l2 = add_rn(l2, mul_rn(dd, dd));          // SubspaceLoss.py:55-63, left to right
                l2 = add_rn(l2, mul_rn(dh, dh));
                l2 = add_rn(l2, mul_rn(dw, dw));
                vm[c] = cc; vc[c] = vp;
            }
            acc += (double)l2;
        }
    }
    block_accumulate_f64(acc, sum);
}

// d reg / d disp.  With D the difference operator of one axis (rows q, columns p) and s its scale,
//     reg = (1/M) sum_q (s (D I)_q)^2   =>   d reg / d I_p = (2 s^2 / M) sum_q D_qp (D I)_q ;
// row q of D has +1 at q+1 and -1 at q-1 in the interior, and (linear mode) -2, +2 at (0, 1) resp. (n-2, n-1) on the faces.
// Interior: sum_q D_qp (D I)_q = (I_p - I_{p-2}) - (I_{p+2} - I_p).  Within two entries of a face the rows of D that
// follow the face rule enter with their own coefficients (the rare predicated block below).
template <int MODE>
__device__ __forceinline__ float fd_adjoint(const float *__restrict__ base, unsigned p, float c, int i, int n, unsigned stride) {
    if (i >= 2 && i <= n - 3) return sub_rn(sub_rn(c, __ldg(base + (p - 2u * stride))), sub_rn(__ldg(base + (p + 2u * stride)), c));
    float tm = 0.0f, tp = 0.0f, t0 = 0.0f;
    if (i >= 2) tm = sub_rn(c, __ldg(base + (p - 2u * stride)));          // row p-1 is an interior row
    if (i <= n - 3) tp = sub_rn(__ldg(base + (p + 2u * stride)), c);      // row p+1 is an interior row
    if (MODE == 0) {
        const float bb = i >= 1 ? __ldg(base + (p - stride)) : c, dd = i <= n - 2 ? __ldg(base + (p + stride)) : c;
        if (i == 1) tm = 2.0f * sub_rn(c, fmaf(2.0f, bb, -c));            // +2 * row 0:   I[1] - (2 I[0] - I[1])
        if (i == n - 2) tp = 2.0f * sub_rn(fmaf(2.0f, dd, -c), c);        // -2 * row n-1: (2 I[n-1] - I[n-2]) - I[n-2]  (sign below)
        if (i == 0) t0 = -2.0f * sub_rn(dd, fmaf(2.0f, c, -dd));          // -2 * row 0
        if (i == n - 1) t0 = add_rn(t0, 2.0f * sub_rn(fmaf(2.0f, c, -bb), bb));   // +2 * row n-1
    }
    return add_rn(sub_rn(tm, tp), t0);
}

template <int MODE>
__global__ void __launch_bounds__(NCC_THREADS) diffusion_reg_backward_kernel(const float *__restrict__ disp, RegDims g, int B,
                                                                             const float *__restrict__ grad_loss,
                                                                             float *__restrict__ grad_disp) {
    const int x = blockIdx.x * REG_TX + (threadIdx.x & 31), y = blockIdx.y * REG_TY + (threadIdx.x >> 5);
    const int zc = blockIdx.z % g.n_zchunks, b = blockIdx.z / g.n_zchunks;
    const int z0 = zc * g.zchunk, z1 = min(g.d, z0 + g.zchunk);
    const int64_t plane = (int64_t)g.h * g.w, cstride = plane * g.d;
    if (x >= g.w || y >= g.h) return;
    const float k = (float)(2.0 * (double)grad_loss[0] / ((double)B * (double)g.d * (double)plane));
    const float kd = k * g.sd * g.sd, kh = k * g.sh * g.sh, kw = k * g.sw * g.sw;
    const unsigned pl = (unsigned)plane, cs = (unsigned)cstride;      // 32-bit element indices, as in the forward
    unsigned off = ((unsigned)b * 3u * (unsigned)g.d + (unsigned)z0) * pl + (unsigned)y * (unsigned)g.w + (unsigned)x;
    for (int z = z0; z < z1; ++z, off += pl) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const unsigned p = off + c * cs;
            const float cc = __ldg(disp + p);
            if (LR_REG_PF > 0 && z + LR_REG_PF + 2 < min(g.d, z1 + 2)) prefetch_l2(disp + (p + (LR_REG_PF + 2) * pl));
            float gr = kd * fd_adjoint<MODE>(disp, p, cc, z, g.d, pl);
            gr = fmaf(kh, fd_adjoint<MODE>(disp, p, cc, y, g.h, (unsigned)g.w), gr);
            gr = fmaf(kw, fd_adjoint<MODE>(disp, p, cc, x, g.w, 1u), gr);
            st_stream(grad_disp + p, gr);
        }
    }
}

// ---- two voxels per thread (W even, 8-byte-aligned field): 64-bit loads and packed fp32x2 arithmetic -------------------
// The scalar kernels above issue ~140 instructions per voxel, most of them addresses and face selects, and are bound by
// the issue rate (ncu: 55 % issue-active at 0.2 of the HBM roofline).  Here a thread owns the voxels (x, x+1), x even:
// every load of the z / y neighbours is one aligned LDG.64, the differences of both voxels run as one FADD2 / FMUL2 /
// FFMA2 stream, and the face rules are a few predicated instructions (x: the first and last pair of a row).
constexpr int REGP_TX = 16, REGP_TY = 16;        // block tile: 16 pairs (32 voxels, one 128-byte line) x 16 rows
#ifndef LR_REGP_MINB
#define LR_REGP_MINB 1
#endif
// measured at 160^3 (profiles/README.md): the adjoint is fastest with 6 resident blocks, two waves of shorter chunks
// and a deeper L2 prefetch (37 us vs 42); the forward with the compiler's own register budget and one wave (26.6 us)
#ifndef LR_REGP_BWD_MINB
#define LR_REGP_BWD_MINB 6
#endif
#ifndef LR_REG_BWD_PF
#define LR_REG_BWD_PF 8
#endif
#ifndef LR_REG_BWD_WAVES
#define LR_REG_BWD_WAVES 2
#endif

__device__ __forceinline__ f32x2 ldg2(const float *p) { return __ldg(reinterpret_cast<const unsigned long long *>(p)); }
__device__ __forceinline__ f32x2 twice_minus(f32x2 c, f32x2 d) { return sub2(add2(c, c), d); }      // 2c - d, 2c exact

template <int MODE>
__device__ __forceinline__ f32x2 fd_delta2(f32x2 u, f32x2 d, f32x2 c, bool lo, bool hi) {
    if (MODE != 0) return (lo || hi) ? 0ull : sub2(u, d);
    if (hi) u = twice_minus(c, d);
    else if (lo) d = twice_minus(c, u);
    return sub2(u, d);
}

template <int MODE>
__global__ void __launch_bounds__(NCC_THREADS, LR_REGP_MINB) diffusion_reg_pair_kernel(const float *__restrict__ disp, RegDims g, double *__restrict__ sum) {
    const int x = (blockIdx.x * REGP_TX + (threadIdx.x & (REGP_TX - 1))) * 2, y = blockIdx.y * REGP_TY + (threadIdx.x / REGP_TX);
    const int zc = blockIdx.z % g.n_zchunks, b = blockIdx.z / g.n_zchunks;
    const int z0 = zc * g.zchunk, z1 = min(g.d, z0 + g.zchunk);
    double acc = 0.0;
    if (x < g.w && y < g.h) {
        const bool xlo = x == 0, xhi = x + 2 == g.w, ylo = y == 0, yhi = y == g.h - 1;
        const int oxl = xlo ? 0 : -1, oxr = xhi ? 1 : 2;                 // I[x-1], I[x+2], clamped into the row
        const int oyu = yhi ? 0 : g.w, oyd = ylo ? 0 : -g.w;
        const unsigned pl = (unsigned)(g.h * g.w), cs = pl * (unsigned)g.d;
        unsigned i0 = ((unsigned)b * 3u * (unsigned)g.d + (unsigned)z0) * pl + (unsigned)y * (unsigned)g.w + (unsigned)x;
        const f32x2 sd2 = splat2(g.sd), sh2 = splat2(g.sh), sw2 = splat2(g.sw);
        f32x2 vm[3], vc[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            vc[c] = ldg2(disp + (i0 + c * cs));
            vm[c] = z0 > 0 ? ldg2(disp + (i0 + c * cs - pl)) : vc[c];
        }
        f32x2 part = 0ull;                                               // fp32 partial sums of at most 16 planes
        for (int z = z0; z < z1; ++z, i0 += pl) {
            const bool zlo = z == 0, zhi = z == g.d - 1;
            f32x2 l2 = 0ull;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const unsigned ic = i0 + c * cs;
                const f32x2 cc = vc[c];
                const f32x2 vp = zhi ? cc : ldg2(disp + (ic + pl));      // allocating load: next iteration's row neighbours hit L1
                if (LR_REG_PF > 0 && z + LR_REG_PF <= z1) prefetch_l2(disp + (ic + LR_REG_PF * pl));
                const f32x2 yu = ldg2(disp + (ic + oyu)), yd = ldg2(disp + (ic + oyd));
                float xl = __ldg(disp + (ic + oxl)), xr = __ldg(disp + (ic + oxr));
                float c0, c1;
                unpack2(cc, c0, c1);
                f32x2 dx;
                if (MODE == 0) {
                    if (xlo) xl = fmaf(2.0f, c0, -c1);                   // xm of voxel 0:     2 I[0] - I[1]
                    if (xhi) xr = fmaf(2.0f, c1, -c0);                   // xp of voxel W-1:   2 I[W-1] - I[W-2]
                    dx = sub2(pack2(c1, xr), pack2(xl, c0));
                } else {
                    dx = pack2(xlo ? 0.0f : sub_rn(c1, xl), xhi ? 0.0f : sub_rn(xr, c0));
                }
                const f32x2 dd = mul2(fd_delta2<MODE>(vp, vm[c], cc, zlo, zhi), sd2);
                const f32x2 dh = mul2(fd_delta2<MODE>(yu, yd, cc, ylo, yhi), sh2);
                const f32x2 dw = mul2(dx, sw2);
                l2 = fma2(dd, dd, l2);                                   // SubspaceLoss.py:55-63 in order, squares fused into the sum
                l2 = fma2(dh, dh, l2);
                l2 = fma2(dw, dw, l2);
                vm[c] = cc; vc[c] = vp;
            }
            part = add2(part, l2);
            if (((z - z0) & 15) == 15 || z == z1 - 1) {
                float p0, p1;
                unpack2(part, p0, p1);
                acc += (double)p0 + (double)p1;
                part = 0ull;
            }
        }
    }
    block_accumulate_f64(acc, sum);      // one fp64 atomic per block (spreading them over 64 addresses changed nothing)
}

// x term of the adjoint for the pair (x, x+1): interior (I_p - I_{p-2}) - (I_{p+2} - I_p); the first pair of a row sees
// row 0 of the difference operator, the last pair row W-1 (see fd_adjoint)
template <int MODE>
__device__ __forceinline__ f32x2 fd_adjoint_x2(const float *__restrict__ base, unsigned p, f32x2 cc, int x, int w) {
    if (x >= 2 && x + 4 <= w) return sub2(sub2(cc, ldg2(base + (p - 2u))), sub2(ldg2(base + (p + 2u)), cc));
    float c0, c1, tm0 = 0.0f, tm1 = 0.0f, tp0 = 0.0f, tp1 = 0.0f, t00 = 0.0f, t01 = 0.0f;
    unpack2(cc, c0, c1);
    if (x >= 2) {
        float a0, a1;
        unpack2(ldg2(base + (p - 2u)), a0, a1);
        tm0 = sub_rn(c0, a0); tm1 = sub_rn(c1, a1);
    } else if (MODE == 0) {
        const float q = sub_rn(c1, fmaf(2.0f, c0, -c1));                 // row 0:   I[1] - (2 I[0] - I[1])
        tm1 = 2.0f * q; t00 = -2.0f * q;
    }
    if (x + 4 <= w) {
        float e0, e1;
        unpack2(ldg2(base + (p + 2u)), e0, e1);
        tp0 = sub_rn(e0, c0); tp1 = sub_rn(e1, c1);
    } else if (MODE == 0) {
        const float r = sub_rn(fmaf(2.0f, c1, -c0), c0);                 // row W-1: (2 I[W-1] - I[W-2]) - I[W-2]
        tp0 = 2.0f * r; t01 = 2.0f * r;
    }
    return pack2(add_rn(sub_rn(tm0, tp0), t00), add_rn(sub_rn(tm1, tp1), t01));
}

// y / z term for the pair: both voxels share the index i along the axis
template <int MODE>
__device__ __forceinline__ f32x2 fd_adjoint_s2(const float *__restrict__ base, unsigned p, f32x2 cc, int i, int n, unsigned stride) {
    if (i >= 2 && i <= n - 3) return sub2(sub2(cc, ldg2(base + (p - 2u * stride))), sub2(ldg2(base + (p + 2u * stride)), cc));
    float c0, c1;
    unpack2(cc, c0, c1);
    return pack2(fd_adjoint<MODE>(base, p, c0, i, n, stride), fd_adjoint<MODE>(base, p + 1u, c1, i, n, stride));
}

template <int MODE>
__global__ void __launch_bounds__(NCC_THREADS, LR_REGP_BWD_MINB) diffusion_reg_backward_pair_kernel(const float *__restrict__ disp, RegDims g, int B,
                                                                                  const float *__restrict__ grad_loss,
                                                                                  float *__restrict__ grad_disp) {
    const int x = (blockIdx.x * REGP_TX + (threadIdx.x & (REGP_TX - 1))) * 2, y = blockIdx.y * REGP_TY + (threadIdx.x / REGP_TX);
    const int zc = blockIdx.z % g.n_zchunks, b = blockIdx.z / g.n_zchunks;
    const int z0 = zc * g.zchunk, z1 = min(g.d, z0 + g.zchunk);
    if (x >= g.w || y >= g.h) return;
    const unsigned pl = (unsigned)(g.h * g.w), cs = pl * (unsigned)g.d;
    const float k = (float)(2.0 * (double)grad_loss[0] / ((double)B * (double)g.d * (double)pl));
    const f32x2 kd = splat2(k * g.sd * g.sd), kh = splat2(k * g.sh * g.sh), kw = splat2(k * g.sw * g.sw);
    unsigned off = ((unsigned)b * 3u * (unsigned)g.d + (unsigned)z0) * pl + (unsigned)y * (unsigned)g.w + (unsigned)x;
    for (int z = z0; z < z1; ++z, off += pl) {
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const unsigned p = off + c * cs;
            const f32x2 cc = ldg2(disp + p);
            if (LR_REG_BWD_PF > 0 && z + LR_REG_BWD_PF + 2 < min(g.d, z1 + 2)) prefetch_l2(disp + (p + (LR_REG_BWD_PF + 2) * pl));
            f32x2 gr = mul2(kd, fd_adjoint_s2<MODE>(disp, p, cc, z, g.d, pl));
            gr = fma2(kh, fd_adjoint_s2<MODE>(disp, p, cc, y, g.h, (unsigned)g.w), gr);
            gr = fma2(kw, fd_adjoint_x2<MODE>(disp, p, cc, x, g.w), gr);
            float g0, g1;
            unpack2(gr, g0, g1);
            __stcs(reinterpret_cast<float2 *>(grad_disp + p), make_float2(g0, g1));
        }
    }
}

// Plane-march launch shape of a kernel whose block of `threads` threads owns a tile_w x tile_h tile of (last, second)
// axis positions: the per-axis scales, the chunking of the first axis and the grid.  `channels` is the number of
// (D,H,W) volumes per item the kernel indexes with 32 bits.
template <typename K>
static int march_dims(K kernel, int threads, int tile_w, int tile_h, int waves, int B, int D, int H, int W, RegDims &g, dim3 &grid,
                      int channels = 3) {
    g.d = D; g.h = H; g.w = W;
    const double sp[3] = {1.0 / (double)(D - 1) * 2.0, 1.0 / (double)(H - 1) * 2.0, 1.0 / (double)(W - 1) * 2.0};   // spacing*2 (:53-54)
    g.sd = (float)(0.5 / sp[0]); g.sh = (float)(0.5 / sp[1]); g.sw = (float)(0.5 / sp[2]);
    const int64_t tiles = (int64_t)((W + tile_w - 1) / tile_w) * ((H + tile_h - 1) / tile_h) * B;
    // ONE wave of blocks when the tiles allow it (a second, nearly empty wave would double the time of this short
    // kernel): as many chunks of planes as fit the resident-block capacity, chunks of at least 4 planes
    const int64_t capacity = (int64_t)sm_count() * blocks_per_sm(kernel, threads, 0, 4) * waves;
    int64_t chunks = capacity / tiles;
    if (chunks < 1) chunks = 1;
    if (chunks > (D + 3) / 4) chunks = (D + 3) / 4;
    g.zchunk = (int)((D + chunks - 1) / chunks);
    g.n_zchunks = (D + g.zchunk - 1) / g.zchunk;
    const int64_t gz = (int64_t)g.n_zchunks * B;
    if (gz > 65535 || (H + tile_h - 1) / tile_h > 65535) return -1;
    if ((int64_t)B * channels * D * H * W >= ((int64_t)1 << 31)) return -1;   // the kernels index with 32 bits
    grid = dim3((unsigned)((W + tile_w - 1) / tile_w), (unsigned)((H + tile_h - 1) / tile_h), (unsigned)gz);
    return 0;
}

template <typename K>
static int reg_dims(K kernel, bool pairs, int waves, int B, int D, int H, int W, RegDims &g, dim3 &grid) {
    return march_dims(kernel, NCC_THREADS, pairs ? 2 * REGP_TX : REG_TX, pairs ? REGP_TY : REG_TY, waves, B, D, H, W, g, grid);
}

static unsigned ncc_blocks(int64_t N, int B) {
    int64_t want = (N + NCC_THREADS * 8 - 1) / (NCC_THREADS * 8);          // >= 8 elements per thread
    const int64_t cap = (int64_t)sm_count() * 8 / (B < 8 ? B : 8) + 1;      // ~8 resident blocks per SM over the whole grid
    if (want > cap) want = cap;
    return (unsigned)(want < 1 ? 1 : want);
}

// the pair kernels need an even row length and 8-byte-aligned rows
static bool reg_use_pairs(const void *a, const void *b, int W) {
    return (W % 2 == 0) && ((uintptr_t)a % 8 == 0) && ((uintptr_t)b % 8 == 0);
}

// ---------------------------------------------------------------------------------------------------------------
// Validation metrics (the host-side scoring of RegistrationNet.py:198-218).  PARITY UNPINNED: the reference's
// utils.py:20-55 (Jacobian folding) and metrics.py:6-121 (label overlap) import mermaid and SimpleITK and are not part of
// this tree; the definitions here are stated from first principles (include/liftreg_b200.h).
//
// Jacobian determinant of a map phi (B,3,D,H,W) in [-1,1], channel c addressing volume axis c: J[c][a] is the
// regulariser's central difference of channel c along axis a, same face rules and scales (0.5/(2/(n-1)), so the identity
// has J = I whatever the per-axis normalisation), and the 3x3 determinant is expanded along the first row with every
// product and difference rounded on its own, left to right, so an fp32 torch restatement reproduces it bit for bit.
constexpr int JAC_STATS = 7;     // per item: #det<0, sum |det| over det<0, min, max, sum det, sum det^2, #non-finite

__device__ __forceinline__ float det3(const float (&j)[3][3]) {
    const float a = mul_rn(j[0][0], sub_rn(mul_rn(j[1][1], j[2][2]), mul_rn(j[1][2], j[2][1])));
    const float b = mul_rn(j[0][1], sub_rn(mul_rn(j[1][0], j[2][2]), mul_rn(j[1][2], j[2][0])));
    const float c = mul_rn(j[0][2], sub_rn(mul_rn(j[1][0], j[2][1]), mul_rn(j[1][1], j[2][0])));
    return add_rn(sub_rn(a, b), c);
}

// per-thread statistics; sums in fp64 (the det is fp32, so det^2 is exact in fp64), counts in integers
struct JacAcc {
    unsigned neg = 0, nonfinite = 0;
    double neg_abs = 0.0, sum = 0.0, sum2 = 0.0;
    float mn = INFINITY, mx = -INFINITY;
    __device__ __forceinline__ void add(float v, bool in) {
        if (!in) return;
        if (!isfinite(v)) { ++nonfinite; return; }
        const double d = (double)v;
        sum += d;
        sum2 = fma(d, d, sum2);
        if (v < 0.0f) { ++neg; neg_abs -= d; }
        mn = fminf(mn, v); mx = fmaxf(mx, v);
    }
};

__device__ __forceinline__ void atomic_min_f64(double *p, double v) {
    unsigned long long *a = reinterpret_cast<unsigned long long *>(p), old = *a;
    while (v < __longlong_as_double((long long)old)) {
        const unsigned long long seen = atomicCAS(a, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}
__device__ __forceinline__ void atomic_max_f64(double *p, double v) {
    unsigned long long *a = reinterpret_cast<unsigned long long *>(p), old = *a;
    while (v > __longlong_as_double((long long)old)) {
        const unsigned long long seen = atomicCAS(a, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}

// block reduction of the per-thread statistics, then one atomic per statistic and block (skipped when it cannot change
// the result: most blocks have no folds and no non-finite values)
__device__ __forceinline__ void jac_block_flush(const JacAcc &t, double *__restrict__ st) {
    __shared__ double sd[NCC_THREADS / 32][3];
    __shared__ float sf[NCC_THREADS / 32][2];
    __shared__ unsigned su[NCC_THREADS / 32][2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const double a = warp_sum(t.neg_abs), s = warp_sum(t.sum), s2 = warp_sum(t.sum2);
    const unsigned n = __reduce_add_sync(0xffffffffu, t.neg), nf = __reduce_add_sync(0xffffffffu, t.nonfinite);
    float mn = t.mn, mx = t.mx;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if (lane == 0) {
        sd[warp][0] = a; sd[warp][1] = s; sd[warp][2] = s2;
        sf[warp][0] = mn; sf[warp][1] = mx;
        su[warp][0] = n; su[warp][1] = nf;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double ta = 0.0, ts = 0.0, ts2 = 0.0;
        unsigned tn = 0, tnf = 0;
        float tmn = INFINITY, tmx = -INFINITY;
#pragma unroll
        for (int w = 0; w < NCC_THREADS / 32; ++w) {
            ta += sd[w][0]; ts += sd[w][1]; ts2 += sd[w][2];
            tn += su[w][0]; tnf += su[w][1];
            tmn = fminf(tmn, sf[w][0]); tmx = fmaxf(tmx, sf[w][1]);
        }
        if (tn) { atomicAdd(st + 0, (double)tn); atomicAdd(st + 1, ta); }
        if (tmn <= tmx) { atomic_min_f64(st + 2, (double)tmn); atomic_max_f64(st + 3, (double)tmx); }
        if (ts != 0.0) atomicAdd(st + 4, ts);
        if (ts2 != 0.0) atomicAdd(st + 5, ts2);
        if (tnf) atomicAdd(st + 6, (double)tnf);
    }
}

__global__ void jac_init_kernel(double *__restrict__ stats, int B) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < B * JAC_STATS) {
        const int k = i % JAC_STATS;
        stats[i] = k == 2 ? INFINITY : (k == 3 ? -INFINITY : 0.0);
    }
}

// one voxel per thread: the march of diffusion_reg_kernel, the nine differences kept instead of squared and summed
template <int MODE>
__global__ void __launch_bounds__(NCC_THREADS) jacobian_det_kernel(const float *__restrict__ phi, RegDims g, int margin,
                                                                   float *__restrict__ det, double *__restrict__ stats) {
    const int x = blockIdx.x * REG_TX + (threadIdx.x & 31), y = blockIdx.y * REG_TY + (threadIdx.x >> 5);
    const int zc = blockIdx.z % g.n_zchunks, b = blockIdx.z / g.n_zchunks;
    const int z0 = zc * g.zchunk, z1 = min(g.d, z0 + g.zchunk);
    JacAcc acc;
    if (x < g.w && y < g.h) {
        const bool xlo = x == 0, xhi = x == g.w - 1, ylo = y == 0, yhi = y == g.h - 1;
        const int oxu = xhi ? 0 : 1, oxd = xlo ? 0 : -1;
        const int oyu = yhi ? 0 : g.w, oyd = ylo ? 0 : -g.w;
        const bool in_xy = x >= margin && x < g.w - margin && y >= margin && y < g.h - margin;
        const unsigned pl = (unsigned)(g.h * g.w), cs = pl * (unsigned)g.d;       // 32-bit indices (B*3*D*H*W < 2^31)
        unsigned i0 = ((unsigned)b * 3u * (unsigned)g.d + (unsigned)z0) * pl + (unsigned)y * (unsigned)g.w + (unsigned)x;
        unsigned o0 = ((unsigned)b * (unsigned)g.d + (unsigned)z0) * pl + (unsigned)y * (unsigned)g.w + (unsigned)x;
        float vm[3], vc[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            vc[c] = __ldg(phi + (i0 + c * cs));
            vm[c] = z0 > 0 ? __ldg(phi + (i0 + c * cs - pl)) : vc[c];
        }
        for (int z = z0; z < z1; ++z, i0 += pl, o0 += pl) {
            const bool zlo = z == 0, zhi = z == g.d - 1;
            float j[3][3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const unsigned ic = i0 + c * cs;
                const float cc = vc[c];
                const float vp = zhi ? cc : __ldg(phi + (ic + pl));
                if (LR_REG_PF > 0 && z + LR_REG_PF <= z1) prefetch_l2(phi + (ic + LR_REG_PF * pl));
                const float yu = __ldg(phi + (ic + oyu)), yd = __ldg(phi + (ic + oyd));
                const float xu = __ldg(phi + (ic + oxu)), xd = __ldg(phi + (ic + oxd));
                j[c][0] = mul_rn(fd_delta<MODE>(vp, vm[c], cc, zlo, zhi), g.sd);
                j[c][1] = mul_rn(fd_delta<MODE>(yu, yd, cc, ylo, yhi), g.sh);
                j[c][2] = mul_rn(fd_delta<MODE>(xu, xd, cc, xlo, xhi), g.sw);
                vm[c] = cc; vc[c] = vp;
            }
            const float v = det3(j);
            if (det) st_stream(det + o0, v);
            acc.add(v, in_xy && z >= margin && z < g.d - margin);
        }
    }
    jac_block_flush(acc, stats + b * JAC_STATS);
}

// two voxels per thread (W even, 8-byte-aligned map and output): the loads and differences of diffusion_reg_pair_kernel,
// the determinant per voxel in scalar fp32 (packed products would be contracted into the subtractions by ptxas)
template <int MODE>
__global__ void __launch_bounds__(NCC_THREADS, LR_REGP_MINB) jacobian_det_pair_kernel(const float *__restrict__ phi, RegDims g, int margin,
                                                                                     float *__restrict__ det, double *__restrict__ stats) {
    const int x = (blockIdx.x * REGP_TX + (threadIdx.x & (REGP_TX - 1))) * 2, y = blockIdx.y * REGP_TY + (threadIdx.x / REGP_TX);
    const int zc = blockIdx.z % g.n_zchunks, b = blockIdx.z / g.n_zchunks;
    const int z0 = zc * g.zchunk, z1 = min(g.d, z0 + g.zchunk);
    JacAcc acc;
    if (x < g.w && y < g.h) {
        const bool xlo = x == 0, xhi = x + 2 == g.w, ylo = y == 0, yhi = y == g.h - 1;
        const int oxl = xlo ? 0 : -1, oxr = xhi ? 1 : 2;
        const int oyu = yhi ? 0 : g.w, oyd = ylo ? 0 : -g.w;
        const bool in_y = y >= margin && y < g.h - margin;
        const bool in0 = in_y && x >= margin && x < g.w - margin, in1 = in_y && x + 1 >= margin && x + 1 < g.w - margin;
        const unsigned pl = (unsigned)(g.h * g.w), cs = pl * (unsigned)g.d;
        unsigned i0 = ((unsigned)b * 3u * (unsigned)g.d + (unsigned)z0) * pl + (unsigned)y * (unsigned)g.w + (unsigned)x;
        unsigned o0 = ((unsigned)b * (unsigned)g.d + (unsigned)z0) * pl + (unsigned)y * (unsigned)g.w + (unsigned)x;
        const f32x2 sd2 = splat2(g.sd), sh2 = splat2(g.sh), sw2 = splat2(g.sw);
        f32x2 vm[3], vc[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            vc[c] = ldg2(phi + (i0 + c * cs));
            vm[c] = z0 > 0 ? ldg2(phi + (i0 + c * cs - pl)) : vc[c];
        }
        for (int z = z0; z < z1; ++z, i0 += pl, o0 += pl) {
            const bool zlo = z == 0, zhi = z == g.d - 1;
            float j0[3][3], j1[3][3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const unsigned ic = i0 + c * cs;
                const f32x2 cc = vc[c];
                const f32x2 vp = zhi ? cc : ldg2(phi + (ic + pl));
                if (LR_REG_PF > 0 && z + LR_REG_PF <= z1) prefetch_l2(phi + (ic + LR_REG_PF * pl));
                const f32x2 yu = ldg2(phi + (ic + oyu)), yd = ldg2(phi + (ic + oyd));
                float xl = __ldg(phi + (ic + oxl)), xr = __ldg(phi + (ic + oxr));
                float c0, c1;
                unpack2(cc, c0, c1);
                f32x2 dx;
                if (MODE == 0) {
                    if (xlo) xl = fmaf(2.0f, c0, -c1);
                    if (xhi) xr = fmaf(2.0f, c1, -c0);
                    dx = sub2(pack2(c1, xr), pack2(xl, c0));
                } else {
                    dx = pack2(xlo ? 0.0f : sub_rn(c1, xl), xhi ? 0.0f : sub_rn(xr, c0));
                }
                unpack2(mul2(fd_delta2<MODE>(vp, vm[c], cc, zlo, zhi), sd2), j0[c][0], j1[c][0]);
                unpack2(mul2(fd_delta2<MODE>(yu, yd, cc, ylo, yhi), sh2), j0[c][1], j1[c][1]);
                unpack2(mul2(dx, sw2), j0[c][2], j1[c][2]);
                vm[c] = cc; vc[c] = vp;
            }
            const float v0 = det3(j0), v1 = det3(j1);
            if (det) __stcs(reinterpret_cast<float2 *>(det + o0), make_float2(v0, v1));
            const bool in_z = z >= margin && z < g.d - margin;
            acc.add(v0, in0 && in_z);
            acc.add(v1, in1 && in_z);
        }
    }
    jac_block_flush(acc, stats + b * JAC_STATS);
}

// ---- d fold / d phi, fold = 1/(B*D*H*W) * sum over voxels of max(0, -det) (include/liftreg_b200.h) -----------------
// With G[c][a](u) = m(u) * C[c][a](u), C the cofactor d det / d J[c][a] and m(u) = 1 where det(u) is finite and < 0:
//     d fold / d phi_c = -(1/(B*D*H*W)) * sum_a s_a * D_a^T G[c][a]
// where D_a is the regulariser's difference operator along axis a (see fd_adjoint for its transpose).  Voxel v needs
// G[.][a] at v - e_a and v + e_a (and at v itself on the faces), so G is computed once per voxel and shared:
//   first axis  (a = 0): the block marches planes; G[.][0] of planes z-1, z, z+1 rolls through registers;
//   second axis (a = 1): the warps of a block are 16 consecutive rows; G[.][1] of the plane goes through shared memory;
//   last axis   (a = 2): a warp is 32 consecutive voxels of a row; G[.][2] comes from the neighbouring lanes.
// The outermost lanes and warps compute the halo (G of the voxels next to the tile), so a block writes the 30 x 14
// voxels of lanes 1..30 of warps 1..14: each output element is written once, by one thread, with no atomics.
constexpr int FOLD_WARPS = 16, FOLD_THREADS = 32 * FOLD_WARPS;
constexpr int FOLD_OX = 30, FOLD_OY = FOLD_WARPS - 2;

// J of the thread's column at plane z (the march and differences of jacobian_det_kernel, so det is bit for bit the
// forward's), then G = m * C; advances the plane window (vm, vc) by one plane
template <int MODE>
__device__ __forceinline__ void fold_cofactors(const float *__restrict__ phi, const RegDims &g, unsigned i0, unsigned cs, unsigned pl,
                                               int z, int oxu, int oxd, int oyu, int oyd, bool xlo, bool xhi, bool ylo, bool yhi,
                                               bool inside, float (&vm)[3], float (&vc)[3], float (&G)[3][3]) {
    const bool zlo = z == 0, zhi = z == g.d - 1;
    float j[3][3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const unsigned ic = i0 + c * cs;
        const float cc = vc[c];
        const float vp = zhi ? cc : __ldg(phi + (ic + pl));
        if (LR_REG_PF > 0 && z + LR_REG_PF < g.d) prefetch_l2(phi + (ic + LR_REG_PF * pl));
        const float yu = __ldg(phi + (ic + oyu)), yd = __ldg(phi + (ic + oyd));
        const float xu = __ldg(phi + (ic + oxu)), xd = __ldg(phi + (ic + oxd));
        j[c][0] = mul_rn(fd_delta<MODE>(vp, vm[c], cc, zlo, zhi), g.sd);
        j[c][1] = mul_rn(fd_delta<MODE>(yu, yd, cc, ylo, yhi), g.sh);
        j[c][2] = mul_rn(fd_delta<MODE>(xu, xd, cc, xlo, xhi), g.sw);
        vm[c] = cc; vc[c] = vp;
    }
    const float det = det3(j);
    const bool fold = inside && det < 0.0f && isfinite(det);
#pragma unroll
    for (int c = 0; c < 3; ++c) {
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            const int c1 = (c + 1) % 3, c2 = (c + 2) % 3, a1 = (a + 1) % 3, a2 = (a + 2) % 3;
            const float C = sub_rn(mul_rn(j[c1][a1], j[c2][a2]), mul_rn(j[c1][a2], j[c2][a1]));
            G[c][a] = fold ? C : 0.0f;
        }
    }
}

// (D^T G)(v) along one axis from G at v - e, v, v + e, for v at index i of n: interior G(v-e) - G(v+e); in linear mode
// rows 0 and n-1 of D enter with +-2 (fd_adjoint), in neumann_zero mode they are zero.  Terms outside the axis are
// selected away, never multiplied by zero, so a non-finite value there cannot leak in.
template <int MODE>
__device__ __forceinline__ float fold_adjoint(float gm, float g0, float gp, int i, int n) {
    float t = 0.0f;
    if (i >= 2) t = gm;
    else if (MODE == 0 && i == 1) t = 2.0f * gm;
    if (i <= n - 3) t = sub_rn(t, gp);
    else if (MODE == 0 && i == n - 2) t = sub_rn(t, 2.0f * gp);
    if (MODE == 0 && i == 0) t = sub_rn(t, 2.0f * g0);
    if (MODE == 0 && i == n - 1) t = add_rn(t, 2.0f * g0);
    return t;
}

template <int MODE>
__global__ void __launch_bounds__(FOLD_THREADS) jacobian_fold_backward_kernel(const float *__restrict__ phi, RegDims g, int B,
                                                                              const float *__restrict__ grad_loss,
                                                                              float *__restrict__ grad_phi) {
    __shared__ float g1s[2][3][FOLD_WARPS][32];       // G[.][1] of one plane, double-buffered over planes
    const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
    const int x = blockIdx.x * FOLD_OX - 1 + lane, y = blockIdx.y * FOLD_OY - 1 + wy;
    const int zc = blockIdx.z % g.n_zchunks, b = blockIdx.z / g.n_zchunks;
    const int z0 = zc * g.zchunk, z1 = min(g.d, z0 + g.zchunk);
    const bool inside = x >= 0 && x < g.w && y >= 0 && y < g.h;
    const bool writer = inside && lane >= 1 && lane <= FOLD_OX && wy >= 1 && wy <= FOLD_OY;
    // halo threads outside the volume run the march on the nearest voxel (in-bounds loads) and contribute G = 0
    const int xc = min(max(x, 0), g.w - 1), yc = min(max(y, 0), g.h - 1);
    const bool xlo = xc == 0, xhi = xc == g.w - 1, ylo = yc == 0, yhi = yc == g.h - 1;
    const int oxu = xhi ? 0 : 1, oxd = xlo ? 0 : -1;
    const int oyu = yhi ? 0 : g.w, oyd = ylo ? 0 : -g.w;
    const unsigned pl = (unsigned)(g.h * g.w), cs = pl * (unsigned)g.d;       // 32-bit indices (B*3*D*H*W < 2^31)
    const unsigned col = (unsigned)yc * (unsigned)g.w + (unsigned)xc, item = (unsigned)b * 3u * (unsigned)g.d * pl;
    const float k = (float)((double)grad_loss[0] / ((double)B * (double)g.d * (double)pl));
    const float kd = -k * g.sd, kh = -k * g.sh, kw = -k * g.sw;

    // prologue: G[.][0] of plane z0-1 and all of G at plane z0
    const int zs = z0 > 0 ? z0 - 1 : 0;
    float vm[3], vc[3], Gc[3][3], g0m[3] = {0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        vc[c] = __ldg(phi + (item + c * cs + (unsigned)zs * pl + col));
        vm[c] = zs > 0 ? __ldg(phi + (item + c * cs + (unsigned)(zs - 1) * pl + col)) : vc[c];
    }
    if (z0 > 0) {
        fold_cofactors<MODE>(phi, g, item + (unsigned)zs * pl + col, cs, pl, zs, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, inside, vm, vc, Gc);
#pragma unroll
        for (int c = 0; c < 3; ++c) g0m[c] = Gc[c][0];
    }
    fold_cofactors<MODE>(phi, g, item + (unsigned)z0 * pl + col, cs, pl, z0, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, inside, vm, vc, Gc);
#pragma unroll
    for (int c = 0; c < 3; ++c) g1s[z0 & 1][c][wy][lane] = Gc[c][1];
    __syncthreads();

    for (int z = z0; z < z1; ++z) {
        float gy[3][2], gx[3][2];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            gy[c][0] = g1s[z & 1][c][max(wy - 1, 0)][lane];
            gy[c][1] = g1s[z & 1][c][min(wy + 1, FOLD_WARPS - 1)][lane];
            gx[c][0] = __shfl_up_sync(0xffffffffu, Gc[c][2], 1);
            gx[c][1] = __shfl_down_sync(0xffffffffu, Gc[c][2], 1);
        }
        float Gn[3][3];
        if (z + 1 < g.d) {
            fold_cofactors<MODE>(phi, g, item + (unsigned)(z + 1) * pl + col, cs, pl, z + 1, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, inside,
                                 vm, vc, Gn);
        } else {
#pragma unroll
            for (int c = 0; c < 3; ++c) Gn[c][0] = Gn[c][1] = Gn[c][2] = 0.0f;
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) g1s[(z + 1) & 1][c][wy][lane] = Gn[c][1];
        if (writer) {
            const unsigned o = item + (unsigned)z * pl + col;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                float gr = mul_rn(kd, fold_adjoint<MODE>(g0m[c], Gc[c][0], Gn[c][0], z, g.d));
                gr = fmaf(kh, fold_adjoint<MODE>(gy[c][0], Gc[c][1], gy[c][1], y, g.h), gr);
                gr = fmaf(kw, fold_adjoint<MODE>(gx[c][0], Gc[c][2], gx[c][1], x, g.w), gr);
                st_stream(grad_phi + (o + c * cs), gr);
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            g0m[c] = Gc[c][0];
            Gc[c][0] = Gn[c][0]; Gc[c][1] = Gn[c][1]; Gc[c][2] = Gn[c][2];
        }
        __syncthreads();
    }
}

// ---- label confusion matrix: counts[b][p][t] = #voxels with pred == p and target == t ------------------------------
// Every (pred, target) pair that is not two integers in [0, L) goes to one extra bin, key L*L, reported as `invalid`.
// The histogram is privatised in shared memory ((L*L+1) 32-bit bins, <= 64 KB at L = 128) and merged into the int64
// output with one 64-bit atomic per non-empty bin and block.  Label maps are mostly background, so equal keys are
// first aggregated within the warp (all lanes equal: one atomic; otherwise __match_any_sync groups) before the shared
// atomic: without that, L = 2 would serialise every warp on one bin.
constexpr int CONF_THREADS = 256;

// key of a (pred, target) pair; (v + 1.5*2^23) - 1.5*2^23 == v holds exactly for the integers |v| < 2^22, and the
// integer is in the mantissa (rint_i): no F2I / FRND on the XU pipe
__device__ __forceinline__ int label_key(float p, float t, int L, float fL) {
    const float M = 12582912.0f;
    const float tp = __fadd_rn(p, M), tt = __fadd_rn(t, M);
    const bool ok = p >= 0.0f && p < fL && t >= 0.0f && t < fL && __fsub_rn(tp, M) == p && __fsub_rn(tt, M) == t;
    return ok ? (__float_as_int(tp) - 0x4B400000) * L + (__float_as_int(tt) - 0x4B400000) : L * L;
}

// the same test for one value: its label l if it is an integer in [0, L), else -1.  (Written out again rather than
// called from label_key, which then compiles differently.)
__device__ __forceinline__ int label_of(float v, float fL) {
    const float M = 12582912.0f;
    const float t = __fadd_rn(v, M);
    return v >= 0.0f && v < fL && __fsub_rn(t, M) == v ? __float_as_int(t) - 0x4B400000 : -1;
}

// one key per lane (key < 0: lane has nothing), called by the whole warp
__device__ __forceinline__ void hist_add_warp(unsigned *__restrict__ h, int key, int lane) {
    const int k0 = __shfl_sync(0xffffffffu, key, 0);
    if (__all_sync(0xffffffffu, key == k0)) {
        if (lane == 0 && k0 >= 0) atomicAdd(h + k0, 32u);
        return;
    }
    const unsigned peers = __match_any_sync(0xffffffffu, key);
    if (key >= 0 && lane == __ffs(peers) - 1) atomicAdd(h + key, (unsigned)__popc(peers));
}

__global__ void __launch_bounds__(CONF_THREADS) label_confusion_kernel(const float *__restrict__ pred, const float *__restrict__ target,
                                                                       int64_t N, int L, unsigned long long *__restrict__ counts,
                                                                       unsigned long long *__restrict__ invalid) {
    extern __shared__ unsigned hist[];
    const int nbins = L * L + 1, b = blockIdx.y, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < nbins; i += CONF_THREADS) hist[i] = 0u;
    __syncthreads();
    const float fL = (float)L;
    const float *pb = pred + (int64_t)b * N, *tb = target + (int64_t)b * N;
    // warp-uniform trip counts (every lane of a warp runs every iteration; lanes past the end carry key -1)
    const int64_t wid = ((int64_t)blockIdx.x * CONF_THREADS + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * CONF_THREADS) >> 5;
    const int64_t n4 = (((uintptr_t)pb | (uintptr_t)tb) % 16 == 0) ? N / 4 : 0;
    for (int64_t base = wid * 32; base < n4; base += nwarps * 32) {
        const int64_t i = base + lane;
        int k[4] = {-1, -1, -1, -1};
        if (i < n4) {
            const float4 p = ld_stream4(reinterpret_cast<const float4 *>(pb) + i), t = ld_stream4(reinterpret_cast<const float4 *>(tb) + i);
            k[0] = label_key(p.x, t.x, L, fL); k[1] = label_key(p.y, t.y, L, fL);
            k[2] = label_key(p.z, t.z, L, fL); k[3] = label_key(p.w, t.w, L, fL);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) hist_add_warp(hist, k[j], lane);
    }
    for (int64_t base = 4 * n4 + wid * 32; base < N; base += nwarps * 32) {
        const int64_t i = base + lane;
        hist_add_warp(hist, i < N ? label_key(ld_stream(pb + i), ld_stream(tb + i), L, fL) : -1, lane);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < nbins; i += CONF_THREADS) {
        const unsigned c = hist[i];
        if (c) atomicAdd(i < nbins - 1 ? counts + (int64_t)b * (nbins - 1) + i : invalid + b, (unsigned long long)c);
    }
}

static unsigned conf_blocks(int64_t N, int B, int L, int per_sm) {
    int64_t want = (N + CONF_THREADS * 16 - 1) / (CONF_THREADS * 16);          // >= 16 voxels per thread
    const int64_t by_bins = N / (4 * (int64_t)L * L);                          // the merge stays small next to the streaming
    if (want > by_bins) want = by_bins;
    const int64_t cap = ((int64_t)sm_count() * per_sm + B - 1) / B;              // one wave over the whole grid
    if (want > cap) want = cap;
    return (unsigned)(want < 1 ? 1 : want);
}

// ---- local (windowed) NCC, a training similarity (include/liftreg_b200.h; PARITY UNPINNED: the reference has none) ----
// Every quantity is a zero-padded box sum over the w x w x w cube centred on a voxel: the forward sums the five moments
// x, y, x^2, y^2, xy; the adjoint sums the three per-centre coefficients alpha, beta, gamma.  One plane-march kernel
// serves all three passes (LNCC_FWD: cc summed per item; LNCC_COEF: alpha, beta, gamma written to the workspace;
// LNCC_GRAD: their box sums combined with x and y into grad_x).  A block owns a 32 x 8 tile of (last, second) axis
// positions and marches a chunk of planes of the first axis.  Per input plane it
//   stages the plane's moments over the tile plus a halo of w-1 in shared memory (fp64: the products x*x, x*y of fp32
//     values are exact there),
//   sums w consecutive entries along the last axis (row pass, shared memory) and then w rows (column pass),
//   and keeps the 2-D sum in a ring of w planes per thread (shared memory), from which an output's window sum is the
//     sum of its w planes in plane order.
// Every window sum is thus a plain fp64 sum of its own terms in a fixed order -- no running add / subtract along an
// axis, no dependence on the tiling, the z chunking or the batch size -- so results repeat bit for bit and the
// cancellation in var = Sxx - Sx^2/n (the CT body at ~1 with 0.01 noise: var / Sxx ~ 1e-4) costs fp64, not fp32, digits.
// Each output element is written once, with no atomics.
constexpr int LNCC_TX = 32, LNCC_TY = 8, LNCC_THREADS = LNCC_TX * LNCC_TY, LNCC_WMAX = 15;
static_assert(LNCC_THREADS == NCC_THREADS, "local_ncc_kernel<fwd> reduces with block_accumulate_f64, sized for NCC_THREADS");
enum { LNCC_FWD = 0, LNCC_COEF = 1, LNCC_GRAD = 2 };

struct LnccDims {
    int D, H, W, w, tiles_x, tiles_y, zchunk, n_zchunks;
    unsigned N, total;     // voxels per item and in all B items (B*D*H*W < 2^31)
    double n, eps, count;  // n = w^3, count = B*D*H*W
};

template <int KIND> struct LnccMoments { static constexpr int NM = KIND == LNCC_GRAD ? 3 : 5; };

// dynamic shared memory of one block: ring[w][NM][threads] + rows[NM][TY+w-1][TX] + tile[NM][TY+w-1][TX+w-1], fp64
template <int KIND>
static size_t lncc_smem_bytes(int w) {
    const int nm = LnccMoments<KIND>::NM;
    return sizeof(double) * (size_t)nm * ((size_t)w * LNCC_THREADS + (size_t)(LNCC_TY + w - 1) * LNCC_TX +
                                          (size_t)(LNCC_TY + w - 1) * (LNCC_TX + w - 1));
}

template <int KIND>
__global__ void __launch_bounds__(LNCC_THREADS) local_ncc_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                                 const float *__restrict__ coef, LnccDims g,
                                                                 const float *__restrict__ grad_loss, double *__restrict__ sum,
                                                                 float *__restrict__ out) {
    constexpr int NM = LnccMoments<KIND>::NM;
    extern __shared__ double lncc_smem[];
    const int w = g.w, r = w >> 1, th = LNCC_TY + w - 1, tw = LNCC_TX + w - 1;
    double *ring = lncc_smem;                                   // [w][NM][LNCC_THREADS], private to each thread
    double *rows = ring + (size_t)w * NM * LNCC_THREADS;        // [NM][th][LNCC_TX]
    double *tile = rows + (size_t)NM * th * LNCC_TX;            // [NM][th][tw]
    const int tid = threadIdx.x, lane = tid & 31, wy = tid >> 5;

    unsigned blk = blockIdx.x;                                  // (tile x, tile y, z chunk, item), x fastest
    const int tx = blk % g.tiles_x; blk /= g.tiles_x;
    const int ty = blk % g.tiles_y; blk /= g.tiles_y;
    const int zc = blk % g.n_zchunks;
    const int b = blk / g.n_zchunks;
    const int x0 = tx * LNCC_TX, y0 = ty * LNCC_TY, z0 = zc * g.zchunk, z1 = min(g.D, z0 + g.zchunk);
    const int ox = x0 + lane, oy = y0 + wy;
    const bool writer = ox < g.W && oy < g.H;
    const unsigned plane = (unsigned)g.H * (unsigned)g.W, item = (unsigned)b * g.N;
    const float *c0 = coef, *c1 = coef + g.total, *c2 = coef + 2 * (size_t)g.total;     // alpha, beta, gamma (LNCC_GRAD)
    double acc = 0.0;

    for (int p = z0 - r; p < z1 + r; ++p) {
        const int slot = (p + w) % w;                           // p >= -r > -w
        double P[NM];
        if (p < 0 || p >= g.D) {                                // a plane of the zero padding
#pragma unroll
            for (int m = 0; m < NM; ++m) P[m] = 0.0;
        } else {
            // stage the plane's moments over tile + halo (zero outside the volume)
            const unsigned pbase = item + (unsigned)p * plane;
            for (int i = tid; i < th * tw; i += LNCC_THREADS) {
                const int gy = y0 - r + i / tw, gx = x0 - r + i % tw;
                double v[NM];
#pragma unroll
                for (int m = 0; m < NM; ++m) v[m] = 0.0;
                if (gy >= 0 && gy < g.H && gx >= 0 && gx < g.W) {
                    const unsigned e = pbase + (unsigned)gy * (unsigned)g.W + (unsigned)gx;
                    if (KIND == LNCC_GRAD) {
                        v[0] = (double)__ldg(c0 + e); v[1] = (double)__ldg(c1 + e); v[2] = (double)__ldg(c2 + e);
                    } else {
                        const double a = (double)__ldg(x + e), c = (double)__ldg(y + e);
                        v[0] = a; v[1] = c; v[2] = a * a; v[3] = c * c; v[NM - 1] = a * c;      // exact products
                    }
                }
#pragma unroll
                for (int m = 0; m < NM; ++m) tile[(size_t)m * th * tw + i] = v[m];
            }
            __syncthreads();
            // row pass: w consecutive entries along the last axis, in index order
            for (int i = tid; i < th * LNCC_TX; i += LNCC_THREADS) {
                const int ry = i / LNCC_TX, rx = i % LNCC_TX;
#pragma unroll
                for (int m = 0; m < NM; ++m) {
                    const double *t = tile + (size_t)m * th * tw + ry * tw + rx;
                    double s = t[0];
                    for (int d = 1; d < w; ++d) s += t[d];
                    rows[(size_t)m * th * LNCC_TX + i] = s;
                }
            }
            __syncthreads();
            // column pass: w rows, in index order
#pragma unroll
            for (int m = 0; m < NM; ++m) {
                const double *t = rows + (size_t)m * th * LNCC_TX + wy * LNCC_TX + lane;
                double s = t[0];
                for (int d = 1; d < w; ++d) s += t[d * LNCC_TX];
                P[m] = s;
            }
        }
#pragma unroll
        for (int m = 0; m < NM; ++m) ring[((size_t)slot * NM + m) * LNCC_THREADS + tid] = P[m];

        const int z = p - r;                                    // the output plane whose window closes with plane p
        if (z < z0 || !writer) continue;
        double S[NM];
#pragma unroll
        for (int m = 0; m < NM; ++m) S[m] = 0.0;
        for (int q = z - r; q <= z + r; ++q) {                  // plane order, whatever the ring's phase
            const double *s = ring + (size_t)((q + w) % w) * NM * LNCC_THREADS + tid;
#pragma unroll
            for (int m = 0; m < NM; ++m) S[m] += s[(size_t)m * LNCC_THREADS];
        }
        const unsigned e = item + (unsigned)z * plane + (unsigned)oy * (unsigned)g.W + (unsigned)ox;
        if (KIND == LNCC_GRAD) {
            // grad_x = -(g / (B*D*H*W)) * (y * sum alpha - x * sum beta + sum gamma)
            const double k = (double)grad_loss[0] / g.count;
            const double t = (double)__ldg(y + e) * S[0] - (double)__ldg(x + e) * S[1] + S[2];
            out[e] = (float)(-k * t);
        } else {
            const double cross = S[4] - S[0] * S[1] / g.n;
            const double vx = S[2] - S[0] * S[0] / g.n, vy = S[3] - S[1] * S[1] / g.n;
            const double d = vx * vy + g.eps;
            if (KIND == LNCC_FWD) {
                if (d > 0.0) acc += cross * cross / d;
            } else {
                double al = 0.0, be = 0.0, ga = 0.0;
                if (d > 0.0) {
                    al = 2.0 * cross / d;
                    be = 2.0 * cross * cross * vy / (d * d);
                    ga = be * (S[0] / g.n) - al * (S[1] / g.n);
                }
                out[e] = (float)al; out[e + (size_t)g.total] = (float)be; out[e + 2 * (size_t)g.total] = (float)ga;
            }
        }
    }
    if (KIND == LNCC_FWD) block_accumulate_f64(acc, sum + b);
}

// ---- soft Dice of the trilinearly warped label map, a training term (include/liftreg_b200.h; PARITY UNPINNED) ----------
// VoxelMorph's semi-supervised term without its L one-hot channels: a voxel's soft probability of label l is the total
// weight of its 8 taps whose moving label is l, so the sums need only the tap weights keyed by the tap's label, and the
// adjoint one coefficient per tap (a[l], or a[l] + e[l] where the tap's label is the target's).  Both kernels march a
// chunk of planes of a 32 x 8 tile of (last, second) axis positions, one voxel per thread; neither cost depends on L.
constexpr int DICE_TX = 32, DICE_TY = 8, DICE_THREADS = DICE_TX * DICE_TY, DICE_LMAX = 128;
static_assert(DICE_THREADS >= DICE_LMAX, "the adjoint derives one label's coefficients per thread");

struct DiceDims {
    RegDims m;                // d, h, w and the chunking of the first axis (march_dims)
    float hx, hy, hz;         // (S-1)/2 per axis, the warp's unnormalisation
    float cx, cy, cz;         // (S-1) + 2, the warp's clamp_index bound under zeros padding
    int L;
};

// The sample position of voxel `vox` of an item under its map phi_b exactly as lr_warp_forward computes it (zeros
// padding, no using_scale): the fractions w?[0] (lower tap) and w?[1] (upper tap) of each axis, and the label of each
// of the 8 taps, t = tx + 2 ty + 4 tz (-1: outside the volume, or no label).
__device__ __forceinline__ void dice_taps(const float *__restrict__ phi_b, const float *__restrict__ src_b, const DiceDims &g,
                                          unsigned vox, unsigned N, float fL, float (&wx)[2], float (&wy)[2], float (&wz)[2],
                                          int (&lab)[8]) {
    // channel c of phi addresses volume axis c
    const float iz = clamp_index(source_index<LR_PAD_ZEROS>(ld_stream(phi_b + vox), g.hz, 0.0f), g.cz);
    const float iy = clamp_index(source_index<LR_PAD_ZEROS>(ld_stream(phi_b + N + vox), g.hy, 0.0f), g.cy);
    const float ix = clamp_index(source_index<LR_PAD_ZEROS>(ld_stream(phi_b + 2u * N + vox), g.hx, 0.0f), g.cx);
    float fx, fy, fz;
    int x0, y0, z0;
    floor_fi(ix, fx, x0);
    floor_fi(iy, fy, y0);
    floor_fi(iz, fz, z0);
    wx[0] = sub_rn(add_rn(fx, 1.0f), ix); wx[1] = sub_rn(ix, fx);
    wy[0] = sub_rn(add_rn(fy, 1.0f), iy); wy[1] = sub_rn(iy, fy);
    wz[0] = sub_rn(add_rn(fz, 1.0f), iz); wz[1] = sub_rn(iz, fz);
    const int W = g.m.w, HW = g.m.h * g.m.w;
    const int base = z0 * HW + y0 * W + x0;                   // may be negative: only in-bounds taps are read
#pragma unroll
    for (int t = 0; t < 8; ++t) {
        const int tx = t & 1, ty = (t >> 1) & 1, tz = t >> 2;
        const bool ok = (unsigned)(x0 + tx) < (unsigned)W && (unsigned)(y0 + ty) < (unsigned)g.m.h && (unsigned)(z0 + tz) < (unsigned)g.m.d;
        lab[t] = ok ? label_of(__ldg(src_b + (base + tx + ty * W + tz * HW)), fL) : -1;
    }
}

// end-of-thread flush of the run accumulators into the block's bins: one shared atomic per warp when every lane holds
// the same label (the common case), else one per lane
__device__ __forceinline__ void dice_flush(int kp, double ap, double ai, int kt, unsigned at, double *sp, double *si,
                                           unsigned *st, int lane) {
    const int p0 = __shfl_sync(0xffffffffu, kp, 0);
    if (__all_sync(0xffffffffu, kp == p0)) {
        ap = warp_sum(ap); ai = warp_sum(ai);
        if (lane == 0 && p0 >= 0) { atomicAdd(sp + p0, ap); atomicAdd(si + p0, ai); }
    } else if (kp >= 0) {
        atomicAdd(sp + kp, ap); atomicAdd(si + kp, ai);
    }
    const int t0 = __shfl_sync(0xffffffffu, kt, 0);
    if (__all_sync(0xffffffffu, kt == t0)) {
        const unsigned n = __reduce_add_sync(0xffffffffu, at);
        if (lane == 0 && t0 >= 0) atomicAdd(st + t0, n);
    } else if (kt >= 0) {
        atomicAdd(st + kt, at);
    }
}

// Forward: sums[b][l] = {I, P, T}.  Each thread keeps run accumulators for the last tap label (P and I, fp64 from the
// fp32 tap weights) and the last target label (T, an integer count) and flushes a run to the block's shared bins when
// the label changes; label maps are mostly large regions, so a thread marching planes rarely does.  The block then adds
// each non-empty bin to sums with one fp64 atomic.
__global__ void __launch_bounds__(DICE_THREADS) label_dice_sums_kernel(const float *__restrict__ phi, const float *__restrict__ src,
                                                                      const float *__restrict__ tgt, DiceDims g, double *__restrict__ sums) {
    __shared__ double sp[DICE_LMAX], si[DICE_LMAX];
    __shared__ unsigned st[DICE_LMAX];
    const int tid = threadIdx.x, lane = tid & 31;
    for (int l = tid; l < g.L; l += DICE_THREADS) { sp[l] = 0.0; si[l] = 0.0; st[l] = 0u; }
    __syncthreads();
    const int x = blockIdx.x * DICE_TX + lane, y = blockIdx.y * DICE_TY + (tid >> 5);
    const int zc = blockIdx.z % g.m.n_zchunks, b = blockIdx.z / g.m.n_zchunks;
    const int z0 = zc * g.m.zchunk, z1 = min(g.m.d, z0 + g.m.zchunk);
    const float fL = (float)g.L;
    int kp = -1, kt = -1;
    double ap = 0.0, ai = 0.0;
    unsigned at = 0u;
    if (x < g.m.w && y < g.m.h) {
        const unsigned plane = (unsigned)g.m.h * (unsigned)g.m.w, N = plane * (unsigned)g.m.d;     // B*3*N < 2^31
        const float *phi_b = phi + 3u * (unsigned)b * N, *src_b = src + (unsigned)b * N, *tgt_b = tgt + (unsigned)b * N;
        unsigned vox = (unsigned)z0 * plane + (unsigned)y * (unsigned)g.m.w + (unsigned)x;
        for (int z = z0; z < z1; ++z, vox += plane) {
            float wx[2], wy[2], wz[2];
            int lab[8];
            dice_taps(phi_b, src_b, g, vox, N, fL, wx, wy, wz, lab);
            const int lt = label_of(ld_stream(tgt_b + vox), fL);
            if (lt != kt) {
                if (kt >= 0) atomicAdd(st + kt, at);
                kt = lt; at = 0u;
            }
            ++at;
            // the weights of warp_one: (wx * wy) * wz
            const float a00 = mul_rn(wx[0], wy[0]), a10 = mul_rn(wx[1], wy[0]), a01 = mul_rn(wx[0], wy[1]), a11 = mul_rn(wx[1], wy[1]);
            const float wt[8] = {mul_rn(a00, wz[0]), mul_rn(a10, wz[0]), mul_rn(a01, wz[0]), mul_rn(a11, wz[0]),
                                 mul_rn(a00, wz[1]), mul_rn(a10, wz[1]), mul_rn(a01, wz[1]), mul_rn(a11, wz[1])};
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                const int l = lab[t];
                if (l < 0) continue;
                if (l != kp) {
                    if (kp >= 0) { atomicAdd(sp + kp, ap); atomicAdd(si + kp, ai); }
                    kp = l; ap = 0.0; ai = 0.0;
                }
                const double w = (double)wt[t];
                ap += w;
                if (l == lt) ai += w;
            }
        }
    }
    dice_flush(kp, ap, ai, kt, at, sp, si, st, lane);
    __syncthreads();
    double *s = sums + (size_t)b * g.L * 3;
    for (int l = tid; l < g.L; l += DICE_THREADS) {
        if (si[l] != 0.0) atomicAdd(s + 3 * l, si[l]);
        if (sp[l] != 0.0) atomicAdd(s + 3 * l + 1, sp[l]);
        if (st[l] != 0u) atomicAdd(s + 3 * l + 2, (double)st[l]);
    }
}

// Adjoint.  loss = 1 - (1/B) sum_b (1/|S_b|) sum_{l in S_b} 2 I / (P + T), so per label of S_b
//     a = d loss / d P = 2 I / (B |S_b| (P + T)^2),   e = d loss / d I = -2 / (B |S_b| (P + T)),
// both times grad_loss, formed in fp64 and rounded once to fp32 (a, and a + e for the taps whose label is the
// target's).  The block derives them for its item into shared memory; then each thread gathers the 8 taps of its voxel
// and evaluates d/di_c of the trilinear blend of the tap coefficients as the warp's d/dphi does: a tree of fused lerps
// over tap differences, so a voxel whose 8 coefficients are equal gets exactly 0.  Each output is written once.
__global__ void __launch_bounds__(DICE_THREADS) label_dice_backward_kernel(const float *__restrict__ phi, const float *__restrict__ src,
                                                                          const float *__restrict__ tgt, DiceDims g, int B,
                                                                          const double *__restrict__ sums,
                                                                          const float *__restrict__ grad_loss,
                                                                          float *__restrict__ grad_phi) {
    __shared__ float sa[DICE_LMAX], sae[DICE_LMAX];
    const int tid = threadIdx.x, lane = tid & 31;
    const int zc = blockIdx.z % g.m.n_zchunks, b = blockIdx.z / g.m.n_zchunks;
    const double *s = sums + (size_t)b * g.L * 3;
    double I = 0.0, den = 0.0;
    bool in = false;                                          // l in S_b: l >= 1 and P + T > 0
    if (tid >= 1 && tid < g.L) {
        I = s[3 * tid]; den = s[3 * tid + 1] + s[3 * tid + 2];
        in = den > 0.0;
    }
    const int n_in = __syncthreads_count(in);
    if (tid < g.L) {
        double a = 0.0, e = 0.0;
        if (in) {
            const double k = 2.0 * (double)grad_loss[0] / ((double)B * (double)n_in);
            a = k * I / (den * den);
            e = -k / den;
        }
        sa[tid] = (float)a;
        sae[tid] = (float)(a + e);
    }
    __syncthreads();
    const int x = blockIdx.x * DICE_TX + lane, y = blockIdx.y * DICE_TY + (tid >> 5);
    if (x >= g.m.w || y >= g.m.h) return;
    const int z0 = zc * g.m.zchunk, z1 = min(g.m.d, z0 + g.m.zchunk);
    const float fL = (float)g.L;
    const unsigned plane = (unsigned)g.m.h * (unsigned)g.m.w, N = plane * (unsigned)g.m.d;
    const float *phi_b = phi + 3u * (unsigned)b * N, *src_b = src + (unsigned)b * N, *tgt_b = tgt + (unsigned)b * N;
    float *gp = grad_phi + 3u * (unsigned)b * N;
    unsigned vox = (unsigned)z0 * plane + (unsigned)y * (unsigned)g.m.w + (unsigned)x;
    for (int z = z0; z < z1; ++z, vox += plane) {
        float wx[2], wy[2], wz[2];
        int lab[8];
        dice_taps(phi_b, src_b, g, vox, N, fL, wx, wy, wz, lab);
        const int lt = label_of(ld_stream(tgt_b + vox), fL);
        float v[8];
#pragma unroll
        for (int t = 0; t < 8; ++t) {
            const int l = max(lab[t], 0);
            const float c = lab[t] == lt ? sae[l] : sa[l];
            v[t] = lab[t] < 0 ? 0.0f : c;
        }
        // d/di_c = sum over the 4 tap pairs along axis c of (upper - lower coefficient) * (the pair's weight in the other
        // two axes).  The differences come first, so equal coefficients give exactly 0; the pair weights are the fp32
        // fractions' products (not the lerp form of the warp's d/dphi, whose implied 1 - w differs from w0), so each
        // rounding is relative to a term of the abs-scale (DESIGN.md section 3)
        float gxyz[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {                         // c: 0 = x (last axis), 1 = y, 2 = z
            const int step = 1 << c;                          // tap index step along axis c
            float acc = 0.0f;
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const int lo = c == 0 ? 2 * p : (c == 1 ? (p & 1) + 4 * (p >> 1) : p);       // lower tap of pair p
                const int tx = lo & 1, ty = (lo >> 1) & 1, tz = lo >> 2;
                const float w = c == 0 ? mul_rn(wy[ty], wz[tz]) : (c == 1 ? mul_rn(wx[tx], wz[tz]) : mul_rn(wx[tx], wy[ty]));
                const float d = sub_rn(v[lo + step], v[lo]);
                acc = p == 0 ? mul_rn(w, d) : fma_rn(w, d, acc);
            }
            gxyz[c] = acc;
        }
        st_stream(gp + vox, mul_rn(g.hz, gxyz[2]));
        st_stream(gp + N + vox, mul_rn(g.hy, gxyz[1]));
        st_stream(gp + 2u * N + vox, mul_rn(g.hx, gxyz[0]));
    }
}

// ---- normalized gradient field (NGF) similarity (include/liftreg_b200.h, lr_ngf_sum; PARITY UNPINNED) -------------
// g = s * D x and h = s * D y are the fp32 differences lr_jacobian_det forms for one channel.  Per voxel, in fp64,
//     a = g.h,  p = |g|^2 + eps^2,  q = |h|^2 + eps^2,  f = a^2 / (p q);   loss = 1 - mean f
//     d loss / d x = -(1/(B*D*H*W)) * sum_a s_a * D_a^T c_a,   c_a = (2a/(pq)) * (h_a - (a/p) * g_a)
// The adjoint has the fold adjoint's shape with a 3-vector c per voxel in place of the nine cofactors, so it uses
// jacobian_fold_backward_kernel's layout.  Every voxel is evaluated by one fixed sequence of operations (fp64 products
// of fp32 values, left to right, no contraction), so f and c do not depend on the launch shape or the batch.

// one volume's scaled differences at plane z of the thread's column (element index i); advances its plane window
template <int MODE>
__device__ __forceinline__ void ngf_diffs(const float *__restrict__ v, const RegDims &g, unsigned i, unsigned pl, int z, int oxu,
                                          int oxd, int oyu, int oyd, bool xlo, bool xhi, bool ylo, bool yhi, float &vm, float &vc,
                                          float (&d)[3]) {
    const bool zlo = z == 0, zhi = z == g.d - 1;
    const float cc = vc;
    const float vp = zhi ? cc : __ldg(v + (i + pl));
    if (LR_REG_PF > 0 && z + LR_REG_PF < g.d) prefetch_l2(v + (i + LR_REG_PF * pl));
    const float yu = __ldg(v + (i + oyu)), yd = __ldg(v + (i + oyd));
    const float xu = __ldg(v + (i + oxu)), xd = __ldg(v + (i + oxd));
    d[0] = mul_rn(fd_delta<MODE>(vp, vm, cc, zlo, zhi), g.sd);
    d[1] = mul_rn(fd_delta<MODE>(yu, yd, cc, ylo, yhi), g.sh);
    d[2] = mul_rn(fd_delta<MODE>(xu, xd, cc, xlo, xhi), g.sw);
    vm = cc; vc = vp;
}

// a, p, q of one voxel in fp64 (the products of fp32 values are exact; the sums are rounded left to right)
__device__ __forceinline__ void ngf_terms(const float (&gx)[3], const float (&hy)[3], double eps2, double &a, double &p, double &q) {
    const double g0 = gx[0], g1 = gx[1], g2 = gx[2], h0 = hy[0], h1 = hy[1], h2 = hy[2];
    a = g0 * h0 + g1 * h1 + g2 * h2;
    p = g0 * g0 + g1 * g1 + g2 * g2 + eps2;
    q = h0 * h0 + h1 * h1 + h2 * h2 + eps2;
}

// forward: the march of jacobian_det_kernel over two single-channel volumes, f summed per thread in fp64
template <int MODE>
__global__ void __launch_bounds__(NCC_THREADS) ngf_sum_kernel(const float *__restrict__ x, const float *__restrict__ y, RegDims g,
                                                              double eps2, double *__restrict__ sum) {
    const int xi = blockIdx.x * REG_TX + (threadIdx.x & 31), yi = blockIdx.y * REG_TY + (threadIdx.x >> 5);
    const int zc = blockIdx.z % g.n_zchunks, b = blockIdx.z / g.n_zchunks;
    const int z0 = zc * g.zchunk, z1 = min(g.d, z0 + g.zchunk);
    double acc = 0.0;
    if (xi < g.w && yi < g.h) {
        const bool xlo = xi == 0, xhi = xi == g.w - 1, ylo = yi == 0, yhi = yi == g.h - 1;
        const int oxu = xhi ? 0 : 1, oxd = xlo ? 0 : -1;
        const int oyu = yhi ? 0 : g.w, oyd = ylo ? 0 : -g.w;
        const unsigned pl = (unsigned)(g.h * g.w);                                // 32-bit indices (B*D*H*W < 2^31)
        unsigned i0 = ((unsigned)b * (unsigned)g.d + (unsigned)z0) * pl + (unsigned)yi * (unsigned)g.w + (unsigned)xi;
        float xm, xc = __ldg(x + i0), ym, yc = __ldg(y + i0);
        xm = z0 > 0 ? __ldg(x + (i0 - pl)) : xc;
        ym = z0 > 0 ? __ldg(y + (i0 - pl)) : yc;
        for (int z = z0; z < z1; ++z, i0 += pl) {
            float gx[3], hy[3];
            ngf_diffs<MODE>(x, g, i0, pl, z, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, xm, xc, gx);
            ngf_diffs<MODE>(y, g, i0, pl, z, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, ym, yc, hy);
            double a, p, q;
            ngf_terms(gx, hy, eps2, a, p, q);
            acc += a * a / (p * q);
        }
    }
    block_accumulate_f64(acc, sum + b);
}

// c of the thread's column at plane z (0 for a halo thread outside the volume); advances both plane windows
template <int MODE>
__device__ __forceinline__ void ngf_coefs(const float *__restrict__ x, const float *__restrict__ y, const RegDims &g, unsigned i,
                                          unsigned pl, int z, int oxu, int oxd, int oyu, int oyd, bool xlo, bool xhi, bool ylo,
                                          bool yhi, bool inside, double eps2, float (&vm)[2], float (&vc)[2], float (&c)[3]) {
    float gx[3], hy[3];
    ngf_diffs<MODE>(x, g, i, pl, z, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, vm[0], vc[0], gx);
    ngf_diffs<MODE>(y, g, i, pl, z, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, vm[1], vc[1], hy);
    double a, p, q;
    ngf_terms(gx, hy, eps2, a, p, q);
    const double t = 2.0 * a / (p * q), r = a / p;
#pragma unroll
    for (int k = 0; k < 3; ++k) c[k] = inside ? (float)(t * ((double)hy[k] - r * (double)gx[k])) : 0.0f;
}

// adjoint: jacobian_fold_backward_kernel's layout (16 warps, 30 x 14 outputs per block, halo threads clamped to the
// nearest voxel): D_z^T from a 3-plane register window of c0, D_y^T through a double-buffered shared plane of c1,
// D_x^T from lane shuffles of c2; each output element written once, no atomics
template <int MODE>
__global__ void __launch_bounds__(FOLD_THREADS) ngf_backward_kernel(const float *__restrict__ x, const float *__restrict__ y, RegDims g,
                                                                    int B, double eps2, const float *__restrict__ grad_loss,
                                                                    float *__restrict__ grad_x) {
    __shared__ float c1s[2][FOLD_WARPS][32];          // c1 of one plane, double-buffered over planes
    const int lane = threadIdx.x & 31, wy = threadIdx.x >> 5;
    const int xi = blockIdx.x * FOLD_OX - 1 + lane, yi = blockIdx.y * FOLD_OY - 1 + wy;
    const int zc = blockIdx.z % g.n_zchunks, b = blockIdx.z / g.n_zchunks;
    const int z0 = zc * g.zchunk, z1 = min(g.d, z0 + g.zchunk);
    const bool inside = xi >= 0 && xi < g.w && yi >= 0 && yi < g.h;
    const bool writer = inside && lane >= 1 && lane <= FOLD_OX && wy >= 1 && wy <= FOLD_OY;
    const int xc = min(max(xi, 0), g.w - 1), yc = min(max(yi, 0), g.h - 1);
    const bool xlo = xc == 0, xhi = xc == g.w - 1, ylo = yc == 0, yhi = yc == g.h - 1;
    const int oxu = xhi ? 0 : 1, oxd = xlo ? 0 : -1;
    const int oyu = yhi ? 0 : g.w, oyd = ylo ? 0 : -g.w;
    const unsigned pl = (unsigned)(g.h * g.w);                                    // 32-bit indices (B*D*H*W < 2^31)
    const unsigned col = (unsigned)yc * (unsigned)g.w + (unsigned)xc, item = (unsigned)b * (unsigned)g.d * pl;
    const float k = (float)((double)grad_loss[0] / ((double)B * (double)g.d * (double)pl));
    const float kd = -k * g.sd, kh = -k * g.sh, kw = -k * g.sw;

    // prologue: c0 of plane z0-1 and all of c at plane z0
    const int zs = z0 > 0 ? z0 - 1 : 0;
    float vm[2], vc[2], Cc[3], c0m = 0.0f;
    vc[0] = __ldg(x + (item + (unsigned)zs * pl + col));
    vc[1] = __ldg(y + (item + (unsigned)zs * pl + col));
    vm[0] = zs > 0 ? __ldg(x + (item + (unsigned)(zs - 1) * pl + col)) : vc[0];
    vm[1] = zs > 0 ? __ldg(y + (item + (unsigned)(zs - 1) * pl + col)) : vc[1];
    if (z0 > 0) {
        ngf_coefs<MODE>(x, y, g, item + (unsigned)zs * pl + col, pl, zs, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, inside, eps2, vm, vc, Cc);
        c0m = Cc[0];
    }
    ngf_coefs<MODE>(x, y, g, item + (unsigned)z0 * pl + col, pl, z0, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, inside, eps2, vm, vc, Cc);
    c1s[z0 & 1][wy][lane] = Cc[1];
    __syncthreads();

    for (int z = z0; z < z1; ++z) {
        const float cym = c1s[z & 1][max(wy - 1, 0)][lane], cyp = c1s[z & 1][min(wy + 1, FOLD_WARPS - 1)][lane];
        const float cxm = __shfl_up_sync(0xffffffffu, Cc[2], 1), cxp = __shfl_down_sync(0xffffffffu, Cc[2], 1);
        float Cn[3] = {0.0f, 0.0f, 0.0f};
        if (z + 1 < g.d)
            ngf_coefs<MODE>(x, y, g, item + (unsigned)(z + 1) * pl + col, pl, z + 1, oxu, oxd, oyu, oyd, xlo, xhi, ylo, yhi, inside, eps2,
                            vm, vc, Cn);
        c1s[(z + 1) & 1][wy][lane] = Cn[1];
        if (writer) {
            float gr = mul_rn(kd, fold_adjoint<MODE>(c0m, Cc[0], Cn[0], z, g.d));
            gr = fmaf(kh, fold_adjoint<MODE>(cym, Cc[1], cyp, yi, g.h), gr);
            gr = fmaf(kw, fold_adjoint<MODE>(cxm, Cc[2], cxp, xi, g.w), gr);
            st_stream(grad_x + (item + (unsigned)z * pl + col), gr);
        }
        c0m = Cc[0];
        Cc[0] = Cn[0]; Cc[1] = Cn[1]; Cc[2] = Cn[2];
        __syncthreads();
    }
}

// ---- mutual information (MI) similarity, Parzen joint histogram (include/liftreg_b200.h, lr_mi_hist; PARITY UNPINNED) --
// Per voxel the fp32 chain u = (clamp(v) - lo) * s of x and y gives the target row iota = floor(u_y + 1/2) and the
// moving cubic B-spline taps k0 - 1 .. k0 + 2 with fraction f = u_x - k0; the histogram row iota gets the four fp64 tap
// weights in columns k0 .. k0 + 3.  A CT image puts most voxels into very few keys (iota, k0) -- air and bone saturate
// the [-1, 1] range -- so the forward keeps one run of equal keys per lane and adds a run to the block's fp64 shared
// histogram only when the key changes (one warp sum and one set of atomics when every flushing lane of the warp holds
// the same key).  The adjoint needs only c(iota, kappa) = log(p / p_x) per bin: each block derives the item's table
// c * (-g s / (B N)) in fp64 and rounds it once to fp32, then streams x and y and writes each gradient element once.
constexpr int MI_THREADS = 256, MI_BWD_THREADS = 512, MI_NBMAX = 64;

struct MiMap {
    float lo, hi, s;
    int nb;
};

// u = (clamp(v, lo, hi) - lo) * s, each op rounded; NaN clamps to lo
__device__ __forceinline__ float mi_u(float v, const MiMap &m) { return mul_rn(sub_rn(fminf(fmaxf(v, m.lo), m.hi), m.lo), m.s); }

// the voxel's histogram key: bin index of its first tap, row iota and column k0 of the (nb, nb + 2) histogram, and f.
// u <= (nb-1)(1 + 3 * 2^-24), so iota <= nb - 1 already; the min only guards the index.
__device__ __forceinline__ int mi_key(float vx, float vy, const MiMap &m, float &f) {
    const float ux = mi_u(vx, m), uy = mi_u(vy, m);
    const int row = min((int)floorf(add_rn(uy, 0.5f)), m.nb - 1);
    const int k0 = min((int)floorf(ux), m.nb - 2);
    f = sub_rn(ux, (float)k0);                               // exact
    return row * (m.nb + 2) + k0;
}

// cubic B-spline weights of the taps k0 - 1 .. k0 + 2 in fp64 from the fp32 f, in the header's order
__device__ __forceinline__ void mi_weights(float f, double (&w)[4]) {
    const double F = (double)f, G = 1.0 - F, F2 = F * F, F3 = F2 * F, r6 = 1.0 / 6.0;
    w[0] = G * G * G * r6;
    w[1] = ((4.0 - 6.0 * F2) + 3.0 * F3) * r6;
    w[2] = (((1.0 + 3.0 * F) + 3.0 * F2) - 3.0 * F3) * r6;
    w[3] = F3 * r6;
}

// adds the runs of the lanes with `part` set to the block's bins (called by the whole warp)
__device__ __forceinline__ void mi_flush(double *__restrict__ h, int key, const double (&a)[4], bool part, int lane) {
    const unsigned m = __ballot_sync(0xffffffffu, part);
    if (!m) return;
    const int k0 = __shfl_sync(0xffffffffu, key, __ffs(m) - 1);
    if (__all_sync(0xffffffffu, !part || key == k0)) {
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const double t = warp_sum(part ? a[j] : 0.0);
            if (lane == 0) atomicAdd(h + k0 + j, t);
        }
    } else if (part) {
#pragma unroll
        for (int j = 0; j < 4; ++j) atomicAdd(h + key + j, a[j]);
    }
}

// one voxel of the forward for every lane of the warp (valid: the lane has a voxel)
__device__ __forceinline__ void mi_step(bool valid, float vx, float vy, const MiMap &m, double *__restrict__ h, int &key,
                                        double (&a)[4], int lane) {
    int k = -1;
    double w[4] = {0.0, 0.0, 0.0, 0.0};
    if (valid) {
        float f;
        k = mi_key(vx, vy, m, f);
        mi_weights(f, w);
    }
    const bool change = k != key;
    mi_flush(h, key, a, change && key >= 0, lane);
#pragma unroll
    for (int j = 0; j < 4; ++j) a[j] = change ? w[j] : a[j] + w[j];
    key = k;
}

// hist[b] += the fp64 tap weights of item b; label_confusion_kernel's traversal (warp-uniform trip counts over float4
// groups of both images, a scalar loop for the rest or for unaligned items), one fp64 atomic per block and non-empty bin
__global__ void __launch_bounds__(MI_THREADS) mi_hist_kernel(const float *__restrict__ x, const float *__restrict__ y, int64_t N,
                                                             MiMap m, double *__restrict__ hist) {
    extern __shared__ double mi_bins[];
    const int nbins = m.nb * (m.nb + 2), b = blockIdx.y, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < nbins; i += MI_THREADS) mi_bins[i] = 0.0;
    __syncthreads();
    const float *xb = x + (int64_t)b * N, *yb = y + (int64_t)b * N;
    const int64_t wid = ((int64_t)blockIdx.x * MI_THREADS + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * MI_THREADS) >> 5;
    const int64_t n4 = (((uintptr_t)xb | (uintptr_t)yb) % 16 == 0) ? N / 4 : 0;
    int key = -1;
    double a[4] = {0.0, 0.0, 0.0, 0.0};
    for (int64_t base = wid * 32; base < n4; base += nwarps * 32) {
        const int64_t i = base + lane;
        const bool ok = i < n4;
        float4 p = make_float4(0.f, 0.f, 0.f, 0.f), t = p;
        if (ok) {
            p = ld_stream4(reinterpret_cast<const float4 *>(xb) + i);
            t = ld_stream4(reinterpret_cast<const float4 *>(yb) + i);
        }
        mi_step(ok, p.x, t.x, m, mi_bins, key, a, lane);
        mi_step(ok, p.y, t.y, m, mi_bins, key, a, lane);
        mi_step(ok, p.z, t.z, m, mi_bins, key, a, lane);
        mi_step(ok, p.w, t.w, m, mi_bins, key, a, lane);
    }
    for (int64_t base = 4 * n4 + wid * 32; base < N; base += nwarps * 32) {
        const int64_t i = base + lane;
        const bool ok = i < N;
        mi_step(ok, ok ? ld_stream(xb + i) : 0.f, ok ? ld_stream(yb + i) : 0.f, m, mi_bins, key, a, lane);
    }
    mi_flush(mi_bins, key, a, key >= 0, lane);
    __syncthreads();
    double *hb = hist + (int64_t)b * nbins;
    for (int i = threadIdx.x; i < nbins; i += MI_THREADS) {
        const double v = mi_bins[i];
        if (v != 0.0) atomicAdd(hb + i, v);
    }
}

// d w_m / d f in fp32, the header's product forms (no cancellation near f = 0 or 1)
__device__ __forceinline__ float mi_grad_one(float vx, float vy, const MiMap &m, const float *__restrict__ tab) {
    float f;
    const int k = mi_key(vx, vy, m, f);
    const float g = sub_rn(1.0f, f);
    const float d0 = -mul_rn(mul_rn(g, g), 0.5f);
    const float d1 = -mul_rn(mul_rn(f, sub_rn(4.0f, mul_rn(3.0f, f))), 0.5f);
    const float d2 = mul_rn(mul_rn(g, add_rn(1.0f, mul_rn(3.0f, f))), 0.5f);
    const float d3 = mul_rn(mul_rn(f, f), 0.5f);
    const float acc = fma_rn(tab[k + 3], d3, fma_rn(tab[k + 2], d2, fma_rn(tab[k + 1], d1, mul_rn(tab[k], d0))));
    return vx >= m.lo && vx <= m.hi ? acc : 0.0f;             // torch.clamp's mask: NaN and values outside get 0
}

// grad_x = grad_loss * d loss / d x for the given histogram; every element written once, no atomics
__global__ void __launch_bounds__(MI_BWD_THREADS) mi_backward_kernel(const float *__restrict__ x, const float *__restrict__ y,
                                                                     int64_t N, int B, MiMap m, const double *__restrict__ hist,
                                                                     const float *__restrict__ grad_loss, float *__restrict__ gx) {
    extern __shared__ float mi_tab[];
    __shared__ double col[MI_NBMAX + 2];
    const int b = blockIdx.y, nc = m.nb + 2, nbins = m.nb * nc;
    const double *hb = hist + (int64_t)b * nbins;
    for (int j = threadIdx.x; j < nc; j += MI_BWD_THREADS) {   // p_x * N, summed over the rows in order
        double s = 0.0;
        for (int r = 0; r < m.nb; ++r) s += hb[r * nc + j];
        col[j] = s;
    }
    __syncthreads();
    const double k = -((double)grad_loss[0] * (double)m.s) / ((double)B * (double)N);
    for (int i = threadIdx.x; i < nbins; i += MI_BWD_THREADS) {
        const double h = hb[i];
        mi_tab[i] = h > 0.0 ? (float)(log(h / col[i % nc]) * k) : 0.0f;
    }
    __syncthreads();
    const float *xb = x + (int64_t)b * N, *yb = y + (int64_t)b * N;
    float *gb = gx + (int64_t)b * N;
    const int64_t t = (int64_t)blockIdx.x * MI_BWD_THREADS + threadIdx.x, stride = (int64_t)gridDim.x * MI_BWD_THREADS;
    const int64_t n4 = (((uintptr_t)xb | (uintptr_t)yb | (uintptr_t)gb) % 16 == 0) ? N / 4 : 0;
    for (int64_t i = t; i < n4; i += stride) {
        const float4 xv = ld_stream4(reinterpret_cast<const float4 *>(xb) + i), yv = ld_stream4(reinterpret_cast<const float4 *>(yb) + i);
        float4 o;
        o.x = mi_grad_one(xv.x, yv.x, m, mi_tab);
        o.y = mi_grad_one(xv.y, yv.y, m, mi_tab);
        o.z = mi_grad_one(xv.z, yv.z, m, mi_tab);
        o.w = mi_grad_one(xv.w, yv.w, m, mi_tab);
        st_stream4(reinterpret_cast<float4 *>(gb) + i, o);
    }
    for (int64_t i = 4 * n4 + t; i < N; i += stride) st_stream(gb + i, mi_grad_one(ld_stream(xb + i), ld_stream(yb + i), m, mi_tab));
}

}  // namespace lr

using namespace lr;

extern "C" int lr_ncc_sums(const float *x, const float *y, int B, int64_t N, double *sums, lr_stream_t stream) {
    LR_REQUIRE(x && y && sums, "ncc_sums: null pointer");
    LR_REQUIRE(B > 0 && B <= 65535 && N > 0, "ncc_sums: bad size (B=%d N=%lld)", B, (long long)N);
    cudaStream_t st = as_stream(stream);
    if (int e = cuda_ok(cudaMemsetAsync(sums, 0, sizeof(double) * NCC_SUMS * (size_t)B, st), "ncc_sums: memset failed")) return e;
    const dim3 grid(ncc_blocks(N, B), (unsigned)B);
    ncc_shifted_kernel<<<grid, NCC_THREADS, 0, st>>>(x, y, N, sums);
    if (int e = check_launch("ncc_shifted_kernel")) return e;
    ncc_finalize_kernel<<<(B + 127) / 128, 128, 0, st>>>(x, y, N, B, sums);
    return check_launch("ncc_finalize_kernel");
}

extern "C" int lr_ncc_backward(const float *x, const float *y, int B, int64_t N, const double *sums, const float *grad_loss,
                               float *grad_x, lr_stream_t stream) {
    LR_REQUIRE(x && y && sums && grad_loss && grad_x, "ncc_backward: null pointer");
    LR_REQUIRE(B > 0 && B <= 65535 && N > 0, "ncc_backward: bad size (B=%d N=%lld)", B, (long long)N);
    const dim3 grid(ncc_blocks(N, B), (unsigned)B);
    ncc_backward_kernel<<<grid, NCC_THREADS, 0, as_stream(stream)>>>(x, y, N, sums, grad_loss, B, grad_x);
    return check_launch("ncc_backward_kernel");
}

// argument rules shared by the finite-difference entries over `channels` (D,H,W) volumes per item, which the kernels
// index with 32 bits, of which the `margin` voxels next to every face are left out (only jacobian_det skips any); 0 when
// they hold
static int fd_check(const char *who, int B, int D, int H, int W, int boundary, int channels, int margin = 0) {
    LR_REQUIRE(B > 0 && D >= 2 && H >= 2 && W >= 2, "%s: every axis needs >= 2 entries (B=%d, %dx%dx%d)", who, B, D, H, W);
    LR_REQUIRE(boundary == LR_FD_LINEAR || boundary == LR_FD_NEUMANN_ZERO, "%s: unknown boundary mode %d", who, boundary);
    LR_REQUIRE(margin >= 0 && 2 * (int64_t)margin < D && 2 * (int64_t)margin < H && 2 * (int64_t)margin < W,
               "%s: margin %d leaves no interior voxel of %dx%dx%d (2*margin must be < every axis)", who, margin, D, H, W);
    LR_REQUIRE((int64_t)B * channels * D * H * W < ((int64_t)1 << 31),
               channels == 3 ? "%s: field too large for one launch (B=%d, %dx%dx%d; B*3*D*H*W must stay below 2^31)"
                             : "%s: too large for one launch (B=%d, %dx%dx%d; B*D*H*W must stay below 2^31)",
               who, B, D, H, W);
    return 0;
}

template <int MODE>
static int diffusion_reg_launch(const float *disp, int B, int D, int H, int W, double *sum, cudaStream_t st) {
    RegDims g; dim3 grid;
    const bool pairs = reg_use_pairs(disp, nullptr, W);
    const int rd = pairs ? reg_dims(diffusion_reg_pair_kernel<MODE>, true, LR_REG_WAVES, B, D, H, W, g, grid)
                         : reg_dims(diffusion_reg_kernel<MODE>, false, LR_REG_WAVES, B, D, H, W, g, grid);
    LR_REQUIRE(rd == 0, "diffusion_reg_sum: field too large for one launch (B=%d, %dx%dx%d; B*3*D*H*W must stay below 2^31)", B, D, H, W);
    if (int e = cuda_ok(cudaMemsetAsync(sum, 0, sizeof(double), st), "diffusion_reg_sum: memset failed")) return e;
    if (pairs) {
        diffusion_reg_pair_kernel<MODE><<<grid, NCC_THREADS, 0, st>>>(disp, g, sum);
        return check_launch("diffusion_reg_pair_kernel");
    }
    diffusion_reg_kernel<MODE><<<grid, NCC_THREADS, 0, st>>>(disp, g, sum);
    return check_launch("diffusion_reg_kernel");
}

extern "C" int lr_diffusion_reg_sum(const float *disp, int B, int D, int H, int W, int boundary, double *sum, lr_stream_t stream) {
    LR_REQUIRE(disp && sum, "diffusion_reg_sum: null pointer");
    if (int e = fd_check("diffusion_reg_sum", B, D, H, W, boundary, 3)) return e;
    cudaStream_t st = as_stream(stream);
    return boundary == LR_FD_LINEAR ? diffusion_reg_launch<0>(disp, B, D, H, W, sum, st)
                                    : diffusion_reg_launch<1>(disp, B, D, H, W, sum, st);
}

template <int MODE>
static int diffusion_reg_backward_launch(const float *disp, int B, int D, int H, int W, const float *grad_loss, float *grad_disp,
                                         cudaStream_t st) {
    RegDims g; dim3 grid;
    const bool pairs = reg_use_pairs(disp, grad_disp, W);
    const int rd = pairs ? reg_dims(diffusion_reg_backward_pair_kernel<MODE>, true, LR_REG_BWD_WAVES, B, D, H, W, g, grid)
                         : reg_dims(diffusion_reg_backward_kernel<MODE>, false, LR_REG_BWD_WAVES, B, D, H, W, g, grid);
    LR_REQUIRE(rd == 0, "diffusion_reg_backward: field too large for one launch (B=%d, %dx%dx%d; B*3*D*H*W must stay below 2^31)", B, D, H, W);
    if (pairs) {
        diffusion_reg_backward_pair_kernel<MODE><<<grid, NCC_THREADS, 0, st>>>(disp, g, B, grad_loss, grad_disp);
        return check_launch("diffusion_reg_backward_pair_kernel");
    }
    diffusion_reg_backward_kernel<MODE><<<grid, NCC_THREADS, 0, st>>>(disp, g, B, grad_loss, grad_disp);
    return check_launch("diffusion_reg_backward_kernel");
}

extern "C" int lr_diffusion_reg_backward(const float *disp, int B, int D, int H, int W, int boundary, const float *grad_loss,
                                         float *grad_disp, lr_stream_t stream) {
    LR_REQUIRE(disp && grad_loss && grad_disp, "diffusion_reg_backward: null pointer");
    if (int e = fd_check("diffusion_reg_backward", B, D, H, W, boundary, 3)) return e;
    cudaStream_t st = as_stream(stream);
    return boundary == LR_FD_LINEAR ? diffusion_reg_backward_launch<0>(disp, B, D, H, W, grad_loss, grad_disp, st)
                                    : diffusion_reg_backward_launch<1>(disp, B, D, H, W, grad_loss, grad_disp, st);
}

template <int MODE>
static int jacobian_launch(const float *phi, int B, int D, int H, int W, int margin, float *det, double *stats, cudaStream_t st) {
    RegDims g; dim3 grid;
    const bool pairs = reg_use_pairs(phi, det, W);
    const int rd = pairs ? reg_dims(jacobian_det_pair_kernel<MODE>, true, LR_REG_WAVES, B, D, H, W, g, grid)
                         : reg_dims(jacobian_det_kernel<MODE>, false, LR_REG_WAVES, B, D, H, W, g, grid);
    LR_REQUIRE(rd == 0, "jacobian_det: field too large for one launch (B=%d, %dx%dx%d; B*3*D*H*W must stay below 2^31)", B, D, H, W);
    jac_init_kernel<<<(B * JAC_STATS + 127) / 128, 128, 0, st>>>(stats, B);
    if (int e = check_launch("jac_init_kernel")) return e;
    if (pairs) {
        jacobian_det_pair_kernel<MODE><<<grid, NCC_THREADS, 0, st>>>(phi, g, margin, det, stats);
        return check_launch("jacobian_det_pair_kernel");
    }
    jacobian_det_kernel<MODE><<<grid, NCC_THREADS, 0, st>>>(phi, g, margin, det, stats);
    return check_launch("jacobian_det_kernel");
}

extern "C" int lr_jacobian_det(const float *phi, int B, int D, int H, int W, int boundary, int margin, float *det, double *stats,
                               lr_stream_t stream) {
    LR_REQUIRE(phi && stats, "jacobian_det: null pointer");
    if (int e = fd_check("jacobian_det", B, D, H, W, boundary, 3, margin)) return e;
    cudaStream_t st = as_stream(stream);
    return boundary == LR_FD_LINEAR ? jacobian_launch<0>(phi, B, D, H, W, margin, det, stats, st)
                                    : jacobian_launch<1>(phi, B, D, H, W, margin, det, stats, st);
}

template <int MODE>
static int fold_backward_launch(const float *phi, int B, int D, int H, int W, const float *grad_loss, float *grad_phi, cudaStream_t st) {
    RegDims g; dim3 grid;
    const int rd = march_dims(jacobian_fold_backward_kernel<MODE>, FOLD_THREADS, FOLD_OX, FOLD_OY, LR_REG_WAVES, B, D, H, W, g, grid);
    LR_REQUIRE(rd == 0, "jacobian_fold_backward: field too large for one launch (B=%d, %dx%dx%d; B*3*D*H*W must stay below 2^31)", B, D, H, W);
    jacobian_fold_backward_kernel<MODE><<<grid, FOLD_THREADS, 0, st>>>(phi, g, B, grad_loss, grad_phi);
    return check_launch("jacobian_fold_backward_kernel");
}

extern "C" int lr_jacobian_fold_backward(const float *phi, int B, int D, int H, int W, int boundary, const float *grad_loss,
                                         float *grad_phi, lr_stream_t stream) {
    LR_REQUIRE(phi && grad_loss && grad_phi, "jacobian_fold_backward: null pointer");
    if (int e = fd_check("jacobian_fold_backward", B, D, H, W, boundary, 3)) return e;
    cudaStream_t st = as_stream(stream);
    return boundary == LR_FD_LINEAR ? fold_backward_launch<0>(phi, B, D, H, W, grad_loss, grad_phi, st)
                                    : fold_backward_launch<1>(phi, B, D, H, W, grad_loss, grad_phi, st);
}

extern "C" int lr_label_confusion(const float *pred, const float *target, int B, int64_t N, int L, int64_t *counts, int64_t *invalid,
                                  lr_stream_t stream) {
    LR_REQUIRE(pred && target && counts && invalid, "label_confusion: null pointer");
    LR_REQUIRE(L >= 1 && L <= 128, "label_confusion: number of labels L=%d must be in [1, 128]", L);
    LR_REQUIRE(B > 0 && B <= 65535 && N > 0, "label_confusion: bad size (B=%d N=%lld)", B, (long long)N);
    cudaStream_t st = as_stream(stream);
    const size_t smem = sizeof(unsigned) * ((size_t)L * L + 1);
    static thread_local int smem_dev = -1;
    if (int e = cuda_ok(opt_in_smem(label_confusion_kernel, (int)(sizeof(unsigned) * (128 * 128 + 1)), smem_dev), "label_confusion")) return e;
    const int per_sm = blocks_per_sm(label_confusion_kernel, CONF_THREADS, smem, 1);
    if (int e = cuda_ok(cudaMemsetAsync(counts, 0, sizeof(int64_t) * (size_t)B * L * L, st), "label_confusion: memset failed")) return e;
    if (int e = cuda_ok(cudaMemsetAsync(invalid, 0, sizeof(int64_t) * (size_t)B, st), "label_confusion: memset failed")) return e;
    const dim3 grid(conf_blocks(N, B, L, per_sm), (unsigned)B);
    label_confusion_kernel<<<grid, CONF_THREADS, smem, st>>>(pred, target, N, L, reinterpret_cast<unsigned long long *>(counts),
                                                              reinterpret_cast<unsigned long long *>(invalid));
    return check_launch("label_confusion_kernel");
}

// argument rules shared by the local NCC entries; 0 when they hold
static int lncc_check(const char *who, int B, int D, int H, int W, int win, double eps) {
    LR_REQUIRE(win % 2 == 1 && win >= 3 && win <= LNCC_WMAX, "%s: window %d must be odd and in [3, %d]", who, win, LNCC_WMAX);
    LR_REQUIRE(eps >= 0.0 && eps <= DBL_MAX, "%s: eps must be finite and >= 0 (got %g)", who, eps);
    LR_REQUIRE(B >= 1 && D >= 1 && H >= 1 && W >= 1, "%s: every axis needs >= 1 entry (B=%d, %dx%dx%d)", who, B, D, H, W);
    // tile origins plus the 32 + 14 tile-and-halo offsets stay in int
    LR_REQUIRE(D <= (1 << 30) && H <= (1 << 30) && W <= (1 << 30), "%s: every axis must be <= 2^30 (%dx%dx%d)", who, D, H, W);
    LR_REQUIRE((int64_t)B * D * H * W < ((int64_t)1 << 31), "%s: too large for one launch (B=%d, %dx%dx%d; B*D*H*W must stay below 2^31)",
               who, B, D, H, W);
    return 0;
}

template <int KIND>
static int lncc_launch(const float *x, const float *y, const float *coef, int B, int D, int H, int W, int win, double eps,
                       const float *grad_loss, double *sum, float *out, cudaStream_t st, const char *name) {
    static thread_local int smem_dev = -1;
    if (int e = cuda_ok(opt_in_smem(local_ncc_kernel<KIND>, (int)lncc_smem_bytes<KIND>(LNCC_WMAX), smem_dev), name)) return e;
    const size_t smem = lncc_smem_bytes<KIND>(win);
    const int per_sm = blocks_per_sm(local_ncc_kernel<KIND>, LNCC_THREADS, smem, 1);
    LnccDims g;
    g.D = D; g.H = H; g.W = W; g.w = win;
    g.N = (unsigned)D * (unsigned)H * (unsigned)W;
    g.total = g.N * (unsigned)B;
    g.n = (double)win * win * win; g.eps = eps; g.count = (double)g.total;
    g.tiles_x = (W + LNCC_TX - 1) / LNCC_TX;
    g.tiles_y = (H + LNCC_TY - 1) / LNCC_TY;
    // enough z chunks for two waves of resident blocks, but a chunk of at least w planes (a chunk re-reads w-1 planes)
    const int64_t tiles = (int64_t)g.tiles_x * g.tiles_y * B;
    int64_t chunks = (2 * (int64_t)sm_count() * per_sm + tiles - 1) / tiles;
    if (chunks > D / win) chunks = D / win;
    if (chunks < 1) chunks = 1;
    g.zchunk = (int)((D + chunks - 1) / chunks);
    g.n_zchunks = (D + g.zchunk - 1) / g.zchunk;
    const int64_t blocks = tiles * g.n_zchunks;     // <= B*D*H*W < 2^31
    local_ncc_kernel<KIND><<<(unsigned)blocks, LNCC_THREADS, smem, st>>>(x, y, coef, g, grad_loss, sum, out);
    return check_launch(name);
}

extern "C" int lr_local_ncc_sum(const float *x, const float *y, int B, int D, int H, int W, int win, double eps, double *sum,
                                lr_stream_t stream) {
    LR_REQUIRE(x && y && sum, "local_ncc_sum: null pointer");
    if (int e = lncc_check("local_ncc_sum", B, D, H, W, win, eps)) return e;
    cudaStream_t st = as_stream(stream);
    if (int e = cuda_ok(cudaMemsetAsync(sum, 0, sizeof(double) * (size_t)B, st), "local_ncc_sum: memset failed")) return e;
    return lncc_launch<LNCC_FWD>(x, y, nullptr, B, D, H, W, win, eps, nullptr, sum, nullptr, st, "local_ncc_kernel<fwd>");
}

extern "C" size_t lr_local_ncc_workspace_bytes(int B, int D, int H, int W, int win) {
    if (win % 2 != 1 || win < 3 || win > LNCC_WMAX || B < 1 || D < 1 || H < 1 || W < 1) return 0;
    if (D > (1 << 30) || H > (1 << 30) || W > (1 << 30)) return 0;
    if ((int64_t)B * D * H * W >= ((int64_t)1 << 31)) return 0;
    return 3 * sizeof(float) * (size_t)B * D * H * W;          // alpha, beta, gamma per voxel
}

extern "C" int lr_local_ncc_backward(const float *x, const float *y, int B, int D, int H, int W, int win, double eps,
                                     const float *grad_loss, float *grad_x, void *workspace, size_t workspace_bytes,
                                     lr_stream_t stream) {
    LR_REQUIRE(x && y && grad_loss && grad_x && workspace, "local_ncc_backward: null pointer");
    if (int e = lncc_check("local_ncc_backward", B, D, H, W, win, eps)) return e;
    const size_t need = lr_local_ncc_workspace_bytes(B, D, H, W, win);
    LR_REQUIRE(workspace_bytes >= need, "local_ncc_backward: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
    cudaStream_t st = as_stream(stream);
    float *coef = static_cast<float *>(workspace);
    if (int e = lncc_launch<LNCC_COEF>(x, y, nullptr, B, D, H, W, win, eps, nullptr, nullptr, coef, st, "local_ncc_kernel<coef>")) return e;
    return lncc_launch<LNCC_GRAD>(x, y, coef, B, D, H, W, win, eps, grad_loss, nullptr, grad_x, st, "local_ncc_kernel<grad>");
}

// argument rules shared by the Dice entries (the warp's size limits); 0 when they hold
static int dice_check(const char *who, int B, int D, int H, int W, int L) {
    LR_REQUIRE(L >= 2 && L <= DICE_LMAX, "%s: number of labels L=%d must be in [2, %d]", who, L, DICE_LMAX);
    LR_REQUIRE(B >= 1 && D >= 1 && H >= 1 && W >= 1, "%s: every axis needs >= 1 entry (B=%d, %dx%dx%d)", who, B, D, H, W);
    LR_REQUIRE(D < (1 << 21) && H < (1 << 21) && W < (1 << 21), "%s: D, H and W must be < 2^21 (%dx%dx%d)", who, D, H, W);
    LR_REQUIRE((int64_t)B * 3 * D * H * W < ((int64_t)1 << 31),
               "%s: field too large for one launch (B=%d, %dx%dx%d; B*3*D*H*W must stay below 2^31)", who, B, D, H, W);
    return 0;
}

template <typename K>
static int dice_dims(K kernel, const char *who, int B, int D, int H, int W, int L, DiceDims &g, dim3 &grid) {
    LR_REQUIRE(march_dims(kernel, DICE_THREADS, DICE_TX, DICE_TY, LR_REG_WAVES, B, D, H, W, g.m, grid) == 0,
               "%s: too many blocks for one launch (B=%d, %dx%dx%d)", who, B, D, H, W);
    g.hx = (float)(W - 1) / 2.0f; g.hy = (float)(H - 1) / 2.0f; g.hz = (float)(D - 1) / 2.0f;
    g.cx = (float)(W - 1) + 2.0f; g.cy = (float)(H - 1) + 2.0f; g.cz = (float)(D - 1) + 2.0f;
    g.L = L;
    return 0;
}

extern "C" int lr_label_dice_sums(const float *phi, const float *src, const float *tgt, int B, int D, int H, int W, int L,
                                  double *sums, lr_stream_t stream) {
    LR_REQUIRE(phi && src && tgt && sums, "label_dice_sums: null pointer");
    if (int e = dice_check("label_dice_sums", B, D, H, W, L)) return e;
    DiceDims g; dim3 grid;
    if (int e = dice_dims(label_dice_sums_kernel, "label_dice_sums", B, D, H, W, L, g, grid)) return e;
    cudaStream_t st = as_stream(stream);
    if (int e = cuda_ok(cudaMemsetAsync(sums, 0, sizeof(double) * 3 * (size_t)B * L, st), "label_dice_sums: memset failed")) return e;
    label_dice_sums_kernel<<<grid, DICE_THREADS, 0, st>>>(phi, src, tgt, g, sums);
    return check_launch("label_dice_sums_kernel");
}

extern "C" int lr_label_dice_backward(const float *phi, const float *src, const float *tgt, int B, int D, int H, int W, int L,
                                      const double *sums, const float *grad_loss, float *grad_phi, lr_stream_t stream) {
    LR_REQUIRE(phi && src && tgt && sums && grad_loss && grad_phi, "label_dice_backward: null pointer");
    if (int e = dice_check("label_dice_backward", B, D, H, W, L)) return e;
    DiceDims g; dim3 grid;
    if (int e = dice_dims(label_dice_backward_kernel, "label_dice_backward", B, D, H, W, L, g, grid)) return e;
    label_dice_backward_kernel<<<grid, DICE_THREADS, 0, as_stream(stream)>>>(phi, src, tgt, g, B, sums, grad_loss, grad_phi);
    return check_launch("label_dice_backward_kernel");
}

// argument rules shared by the NGF entries; 0 when they hold.  eps >= 1e-77 keeps p*q >= eps^4 > 0 in fp64.
static int ngf_check(const char *who, int B, int D, int H, int W, int boundary, double eps) {
    LR_REQUIRE(eps >= 1e-77 && eps <= DBL_MAX, "%s: eps must be finite and > 0 (>= 1e-77; got %g)", who, eps);
    return fd_check(who, B, D, H, W, boundary, 1);
}

template <int MODE>
static int ngf_sum_launch(const float *x, const float *y, int B, int D, int H, int W, double eps, double *sum, cudaStream_t st) {
    RegDims g; dim3 grid;
    LR_REQUIRE(march_dims(ngf_sum_kernel<MODE>, NCC_THREADS, REG_TX, REG_TY, LR_REG_WAVES, B, D, H, W, g, grid, 1) == 0,
               "ngf_sum: too many blocks for one launch (B=%d, %dx%dx%d)", B, D, H, W);
    if (int e = cuda_ok(cudaMemsetAsync(sum, 0, sizeof(double) * (size_t)B, st), "ngf_sum: memset failed")) return e;
    ngf_sum_kernel<MODE><<<grid, NCC_THREADS, 0, st>>>(x, y, g, eps * eps, sum);
    return check_launch("ngf_sum_kernel");
}

template <int MODE>
static int ngf_backward_launch(const float *x, const float *y, int B, int D, int H, int W, double eps, const float *grad_loss,
                               float *grad_x, cudaStream_t st) {
    RegDims g; dim3 grid;
    LR_REQUIRE(march_dims(ngf_backward_kernel<MODE>, FOLD_THREADS, FOLD_OX, FOLD_OY, LR_REG_WAVES, B, D, H, W, g, grid, 1) == 0,
               "ngf_backward: too many blocks for one launch (B=%d, %dx%dx%d)", B, D, H, W);
    ngf_backward_kernel<MODE><<<grid, FOLD_THREADS, 0, st>>>(x, y, g, B, eps * eps, grad_loss, grad_x);
    return check_launch("ngf_backward_kernel");
}

extern "C" int lr_ngf_sum(const float *x, const float *y, int B, int D, int H, int W, int boundary, double eps, double *sum,
                          lr_stream_t stream) {
    LR_REQUIRE(x && y && sum, "ngf_sum: null pointer");
    if (int e = ngf_check("ngf_sum", B, D, H, W, boundary, eps)) return e;
    cudaStream_t st = as_stream(stream);
    return boundary == LR_FD_LINEAR ? ngf_sum_launch<0>(x, y, B, D, H, W, eps, sum, st)
                                    : ngf_sum_launch<1>(x, y, B, D, H, W, eps, sum, st);
}

extern "C" int lr_ngf_backward(const float *x, const float *y, int B, int D, int H, int W, int boundary, double eps,
                               const float *grad_loss, float *grad_x, lr_stream_t stream) {
    LR_REQUIRE(x && y && grad_loss && grad_x, "ngf_backward: null pointer");
    if (int e = ngf_check("ngf_backward", B, D, H, W, boundary, eps)) return e;
    cudaStream_t st = as_stream(stream);
    return boundary == LR_FD_LINEAR ? ngf_backward_launch<0>(x, y, B, D, H, W, eps, grad_loss, grad_x, st)
                                    : ngf_backward_launch<1>(x, y, B, D, H, W, eps, grad_loss, grad_x, st);
}

// argument rules shared by the MI entries; 0 when they hold, with the map's fp32 s = (nb - 1) / (hi - lo)
static int mi_check(const char *who, int B, int64_t N, int nb, float lo, float hi, MiMap &m) {
    LR_REQUIRE(B >= 1 && B <= 65535 && N >= 1, "%s: bad size (B=%d N=%lld; 1 <= B <= 65535, N >= 1)", who, B, (long long)N);
    LR_REQUIRE(nb >= 4 && nb <= MI_NBMAX, "%s: num_bins=%d must be in [4, %d]", who, nb, MI_NBMAX);
    LR_REQUIRE(lo >= -FLT_MAX && hi <= FLT_MAX && lo < hi, "%s: value range (%g, %g) must be finite with lo < hi", who, (double)lo, (double)hi);
    const float s = (float)((double)(nb - 1) / ((double)hi - (double)lo));
    LR_REQUIRE(s > 0.0f && s <= FLT_MAX, "%s: (num_bins - 1) / (hi - lo) = %g is not a finite positive float", who, (double)s);
    m.lo = lo; m.hi = hi; m.s = s; m.nb = nb;
    return 0;
}

// blocks per item: >= 16 voxels per thread, one wave over the whole grid
static unsigned mi_blocks(int64_t N, int B, int threads, int per_sm) {
    int64_t want = (N + threads * 16 - 1) / (threads * 16);
    const int64_t cap = ((int64_t)sm_count() * per_sm + B - 1) / B;
    if (want > cap) want = cap;
    return (unsigned)(want < 1 ? 1 : want);
}

extern "C" int lr_mi_hist(const float *x, const float *y, int B, int64_t N, int num_bins, float lo, float hi, double *hist,
                          lr_stream_t stream) {
    LR_REQUIRE(x && y && hist, "mi_hist: null pointer");
    MiMap m;
    if (int e = mi_check("mi_hist", B, N, num_bins, lo, hi, m)) return e;
    cudaStream_t st = as_stream(stream);
    const size_t nbins = (size_t)num_bins * (num_bins + 2), smem = sizeof(double) * nbins;
    if (int e = cuda_ok(cudaMemsetAsync(hist, 0, sizeof(double) * nbins * (size_t)B, st), "mi_hist: memset failed")) return e;
    const dim3 grid(mi_blocks(N, B, MI_THREADS, blocks_per_sm(mi_hist_kernel, MI_THREADS, smem, 1)), (unsigned)B);
    mi_hist_kernel<<<grid, MI_THREADS, smem, st>>>(x, y, N, m, hist);
    return check_launch("mi_hist_kernel");
}

extern "C" int lr_mi_backward(const float *x, const float *y, int B, int64_t N, int num_bins, float lo, float hi,
                              const double *hist, const float *grad_loss, float *grad_x, lr_stream_t stream) {
    LR_REQUIRE(x && y && hist && grad_loss && grad_x, "mi_backward: null pointer");
    MiMap m;
    if (int e = mi_check("mi_backward", B, N, num_bins, lo, hi, m)) return e;
    const size_t smem = sizeof(float) * (size_t)num_bins * (num_bins + 2);
    const dim3 grid(mi_blocks(N, B, MI_BWD_THREADS, blocks_per_sm(mi_backward_kernel, MI_BWD_THREADS, smem, 1)), (unsigned)B);
    mi_backward_kernel<<<grid, MI_BWD_THREADS, smem, as_stream(stream)>>>(x, y, N, B, m, hist, grad_loss, grad_x);
    return check_launch("mi_backward_kernel");
}
