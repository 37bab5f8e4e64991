// PCA-subspace displacement decode: disp = coefs @ basis^T + mean (+ identity map), sm_100a.
//
// Replaces reference src/liftreg/models/LiftRegDeformSubspaceBackproj.py:102
//     disp_field = F.linear(x, self.pca_vectors, self.pca_mean).reshape(B, 3, D, W, H)
// and, optionally, the `+ self.id_transform` of :68 (SURVEY.md 8f row f2).  pca_vectors is (N, K) row-major with
// N = 3*D*W*H = 12.3 M and K = 56 at 160^3: a 2.75 GB basis streamed once per forward -- by far the largest HBM
// consumer of the model's forward pass and purely bandwidth-bound (algorithmic bytes = 4*N*K + 4*N + 4*B*(N + K)).
//
// Layout: a block owns tiles of 256 consecutive basis rows (256*K contiguous floats).  The tile is copied with
// perfectly coalesced 16-byte streaming loads into shared memory (STS.128) with a row pitch whose quarter is odd, so
// that in the compute phase lane = row reads its row four coefficients at a time (LDS.128) without bank conflicts; the
// batch's coefficients sit in shared memory as [k][b] and are read four batch items at a time (LDS.128 broadcast).
// Accumulation is a sequential fp32 FMA chain over k (ascending), then + mean, then (optionally) + identity -- the
// order the oracle restates.
#include "common.cuh"

namespace lr {

#ifndef LR_PD_ROWS
#define LR_PD_ROWS 256
#endif
constexpr int PD_ROWS = LR_PD_ROWS;     // basis rows per tile = threads per block
// shared-memory row pitch in floats: a multiple of 4 (aligned STS.128 / LDS.128) whose quarter is odd (8 consecutive
// lanes x 16 B then cover all 32 banks exactly once)
__host__ __device__ inline int pd_pitch(int K) { return (K / 4) % 2 == 0 ? K + 4 : K + 8; }

struct PcaDims {
    int B, K;
    int64_t N;                   // rows of the basis = 3*D*H*W when add_identity
    int add_identity;
    int D, H, W, nvox;           // identity map geometry (axis c of output row n = n / nvox)
    double sp0, sp1, sp2;        // 1/(D-1), 1/(H-1), 1/(W-1) in float64 (net_utils.py:81)
    int64_t n_tiles;
};

// net_utils.py:81-85 with numpy>=2 casting (same helper as warp.cu)
__device__ __forceinline__ float pd_identity_coord(int idx, double spacing) {
    float v = __double2float_rn((double)idx * spacing);
    return sub_rn(mul_rn(v, 2.0f), 1.0f);
}

// Fallback for K % 4 != 0 or an unaligned basis: scalar staging with an odd row pitch (conflict-free scalar reads).
template <int BT>
__global__ void __launch_bounds__(PD_ROWS)
    pca_decode_scalar_kernel(const float *__restrict__ coefs, const float *__restrict__ basis, const float *__restrict__ mean,
                             float *__restrict__ out, PcaDims g) {
    extern __shared__ float smem[];
    const int pitch = g.K | 1;
    float *tile = smem;
    float *cf = smem + (size_t)PD_ROWS * pitch;
    const int tid = threadIdx.x;
    for (int i = tid; i < g.K * BT; i += PD_ROWS) {
        const int k = i / BT, b = i - k * BT;
        cf[i] = b < g.B ? coefs[(int64_t)b * g.K + k] : 0.0f;
    }
    for (int64_t t = blockIdx.x; t < g.n_tiles; t += gridDim.x) {
        const int64_t row0 = t * PD_ROWS;
        const int rows = (int)min((int64_t)PD_ROWS, g.N - row0);
        __syncthreads();
        const float *src = basis + row0 * g.K;
        for (int f = tid; f < rows * g.K; f += PD_ROWS) {
            const int r = f / g.K;
            tile[r * pitch + (f - r * g.K)] = ld_stream(src + f);
        }
        __syncthreads();
        if (tid < rows) {
            float acc[BT];
#pragma unroll
            for (int b = 0; b < BT; ++b) acc[b] = 0.0f;
            for (int k = 0; k < g.K; ++k) {
                const float w = tile[tid * pitch + k];
#pragma unroll
                for (int b = 0; b < BT; ++b) acc[b] = fma_rn(cf[k * BT + b], w, acc[b]);
            }
            const int64_t n = row0 + tid;
            const float m = mean ? ld_stream(mean + n) : 0.0f;
            float idv = 0.0f;
            if (g.add_identity) {
                const int c = (int)(n / g.nvox);
                const int v = (int)(n - (int64_t)c * g.nvox);
                const int z = v / (g.H * g.W), rem = v - z * (g.H * g.W), y = rem / g.W, x = rem - y * g.W;
                idv = c == 0 ? pd_identity_coord(z, g.sp0) : (c == 1 ? pd_identity_coord(y, g.sp1) : pd_identity_coord(x, g.sp2));
            }
#pragma unroll
            for (int b = 0; b < BT; ++b) {
                if (b < g.B) {
                    float o = add_rn(acc[b], m);
                    if (g.add_identity) o = add_rn(o, idv);
                    st_stream(out + (int64_t)b * g.N + n, o);
                }
            }
        }
    }
}

template <int BT>   // batch items held in registers per pass (B <= BT)
__global__ void __launch_bounds__(PD_ROWS)
    pca_decode_kernel(const float *__restrict__ coefs, const float *__restrict__ basis, const float *__restrict__ mean,
                      float *__restrict__ out, PcaDims g) {
    extern __shared__ float smem[];
    const int pitch = pd_pitch(g.K);
    float *tile = smem;                                  // [PD_ROWS][pitch]
    float *cf = smem + (size_t)PD_ROWS * pitch;          // [K][BT], zero-padded beyond B
    const int tid = threadIdx.x;
    for (int i = tid; i < g.K * BT; i += PD_ROWS) {
        const int k = i / BT, b = i - k * BT;
        cf[i] = b < g.B ? coefs[(int64_t)b * g.K + k] : 0.0f;
    }
    const int k4 = g.K / 4;                              // float4 per row (K % 4 == 0 on this path)
    const int tile_f4 = PD_ROWS * k4;

    for (int64_t t = blockIdx.x; t < g.n_tiles; t += gridDim.x) {
        const int64_t row0 = t * PD_ROWS;
        const int rows = (int)min((int64_t)PD_ROWS, g.N - row0);
        __syncthreads();                                 // previous tile fully consumed (and cf written)
        // ---- stage: rows*K contiguous floats, coalesced 16 B streaming loads, transposed into shared memory
        const float4 *src = reinterpret_cast<const float4 *>(basis + row0 * g.K);
        const int n_f4 = rows * k4;
#ifndef LR_PD_UNR
#define LR_PD_UNR 7
#endif
        constexpr int UNR = LR_PD_UNR;                           // loads in flight per thread before the first store
        for (int f0 = tid; f0 < tile_f4; f0 += UNR * PD_ROWS) {
            float4 v[UNR];
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const int f = f0 + u * PD_ROWS;
                if (f < n_f4) v[u] = ld_stream4(src + f);
            }
#pragma unroll
            for (int u = 0; u < UNR; ++u) {
                const int f = f0 + u * PD_ROWS;
                if (f < n_f4) {
                    const int r = f / k4, k = (f - r * k4) * 4;
                    *reinterpret_cast<float4 *>(tile + r * pitch + k) = v[u];
                }
            }
        }
        __syncthreads();
        if (tid < rows) {
            float acc[BT];
#pragma unroll
            for (int b = 0; b < BT; ++b) acc[b] = 0.0f;
            const float *myrow = tile + tid * pitch;
            for (int k = 0; k < g.K; k += 4) {
                const float4 w4 = *reinterpret_cast<const float4 *>(myrow + k);
                const float w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {          // k ascending: one sequential fp32 FMA chain per output
                    if (BT >= 4) {
#pragma unroll
                        for (int b = 0; b < BT; b += 4) {
                            const float4 c = *reinterpret_cast<const float4 *>(cf + (k + kk) * BT + b);
                            acc[b] = fma_rn(c.x, w[kk], acc[b]); acc[b + 1] = fma_rn(c.y, w[kk], acc[b + 1]);
                            acc[b + 2] = fma_rn(c.z, w[kk], acc[b + 2]); acc[b + 3] = fma_rn(c.w, w[kk], acc[b + 3]);
                        }
                    } else {
#pragma unroll
                        for (int b = 0; b < BT; ++b) acc[b] = fma_rn(cf[(k + kk) * BT + b], w[kk], acc[b]);
                    }
                }
            }
            const int64_t n = row0 + tid;
            const float m = mean ? ld_stream(mean + n) : 0.0f;
            float idv = 0.0f;
            if (g.add_identity) {                         // model :68: deform_field = disp_field + id_transform
                const int c = (int)(n / g.nvox);
                const int v = (int)(n - (int64_t)c * g.nvox);
                const int z = v / (g.H * g.W), rem = v - z * (g.H * g.W), y = rem / g.W, x = rem - y * g.W;
                idv = c == 0 ? pd_identity_coord(z, g.sp0) : (c == 1 ? pd_identity_coord(y, g.sp1) : pd_identity_coord(x, g.sp2));
            }
#pragma unroll
            for (int b = 0; b < BT; ++b) {
                if (b < g.B) {
                    float o = add_rn(acc[b], m);
                    if (g.add_identity) o = add_rn(o, idv);
                    st_stream(out + (int64_t)b * g.N + n, o);
                }
            }
        }
    }
}

// ---- TMA-pipelined forward ---------------------------------------------------------------------------------------
// The staging loop above is load -> barrier -> compute -> barrier with one tile per block in flight; HBM sits idle
// while a block computes and the loads restart cold every tile (5.2 TB/s = 80 % of the copy peak).  Here the basis
// tiles (PT_ROWS rows = PT_ROWS*K contiguous floats each) are pulled into a ring of shared-memory stages by the TMA
// engine (cp.async.bulk global -> shared, one bulk copy per tile, completion on an mbarrier), PT_STAGES-1 tiles ahead
// of the compute: the copies cost no LSU instructions and no registers, and every SM keeps ~2 x 57 KB in flight.
// The tile lands unpadded (row pitch K floats), so lane = row reads its row with LDS.128 at a pitch of K/4 16-byte
// slots: conflict degree gcd(K/4, 8) -- 2 for K = 56, which shared memory absorbs easily (a tile is read once per
// ~2600 cycles of HBM time).  K whose degree exceeds 2 (K a multiple of 16) stay on the padded staging kernel.
// Same arithmetic as pca_decode_kernel: one sequential fp32 FMA chain over k ascending, + mean, (+ identity).
#ifndef LR_PT_ROWS
#define LR_PT_ROWS 128
#endif
#ifndef LR_PT_STAGES
#define LR_PT_STAGES 3
#endif
constexpr int PT_ROWS = LR_PT_ROWS;
constexpr int PT_STAGES = LR_PT_STAGES;

__device__ __forceinline__ uint32_t pd_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(pd_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(pd_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "LR_WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra LR_DONE_%=;\n"
        "bra LR_WAIT_%=;\n"
        "LR_DONE_%=:\n"
        "}\n" ::"r"(pd_smem_u32(bar)), "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_1d(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(pd_smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(pd_smem_u32(bar))
                 : "memory");
}

template <int BT>
__global__ void __launch_bounds__(PT_ROWS)
    pca_decode_tma_kernel(const float *__restrict__ coefs, const float *__restrict__ basis, const float *__restrict__ mean,
                          float *__restrict__ out, PcaDims g) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t full[PT_STAGES];
    const int tile_floats = PT_ROWS * g.K;               // K % 4 == 0: every stage is 16-byte aligned
    float *cf = smem + (size_t)PT_STAGES * tile_floats;  // [K][BT], zero-padded beyond B
    const int tid = threadIdx.x;
    for (int i = tid; i < g.K * BT; i += PT_ROWS) {
        const int k = i / BT, b = i - k * BT;
        cf[i] = b < g.B ? coefs[(int64_t)b * g.K + k] : 0.0f;
    }
    if (tid == 0) {
        for (int s2 = 0; s2 < PT_STAGES; ++s2) mbar_init(&full[s2], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();

    const int64_t n_tiles = (g.N + PT_ROWS - 1) / PT_ROWS;
    const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    auto issue = [&](int64_t it) {          // thread 0: start the copy of this block's it-th tile into stage it % PT_STAGES
        const int64_t row0 = (blockIdx.x + it * gridDim.x) * PT_ROWS;
        const uint32_t bytes = (uint32_t)(min((int64_t)PT_ROWS, g.N - row0) * g.K * 4);
        const int st = (int)(it % PT_STAGES);
        mbar_expect_tx(&full[st], bytes);
        tma_load_1d(smem + (size_t)st * tile_floats, basis + row0 * g.K, bytes, &full[st]);
    };
    if (tid == 0)
        for (int64_t it = 0; it < PT_STAGES - 1 && it < my_tiles; ++it) issue(it);

    for (int64_t it = 0; it < my_tiles; ++it) {
        const int st = (int)(it % PT_STAGES);
        // the stage refilled now was consumed in iteration it-1 (the barrier at the end of the loop body orders it)
        if (tid == 0 && it + PT_STAGES - 1 < my_tiles) issue(it + PT_STAGES - 1);
        mbar_wait(&full[st], (uint32_t)((it / PT_STAGES) & 1));
        const int64_t row0 = (blockIdx.x + it * gridDim.x) * PT_ROWS;
        const int rows = (int)min((int64_t)PT_ROWS, g.N - row0);
        if (tid < rows) {
            float acc[BT];
#pragma unroll
            for (int b = 0; b < BT; ++b) acc[b] = 0.0f;
            const float *myrow = smem + (size_t)st * tile_floats + tid * g.K;
            for (int k = 0; k < g.K; k += 4) {
                const float4 w4 = *reinterpret_cast<const float4 *>(myrow + k);
                const float w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {          // k ascending: one sequential fp32 FMA chain per output
                    if (BT >= 4) {
#pragma unroll
                        for (int b = 0; b < BT; b += 4) {
                            const float4 c = *reinterpret_cast<const float4 *>(cf + (k + kk) * BT + b);
                            acc[b] = fma_rn(c.x, w[kk], acc[b]); acc[b + 1] = fma_rn(c.y, w[kk], acc[b + 1]);
                            acc[b + 2] = fma_rn(c.z, w[kk], acc[b + 2]); acc[b + 3] = fma_rn(c.w, w[kk], acc[b + 3]);
                        }
                    } else {
#pragma unroll
                        for (int b = 0; b < BT; ++b) acc[b] = fma_rn(cf[(k + kk) * BT + b], w[kk], acc[b]);
                    }
                }
            }
            const int64_t n = row0 + tid;
            const float m = mean ? ld_stream(mean + n) : 0.0f;
            float idv = 0.0f;
            if (g.add_identity) {                         // model :68: deform_field = disp_field + id_transform
                const int c = (int)(n / g.nvox);
                const int v = (int)(n - (int64_t)c * g.nvox);
                const int z = v / (g.H * g.W), rem = v - z * (g.H * g.W), y = rem / g.W, x = rem - y * g.W;
                idv = c == 0 ? pd_identity_coord(z, g.sp0) : (c == 1 ? pd_identity_coord(y, g.sp1) : pd_identity_coord(x, g.sp2));
            }
#pragma unroll
            for (int b = 0; b < BT; ++b) {
                if (b < g.B) {
                    float o = add_rn(acc[b], m);
                    if (g.add_identity) o = add_rn(o, idv);
                    st_stream(out + (int64_t)b * g.N + n, o);
                }
            }
        }
        __syncthreads();                                  // every thread is done with this stage before it is refilled
    }
}

// Adjoint wrt the coefficients: grad_coefs[b,k] += sum_n grad_out[b,n] * basis[n,k] -- the second full pass over the
// basis that a training step makes (autograd of F.linear at model :102).  Same tile staging as the forward; thread
// (k, row-group) accumulates its column over a quarter of the tile's rows for all batch items, partial sums stay in
// registers across the block's tiles and are reduced once at the end (shared memory, then RED.ADD.F32: the summation
// order across blocks is not fixed, results agree with a sequential sum to fp32 round-off).
template <int BT, bool VEC>      // VEC: K % 4 == 0 and a 16-byte aligned basis (float4 staging); else scalar staging, odd pitch
__global__ void __launch_bounds__(PD_ROWS)
    pca_decode_backward_kernel(const float *__restrict__ gout, const float *__restrict__ basis, float *__restrict__ gcoefs,
                               PcaDims g) {
    extern __shared__ float smem[];
    const int pitch = VEC ? pd_pitch(g.K) : (g.K | 1);
    float *tile = smem;                                  // [PD_ROWS][pitch]
    float *gs = smem + (size_t)PD_ROWS * pitch;          // [PD_ROWS][BT] grad_out of the tile's rows
    const int tid = threadIdx.x;
    const int kpad = ((g.K + 31) / 32) * 32;             // threads per row-group (whole warps)
    const int n_groups = PD_ROWS / kpad > 0 ? PD_ROWS / kpad : 1;
    const int grp = tid / kpad, k = tid - grp * kpad;
    const bool worker = grp < n_groups && k < g.K;
    const int rows_per_grp = PD_ROWS / n_groups;
    const int k4 = g.K / 4;
    const int tile_f4 = PD_ROWS * k4;
    float acc[BT];
#pragma unroll
    for (int b = 0; b < BT; ++b) acc[b] = 0.0f;

    for (int64_t t = blockIdx.x; t < g.n_tiles; t += gridDim.x) {
        const int64_t row0 = t * PD_ROWS;
        const int rows = (int)min((int64_t)PD_ROWS, g.N - row0);
        __syncthreads();
        if (VEC) {
            const float4 *src = reinterpret_cast<const float4 *>(basis + row0 * g.K);
            const int n_f4 = rows * k4;
            constexpr int UNR = 7;
            for (int f0 = tid; f0 < tile_f4; f0 += UNR * PD_ROWS) {
                float4 v[UNR];
#pragma unroll
                for (int u = 0; u < UNR; ++u) {
                    const int f = f0 + u * PD_ROWS;
                    if (f < n_f4) v[u] = ld_stream4(src + f);
                }
#pragma unroll
                for (int u = 0; u < UNR; ++u) {
                    const int f = f0 + u * PD_ROWS;
                    if (f < n_f4) {
                        const int r = f / k4, kk = (f - r * k4) * 4;
                        *reinterpret_cast<float4 *>(tile + r * pitch + kk) = v[u];
                    }
                }
            }
        } else {
            const float *src = basis + row0 * g.K;
            for (int f = tid; f < rows * g.K; f += PD_ROWS) {
                const int r = f / g.K;
                tile[r * pitch + (f - r * g.K)] = ld_stream(src + f);
            }
        }
#pragma unroll
        for (int b = 0; b < BT; ++b)                      // thread = row: its grad_out values (0 beyond the end)
            gs[tid * BT + b] = (tid < rows && b < g.B) ? ld_stream(gout + (int64_t)b * g.N + row0 + tid) : 0.0f;
        __syncthreads();
        if (worker) {
            const int r_lo = grp * rows_per_grp, r_hi = min(rows, r_lo + rows_per_grp);
            for (int r = r_lo; r < r_hi; ++r) {
                const float w = tile[r * pitch + k];
#pragma unroll
                for (int b = 0; b < BT; ++b) acc[b] = fmaf(gs[r * BT + b], w, acc[b]);
            }
        }
    }
    // block reduction over the row groups, then one RED per (b,k)
    __syncthreads();
    float *red = smem;                                   // [n_groups][K][BT] (reuses the tile)
    if (worker) {
#pragma unroll
        for (int b = 0; b < BT; ++b) red[(grp * g.K + k) * BT + b] = acc[b];
    }
    __syncthreads();
    for (int i = tid; i < g.K * BT; i += PD_ROWS) {
        const int kk = i / BT, b = i - kk * BT;
        if (b < g.B) {
            float sum = 0.0f;
            for (int q = 0; q < n_groups; ++q) sum += red[(q * g.K + kk) * BT + b];
            red_add(gcoefs + (int64_t)b * g.K + kk, sum);
        }
    }
}

static int gcd_int(int a, int b) { return b == 0 ? a : gcd_int(b, a % b); }

template <int BT>
static int launch_pca(const float *coefs, const float *basis, const float *mean, float *out, const PcaDims &g,
                      cudaStream_t st) {
    const bool vec = g.K % 4 == 0 && ((uintptr_t)basis & 15) == 0;
    if (vec && gcd_int(g.K / 4, 8) <= 2) {
        // + 4 floats: the compiler reads the coefficient table four at a time in the k-loop's remainder iterations
        const size_t smem_t = sizeof(float) * ((size_t)PT_STAGES * PT_ROWS * g.K + (size_t)g.K * BT + 4);
        if (smem_t <= 110 * 1024) {
            if (smem_t > 48 * 1024) {
                static thread_local int smem_dev = -1;
                const cudaError_t ce = opt_in_smem(pca_decode_tma_kernel<BT>, 110 * 1024, smem_dev);
                if (int e = cuda_ok(ce, "pca_decode: cannot raise shared memory limit")) return e;
            }
            const int64_t n_tiles = (g.N + PT_ROWS - 1) / PT_ROWS;
            int per_sm = (int)((224 * 1024) / (smem_t + 1024));
            if (per_sm > 4) per_sm = 4;
            int64_t grid = (int64_t)sm_count() * per_sm;
            if (grid > n_tiles) grid = n_tiles;
            pca_decode_tma_kernel<BT><<<(unsigned)grid, PT_ROWS, smem_t, st>>>(coefs, basis, mean, out, g);
            return check_launch("pca_decode_tma_kernel");
        }
    }
    const int pitch = vec ? pd_pitch(g.K) : (g.K | 1);
    // + 4 floats: the compiler reads the coefficient table four at a time in the k-loop's remainder iterations
    const size_t smem = sizeof(float) * ((size_t)PD_ROWS * pitch + (size_t)g.K * BT + 4);
    if (smem > 200 * 1024) { set_error("pca_decode: K=%d needs %zu bytes of shared memory", g.K, smem); return LR_ERR_BAD_ARGUMENT; }
    if (smem > 48 * 1024) {
        static thread_local int vec_dev = -1, scalar_dev = -1;
        const cudaError_t ce = vec ? opt_in_smem(pca_decode_kernel<BT>, 200 * 1024, vec_dev)
                                   : opt_in_smem(pca_decode_scalar_kernel<BT>, 200 * 1024, scalar_dev);
        if (int e = cuda_ok(ce, "pca_decode: cannot raise shared memory limit")) return e;
    }
    int per_sm = (int)((220 * 1024) / (smem + 1024));
    if (per_sm > 8) per_sm = 8;
    if (per_sm < 1) per_sm = 1;
    int64_t grid = (int64_t)148 * per_sm;
    if (grid > g.n_tiles) grid = g.n_tiles;
    if (vec) pca_decode_kernel<BT><<<(unsigned)grid, PD_ROWS, smem, st>>>(coefs, basis, mean, out, g);
    else pca_decode_scalar_kernel<BT><<<(unsigned)grid, PD_ROWS, smem, st>>>(coefs, basis, mean, out, g);
    return check_launch("pca_decode_kernel");
}

// TMA-pipelined adjoint: the same ring of stages as pca_decode_tma_kernel; a stage holds the basis tile (unpadded:
// thread = coefficient k reads column k of consecutive rows, conflict-free) and the tile's grad_out rows of every batch
// item ([b][row], one 512-byte bulk copy per item).
template <int BT>
__global__ void __launch_bounds__(PT_ROWS)
    pca_decode_backward_tma_kernel(const float *__restrict__ gout, const float *__restrict__ basis, float *__restrict__ gcoefs,
                                   PcaDims g) {
    extern __shared__ __align__(128) float smem[];
    __shared__ __align__(8) uint64_t full[PT_STAGES];
    const int tile_floats = PT_ROWS * g.K, stage_floats = tile_floats + BT * PT_ROWS;
    const int tid = threadIdx.x;
    const int kpad = ((g.K + 31) / 32) * 32;             // threads per row-group (whole warps)
    const int n_groups = PT_ROWS / kpad > 0 ? PT_ROWS / kpad : 1;
    const int grp = tid / kpad, k = tid - grp * kpad;
    const bool worker = grp < n_groups && k < g.K;
    const int rows_per_grp = PT_ROWS / n_groups;
    if (tid == 0) {
        for (int s2 = 0; s2 < PT_STAGES; ++s2) mbar_init(&full[s2], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const int64_t n_tiles = (g.N + PT_ROWS - 1) / PT_ROWS;
    const int64_t my_tiles = blockIdx.x < n_tiles ? (n_tiles - 1 - blockIdx.x) / gridDim.x + 1 : 0;
    auto issue = [&](int64_t it) {
        const int64_t row0 = (blockIdx.x + it * gridDim.x) * PT_ROWS;
        const int rows = (int)min((int64_t)PT_ROWS, g.N - row0);      // N % 4 == 0 on this path: rows*4 is a multiple of 16
        const int st = (int)(it % PT_STAGES);
        float *stage = smem + (size_t)st * stage_floats;
        mbar_expect_tx(&full[st], (uint32_t)(rows * g.K * 4 + g.B * rows * 4));
        tma_load_1d(stage, basis + row0 * g.K, (uint32_t)(rows * g.K * 4), &full[st]);
        for (int b = 0; b < g.B; ++b) tma_load_1d(stage + tile_floats + b * PT_ROWS, gout + (int64_t)b * g.N + row0, (uint32_t)(rows * 4), &full[st]);
    };
    if (tid == 0)
        for (int64_t it = 0; it < PT_STAGES - 1 && it < my_tiles; ++it) issue(it);
    float acc[BT];
#pragma unroll
    for (int b = 0; b < BT; ++b) acc[b] = 0.0f;
    for (int64_t it = 0; it < my_tiles; ++it) {
        const int st = (int)(it % PT_STAGES);
        if (tid == 0 && it + PT_STAGES - 1 < my_tiles) issue(it + PT_STAGES - 1);
        mbar_wait(&full[st], (uint32_t)((it / PT_STAGES) & 1));
        const int64_t row0 = (blockIdx.x + it * gridDim.x) * PT_ROWS;
        const int rows = (int)min((int64_t)PT_ROWS, g.N - row0);
        if (worker) {
            const float *tile = smem + (size_t)st * stage_floats, *gs = tile + tile_floats;
            const int r_lo = grp * rows_per_grp, r_hi = min(rows, r_lo + rows_per_grp);
#pragma unroll 4
            for (int r = r_lo; r < r_hi; ++r) {
                const float w = tile[r * g.K + k];
#pragma unroll
                for (int b = 0; b < BT; ++b)
                    if (b < g.B) acc[b] = fmaf(gs[b * PT_ROWS + r], w, acc[b]);
            }
        }
        __syncthreads();
    }
    // block reduction over the row groups, then one RED per (b,k)
    float *red = smem;                                   // [n_groups][K][BT] (reuses stage 0; all copies have landed)
    if (worker) {
#pragma unroll
        for (int b = 0; b < BT; ++b) red[(grp * g.K + k) * BT + b] = acc[b];
    }
    __syncthreads();
    for (int i = tid; i < g.K * BT; i += PT_ROWS) {
        const int kk = i / BT, b = i - kk * BT;
        if (b < g.B) {
            float sum = 0.0f;
            for (int q = 0; q < n_groups; ++q) sum += red[(q * g.K + kk) * BT + b];
            red_add(gcoefs + (int64_t)b * g.K + kk, sum);
        }
    }
}

template <int BT>
static int launch_pca_bwd(const float *gout, const float *basis, float *gcoefs, const PcaDims &g, cudaStream_t st) {
    if (g.K % 4 == 0 && ((uintptr_t)basis & 15) == 0 && g.N % 4 == 0 && ((uintptr_t)gout & 15) == 0 && g.K <= PT_ROWS) {
        const size_t smem_t = sizeof(float) * (size_t)PT_STAGES * ((size_t)PT_ROWS * g.K + (size_t)BT * PT_ROWS);
        if (smem_t <= 110 * 1024) {
            if (smem_t > 48 * 1024) {
                static thread_local int smem_dev = -1;
                const cudaError_t ce = opt_in_smem(pca_decode_backward_tma_kernel<BT>, 110 * 1024, smem_dev);
                if (int e = cuda_ok(ce, "pca_decode_backward: cannot raise shared memory limit")) return e;
            }
            const int64_t n_tiles = (g.N + PT_ROWS - 1) / PT_ROWS;
            int per_sm = (int)((224 * 1024) / (smem_t + 1024));
            if (per_sm > 4) per_sm = 4;
            int64_t grid = (int64_t)sm_count() * per_sm;
            if (grid > n_tiles) grid = n_tiles;
            pca_decode_backward_tma_kernel<BT><<<(unsigned)grid, PT_ROWS, smem_t, st>>>(gout, basis, gcoefs, g);
            return check_launch("pca_decode_backward_tma_kernel");
        }
    }
    const bool vec = g.K % 4 == 0 && ((uintptr_t)basis & 15) == 0;
    const size_t tile = (size_t)PD_ROWS * (vec ? pd_pitch(g.K) : (g.K | 1));
    size_t smem_f = tile + (size_t)PD_ROWS * BT;
    const size_t red = (size_t)(PD_ROWS / 32 + 1) * g.K * BT;
    if (red > tile) smem_f += red - tile;
    const size_t smem = sizeof(float) * smem_f;
    if (smem > 200 * 1024) { set_error("pca_decode_backward: needs %zu bytes of shared memory", smem); return LR_ERR_BAD_ARGUMENT; }
    if (smem > 48 * 1024) {
        static thread_local int vec_dev = -1, scalar_dev = -1;
        const cudaError_t ce = vec ? opt_in_smem(pca_decode_backward_kernel<BT, true>, 200 * 1024, vec_dev)
                                   : opt_in_smem(pca_decode_backward_kernel<BT, false>, 200 * 1024, scalar_dev);
        if (int e = cuda_ok(ce, "pca_decode_backward: cannot raise shared memory limit")) return e;
    }
    int per_sm = (int)((220 * 1024) / (smem + 1024));
    if (per_sm > 8) per_sm = 8;
    if (per_sm < 1) per_sm = 1;
    int64_t grid = (int64_t)148 * per_sm;
    if (grid > g.n_tiles) grid = g.n_tiles;
    if (vec) pca_decode_backward_kernel<BT, true><<<(unsigned)grid, PD_ROWS, smem, st>>>(gout, basis, gcoefs, g);
    else pca_decode_backward_kernel<BT, false><<<(unsigned)grid, PD_ROWS, smem, st>>>(gout, basis, gcoefs, g);
    return check_launch("pca_decode_backward_kernel");
}

}  // namespace lr

using namespace lr;

extern "C" int lr_pca_decode_backward(const float *grad_out, const float *basis, int B, int K, int64_t N, float *grad_coefs,
                                      lr_stream_t stream) {
    LR_REQUIRE(grad_out && basis && grad_coefs, "pca_decode_backward: null pointer");
    LR_REQUIRE(B > 0 && K > 0 && N > 0, "pca_decode_backward: non-positive dimension (B=%d K=%d N=%lld)", B, K, (long long)N);
    LR_REQUIRE(K <= 160, "pca_decode_backward: K must be <= 160 (got %d)", K);
    PcaDims g;
    g.K = K; g.N = N; g.add_identity = 0; g.D = g.H = g.W = 0; g.nvox = 1; g.sp0 = g.sp1 = g.sp2 = 0.0;
    g.n_tiles = (N + PD_ROWS - 1) / PD_ROWS;
    cudaStream_t st = as_stream(stream);
    for (int b0 = 0; b0 < B; b0 += 16) {
        const int nb = B - b0 < 16 ? B - b0 : 16;
        g.B = nb;
        const float *go = grad_out + (int64_t)b0 * N;
        float *gc = grad_coefs + (int64_t)b0 * K;
        int e;
        if (nb <= 1) e = launch_pca_bwd<1>(go, basis, gc, g, st);
        else if (nb <= 2) e = launch_pca_bwd<2>(go, basis, gc, g, st);
        else if (nb <= 4) e = launch_pca_bwd<4>(go, basis, gc, g, st);
        else if (nb <= 8) e = launch_pca_bwd<8>(go, basis, gc, g, st);
        else e = launch_pca_bwd<16>(go, basis, gc, g, st);
        if (e) return e;
    }
    return LR_OK;
}

extern "C" int lr_pca_decode(const float *coefs, const float *basis, const float *mean, int B, int K, int64_t N,
                             int add_identity, int D, int H, int W, float *out, lr_stream_t stream) {
    LR_REQUIRE(coefs && basis && out, "pca_decode: null pointer");
    LR_REQUIRE(B > 0 && K > 0 && N > 0, "pca_decode: non-positive dimension (B=%d K=%d N=%lld)", B, K, (long long)N);
    LR_REQUIRE(K <= 160, "pca_decode: K must be <= 160 (got %d)", K);
    if (add_identity) {
        LR_REQUIRE(D > 1 && H > 1 && W > 1 && (int64_t)3 * D * H * W == N && (int64_t)D * H * W < (1ll << 31),
                   "pca_decode: add_identity needs N == 3*D*H*W (N=%lld, D=%d H=%d W=%d)", (long long)N, D, H, W);
    }
    PcaDims g;
    g.K = K; g.N = N; g.add_identity = add_identity != 0;
    g.D = D; g.H = H; g.W = W; g.nvox = add_identity ? D * H * W : 1;
    g.sp0 = D > 1 ? 1.0 / (double)(D - 1) : 0.0; g.sp1 = H > 1 ? 1.0 / (double)(H - 1) : 0.0; g.sp2 = W > 1 ? 1.0 / (double)(W - 1) : 0.0;
    g.n_tiles = (N + PD_ROWS - 1) / PD_ROWS;
    cudaStream_t st = as_stream(stream);
    // batch items beyond 32 take further passes over the basis
    for (int b0 = 0; b0 < B; b0 += 32) {
        const int nb = B - b0 < 32 ? B - b0 : 32;
        g.B = nb;
        const float *c = coefs + (int64_t)b0 * K;
        float *o = out + (int64_t)b0 * N;
        int e;
        if (nb <= 1) e = launch_pca<1>(c, basis, mean, o, g, st);
        else if (nb <= 2) e = launch_pca<2>(c, basis, mean, o, g, st);
        else if (nb <= 4) e = launch_pca<4>(c, basis, mean, o, g, st);
        else if (nb <= 8) e = launch_pca<8>(c, basis, mean, o, g, st);
        else if (nb <= 16) e = launch_pca<16>(c, basis, mean, o, g, st);
        else e = launch_pca<32>(c, basis, mean, o, g, st);
        if (e) return e;
    }
    return LR_OK;
}
