// Shared device helpers for the LiftReg resampling kernels (sm_100a).
//
// Numerical contract: the reference evaluates every coordinate and weight as a chain of separately
// rounded fp32 torch ops (SURVEY.md §7 "coordinate parity").  To keep ray and voxel indexing bit-exact
// the kernels replay that chain with explicitly rounded intrinsics (__fadd_rn/__fmul_rn are never
// contracted into FMAs by nvcc) and use a fused multiply-add only where torch's CPU kernels do.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace lr {

__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ float div_rn(float a, float b) { return __fdiv_rn(a, b); }
__device__ __forceinline__ float fma_rn(float a, float b, float c) { return __fmaf_rn(a, b, c); }

// Correctly rounded x / c for a loop-invariant divisor c, given rc = RN(1/c) (Markstein: q0 = x*rc,
// r = x - c*q0 exactly, q = q0 + r*rc).  Bit-identical to __fdiv_rn for normal operands (validated over
// 6M values per divisor, tests/test_host_logic.py::test_markstein_division); 3 instructions instead of ~10.
struct ConstDiv {
    float c, rc;
};
__host__ __device__ __forceinline__ ConstDiv make_const_div(float c) {
    ConstDiv k;
    k.c = c;
    k.rc = 1.0f / c;
    return k;
}
__device__ __forceinline__ float div_const(float x, ConstDiv k) {
    float q0 = __fmul_rn(x, k.rc);
    float r = __fmaf_rn(-k.c, q0, x);
    return __fmaf_rn(r, k.rc, q0);
}

// floor(x) as float and int for |x| < 2^22, on the FP32/ALU pipes only.  FRND/F2I/I2F run on the XU pipe at 16
// lanes/clk/SM and saturated it in the first version of these kernels (ncu: xu 95 %).  Adding 1.5*2^23 (where one
// ulp is 1) with round-toward-minus-infinity (FADD.RM) lands exactly on 1.5*2^23 + floor(x): the float floor is one
// exact subtraction away and the integer floor sits in the mantissa.  Callers keep |x| < 2^22 (clamp / clip);
// out-of-range or NaN inputs yield an int outside any realistic volume, which the bounds tests then reject.
__device__ __forceinline__ void floor_fi(float x, float &f, int &i) {
    const float M = 12582912.0f;                  // 1.5 * 2^23 = 0x4B400000
    const float t = __fadd_rd(x, M);
    f = __fsub_rn(t, M);                          // exact
    i = __float_as_int(t) - 0x4B400000;
}
// nearbyint(x) (half to even) for |x| < 2^22, same trick without the compare
__device__ __forceinline__ int rint_i(float x) {
    return __float_as_int(__fadd_rn(x, 12582912.0f)) - 0x4B400000;
}
__device__ __forceinline__ float clamp_index(float x, float hi) {   // keep |x| < 2^22; NaN -> -2
    return fminf(fmaxf(x, -2.0f), hi);
}

// ---- packed fp32x2 arithmetic (Blackwell: FADD2 / FMUL2 / FFMA2 issue two IEEE-rounded fp32 ops per slot) -----
// The resampling kernels are bound by instruction issue, not by the FMA pipe, so each thread processes TWO
// independent outputs and runs their (identical) fp32 op sequences as one packed sequence.  Every lane of a
// packed op is rounded exactly like the scalar op (.rn), so bit-exactness against the reference is unaffected.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
    f32x2 r;
    asm("mov.b64 %0, {%1,%2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(f32x2 a, float &lo, float &hi) {
    asm("mov.b64 {%0,%1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a));
}
__device__ __forceinline__ f32x2 splat2(float v) { return pack2(v, v); }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 sub2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
    f32x2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
    return r;
}
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
    f32x2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
    return r;
}
// a*b rounded on its own, for products that feed an add: ptxas (12.9) contracts mul.rn.f32x2 + add.rn.f32x2 into a
// single-rounding FFMA2 whatever the flags (it does not do that to the scalar .rn forms).  `zero` must be a
// run-time +0 that the compiler cannot see through (a kernel parameter): fma(a, b, +0) == RN(a*b).
__device__ __forceinline__ f32x2 mul2_sep(f32x2 a, f32x2 b, f32x2 zero) { return fma2(a, b, zero); }
// packed Markstein division by a loop-invariant (see div_const)
__device__ __forceinline__ f32x2 div_const2(f32x2 x, ConstDiv k) {
    const f32x2 rc = splat2(k.rc);
    const f32x2 q0 = mul2(x, rc);
    const f32x2 r = fma2(splat2(-k.c), q0, x);
    return fma2(r, rc, q0);
}
// packed floor for two values with |x| < 2^22: float floors and int floors (FADD2.RM, see floor_fi)
__device__ __forceinline__ void floor2_fi(f32x2 x, f32x2 &f, int &i_lo, int &i_hi) {
    const f32x2 M = splat2(12582912.0f);
    f32x2 t;
    asm("add.rm.f32x2 %0, %1, %2;" : "=l"(t) : "l"(x), "l"(M));
    f = sub2(t, M);
    float tl, th;
    unpack2(t, tl, th);
    i_lo = __float_as_int(tl) - 0x4B400000;
    i_hi = __float_as_int(th) - 0x4B400000;
}

// Hides how a pointer was computed so that nvcc keeps it in a register pair instead of re-deriving it (as a 64-bit
// multiply-add chain) at every use: `opaque(base) + u32_index` then costs a single IMAD.WIDE.U32.
template <typename T>
__device__ __forceinline__ T *opaque(T *p) {
    asm volatile("" : "+l"(p));
    return p;
}

// Streaming (read-once / write-once) accesses: keep them out of L1 so the gather working set stays resident.
__device__ __forceinline__ float ld_stream(const float *p) {
    float v;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ float4 ld_stream4(const float4 *p) {
    float4 v;
    asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                 : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
                 : "l"(p));
    return v;
}
__device__ __forceinline__ void st_stream(float *p, float v) {
    asm volatile("st.global.L1::no_allocate.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void st_stream4(float4 *p, float4 v) {
    asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y), "f"(v.z),
                 "f"(v.w)
                 : "memory");
}

// fire-and-forget fp32 reduction to global memory (RED.E.ADD.F32)
__device__ __forceinline__ void red_add(float *p, float v) {
    asm volatile("red.global.add.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
// the same under a predicate that lives inside the instruction (@p RED): the compiler branches around an `asm volatile`
// instead of predicating it, which costs BSSY + BRA + BSYNC per conditional reduction
__device__ __forceinline__ void red_add_if(bool on, float *p, float v) {
    asm volatile("{\n\t.reg .pred q;\n\tsetp.ne.u32 q, %2, 0;\n\t@q red.global.add.f32 [%0], %1;\n\t}" ::"l"(p), "f"(v), "r"((unsigned)on) : "memory");
}

}  // namespace lr

// ---- host-side plumbing shared by the .cu files -------------------------------------------------
#include "../../include/liftreg_b200.h"
namespace lr {
void set_error(const char *fmt, ...);
int check_launch(const char *what);  // cudaGetLastError -> lr_status; bumps the per-thread launch counter
int cuda_ok(cudaError_t e, const char *what);  // LR_OK, or LR_ERR_CUDA with the error "what: <cuda message>"
int sm_count();                      // multiprocessors of the current device (cached per device)
int numerics_mode();                 // LR_NUMERICS_FAST / LR_NUMERICS_EXACT (lr_set_numerics)
inline cudaStream_t as_stream(lr_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// Resident blocks per SM of `kernel`, or `fallback` when the occupancy query fails (its error is cleared, so that the
// next check_launch does not report it) or finds none.
template <typename K>
int blocks_per_sm(K kernel, int threads, size_t smem, int fallback) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, smem) != cudaSuccess || n < 1) {
        cudaGetLastError();
        n = fallback;
    }
    return n;
}

// Raise the dynamic shared-memory limit of `kernel` to `bytes` (the > 48 KB opt-in).  The attribute belongs to the
// current device, so it is set again whenever the device differs from `done_dev`, the caller's per-thread record of
// the last device it was set on.
template <typename K>
cudaError_t opt_in_smem(K kernel, int bytes, int &done_dev) {
    int dev = 0;
    cudaError_t ce = cudaGetDevice(&dev);
    if (ce == cudaSuccess && dev != done_dev) {
        ce = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
        if (ce == cudaSuccess) done_dev = dev;
    }
    return ce;
}

// ATen grid_sampler_unnormalize(align_corners) then optional clip_coordinates: the sample coordinate of the warp, and
// of every kernel that samples as the warp does.
template <int PAD>
__device__ __forceinline__ float source_index(float g, float half_sm1, float sm1) {
    // ((g+1)/2)*(S-1) == RN(RN(g+1) * ((S-1)/2)): /2 is exact and (S-1)/2 is representable.
    float i = mul_rn(add_rn(g, 1.0f), half_sm1);
    if (PAD == LR_PAD_BORDER) i = fminf(sm1, fmaxf(i, 0.0f));
    return i;
}
}  // namespace lr

#define LR_REQUIRE(cond, ...)                \
    do {                                     \
        if (!(cond)) {                       \
            lr::set_error(__VA_ARGS__);      \
            return LR_ERR_BAD_ARGUMENT;      \
        }                                    \
    } while (0)
