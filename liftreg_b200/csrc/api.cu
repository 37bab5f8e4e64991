// Library plumbing of libliftreg_b200.so: error reporting, launch accounting and the host-buffer entry
// points (the numpy-in / numpy-out contract of the reference calls, e.g. sdct:59-100 calculate_projection).
#include <atomic>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>

#include <cstring>
#include "common.cuh"

namespace lr {

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};   // process-wide: autograd runs backward on its own thread

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

int check_launch(const char *what) {
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: launch failed: %s", what, cudaGetErrorString(e));
        return LR_ERR_CUDA;
    }
    return LR_OK;
}

int sm_count() {
    static thread_local int cached_dev = -1, cached_n = 148;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) { cudaGetLastError(); return cached_n; }
    if (dev != cached_dev) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) { cached_n = n; cached_dev = dev; }
        else cudaGetLastError();
    }
    return cached_n;
}

// Numerics of the interpolation blends (indices and weights are bit-exact in both modes): see lr_set_numerics.
static std::atomic<int> g_numerics{-1};
int numerics_mode() {
    int m = g_numerics.load(std::memory_order_relaxed);
    if (m < 0) {
        const char *e = getenv("LIFTREG_B200_NUMERICS");
        m = (e && (e[0] == 'e' || e[0] == 'E' || e[0] == '1')) ? LR_NUMERICS_EXACT : LR_NUMERICS_FAST;
        g_numerics.store(m, std::memory_order_relaxed);
    }
    return m;
}

static size_t align256(size_t n) { return (n + 255) & ~(size_t)255; }

// Pinned (page-locked, mapped) host memory can be read / written by kernels directly over PCIe (UVA).  The host
// entry points use that to stream the large read-once / write-once operands straight from / to host memory inside
// the kernel, which overlaps H2D, compute and D2H without any extra stream; pageable buffers take the staged path.
static bool host_ptr_is_mapped(const void *p, const void **dev_alias) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    if (a.type != cudaMemoryTypeHost || a.devicePointer == nullptr) return false;
    *dev_alias = a.devicePointer;
    return true;
}
static bool zero_copy_enabled() {
    static int v = -1;
    if (v < 0) { const char *e = getenv("LIFTREG_B200_ZERO_COPY"); v = (e && e[0] == '0') ? 0 : 1; }
    return v != 0;
}

int cuda_ok(cudaError_t e, const char *what) {
    if (e == cudaSuccess) return LR_OK;
    set_error("%s: %s", what, cudaGetErrorString(e));
    return LR_ERR_CUDA;
}

}  // namespace lr

using namespace lr;

extern "C" int lr_abi_version(void) { return 1; }
extern "C" const char *lr_last_error(void) { return g_err; }
extern "C" long long lr_launch_count(void) { return g_launches.load(); }
extern "C" void lr_launch_count_reset(void) { g_launches.store(0); }

extern "C" int lr_set_numerics(int mode) {
    LR_REQUIRE(mode == LR_NUMERICS_FAST || mode == LR_NUMERICS_EXACT, "set_numerics: mode must be 0 (fast) or 1 (exact)");
    g_numerics.store(mode);
    return LR_OK;
}
extern "C" int lr_get_numerics(void) { return numerics_mode(); }

extern "C" int lr_device_count(void) {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        set_error("cudaGetDeviceCount: %s", cudaGetErrorString(e));
        cudaGetLastError();
        return LR_ERR_NO_DEVICE;
    }
    return n;
}

// ---- DRR, host buffers ----------------------------------------------------------------------------
extern "C" size_t lr_drr_forward_host_workspace_bytes(int B, int d, int w, int h, int P, int rd, int rh) {
    if (B <= 0 || d <= 0 || w <= 0 || h <= 0 || P <= 0 || rd <= 0 || rh <= 0) return 0;
    return align256(sizeof(float) * (size_t)B * d * w * h) + align256(sizeof(float) * (size_t)B * P * rd * rh);
}

extern "C" int lr_drr_forward_host(const float *vol_host, int B, int d, int w, int h, const double *poses,
                                   int n_pose_sets, int P, int rd, int rh, const float spacing[3], int y_norm_mode,
                                   float out_scale, float *proj_host, void *workspace, size_t workspace_bytes,
                                   lr_stream_t stream) {
    LR_REQUIRE(vol_host && proj_host && workspace, "drr_forward_host: null pointer");
    const size_t need = lr_drr_forward_host_workspace_bytes(B, d, w, h, P, rd, rh);
    if (need == 0 || workspace_bytes < need) {
        set_error("drr_forward_host: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return LR_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    const size_t vol_bytes = sizeof(float) * (size_t)B * d * w * h, proj_bytes = sizeof(float) * (size_t)B * P * rd * rh;
    float *d_vol = (float *)workspace;
    float *d_proj = (float *)((char *)workspace + align256(vol_bytes));
    if (int e = cuda_ok(cudaMemcpyAsync(d_vol, vol_host, vol_bytes, cudaMemcpyHostToDevice, st), "drr_forward_host: H2D")) return e;
    if (int e = lr_drr_forward(d_vol, B, d, w, h, poses, n_pose_sets, P, rd, rh, spacing, y_norm_mode, out_scale, d_proj, stream)) return e;
    if (int e = cuda_ok(cudaMemcpyAsync(proj_host, d_proj, proj_bytes, cudaMemcpyDeviceToHost, st), "drr_forward_host: D2H")) return e;
    return cuda_ok(cudaStreamSynchronize(st), "drr_forward_host: sync");   // sdct:97 .cpu() is synchronous
}

// ---- backprojection, host buffers -------------------------------------------------------------------
extern "C" size_t lr_backproject_forward_host_workspace_bytes(int B, int P, int pw, int ph, int d, int w, int h) {
    if (B <= 0 || P <= 0 || pw <= 0 || ph <= 0 || d <= 0 || w <= 0 || h <= 0) return 0;
    return align256(sizeof(float) * (size_t)B * P * pw * ph) + align256(sizeof(float) * (size_t)B * P * d * w * h);
}

// Asynchronous form: H2D, kernel and D2H are enqueued on `stream` and the call returns without waiting.  Two such
// calls on two streams (e.g. this one and lr_warp_forward_host_async) overlap on the full-duplex link; the caller
// synchronises with lr_stream_synchronize (or its own cudaStreamSynchronize) before touching out_host.
extern "C" int lr_backproject_forward_host_async(const float *proj_host, const float *poses, int B, int P, int pw, int ph,
                                                 int d, int w, int h, float *out_host, void *workspace,
                                                 size_t workspace_bytes, lr_stream_t stream) {
    LR_REQUIRE(proj_host && out_host && workspace, "backproject_forward_host: null pointer");
    const size_t need = lr_backproject_forward_host_workspace_bytes(B, P, pw, ph, d, w, h);
    if (need == 0 || workspace_bytes < need) {
        set_error("backproject_forward_host: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return LR_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    const size_t in_bytes = sizeof(float) * (size_t)B * P * pw * ph, out_bytes = sizeof(float) * (size_t)B * P * d * w * h;
    float *d_in = (float *)workspace;
    float *d_out = (float *)((char *)workspace + align256(in_bytes));
    if (int e = cuda_ok(cudaMemcpyAsync(d_in, proj_host, in_bytes, cudaMemcpyHostToDevice, st), "backproject_forward_host: H2D")) return e;
    // (Writing the 65 MB result straight to pinned host memory from the kernel was measured slower than the copy
    // engine: 1.30 vs 1.23 ms at cfg 2, so this path stays staged; the warp below does stream over PCIe itself.)
    if (int e = lr_backproject_forward(d_in, poses, B, P, pw, ph, d, w, h, d_out, (int64_t)P * d * w * h, (int64_t)d * w * h, stream)) return e;
    return cuda_ok(cudaMemcpyAsync(out_host, d_out, out_bytes, cudaMemcpyDeviceToHost, st), "backproject_forward_host: D2H");
}

extern "C" int lr_backproject_forward_host(const float *proj_host, const float *poses, int B, int P, int pw, int ph,
                                           int d, int w, int h, float *out_host, void *workspace,
                                           size_t workspace_bytes, lr_stream_t stream) {
    if (int e = lr_backproject_forward_host_async(proj_host, poses, B, P, pw, ph, d, w, h, out_host, workspace, workspace_bytes, stream)) return e;
    return cuda_ok(cudaStreamSynchronize(as_stream(stream)), "backproject_forward_host: sync");
}

extern "C" int lr_stream_synchronize(lr_stream_t stream) {
    return cuda_ok(cudaStreamSynchronize(as_stream(stream)), "stream_synchronize");
}

// ---- peer-visible buffers for lr_drr_forward_peers (CUDA IPC between the per-GPU processes of one box) ----------------
extern "C" int lr_peer_alloc(size_t bytes, void **dev_ptr, unsigned char handle[LR_IPC_HANDLE_BYTES]) {
    LR_REQUIRE(dev_ptr && handle && bytes > 0, "peer_alloc: null pointer or empty buffer");
    static_assert(sizeof(cudaIpcMemHandle_t) == LR_IPC_HANDLE_BYTES, "IPC handle size");
    void *p = nullptr;
    if (int e = cuda_ok(cudaMalloc(&p, bytes), "peer_alloc: cudaMalloc")) return e;
    cudaIpcMemHandle_t hd;
    const cudaError_t ce = cudaIpcGetMemHandle(&hd, p);
    if (ce != cudaSuccess) {
        cudaFree(p);
        return cuda_ok(ce, "peer_alloc: cudaIpcGetMemHandle");
    }
    memcpy(handle, &hd, sizeof(hd));
    *dev_ptr = p;
    return LR_OK;
}

extern "C" int lr_peer_open(const unsigned char handle[LR_IPC_HANDLE_BYTES], void **dev_ptr) {
    LR_REQUIRE(dev_ptr && handle, "peer_open: null pointer");
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handle, sizeof(hd));
    return cuda_ok(cudaIpcOpenMemHandle(dev_ptr, hd, cudaIpcMemLazyEnablePeerAccess), "peer_open: cudaIpcOpenMemHandle");
}

extern "C" int lr_peer_close(void *dev_ptr) {
    LR_REQUIRE(dev_ptr, "peer_close: null pointer");
    return cuda_ok(cudaIpcCloseMemHandle(dev_ptr), "peer_close: cudaIpcCloseMemHandle");
}

extern "C" int lr_peer_free(void *dev_ptr) {
    LR_REQUIRE(dev_ptr, "peer_free: null pointer");
    return cuda_ok(cudaFree(dev_ptr), "peer_free: cudaFree");
}

// ---- warp, host buffers -----------------------------------------------------------------------------
extern "C" size_t lr_warp_forward_host_workspace_bytes(int B, int C, int D, int H, int W) {
    if (B <= 0 || C <= 0 || D <= 0 || H <= 0 || W <= 0) return 0;
    const size_t nv = (size_t)D * H * W;
    return 2 * align256(sizeof(float) * B * C * nv) + align256(sizeof(float) * B * 3 * nv);
}

static int warp_forward_host_enqueue(const float *img_host, const float *phi_host, int B, int C, int D, int H, int W,
                                     int padding, int mode, int using_scale, int disp_plus_identity, float *out_host,
                                     void *workspace, size_t workspace_bytes, lr_stream_t stream, bool allow_zero_copy) {
    LR_REQUIRE(img_host && phi_host && out_host && workspace, "warp_forward_host: null pointer");
    const size_t need = lr_warp_forward_host_workspace_bytes(B, C, D, H, W);
    if (need == 0 || workspace_bytes < need) {
        set_error("warp_forward_host: workspace too small (%zu < %zu bytes)", workspace_bytes, need);
        return LR_ERR_WORKSPACE;
    }
    cudaStream_t st = as_stream(stream);
    const size_t nv = (size_t)D * H * W;
    const size_t img_bytes = sizeof(float) * B * C * nv, phi_bytes = sizeof(float) * B * 3 * nv;
    float *d_img = (float *)workspace;
    float *d_phi = (float *)((char *)workspace + align256(img_bytes));
    float *d_out = (float *)((char *)d_phi + align256(phi_bytes));
    if (int e = cuda_ok(cudaMemcpyAsync(d_img, img_host, img_bytes, cudaMemcpyHostToDevice, st), "warp_forward_host: H2D img")) return e;
    const void *phi_alias = nullptr, *out_alias = nullptr;
    if (allow_zero_copy && zero_copy_enabled() && host_ptr_is_mapped(phi_host, &phi_alias) && host_ptr_is_mapped(out_host, &out_alias)) {
        // the image is gathered 8x per voxel and must sit in HBM; the map is read once and the result written once, so
        // the kernel streams both over PCIe itself (H2D of phi, compute and D2H of the result overlap in one pass)
        return lr_warp_forward(d_img, (const float *)phi_alias, B, C, D, H, W, padding, mode, using_scale, disp_plus_identity, (float *)out_alias, stream);
    }
    if (int e = cuda_ok(cudaMemcpyAsync(d_phi, phi_host, phi_bytes, cudaMemcpyHostToDevice, st), "warp_forward_host: H2D phi")) return e;
    if (int e = lr_warp_forward(d_img, d_phi, B, C, D, H, W, padding, mode, using_scale, disp_plus_identity, d_out, stream)) return e;
    return cuda_ok(cudaMemcpyAsync(out_host, d_out, img_bytes, cudaMemcpyDeviceToHost, st), "warp_forward_host: D2H");
}

// The asynchronous form always stages through the copy engines: it exists to overlap with OTHER transfers (the
// backprojection's D2H on a second stream), and there the kernel-driven PCIe streaming of the blocking form competes
// with the copy engine for the link (measured at cfg 2, both calls in flight: 1.92 ms with it, 1.71 ms staged).
extern "C" int lr_warp_forward_host_async(const float *img_host, const float *phi_host, int B, int C, int D, int H, int W,
                                          int padding, int mode, int using_scale, int disp_plus_identity,
                                          float *out_host, void *workspace, size_t workspace_bytes, lr_stream_t stream) {
    return warp_forward_host_enqueue(img_host, phi_host, B, C, D, H, W, padding, mode, using_scale, disp_plus_identity, out_host,
                                     workspace, workspace_bytes, stream, false);
}

extern "C" int lr_warp_forward_host(const float *img_host, const float *phi_host, int B, int C, int D, int H, int W,
                                    int padding, int mode, int using_scale, int disp_plus_identity, float *out_host,
                                    void *workspace, size_t workspace_bytes, lr_stream_t stream) {
    if (int e = warp_forward_host_enqueue(img_host, phi_host, B, C, D, H, W, padding, mode, using_scale, disp_plus_identity, out_host, workspace, workspace_bytes, stream, true)) return e;
    return cuda_ok(cudaStreamSynchronize(as_stream(stream)), "warp_forward_host: sync");
}
