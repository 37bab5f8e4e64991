/*
 * liftreg_b200.h -- C-ABI of the B200-native LiftReg resampling library
 * (libliftreg_b200.so, built from liftreg_b200/csrc/ for sm_100a).
 *
 * The reference (uncbiag/LiftReg) is pure Python: its "operator API" for this
 * path is the Python surface of
 *     src/liftreg/utils/sdct_projection_utils.py   ("sdct" below)
 *     src/liftreg/utils/net_utils.py               (Bilinear, identity_map)
 *     src/liftreg/layers/layers.py                 (proj_layer)
 *     src/liftreg/models/LiftRegDeformSubspaceBackproj.py:85-93,68-69
 * and every one of those bottoms out in torch.nn.functional.grid_sample.
 * Each entry point below replaces the cited reference lines; the Python mirror
 * in liftreg_b200/ binds them with ctypes (INTEGRATION.md shows the stub a
 * reference maintainer would add).
 *
 * Conventions
 *   - plain C types only; no torch / C++ types cross this boundary.
 *   - every buffer is owned by the caller; the library never allocates or frees
 *     device memory and keeps no state (geometry is passed by value per call).
 *   - all tensors are dense, C-contiguous fp32 unless a stride is given.
 *   - functions without the _host suffix take DEVICE pointers, are asynchronous
 *     on `stream` (a cudaStream_t) and never synchronise.  As with any CUDA
 *     launch, the calling thread's current device must be the device that owns
 *     `stream` and the buffers (the current device is per host thread).
 *   - _host functions take HOST pointers (pinned for full speed) plus a device
 *     workspace of lr_*_workspace_bytes(); they enqueue H2D, kernels and D2H on
 *     `stream` and synchronise it before returning, like the reference calls
 *     they replace (which end in .cpu().numpy()).  When the host buffers are
 *     pinned+mapped, lr_warp_forward_host lets the kernel stream the map and the
 *     result over PCIe itself (set LIFTREG_B200_ZERO_COPY=0 to force staging).
 *   - return 0 on success, a negative lr_status on failure; never throws or
 *     exits.  lr_last_error() returns a thread-local message.
 *   - volume axes (d,w,h) = (axial, coronal, sagittal); detector (rd,rh);
 *     emitter poses in voxel units, detector plane y = 0 (sdct:59-68).
 */
#ifndef LIFTREG_B200_H
#define LIFTREG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define LR_API __attribute__((visibility("default")))
#else
#define LR_API
#endif

typedef void *lr_stream_t; /* cudaStream_t */

typedef enum {
    LR_OK = 0,
    LR_ERR_BAD_ARGUMENT = -1,
    LR_ERR_CUDA = -2,
    LR_ERR_WORKSPACE = -3,
    LR_ERR_NO_DEVICE = -4
} lr_status;

enum { LR_PAD_ZEROS = 0, LR_PAD_BORDER = 1 };     /* net_utils.py:21  zero_boundary ? zeros : border */
enum { LR_MODE_LINEAR = 0, LR_MODE_NEAREST = 1 }; /* net_utils.py:23  mode = "bilinear" | "nearest"  */
enum { LR_YNORM_WM1 = 0, LR_YNORM_W = 1 };        /* sdct:55 (/(w-1))  vs  layers.py:234 (/w)        */
/* How the interpolation BLEND of lr_backproject_forward and lr_warp_forward (linear mode) is rounded.  Sample
 * coordinates, floor indices and interpolation weights replay the reference's fp32 op chain bit for bit in both modes.
 *   LR_NUMERICS_FAST  (default) the blend is a chain of fused linear interpolations (separable rows-then-columns for
 *                     the backprojection, x-y-z lerps for the warp; `using_scale` folds away where all taps are inside):
 *                     <= 1e-6 relative L2 from ATen's result (BASELINE.json's tolerance is 1e-5), half the instructions.
 *   LR_NUMERICS_EXACT ATen's own operation order (grid_sampler_2d vector kernel / grid_sampler_3d scalar kernel):
 *                     results bit-identical to the reference's torch CPU path.                                    */
enum { LR_NUMERICS_FAST = 0, LR_NUMERICS_EXACT = 1 };

/* ---- library ---------------------------------------------------------- */
LR_API int lr_abi_version(void);
LR_API const char *lr_last_error(void);
/* process-wide numerics mode (also: environment LIFTREG_B200_NUMERICS=exact|fast read at first use) */
LR_API int lr_set_numerics(int mode);
LR_API int lr_get_numerics(void);
/* number of CUDA devices visible, or a negative lr_status */
LR_API int lr_device_count(void);
/* kernels launched by this library (all threads) since the last reset (bench.py's gpu_launches) */
LR_API long long lr_launch_count(void);
LR_API void lr_launch_count_reset(void);

/* ---- cone-beam DRR ---------------------------------------------------- */
/* replaces sdct:59-86 calculate_projection (grid build sdct:15-57, flip :76, grid_sample+sum+*dx :81, *0.1 :85)
 * and layers.py:182-187 proj_layer.forward (y_norm_mode = LR_YNORM_W, out_scale = 1).
 *   vol   (B,d,w,h)       attenuation volume(s)
 *   poses (n_pose_sets,P,3) HOST pointer, float64, voxel units; n_pose_sets is 1 (shared by all B, as in
 *         proj_layer) or B (per item, models/previous/RegNet2D3D.py:161-171)
 *   proj  (B,P,rd,rh) = out_scale * dx[p,u,v] * sum_j trilinear_zeros(vol[b], ray point j)   */
LR_API int lr_drr_forward(const float *vol, int B, int d, int w, int h,
                          const double *poses, int n_pose_sets, int P, int rd, int rh,
                          const float spacing[3], int y_norm_mode, float out_scale,
                          float *proj, lr_stream_t stream);

/* Multi-GPU form of lr_drr_forward for view-sharded sweeps (BASELINE.json north star: "forward projection by view angle
 * ..., all-gather of the detector images over NVLink"; the reference itself is single-GPU, main.py:108-110).  The kernel
 * stores every detector pixel into n_outs buffers -- this rank's gather buffer and the peers' (device pointers obtained
 * with lr_peer_open, written as P2P stores over NVLink) -- so the images need no collective afterwards, only a barrier.
 * View k of the call (k = b*P + p) lands at outs[i] + k * view_stride * rd * rh: with view_stride = world size and
 * outs[i] pointing at this rank's first view, a rank that owns the views r, r+world, ... fills the full (n_views,rd,rh)
 * array in view order on every rank. */
#define LR_MAX_PEERS 8
LR_API int lr_drr_forward_peers(const float *vol, int B, int d, int w, int h,
                                const double *poses, int n_pose_sets, int P, int rd, int rh,
                                const float spacing[3], int y_norm_mode, float out_scale,
                                float *const *outs, int n_outs, int view_stride, lr_stream_t stream);
/* Peer-visible device buffers for the call above (CUDA IPC, one process per GPU on one box).
 * lr_peer_alloc: cudaMalloc on the current device + its 64-byte IPC handle (to be sent to the other ranks by any means).
 * lr_peer_open: maps another rank's buffer into this process (peer access enabled lazily); lr_peer_close unmaps it.
 * lr_peer_free releases a buffer obtained from lr_peer_alloc (after the peers closed it). */
#define LR_IPC_HANDLE_BYTES 64
LR_API int lr_peer_alloc(size_t bytes, void **dev_ptr, unsigned char handle[LR_IPC_HANDLE_BYTES]);
LR_API int lr_peer_open(const unsigned char handle[LR_IPC_HANDLE_BYTES], void **dev_ptr);
LR_API int lr_peer_close(void *dev_ptr);
LR_API int lr_peer_free(void *dev_ptr);

/* adjoint of lr_drr_forward wrt vol (autograd of sdct:81 / layers.py:187; RegNet2D3D.py:161-185 needs it).
 * grad_vol (B,d,w,h) is ACCUMULATED into (caller zero-initialises). */
LR_API int lr_drr_backward(const float *grad_proj, int B, int d, int w, int h,
                           const double *poses, int n_pose_sets, int P, int rd, int rh,
                           const float spacing[3], int y_norm_mode, float out_scale,
                           float *grad_vol, lr_stream_t stream);

/* replaces sdct:15-57 project_grid_multi / layers.py:194-236 (API parity and bit-exactness checks; the DRR
 * kernels never materialise this).  grid (P,rd,rh,w,3) nullable, dx (P,rd,rh) nullable.
 * flip != 0 writes the last axis reversed, as sdct:76 / forward_grids (sdct:223,263) return it. */
LR_API int lr_project_grid(const double *poses, int P, int rd, int rh, int d, int w, int h,
                           const float spacing[3], int y_norm_mode, int flip,
                           float *grid, float *dx, lr_stream_t stream);

/* host-buffer form of lr_drr_forward == calculate_projection's numpy-in / numpy-out contract (sdct:59-100). */
LR_API size_t lr_drr_forward_host_workspace_bytes(int B, int d, int w, int h, int P, int rd, int rh);
LR_API int lr_drr_forward_host(const float *vol_host, int B, int d, int w, int h,
                               const double *poses, int n_pose_sets, int P, int rd, int rh,
                               const float spacing[3], int y_norm_mode, float out_scale,
                               float *proj_host, void *workspace, size_t workspace_bytes, lr_stream_t stream);

/* ---- backprojection ---------------------------------------------------- */
/* replaces sdct:227-250 backproj_grids_with_poses + the grid_sample block at
 * models/LiftRegDeformSubspaceBackproj.py:85-93 (same block: models/previous/RegNet2D3D.py:105-112).
 *   proj  (B,P,pw,ph)
 *   poses (P,3) HOST pointer, float32 (Registration2D3DDataset.py:121 casts to fp32; geometry frozen from
 *         batch item 0, model :85-87)
 *   out[b*out_batch_stride + p*out_chan_stride + (i*w+j)*h+k] = bilinear_zeros(proj[b,p], u(p,i,j), v(p,j,k))
 *   strides are in elements; a dense (B,P,d,w,h) output uses P*d*w*h and d*w*h.  They let the caller aim at
 *   channels 1..P of the (B,1+P,d,w,h) encoder input and skip torch.cat (model :95-98). */
LR_API int lr_backproject_forward(const float *proj, const float *poses, int B, int P, int pw, int ph,
                                  int d, int w, int h, float *out,
                                  int64_t out_batch_stride, int64_t out_chan_stride, lr_stream_t stream);

/* z-slab form for multi-GPU sharding along axis 0 (SURVEY.md 8e): `out` holds planes [i_begin, i_begin+i_count)
 * only, i.e. a (B,P,i_count,w,h) tensor with the given strides; projections (<= 1 MB per item) are replicated on
 * every rank, so the op needs no halo and no collective. */
LR_API int lr_backproject_forward_slab(const float *proj, const float *poses, int B, int P, int pw, int ph,
                                       int d_total, int w, int h, int i_begin, int i_count, float *out,
                                       int64_t out_batch_stride, int64_t out_chan_stride, lr_stream_t stream);

/* adjoint wrt proj; grad_proj (B,P,pw,ph) is ACCUMULATED into (caller zero-initialises). */
LR_API int lr_backproject_backward(const float *grad_out, int64_t go_batch_stride, int64_t go_chan_stride,
                                   const float *poses, int B, int P, int pw, int ph, int d, int w, int h,
                                   float *grad_proj, lr_stream_t stream);

/* replaces sdct:227-250 itself: grid (P,2,d,w,h), channel 0 = detector axis 1 (ph), channel 1 = axis 0 (pw). */
LR_API int lr_backproj_grid(const float *poses, int P, int d, int w, int h, int pw, int ph,
                            float *grid, lr_stream_t stream);

LR_API size_t lr_backproject_forward_host_workspace_bytes(int B, int P, int pw, int ph, int d, int w, int h);
LR_API int lr_backproject_forward_host(const float *proj_host, const float *poses, int B, int P, int pw, int ph,
                                       int d, int w, int h, float *out_host,
                                       void *workspace, size_t workspace_bytes, lr_stream_t stream);
/* Overlapped form of the host-buffer calls: the *_host_async entry points enqueue H2D, kernels and D2H on `stream` and
 * return WITHOUT synchronising, so one host thread can put the backprojection on one stream and the warp on another and
 * the two transfers share the full-duplex PCIe link (the reference's calls, sdct:70-72,97-99, are serial and blocking).
 * Host buffers must be pinned for the copies to be asynchronous and must stay alive until the stream is synchronised:
 * lr_stream_synchronize(stream) (for callers without a CUDA runtime binding) or cudaStreamSynchronize. */
LR_API int lr_backproject_forward_host_async(const float *proj_host, const float *poses, int B, int P, int pw, int ph,
                                             int d, int w, int h, float *out_host,
                                             void *workspace, size_t workspace_bytes, lr_stream_t stream);
LR_API int lr_stream_synchronize(lr_stream_t stream);

/* ---- displacement-field warp ------------------------------------------- */
/* replaces net_utils.py:26-56 Bilinear.forward / forward_stn.
 *   img (B,C,D,H,W); phi (B,3,D,H,W), channel c addresses volume axis c in [-1,1] (the channel reversal of
 *   :27-30 is folded into the addressing); out (B,C,D,H,W).
 *   using_scale: sample (img+1)/2 and return 2*out-1 (:48-52), fused.
 *   disp_plus_identity != 0: phi holds the DISPLACEMENT and the normalised identity map
 *   (net_utils.py:59-87) is added in-kernel, i.e. the `disp_field + self.id_transform` of model :68 is fused;
 *   the sum is rounded to fp32 exactly as the torch add would.  The identity map needs D, H, W >= 2 (as
 *   lr_identity_map); a size-1 axis with disp_plus_identity != 0 is rejected (LR_ERR_BAD_ARGUMENT). */
LR_API int lr_warp_forward(const float *img, const float *phi, int B, int C, int D, int H, int W,
                           int padding, int mode, int using_scale, int disp_plus_identity,
                           float *out, lr_stream_t stream);

/* adjoint (autograd of grid_sample at net_utils.py:32-35 plus the (x+1)/2 and *2-1 factors).
 * grad_img (B,C,D,H,W) nullable, ACCUMULATED into (caller zero-initialises);
 * grad_phi (B,3,D,H,W) nullable, overwritten (zero for LR_MODE_NEAREST). */
LR_API int lr_warp_backward(const float *grad_out, const float *img, const float *phi,
                            int B, int C, int D, int H, int W,
                            int padding, int mode, int using_scale, int disp_plus_identity,
                            float *grad_img, float *grad_phi, lr_stream_t stream);

/* z-slab forms for multi-GPU sharding along axis 0 (SURVEY.md 8e): phi / out / grad_out / grad_phi are
 * (B,*,z_count,H,W) tensors holding output planes [z_begin, z_begin+z_count); img (and grad_img) stay the full
 * (B,C,D,H,W) volume, which every rank holds (16.4 MB at 160^3), so no halo exchange and no reduction is needed. */
LR_API int lr_warp_forward_slab(const float *img, const float *phi, int B, int C, int D, int H, int W,
                                int z_begin, int z_count, int padding, int mode, int using_scale,
                                int disp_plus_identity, float *out, lr_stream_t stream);
LR_API int lr_warp_backward_slab(const float *grad_out, const float *img, const float *phi,
                                 int B, int C, int D, int H, int W, int z_begin, int z_count,
                                 int padding, int mode, int using_scale, int disp_plus_identity,
                                 float *grad_img, float *grad_phi, lr_stream_t stream);

/* replaces net_utils.py:59-87 identity_map: out (3,D,H,W) */
LR_API int lr_identity_map(int D, int H, int W, float *out, lr_stream_t stream);

LR_API size_t lr_warp_forward_host_workspace_bytes(int B, int C, int D, int H, int W);
LR_API int lr_warp_forward_host(const float *img_host, const float *phi_host, int B, int C, int D, int H, int W,
                                int padding, int mode, int using_scale, int disp_plus_identity, float *out_host,
                                void *workspace, size_t workspace_bytes, lr_stream_t stream);
LR_API int lr_warp_forward_host_async(const float *img_host, const float *phi_host, int B, int C, int D, int H, int W,
                                      int padding, int mode, int using_scale, int disp_plus_identity, float *out_host,
                                      void *workspace, size_t workspace_bytes, lr_stream_t stream);

/* ---- PCA-subspace displacement decode (SURVEY.md 8f, row f2) ------------- */
/* replaces models/LiftRegDeformSubspaceBackproj.py:102
 *     disp_field = F.linear(x, self.pca_vectors, self.pca_mean)          (x: (B,K) coefficients)
 * and, if add_identity != 0, the `disp_field + self.id_transform` of :68 (N must then be 3*D*H*W; the (B,N) result
 * reshaped to (B,3,D,H,W) is the map phi that lr_warp_forward consumes).
 *   coefs (B,K); basis (N,K) row-major = pca_vectors as the model stores it (:42); K <= 160; the fast path needs
 *   K % 4 == 0 and a 16-byte aligned basis (anything else takes a scalar staging path);
 *   mean (N) nullable; out (B,N).
 * out[b,n] = (sum_k coefs[b,k]*basis[n,k], fp32 FMA chain, k ascending) + mean[n] (+ identity(n)).
 * The 4*N*K-byte basis (2.75 GB at 160^3, K = 56) is streamed from HBM exactly once for up to 32 batch items. */
LR_API int lr_pca_decode(const float *coefs, const float *basis, const float *mean, int B, int K, int64_t N,
                         int add_identity, int D, int H, int W, float *out, lr_stream_t stream);

/* adjoint wrt the coefficients (autograd of F.linear at model :102): grad_coefs (B,K) is ACCUMULATED into (caller
 * zero-initialises): grad_coefs[b,k] += sum_n grad_out[b,n] * basis[n,k].  K <= 160; K % 4 == 0 with 16-byte aligned
 * basis / grad_out takes the TMA-pipelined path, anything else a scalar staging path. */
LR_API int lr_pca_decode_backward(const float *grad_out, const float *basis, int B, int K, int64_t N,
                                  float *grad_coefs, lr_stream_t stream);

/* ---- HU -> attenuation -------------------------------------------------- */
/* replaces sdct:6-13 calc_relative_atten_coef(_cuda): mu = (max(HU,-1000)+1000)/1000*0.2; in place allowed */
LR_API int lr_atten_coef(const float *hu, int64_t n, float *mu, lr_stream_t stream);

/* ---- launch plans (diagnostics for host-side tests; no device work) ------- */
/* how lr_warp_forward cuts the z_count planes of an item into z-blocks: plan = {size0, n0, size1, n1, size2, n2} */
LR_API int lr_warp_forward_plan(int B, int D, int H, int W, int z_count, int plan[6]);
/* how lr_backproject_forward tiles planes, columns and rows: plan = {ichunk, isub, by, bx, n_chunks, run0, n0, run1, n1,
 * run2, n2, grid} */
LR_API int lr_backproject_forward_plan(int B, int P, int pw, int ph, int d, int w, int h, int plan[12]);

/* ---- measurement probes (diagnostics; bench.py's DRR fractions) -------------- */
/* lr_probe_l1_gather: every block re-reads its own floats_per_block-float (power of two >= 2048) slice of buf `iters`
 * times with coalesced 32-bit loads that hit L1: bytes moved = blocks*256*iters*32.  Timed by the caller, it gives the
 * aggregate L1 gather bandwidth that SURVEY.md 8d names as the DRR kernel's binding resource.
 * lr_probe_issue: blocks*256 threads each issue iters*8 independent FFMAs: the chip's sustained issue rate. */
LR_API int lr_probe_l1_gather(const float *buf, int64_t buf_floats, int blocks, int floats_per_block, int iters,
                              float *sink, lr_stream_t stream);
LR_API int lr_probe_issue(int blocks, int iters, float *sink, lr_stream_t stream);
/* lr_probe_issue_packed: the same with packed fp32x2 FMAs (blocks*256 threads, iters*8 FFMA2 each). */
LR_API int lr_probe_issue_packed(int blocks, int iters, float *sink, lr_stream_t stream);

/* ---- similarity loss on the warp output (SURVEY.md 8f row f4) -------------- */
/* replaces src/liftreg/layers/losses.py:14-29 NCCLoss.forward (training similarity, SubspaceLoss.py:27; validation score,
 * RegistrationNet.py:210-212):  a = x - mean(x) + 1e-10, b = y - mean(y) + 1e-10 per batch item over N voxels,
 * ncc = mean(a*b) / sqrt(mean(a*a) * mean(b*b)).
 * lr_ncc_sums (one pass over x and y) fills sums (B,7) float64, device memory owned by the caller (zeroed by the call):
 *   [sum x, sum y, sum a*b, sum a*a, sum b*b, sum a, sum b]  ->  ncc_b = s2 / sqrt(s3*s4); loss = 1 - mean_b ncc_b.
 * lr_ncc_backward: grad_x (B,N) = d(loss)/dx * grad_loss[0] (grad_loss: one float in device memory), from the same sums. */
LR_API int lr_ncc_sums(const float *x, const float *y, int B, int64_t N, double *sums, lr_stream_t stream);
LR_API int lr_ncc_backward(const float *x, const float *y, int B, int64_t N, const double *sums, const float *grad_loss,
                           float *grad_x, lr_stream_t stream);

/* ---- displacement regulariser of the subspace loss (SURVEY.md 8f row f4) ---- */
/* replaces src/liftreg/losses/SubspaceLoss.py:51-67 compute_reg_loss (same code: losses/RegNet2D3DLoss.py:53-69):
 *   fd = mermaid.finite_differences.FD_torch(spacing*2), spacing = 1/(shape-1);
 *   reg = mean over (B, D, H, W) of sum_{c<3} dXc(disp_c)^2 + dYc(disp_c)^2 + dZc(disp_c)^2
 * disp (B,3,D,H,W) float32, dense.  mermaid (third party, requirements.txt:61) is not part of the reference tree; its
 * central difference is (I[i+1]-I[i-1]) * 0.5/spacing in the interior, and on the faces either a linear extrapolation
 * of the missing neighbour (LR_FD_LINEAR, FD_torch's default mode) or zero (LR_FD_NEUMANN_ZERO).
 * lr_diffusion_reg_sum: *sum (one float64 in device memory, zeroed by the call) = sum over every voxel of the nine
 *   squares; reg = *sum / (B*D*H*W).
 * lr_diffusion_reg_backward: grad_disp (B,3,D,H,W) = d(reg)/d(disp) * grad_loss[0] (one float in device memory). */
#define LR_FD_LINEAR 0
#define LR_FD_NEUMANN_ZERO 1
LR_API int lr_diffusion_reg_sum(const float *disp, int B, int D, int H, int W, int boundary, double *sum, lr_stream_t stream);
LR_API int lr_diffusion_reg_backward(const float *disp, int B, int D, int H, int W, int boundary, const float *grad_loss,
                                     float *grad_disp, lr_stream_t stream);

/* ---- validation metrics (RegistrationNet.py:198-218 _compute_metrics) --------------------------------------------
 * PARITY UNPINNED: the reference's utils/utils.py and utils/metrics.py import mermaid and SimpleITK and are not part of
 * the reference tree, so which determinant, boundary crop, background rule and empty-label score they use is unknown.
 * These entries are defined from first principles, are not signature-compatible replacements, and no golden pins them.
 *
 * lr_jacobian_det replaces the host-side folding statistic of utils/utils.py:20-55 (numpy Jacobian determinant of phi
 * with mermaid's finite differences, each item's 3*D*H*W map copied to the host).
 *   phi (B,3,D,H,W) float32 in [-1,1], channel c addressing volume axis c (lr_warp_forward's convention); D,H,W >= 2.
 *   J[c][a] = central difference of phi_c along axis a * 0.5/(2/(n_a-1)), with the face rule `boundary` of
 *   lr_diffusion_reg_sum (LR_FD_LINEAR / LR_FD_NEUMANN_ZERO); the identity map has J = I.
 *   det = J00*(J11*J22 - J12*J21) - J01*(J10*J22 - J12*J20) + J02*(J10*J21 - J11*J20), each product and difference
 *   rounded to fp32 on its own, left to right.
 *   det (B,D,H,W) nullable: the determinant map.
 *   stats (B,7) float64, zeroed / initialised by the call, over the voxels at least `margin` (2*margin < every axis)
 *   from every face: [#det<0, sum |det| over det<0, min det, max det, sum det, sum det^2, #non-finite det]; sums
 *   accumulate in fp64, counts are exact, and min / max / the sums cover finite values only (min = +inf, max = -inf
 *   when there is none).  B*3*D*H*W must stay below 2^31.
 *
 * lr_label_confusion replaces the Python-set overlap scoring of utils/metrics.py:6-121 (get_multi_metric / cal_metric):
 * every per-label Dice, IoU, recall and precision follows from the L x L confusion matrix of (predicted, target) labels.
 *   pred, target (B,N) float32 label maps (what the nearest-mode warp returns); 1 <= L <= 128.
 *   counts (B,L,L) int64: counts[b][p][t] = #voxels with pred == p and target == t (exact).
 *   invalid (B) int64: #voxels where either value is not an integer in [0, L) (negative, >= L, fractional, NaN).
 *   Both outputs are zeroed by the call. */
LR_API int lr_jacobian_det(const float *phi, int B, int D, int H, int W, int boundary, int margin,
                           float *det, double *stats, lr_stream_t stream);
LR_API int lr_label_confusion(const float *pred, const float *target, int B, int64_t N, int L,
                              int64_t *counts, int64_t *invalid, lr_stream_t stream);

/* ---- surface-distance validation metrics (PARITY UNPINNED: the reference scores no surface metric) ------------------
 * The boundary scores registration papers report next to Dice (Hausdorff, HD95, average symmetric surface distance)
 * all follow from the directed surface distances below; metrics.surface_distance forms them.  These are voxel-based
 * distances, not the surfel-area-weighted ones of DeepMind's surface_distance package.
 *   pred, target / from, to: (B,D,H,W) float32 label maps (what the nearest-mode warp returns); labels 1..L-1 are
 *   scored, L <= 128; a value that is not an integer in [0, L) is "no label".
 *   The surface S_M(l) of label l in map M is the set of voxels with M == l that have at least one of their 6 face
 *   neighbours outside the volume or != l (scipy's m & ~binary_erosion(m, generate_binary_structure(3, 1),
 *   border_value=0)).
 * lr_label_surface_counts: counts (B,2,L) int64 = [|S_pred(l)|, |S_target(l)|] for every l in [0, L) (exact), and
 *   invalid (B) int64 = #voxels where either value is not an integer in [0, L), as lr_label_confusion counts them.
 *   Both outputs are zeroed by the call.
 * lr_surface_distances: for every voxel v of S_from(label), the distance from v to the nearest voxel n of S_to(label)
 *   with spacing (s_d, s_h, s_w), formed from the index offsets as scipy's distance_transform_edt forms it, in fp64:
 *     d(v) = sqrt(((s_d*(v_d - n_d))^2 + (s_h*(v_h - n_h))^2) + (s_w*(v_w - n_w))^2)    (+inf if S_to is empty)
 *   The nearest voxel is found by an exact separable transform (Meijster et al. 2000); with integer spacings every
 *   squared distance is an exact integer in fp64 and d(v) is bit-identical to scipy's whichever voxel a tie picks, and
 *   otherwise it is within 8*2^-53*d(v) of it (DESIGN.md §3).
 *   seg_offset (B+1) int64 in device memory, nondecreasing: item b's distances are written, in no particular order, to
 *   dist[seg_offset[b] .. seg_offset[b+1]); a segment holds |S_from(label)| of the item when the offsets come from
 *   lr_label_surface_counts of the same maps, and a write past a segment's end is dropped.
 *   stats (B,3) float64, overwritten by the call: [count, sum, max] of each item's distances (max 0 when the count is
 *   0).  The sum is reduced in a fixed order (no floating-point atomics), so repeated calls give the same bits.
 *   The call needs a caller-owned device workspace of lr_surface_distance_workspace_bytes(B, D, H, W) bytes (16 per
 *   voxel for the nearest-voxel intermediates and the envelope stacks, plus 24 per item and 128 columns for the
 *   partial statistics; the call never allocates).
 * Arguments: no null pointer; 1 <= B <= 65535; every axis >= 1; B*D*H*W < 2^31; 1 <= L <= 128; for the distances
 * 1 <= label <= 127, H and W <= 65535 (the nearest voxel's (h, w) is packed into 32 bits), the spacings finite and > 0
 * and the workspace large enough.  The checks run before any CUDA call; the workspace query returns 0 for sizes the
 * call rejects.  Nothing depends on lr_set_numerics. */
LR_API int lr_label_surface_counts(const float *pred, const float *target, int B, int D, int H, int W, int L,
                                   int64_t *counts, int64_t *invalid, lr_stream_t stream);
LR_API size_t lr_surface_distance_workspace_bytes(int B, int D, int H, int W);
LR_API int lr_surface_distances(const float *from, const float *to, int B, int D, int H, int W, int label, double s_d,
                                double s_h, double s_w, const int64_t *seg_offset, double *dist, double *stats,
                                void *workspace, size_t workspace_bytes, lr_stream_t stream);

/* ---- folding penalty (a training term; PARITY UNPINNED: the reference has no such term) ----------------------------
 *   fold(phi) = 1/(B*D*H*W) * sum_b sum_v max(0, -det_b(v))
 * det is, bit for bit, the determinant lr_jacobian_det computes for the same phi and boundary, over every voxel (no
 * margin).  A voxel whose det is not finite contributes nothing, to the value or to the gradient (as in the
 * statistics).  The subgradient is taken over the strict fold set det < 0 (the voxels stats[:,0] counts), so det == 0
 * contributes 0.  The value needs no kernel of its own: fold = sum_b stats[b][1] / (B*D*H*W) with the stats of
 * lr_jacobian_det(phi, ..., margin = 0, det = NULL, ...).
 * lr_jacobian_fold_backward: grad_phi (B,3,D,H,W) is OVERWRITTEN with grad_loss[0] * d fold / d phi (grad_loss: one
 * float in device memory).  With J[c][a] = s_a * (D_a phi_c), C[c][a] = d det / d J[c][a] and m = 1 where det is finite
 * and < 0 (0 elsewhere):  grad_phi_c = -(grad_loss / (B*D*H*W)) * sum_a s_a * D_a^T (m * C[c][a]), D_a^T the transpose
 * of the difference operator with its face rows.  Each element is written once, without atomics, so repeated calls
 * give the same bits.  Same argument rules as lr_jacobian_det (D,H,W >= 2, B*3*D*H*W < 2^31). */
LR_API int lr_jacobian_fold_backward(const float *phi, int B, int D, int H, int W, int boundary,
                                     const float *grad_loss, float *grad_phi, lr_stream_t stream);

/* ---- local (windowed) NCC similarity (a training term; PARITY UNPINNED: the reference has none) --------------------
 * VoxelMorph's NCC(win) form, per batch item b, with x = warped, y = target, both (B,1,D,H,W) float32 and an odd
 * window side w in [3, 15]:
 *   N(v) is the w x w x w cube centred on voxel v; voxels outside the volume count as 0 (zero padding) and
 *   n = w^3 is fixed (it is not the number of voxels inside).  Sx, Sy, Sxx, Syy, Sxy are the sums over N(v);
 *   cross = Sxy - Sx*Sy/n,  var_x = Sxx - Sx^2/n,  var_y = Syy - Sy^2/n,  d = var_x*var_y + eps,
 *   cc(v) = cross^2 / d  (cc = 0 where d <= 0: a window with zero variance and eps = 0),
 *   loss = 1 - mean over (B, D, H, W) of cc.
 * The gradient is taken wrt x only (the target is data).  With mu = S/n and, per window centre u with d > 0,
 *   alpha_u = 2*cross/d,  beta_u = 2*cross^2*var_y/d^2,  gamma_u = beta_u*mu_x - alpha_u*mu_y   (all 0 where d <= 0),
 *   d loss / d x_v = -(grad_loss / (B*D*H*W)) * (y_v * sum alpha - x_v * sum beta + sum gamma),
 * each sum over the centres u in N(v) inside the volume (with zero padding and a fixed n, v in N(u) <=> u in N(v), so
 * the adjoint is again a box sum).
 * Every window sum is accumulated in fp64 (the products of the fp32 inputs are exact there) as a plain sum of its terms
 * in a fixed order, so no result depends on the launch shape or the batch size.
 * lr_local_ncc_sum: sum (B) float64, zeroed by the call, = the fp64 sum of cc over each item;
 *   loss = 1 - (sum_b sum[b]) / (B*D*H*W).
 * lr_local_ncc_backward: grad_x (B,1,D,H,W) is OVERWRITTEN with grad_loss[0] * d loss / d x (grad_loss: one float in
 *   device memory); each element is written once, without atomics, so repeated calls give the same bits.  It needs a
 *   caller-owned device workspace of lr_local_ncc_workspace_bytes(B, D, H, W, win) bytes (alpha, beta, gamma as
 *   float32: 12 bytes per voxel; the call never allocates).
 * Arguments: win odd in [3, 15]; eps finite and >= 0; every axis >= 1 (an axis may be smaller than the window)
 * and <= 2^30; B*D*H*W < 2^31; no null pointer.  lr_local_ncc_workspace_bytes returns 0 for arguments the calls reject. */
LR_API int lr_local_ncc_sum(const float *x, const float *y, int B, int D, int H, int W, int win, double eps,
                            double *sum, lr_stream_t stream);
LR_API size_t lr_local_ncc_workspace_bytes(int B, int D, int H, int W, int win);
LR_API int lr_local_ncc_backward(const float *x, const float *y, int B, int D, int H, int W, int win, double eps,
                                 const float *grad_loss, float *grad_x, void *workspace, size_t workspace_bytes,
                                 lr_stream_t stream);

/* ---- soft Dice of the warped label map (a training term; PARITY UNPINNED: the reference has none) -------------------
 * VoxelMorph's semi-supervised Dice term (one-hot moving labels, trilinear warp, 1 - soft Dice) without the one-hot
 * channels.  phi (B,3,D,H,W) float32 in [-1,1], channel c addressing volume axis c (lr_warp_forward's convention);
 * src (moving) and tgt (target) (B,D,H,W) float32 label maps; 2 <= L <= 128.  A value that is not an integer in [0, L)
 * (negative, >= L, fractional, NaN) is "no label", as in lr_label_confusion.
 * Sampling is lr_warp_forward's with zeros padding and no using_scale, bit for bit: per axis i = (g+1)*((S-1)/2) in
 * fp32, clamp_index, floor; fractions w1 = i - floor(i), w0 = (floor(i)+1) - i; the weight of tap (tx,ty,tz) is the fp32
 * product (wx*wy)*wz.  A tap outside the volume carries no label.  Nothing depends on lr_set_numerics.
 * Per item b and label l, over all voxels v and their 8 taps t with weight w_t(v):
 *   P[b,l] = sum_v sum_t w_t(v) [src(t) = l]                 (soft size of the warped label)
 *   I[b,l] = sum_v sum_t w_t(v) [src(t) = l] [tgt(v) = l]    (soft overlap)
 *   T[b,l] = #{v : tgt(v) = l}
 *   S_b = {l in [1, L) : P + T > 0}  (background excluded);  dice_b = mean over S_b of 2 I / (P + T)  (1 if S_b is empty);
 *   loss = 1 - mean_b dice_b.
 * lr_label_dice_sums: sums (B,L,3) float64 = [I, P, T], zeroed by the call; I and P accumulate in fp64 from the fp32
 *   weights (the atomic order varies, so the last bits may differ between calls), T is exact.
 * lr_label_dice_backward: grad_phi (B,3,D,H,W) is OVERWRITTEN with grad_loss[0] * d loss / d phi (grad_loss: one float in
 *   device memory), from the sums of lr_label_dice_sums; the labels are data.  With a = d loss / d P, e = d loss / d I
 *   (both 0 for l not in S_b) and s_c = (S_c - 1)/2:
 *     grad_phi_c(v) = grad_loss * s_c * sum_t d w_t / d i_c * (a[b, src_t] + [src_t = tgt(v)] * e[b, src_t])
 *   over the in-bounds taps with a label.  a and a + e are formed in fp64 (grad_loss and 1/B folded in) and rounded
 *   once to fp32; the sum is evaluated as a tree over tap differences, so it is exactly 0 where the 8 taps carry one
 *   coefficient.  Each element is written once, without atomics: the same sums give the same bits.
 * Arguments: no null pointer; every axis >= 1 and < 2^21; B*3*D*H*W < 2^31; 2 <= L <= 128. */
LR_API int lr_label_dice_sums(const float *phi, const float *src, const float *tgt, int B, int D, int H, int W, int L,
                              double *sums, lr_stream_t stream);
LR_API int lr_label_dice_backward(const float *phi, const float *src, const float *tgt, int B, int D, int H, int W, int L,
                                  const double *sums, const float *grad_loss, float *grad_phi, lr_stream_t stream);

/* ---- normalized gradient field (NGF) similarity (PARITY UNPINNED) ---------------------------------------------------
 * The reference's layers/losses.py names an NGFLoss, but that file is not in its tree (and needs mermaid), so its eps,
 * spacing and face rule are unknown; this definition is from first principles (Haber & Modersitzki 2006).
 * x = warped, y = target, both (B,1,D,H,W) or (B,D,H,W) float32; `boundary` is LR_FD_LINEAR or LR_FD_NEUMANN_ZERO.
 *   g_a = s_a * D_a x,  h_a = s_a * D_a y  (a = 0, 1, 2 over the axes, s_a = 0.5/(2/(n_a-1))): exactly the fp32
 *   differences lr_jacobian_det forms for one channel (the face rule, then the product with the fp32 s_a).
 *   Per voxel, in fp64 from the fp32 g and h (sums left to right):
 *     a = g.h,  p = |g|^2 + eps^2,  q = |h|^2 + eps^2,  f = a^2 / (p*q)  in [0, 1];
 *   loss = 1 - (1/(B*D*H*W)) * sum_b sum_v f.
 * The gradient is taken wrt x only (the target is data):
 *   c_a = (2a/(p*q)) * (h_a - (a/p)*g_a)  formed in fp64 and rounded once to fp32,
 *   d loss / d x = -(1/(B*D*H*W)) * sum_a s_a * D_a^T c_a,  D_a^T the transposed difference with its face rows, as in
 *   lr_jacobian_fold_backward.
 * lr_ngf_sum: sum (B) float64, zeroed by the call, = the fp64 sum of f over each item (the atomic order varies, so the
 *   last bits may differ between calls);  loss = 1 - (sum_b sum[b]) / (B*D*H*W).
 * lr_ngf_backward: grad_x is OVERWRITTEN with grad_loss[0] * d loss / d x (grad_loss: one float in device memory); each
 *   element is written once, without atomics, so repeated calls give the same bits.
 * Nothing depends on lr_set_numerics.  Arguments: eps finite and > 0 (at least 1e-77, so that p*q >= eps^4 > 0;
 * eps = 0 would make 0/0 wherever both gradients vanish); D, H, W >= 2; B*D*H*W < 2^31; boundary 0 or 1; no null
 * pointer.  The checks run before any CUDA call.  ops.ngf_loss uses eps = 1 by default (DESIGN.md §1). */
LR_API int lr_ngf_sum(const float *x, const float *y, int B, int D, int H, int W, int boundary, double eps,
                      double *sum, lr_stream_t stream);
LR_API int lr_ngf_backward(const float *x, const float *y, int B, int D, int H, int W, int boundary, double eps,
                           const float *grad_loss, float *grad_x, lr_stream_t stream);

/* ---- mutual information (MI) similarity, Parzen joint histogram (PARITY UNPINNED) -------------------------------------
 * Mattes et al. (2003) MI, the default metric of elastix; the reference has no MI, so nothing pins it.
 * x = warped, y = target, each B items of N float32 (any shape, flattened per item); nb = num_bins in [4, 64];
 * lo < hi finite fp32 (the value range; ops.mi_loss uses (-1, 1), the range of the unit-normalised CT).  The range is
 * FIXED rather than each image's own min and max as Mattes uses: no min/max pass, no host synchronisation, and the
 * gradient has no term through the range.
 *   s = (float)((nb - 1) / ((double)hi - lo)).  Per voxel v, in fp32 with each op rounded:
 *     u = (fminf(fmaxf(v, lo), hi) - lo) * s        (NaN -> lo, -inf -> lo, +inf -> hi: no input indexes outside)
 *     target row   iota = floor(u_y + 0.5)           (in [0, nb-1]; zero-order Parzen window)
 *     moving taps  k0 = min(floor(u_x), nb - 2),  f = u_x - k0 (exact; in [0, 1] up to the rounding of u near nb-1),
 *                  kappa = k0 - 1 .. k0 + 2 with the cubic B-spline weights, in fp64 from the fp32 f:
 *       F = f, G = 1 - F, F2 = F*F, F3 = F2*F, r6 = 1.0/6.0 (the double nearest 1/6);
 *       w0 = ((G*G)*G)*r6,  w1 = ((4 - 6*F2) + 3*F3)*r6,  w2 = (((1 + 3*F) + 3*F2) - 3*F3)*r6,  w3 = F3*r6.
 *   hist (B, nb, nb+2) float64: hist[b][iota][kappa + 1] += w_m, so every tap lands inside (kappa in [-1, nb]).
 *   p = hist/N, p_y = sum over the columns of p, p_x = sum over the rows, MI_b = sum_{p>0} p (log p - log p_y - log p_x),
 *   loss = -mean_b MI_b (nats).
 * Gradient wrt x only (p_y does not depend on x, and sum_m dw_m/df = 0):
 *   d loss / d x_v = -(g/(B N)) * s * sum_m w_m'(f_v) * c(iota_v, k0_v - 1 + m),  c(iota, kappa) = log(p / p_x) (0 where
 *   p = 0), exactly 0 unless lo <= x_v <= hi (torch.clamp's mask; NaN gets 0).  The cubic B-spline is C^2, so the
 *   gradient does not jump at bin edges.
 * lr_mi_hist: hist (B*nb*(nb+2) float64) is zeroed and filled by the call; the fp64 atomic order varies, so the last
 *   bits may differ between calls.
 * lr_mi_backward: grad_x (B*N) is OVERWRITTEN with grad_loss[0] * d loss / d x for the given hist (grad_loss: one float
 *   in device memory).  Per item, the column sums P_x[j] = sum_{r = 0..nb-1} hist[r][j] (fp64, rows in order) and the
 *   table T = (float)(log(hist / P_x) * k), k = -((double)g * s) / ((double)B * N), are formed in fp64 and T is rounded
 *   once to fp32 (T = 0 where hist = 0).  Per voxel, in fp32 with each op rounded, the derivative weights are
 *     w0' = -((1-f)^2 * 0.5),  w1' = -((f * (4 - 3f)) * 0.5),  w2' = ((1-f) * (1 + 3f)) * 0.5,  w3' = (f*f) * 0.5
 *   (the polynomials -(1-f)^2/2, f(3f-4)/2, (1+2f-3f^2)/2, f^2/2 in product form, free of cancellation), and
 *   grad = fma(T3, w3', fma(T2, w2', fma(T1, w1', T0 * w0'))) with T_m = T[iota][k0 + m].  Each element is written
 *   once, without atomics: the same hist gives the same bits.
 * Arguments: no null pointer; 1 <= B <= 65535, N >= 1; 4 <= nb <= 64; lo, hi finite with lo < hi and s finite and
 * > 0.  The checks run before any CUDA call. */
LR_API int lr_mi_hist(const float *x, const float *y, int B, int64_t N, int num_bins, float lo, float hi, double *hist,
                      lr_stream_t stream);
LR_API int lr_mi_backward(const float *x, const float *y, int B, int64_t N, int num_bins, float lo, float hi,
                          const double *hist, const float *grad_loss, float *grad_x, lr_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* LIFTREG_B200_H */
