"""Functional PyTorch surface over the C-ABI: tensors in, tensors out, autograd wired.

PyTorch is plumbing here (device memory, streams, autograd graph); all arithmetic happens in
libliftreg_b200.so.  CUDA float32 tensors only -- there is no CPU fallback.
"""
import ctypes
import math

import numpy as np
import torch

from . import _native

PAD_ZEROS, PAD_BORDER = 0, 1
MODE_LINEAR, MODE_NEAREST = 0, 1
YNORM_WM1, YNORM_W = 0, 1


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _call(name, device, *args):
    """Call the C-ABI entry `name` on `device` with args and that device's current stream; RuntimeError if it fails."""
    with torch.cuda.device(device):
        _native.check(getattr(_native.lib(), name)(*args, _stream()), name)


def _grad_scalar(grad_loss, device):
    """The incoming gradient of a scalar loss as the one-element float32 tensor on `device` that the adjoints read."""
    return grad_loss.to(device=device, dtype=torch.float32).reshape(1).contiguous()


def _need_cuda_f32(t, name):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, got %s" % (name, type(t).__name__))
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: liftreg_b200 has no CPU path (got device %s)" % (name, t.device))
    if t.dtype != torch.float32:
        raise TypeError("%s must be float32 (got %s)" % (name, t.dtype))
    return t.contiguous()


def _poses64(poses):
    """(P,3) or (n_sets,P,3) -> contiguous float64 numpy (n_sets,P,3)."""
    if isinstance(poses, torch.Tensor):
        poses = poses.detach().cpu().numpy()
    a = np.ascontiguousarray(poses, dtype=np.float64)
    if a.ndim == 2:
        a = a[None]
    if a.ndim != 3 or a.shape[2] != 3:
        raise ValueError("poses must have shape (P,3) or (B,P,3), got %s" % (a.shape,))
    return a


def _poses32(poses):
    if isinstance(poses, torch.Tensor):
        poses = poses.detach().cpu().numpy()
    a = np.ascontiguousarray(poses, dtype=np.float32)
    if a.ndim == 3:
        a = a[0]            # geometry frozen from batch item 0 (reference model :85-87)
    if a.ndim != 2 or a.shape[1] != 3:
        raise ValueError("poses must have shape (P,3) or (B,P,3), got %s" % (a.shape,))
    return np.ascontiguousarray(a)


def _spacing3(spacing):
    if isinstance(spacing, torch.Tensor):
        spacing = spacing.detach().cpu().numpy()
    a = np.ascontiguousarray(np.asarray(spacing, dtype=np.float32).reshape(-1))
    if a.size != 3:
        raise ValueError("spacing must have 3 entries")
    return a


def _fp(a):
    return a.ctypes.data_as(_native.c_float_p)


def _dp(a):
    return a.ctypes.data_as(_native.c_double_p)


# --------------------------------------------------------------------------- DRR
class _DRR(torch.autograd.Function):
    @staticmethod
    def forward(ctx, vol, poses, rd, rh, spacing, y_norm_mode, out_scale, out):
        vol = _need_cuda_f32(vol, "vol")
        B, d, w, h = vol.shape
        n_sets, P, _ = poses.shape
        if out is None:
            proj = torch.empty((B, P, rd, rh), device=vol.device, dtype=torch.float32)
        else:
            if not (out.is_cuda and out.dtype == torch.float32 and out.is_contiguous() and out.numel() == B * P * rd * rh):
                raise ValueError("out must be a contiguous CUDA float32 tensor of %d elements" % (B * P * rd * rh))
            proj = out
            ctx.mark_dirty(out)
        _call("lr_drr_forward", vol.device, _ptr(vol), B, d, w, h, _dp(poses), n_sets, P, rd, rh, _fp(spacing), y_norm_mode,
              out_scale, _ptr(proj))
        ctx.geom = (poses, rd, rh, spacing, y_norm_mode, out_scale, (B, d, w, h))
        return proj

    @staticmethod
    def backward(ctx, grad_proj):
        poses, rd, rh, spacing, y_norm_mode, out_scale, (B, d, w, h) = ctx.geom
        grad_proj = _need_cuda_f32(grad_proj, "grad_proj")
        n_sets, P, _ = poses.shape
        grad_vol = torch.zeros((B, d, w, h), device=grad_proj.device, dtype=torch.float32)
        _call("lr_drr_backward", grad_proj.device, _ptr(grad_proj), B, d, w, h, _dp(poses), n_sets, P, rd, rh, _fp(spacing),
              y_norm_mode, out_scale, _ptr(grad_vol))
        return grad_vol, None, None, None, None, None, None, None


def drr_project(vol, poses, resolution, spacing, y_norm_mode=YNORM_WM1, out_scale=0.1, out=None):
    """Cone-beam DRR of vol (B,d,w,h) -> (B,P,rd,rh); differentiable wrt vol.

    Replaces reference sdct:59-86 (y_norm_mode=0, out_scale=0.1) and layers.py:182-187 (y_norm_mode=1, out_scale=1).
    poses: (P,3) shared by the batch, or (B,P,3); float64, voxel units.
    out: optional pre-allocated contiguous (B,P,rd,rh) CUDA tensor (or any contiguous view with that many elements,
    e.g. a rank's slot of an all-gather buffer) that the kernel writes into; it is returned.
    """
    poses = _poses64(poses)
    if vol.dim() != 4:
        raise ValueError("vol must be (B,d,w,h), got %s" % (tuple(vol.shape),))
    if poses.shape[0] not in (1, vol.shape[0]):
        raise ValueError("poses batch (%d) must be 1 or B (%d)" % (poses.shape[0], vol.shape[0]))
    rd, rh = int(resolution[0]), int(resolution[1])
    return _DRR.apply(vol, poses, rd, rh, _spacing3(spacing), int(y_norm_mode), float(out_scale), out)


def drr_project_peers(vol, poses, resolution, spacing, out_ptrs, view_stride, y_norm_mode=YNORM_WM1, out_scale=0.1):
    """Multi-GPU sweep form of drr_project (no autograd): the kernel stores the images into every buffer of `out_ptrs`
    (raw device addresses: this rank's gather buffer and the peers', see sharding.PeerGather), view k of the call at
    k * view_stride images from each address.  Nothing is returned; the caller orders the ranks with a barrier."""
    poses = _poses64(poses)
    vol = _need_cuda_f32(vol, "vol")
    if vol.dim() != 4 or poses.shape[0] not in (1, vol.shape[0]):
        raise ValueError("vol must be (B,d,w,h) and poses (P,3) or (B,P,3)")
    B, d, w, h = vol.shape
    n_sets, P, _ = poses.shape
    ptrs = (ctypes.c_void_p * len(out_ptrs))(*[int(a) for a in out_ptrs])
    _call("lr_drr_forward_peers", vol.device, _ptr(vol), B, d, w, h, _dp(poses), n_sets, P, int(resolution[0]),
          int(resolution[1]), _fp(_spacing3(spacing)), int(y_norm_mode), float(out_scale), ptrs, len(out_ptrs),
          int(view_stride))


def project_grid(poses, resolution, obj_shape, spacing, device, y_norm_mode=YNORM_WM1, flip=False, want_grid=True):
    """Materialised sample grid (P,rd,rh,w,3) and dx (P,rd,rh) -- reference sdct:15-57, for API parity only."""
    poses = _poses64(poses)[0]
    P = poses.shape[0]
    rd, rh = int(resolution[0]), int(resolution[1])
    d, w, h = (int(s) for s in obj_shape)
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("project_grid needs a CUDA device: liftreg_b200 has no CPU path")
    grid = torch.empty((P, rd, rh, w, 3), device=dev, dtype=torch.float32) if want_grid else None
    dx = torch.empty((P, rd, rh), device=dev, dtype=torch.float32)
    _call("lr_project_grid", dev, _dp(poses), P, rd, rh, d, w, h, _fp(_spacing3(spacing)), int(y_norm_mode), int(bool(flip)),
          _ptr(grid), _ptr(dx))
    return grid, dx


# --------------------------------------------------------------------------- backprojection
class _Backproject(torch.autograd.Function):
    @staticmethod
    def forward(ctx, proj, poses, d_total, w, h, out, channel_offset, i_begin, i_count):
        proj = _need_cuda_f32(proj, "target_proj")
        B, P, pw, ph = proj.shape
        d = i_count
        nv = d * w * h
        if out is None:
            out = torch.empty((B, P, d, w, h), device=proj.device, dtype=torch.float32)
            view, bs, cs = out, P * nv, nv
        else:
            if not (out.is_cuda and out.dtype == torch.float32 and out.is_contiguous()):
                raise ValueError("out must be a contiguous CUDA float32 tensor")
            if out.dim() != 5 or out.shape[0] != B or tuple(out.shape[2:]) != (d, w, h) \
                    or out.shape[1] < channel_offset + P:
                raise ValueError("out must be (B,>=%d,%d,%d,%d), got %s" % (channel_offset + P, d, w, h, tuple(out.shape)))
            view, bs, cs = out[:, channel_offset:channel_offset + P], out.shape[1] * nv, nv
            ctx.mark_dirty(out)
        _call("lr_backproject_forward_slab", proj.device, _ptr(proj), _fp(poses), B, P, pw, ph, d_total, w, h, i_begin, i_count,
              ctypes.c_void_p(view.data_ptr()), bs, cs)
        ctx.geom = (poses, B, P, pw, ph, d, w, h, channel_offset, out.shape[1], d_total, i_begin)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        poses, B, P, pw, ph, d, w, h, off, nchan, d_total, i_begin = ctx.geom
        if d != d_total:
            raise NotImplementedError("gradient wrt the projections is not implemented for slab-sharded backprojection "
                                      "(the reference detaches this output, LiftRegDeformSubspaceBackproj.py:93)")
        grad_out = _need_cuda_f32(grad_out, "grad_out")
        nv = d * w * h
        gview = grad_out[:, off:off + P]
        grad_proj = torch.zeros((B, P, pw, ph), device=grad_out.device, dtype=torch.float32)
        _call("lr_backproject_backward", grad_out.device, ctypes.c_void_p(gview.data_ptr()), nchan * nv, nv, _fp(poses), B, P,
              pw, ph, d, w, h, _ptr(grad_proj))
        # `out` was overwritten in channels [off, off+P): the gradient wrt its previous content passes through elsewhere
        grad_buf = None
        if ctx.needs_input_grad[5]:
            grad_buf = grad_out.clone()
            grad_buf[:, off:off + P] = 0
        return grad_proj, None, None, None, None, grad_buf, None, None, None


def backproject(target_proj, poses, img_shape, out=None, channel_offset=0, slab=None):
    """Lift projections (B,P,pw,ph) into a volume (B,P,d,w,h); differentiable wrt target_proj.

    Replaces reference sdct:227-250 + LiftRegDeformSubspaceBackproj.py:85-93 in one kernel (no 131 MB grid).
    poses: (P,3) or (B,P,3) float32 (item 0 is used, as the reference freezes geometry from the first batch).
    out/channel_offset: optionally write into channels [offset, offset+P) of a pre-allocated (B,Ctot,d,w,h)
    buffer, which removes the torch.cat of model :95-98; the whole buffer is returned.
    slab=(i_begin, i_count): compute only planes [i_begin, i_begin+i_count) of axis 0 (multi-GPU z-slab sharding);
    the result (and `out`) then has i_count planes.
    """
    if target_proj.dim() != 4:
        raise ValueError("target_proj must be (B,P,pw,ph), got %s" % (tuple(target_proj.shape),))
    poses = _poses32(poses)
    if poses.shape[0] != target_proj.shape[1]:
        raise ValueError("poses has %d views but target_proj has %d" % (poses.shape[0], target_proj.shape[1]))
    d, w, h = (int(s) for s in img_shape)
    i_begin, i_count = (0, d) if slab is None else (int(slab[0]), int(slab[1]))
    if not (0 <= i_begin and i_count > 0 and i_begin + i_count <= d):
        raise ValueError("slab %r is not inside [0, %d)" % (slab, d))
    return _Backproject.apply(target_proj, poses, d, w, h, out, int(channel_offset), i_begin, i_count)


def backproj_grid(poses, img_shape, proj_shape, device):
    """Materialised voxel->detector grid (P,2,d,w,h) -- reference sdct:227-250, for API parity only."""
    poses = _poses32(poses)
    d, w, h = (int(s) for s in img_shape)
    pw, ph = (int(s) for s in proj_shape)
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("backproj_grid needs a CUDA device: liftreg_b200 has no CPU path")
    grid = torch.empty((poses.shape[0], 2, d, w, h), device=dev, dtype=torch.float32)
    _call("lr_backproj_grid", dev, _fp(poses), poses.shape[0], d, w, h, pw, ph, _ptr(grid))
    return grid


# --------------------------------------------------------------------------- warp
class _Warp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, img, phi, padding, mode, using_scale, disp_plus_identity, z_begin):
        img = _need_cuda_f32(img, "input1")
        phi = _need_cuda_f32(phi, "input2")
        B, C, D, H, W = img.shape
        z_count = phi.shape[2]
        out = torch.empty((B, C, z_count, H, W), device=img.device, dtype=torch.float32)
        _call("lr_warp_forward_slab", img.device, _ptr(img), _ptr(phi), B, C, D, H, W, z_begin, z_count, padding, mode,
              int(using_scale), int(disp_plus_identity), _ptr(out))
        ctx.save_for_backward(img, phi)
        ctx.cfg = (padding, mode, using_scale, disp_plus_identity, z_begin)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        img, phi = ctx.saved_tensors
        padding, mode, using_scale, ident, z_begin = ctx.cfg
        grad_out = _need_cuda_f32(grad_out, "grad_out")
        B, C, D, H, W = img.shape
        z_count = phi.shape[2]
        need_img, need_phi = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if need_img and mode == MODE_NEAREST:
            raise NotImplementedError("gradient wrt the image is not implemented for nearest-mode warps")
        gimg = torch.zeros_like(img) if need_img else None
        gphi = torch.empty_like(phi) if need_phi else None
        _call("lr_warp_backward_slab", img.device, _ptr(grad_out), _ptr(img), _ptr(phi), B, C, D, H, W, z_begin, z_count,
              padding, mode, int(using_scale), int(ident), _ptr(gimg), _ptr(gphi))
        return gimg, gphi, None, None, None, None, None


def warp(img, phi, zero_boundary=False, using_scale=True, mode="bilinear", disp_plus_identity=False, z_begin=None):
    """Spatial transformer: img (B,C,D,H,W) sampled at phi (B,3,D,H,W) in [-1,1]; differentiable wrt both.

    Replaces reference net_utils.py:26-56.  disp_plus_identity=True treats phi as a displacement and adds the
    identity map in-kernel (fuses LiftRegDeformSubspaceBackproj.py:68).
    z_begin: phi is a z-slab (B,3,Dz,H,W) holding output planes [z_begin, z_begin+Dz) of the full (D,H,W) image
    (multi-GPU z-slab sharding); the result is the matching (B,C,Dz,H,W) slab.
    """
    if mode not in ("bilinear", "nearest"):
        raise ValueError("mode must be 'bilinear' or 'nearest', got %r" % (mode,))
    if img.dim() != 5 or phi.dim() != 5 or phi.shape[1] != 3 or phi.shape[0] != img.shape[0] \
            or tuple(phi.shape[3:]) != tuple(img.shape[3:]):
        raise ValueError("expected input1 (B,C,D,H,W) and input2 (B,3,D,H,W); got %s and %s"
                         % (tuple(img.shape), tuple(phi.shape)))
    if z_begin is None:
        if phi.shape[2] != img.shape[2]:
            raise ValueError("input2 has %d planes but input1 has %d (pass z_begin for a slab)" % (phi.shape[2], img.shape[2]))
        z_begin = 0
    if not (0 <= z_begin and z_begin + phi.shape[2] <= img.shape[2]):
        raise ValueError("slab [%d, %d) is not inside [0, %d)" % (z_begin, z_begin + phi.shape[2], img.shape[2]))
    return _Warp.apply(img, phi, PAD_ZEROS if zero_boundary else PAD_BORDER,
                       MODE_LINEAR if mode == "bilinear" else MODE_NEAREST, bool(using_scale), bool(disp_plus_identity),
                       int(z_begin))


def identity_map(sz, device):
    """Normalised identity map (3,*sz) on `device` -- reference net_utils.py:59-87."""
    D, H, W = (int(s) for s in sz)
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("identity_map needs a CUDA device: liftreg_b200 has no CPU path")
    out = torch.empty((3, D, H, W), device=dev, dtype=torch.float32)
    _call("lr_identity_map", dev, D, H, W, _ptr(out))
    return out


def atten_coef_(img):
    """In-place HU -> attenuation on a CUDA tensor -- reference sdct:11-13."""
    t = _need_cuda_f32(img, "img")
    if t.data_ptr() != img.data_ptr():
        raise ValueError("atten_coef_ needs a contiguous tensor")
    _call("lr_atten_coef", t.device, _ptr(t), t.numel(), _ptr(t))
    return img


# --------------------------------------------------------------------------- PCA-subspace decode (row f2)
class _PcaDecode(torch.autograd.Function):
    @staticmethod
    def forward(ctx, coefs, basis, mean, D, H, W, add_identity):
        coefs = _need_cuda_f32(coefs, "coefs")
        basis = _need_cuda_f32(basis, "pca_vectors")
        mean_c = _need_cuda_f32(mean, "pca_mean") if mean is not None else None
        B, K = coefs.shape
        N = basis.shape[0]
        out = torch.empty((B, N), device=coefs.device, dtype=torch.float32)
        _call("lr_pca_decode", coefs.device, _ptr(coefs), _ptr(basis), _ptr(mean_c), B, K, N, int(add_identity), D, H, W,
              _ptr(out))
        ctx.save_for_backward(basis)
        return out

    @staticmethod
    def backward(ctx, grad_out):
        (basis,) = ctx.saved_tensors
        # d/dcoefs = grad_out (B,N) @ basis (N,K): the second pass over the basis; basis and mean are frozen buffers
        grad_out = _need_cuda_f32(grad_out, "grad_out")
        B, N = grad_out.shape
        K = basis.shape[1]
        gcoefs = torch.zeros((B, K), device=grad_out.device, dtype=torch.float32)
        _call("lr_pca_decode_backward", grad_out.device, _ptr(grad_out), _ptr(basis), B, K, N, _ptr(gcoefs))
        return gcoefs, None, None, None, None, None, None


def pca_decode(coefs, pca_vectors, pca_mean=None, img_shape=None, add_identity=False):
    """disp = F.linear(coefs, pca_vectors, pca_mean) as one streaming kernel (reference model :102); with
    add_identity (needs img_shape = (D,H,W), N = 3*D*H*W) the identity map of model :68 is added too, so the result
    reshaped to (B,3,D,H,W) is the map the warp consumes.  coefs (B,K); pca_vectors (N,K) as the model stores it
    (:42); pca_mean (N).  Differentiable wrt coefs."""
    if coefs.dim() != 2 or pca_vectors.dim() != 2 or coefs.shape[1] != pca_vectors.shape[1]:
        raise ValueError("expected coefs (B,K) and pca_vectors (N,K); got %s and %s" % (tuple(coefs.shape), tuple(pca_vectors.shape)))
    if pca_mean is not None and tuple(pca_mean.shape) != (pca_vectors.shape[0],):
        raise ValueError("pca_mean must be (N,)")
    if not pca_vectors.is_contiguous():
        # a silent .contiguous() here would transpose-copy the whole basis (2.75 GB at 160^3) on EVERY call
        raise ValueError("pca_vectors must be a dense row-major (N,K) tensor; the reference builds an (N,K) view of a "
                         "(K,N) array (model :42) -- call .contiguous() on it once (dropin.install() does)")
    D = H = W = 0
    if add_identity:
        if img_shape is None or 3 * int(np.prod(img_shape)) != pca_vectors.shape[0]:
            raise ValueError("add_identity needs img_shape with 3*D*H*W == N")
        D, H, W = (int(s) for s in img_shape)
    out = _PcaDecode.apply(coefs, pca_vectors, pca_mean, D, H, W, bool(add_identity))
    if img_shape is not None:
        return out.reshape(coefs.shape[0], 3, *[int(s) for s in img_shape])
    return out


# --------------------------------------------------------------------------- NCC similarity (row f4)
class _Ncc(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y):
        x = _need_cuda_f32(x, "input")
        y = _need_cuda_f32(y, "target")
        B = x.shape[0]
        N = x.numel() // B
        sums = torch.empty((B, 7), device=x.device, dtype=torch.float64)
        _call("lr_ncc_sums", x.device, _ptr(x), _ptr(y), B, N, _ptr(sums))
        ncc = sums[:, 2] / torch.sqrt(sums[:, 3] * sums[:, 4])           # the 1/N of the three means cancels
        ctx.save_for_backward(x, y, sums)
        return (1.0 - ncc.mean()).to(torch.float32)

    @staticmethod
    def backward(ctx, grad_loss):
        x, y, sums = ctx.saved_tensors
        B = x.shape[0]
        N = x.numel() // B
        g = _grad_scalar(grad_loss, x.device)
        gx = torch.empty_like(x)
        _call("lr_ncc_backward", x.device, _ptr(x), _ptr(y), B, N, _ptr(sums), _ptr(g), _ptr(gx))
        return gx, None


def ncc_loss(input, target):
    """1 - mean over the batch of the normalised cross correlation -- reference layers/losses.py:14-29 (NCCLoss).
    Differentiable wrt `input` (the warped image); `target` is data."""
    if input.shape != target.shape:
        raise ValueError("input %s and target %s must have the same shape" % (tuple(input.shape), tuple(target.shape)))
    return _Ncc.apply(input, target)


# --------------------------------------------------------------------------- local NCC similarity (training term)
def _volume_shape(t, name, want=None):
    """(B, D, H, W) of a (B,1,D,H,W) or (B,D,H,W) tensor t, which must equal `want` when given; ValueError otherwise.
    Checks the shape only, so that callers raise every ValueError before their device and dtype checks."""
    if isinstance(t, torch.Tensor) and (t.dim() == 4 or (t.dim() == 5 and t.shape[1] == 1)):
        got = (t.shape[0],) + tuple(t.shape[-3:])
        if want is None or got == want:
            return got
    else:
        got = tuple(t.shape) if isinstance(t, torch.Tensor) else type(t).__name__
    raise ValueError("%s must be (B,1,D,H,W) or (B,D,H,W)%s, got %s"
                     % (name, "" if want is None else " with (B,D,H,W) = %s" % (want,), got))


class _LocalNcc(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, window, eps):
        x = _need_cuda_f32(x, "input")
        y = _need_cuda_f32(y, "target")
        B, D, H, W = x.shape[0], *x.shape[-3:]
        sums = torch.empty(B, device=x.device, dtype=torch.float64)
        _call("lr_local_ncc_sum", x.device, _ptr(x), _ptr(y), B, D, H, W, window, eps, _ptr(sums))
        ctx.save_for_backward(x, y)
        ctx.cfg = (window, eps)
        return (1.0 - sums.sum() / float(B * D * H * W)).to(torch.float32)

    @staticmethod
    def backward(ctx, grad_loss):
        x, y = ctx.saved_tensors
        window, eps = ctx.cfg
        B, D, H, W = x.shape[0], *x.shape[-3:]
        g = _grad_scalar(grad_loss, x.device)
        gx = torch.empty_like(x)
        ws = torch.empty(_native.lib().lr_local_ncc_workspace_bytes(B, D, H, W, window), device=x.device, dtype=torch.uint8)
        _call("lr_local_ncc_backward", x.device, _ptr(x), _ptr(y), B, D, H, W, window, eps, _ptr(g), _ptr(gx), _ptr(ws),
              ws.numel())
        return gx, None, None, None


def local_ncc_loss(input, target, window=9, eps=1e-5):
    """1 - mean over (B, D, H, W) of the local (windowed) squared correlation cc of VoxelMorph's NCC(win): window sums
    over the window x window x window cube around each voxel, zero padding, cc = cross^2 / (var_x var_y + eps)
    (definition: include/liftreg_b200.h, lr_local_ncc_sum).  input and target are (B,1,D,H,W) or (B,D,H,W) CUDA
    float32; window is odd, in [3, 15].  Differentiable wrt `input` (the warped image); `target` is data.  The reference
    has no such term, so parity is unpinned."""
    if input.shape != target.shape:
        raise ValueError("input %s and target %s must have the same shape" % (tuple(input.shape), tuple(target.shape)))
    _volume_shape(input, "input")
    return _LocalNcc.apply(input, target, int(window), float(eps))


# --------------------------------------------------------------------------- displacement regulariser (row f4)
FD_BOUNDARY = {"linear": 0, "neumann_zero": 1}       # LR_FD_LINEAR / LR_FD_NEUMANN_ZERO (mermaid FD modes)


def _fd_boundary(boundary):
    """The C-ABI code of the face rule named `boundary`; ValueError for a name not in FD_BOUNDARY."""
    if boundary not in FD_BOUNDARY:
        raise ValueError("boundary must be one of %s, got %r" % (sorted(FD_BOUNDARY), boundary))
    return FD_BOUNDARY[boundary]


class _DiffusionReg(torch.autograd.Function):
    @staticmethod
    def forward(ctx, disp, boundary):
        disp = _need_cuda_f32(disp, "disp")
        B, _, D, H, W = disp.shape
        total = torch.empty(1, device=disp.device, dtype=torch.float64)
        _call("lr_diffusion_reg_sum", disp.device, _ptr(disp), B, D, H, W, boundary, _ptr(total))
        ctx.save_for_backward(disp)
        ctx.boundary = boundary
        return (total[0] / float(B * D * H * W)).to(torch.float32)

    @staticmethod
    def backward(ctx, grad_loss):
        disp, = ctx.saved_tensors
        B, _, D, H, W = disp.shape
        g = _grad_scalar(grad_loss, disp.device)
        gd = torch.empty_like(disp)
        _call("lr_diffusion_reg_backward", disp.device, _ptr(disp), B, D, H, W, ctx.boundary, _ptr(g), _ptr(gd))
        return gd, None


def diffusion_reg(disp, boundary="linear"):
    """mean over (B, D, H, W) of the nine squared central differences of a displacement field (B,3,D,H,W) -- reference
    losses/SubspaceLoss.py:51-67 (compute_reg_loss), one fused pass instead of ~27 kernels; differentiable.

    `boundary` names the rule of mermaid's finite differences on the volume faces: "linear" (FD_torch's default mode:
    the missing neighbour is extrapolated linearly) or "neumann_zero" (zero difference on the faces)."""
    if disp.dim() != 5 or disp.shape[1] != 3:
        raise ValueError("disp must be (B,3,D,H,W), got %s" % (tuple(disp.shape),))
    return _DiffusionReg.apply(disp, _fd_boundary(boundary))


# --------------------------------------------------------------------------- NGF similarity (training term)
class _Ngf(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, eps, boundary):
        x = _need_cuda_f32(x, "input")
        y = _need_cuda_f32(y, "target")
        B, D, H, W = x.shape[0], *x.shape[-3:]
        sums = torch.empty(B, device=x.device, dtype=torch.float64)
        _call("lr_ngf_sum", x.device, _ptr(x), _ptr(y), B, D, H, W, boundary, eps, _ptr(sums))
        ctx.save_for_backward(x, y)
        ctx.cfg = (eps, boundary)
        return (1.0 - sums.sum() / float(B * D * H * W)).to(torch.float32)

    @staticmethod
    def backward(ctx, grad_loss):
        x, y = ctx.saved_tensors
        eps, boundary = ctx.cfg
        B, D, H, W = x.shape[0], *x.shape[-3:]
        g = _grad_scalar(grad_loss, x.device)
        gx = torch.empty_like(x)
        _call("lr_ngf_backward", x.device, _ptr(x), _ptr(y), B, D, H, W, boundary, eps, _ptr(g), _ptr(gx))
        return gx, None, None, None


def ngf_loss(input, target, eps=1.0, boundary="linear"):
    """Normalized gradient field similarity: 1 - mean over (B, D, H, W) of (g.h)^2 / ((|g|^2 + eps^2)(|h|^2 + eps^2)),
    with g and h the regulariser's central differences of input and target (face rule `boundary`, as diffusion_reg);
    it scores edge alignment only, so an intensity change between the images does not affect it (definition:
    include/liftreg_b200.h, lr_ngf_sum).  input and target are (B,1,D,H,W) or (B,D,H,W) CUDA float32 with every
    spatial axis >= 2; eps (finite, > 0) is in the units of g: intensity per unit of the [-1, 1] grid coordinate.
    Differentiable wrt `input` (the warped image); `target` is data.  A float32 scalar computed without a host
    synchronisation.  The reference's NGFLoss is not in its tree, so parity is unpinned."""
    _volume_shape(input, "input")
    _volume_shape(target, "target")
    if input.shape != target.shape:
        raise ValueError("input %s and target %s must have the same shape" % (tuple(input.shape), tuple(target.shape)))
    if min(input.shape[-3:]) < 2:
        raise ValueError("every spatial axis needs >= 2 entries, got %s" % (tuple(input.shape[-3:]),))
    eps = float(eps)
    if not (math.isfinite(eps) and eps >= 1e-77):
        raise ValueError("eps must be finite and > 0 (>= 1e-77), got %r" % eps)
    return _Ngf.apply(input, target, eps, _fd_boundary(boundary))


# --------------------------------------------------------------------------- mutual information similarity (training term)
def _mi_loss_from_hist(hist, N):
    """-mean_b MI_b from hist (B, nb, nb+2) float64 of N voxels per item: float64 on the histogram's device, no host
    synchronisation"""
    p = hist / float(N)
    pos = p > 0
    one = torch.ones((), dtype=p.dtype, device=p.device)
    py = p.sum(2, keepdim=True).expand_as(p)
    px = p.sum(1, keepdim=True).expand_as(p)
    log = lambda t: torch.log(torch.where(pos, t, one))
    mi = torch.where(pos, p * (log(p) - log(py) - log(px)), 0.0).sum((1, 2))
    return -mi.mean()


class _Mi(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, y, nb, lo, hi):
        x = _need_cuda_f32(x, "input")
        y = _need_cuda_f32(y, "target")
        B, N = x.shape[0], x.numel() // x.shape[0]
        hist = torch.empty((B, nb, nb + 2), device=x.device, dtype=torch.float64)
        _call("lr_mi_hist", x.device, _ptr(x), _ptr(y), B, N, nb, lo, hi, _ptr(hist))
        ctx.save_for_backward(x, y, hist)
        ctx.cfg = (nb, lo, hi)
        return _mi_loss_from_hist(hist, N).to(torch.float32)

    @staticmethod
    def backward(ctx, grad_loss):
        x, y, hist = ctx.saved_tensors
        nb, lo, hi = ctx.cfg
        B, N = x.shape[0], x.numel() // x.shape[0]
        g = _grad_scalar(grad_loss, x.device)
        gx = torch.empty_like(x)
        _call("lr_mi_backward", x.device, _ptr(x), _ptr(y), B, N, nb, lo, hi, _ptr(hist), _ptr(g), _ptr(gx))
        return gx, None, None, None, None


def mi_loss(input, target, num_bins=32, value_range=(-1.0, 1.0)):
    """-mean_b of the mutual information (nats) of the Parzen joint histogram of input_b and target_b (Mattes et al.
    2003): a cubic B-spline window on the input, a zero-order window on the target, num_bins bins over the FIXED
    value_range (lo, hi), values outside clamped to it (definition: include/liftreg_b200.h, lr_mi_hist).  input and
    target are (B, ...) CUDA float32 of one shape, each item flattened.  Differentiable wrt `input` (the warped image);
    `target` is data.  A float32 scalar computed without a host synchronisation.  The reference has no MI, so parity
    is unpinned."""
    for t, name in ((input, "input"), (target, "target")):
        if not isinstance(t, torch.Tensor) or t.dim() < 1 or t.numel() == 0:
            raise ValueError("%s must be a non-empty (B, ...) tensor, got %s"
                             % (name, tuple(t.shape) if isinstance(t, torch.Tensor) else type(t).__name__))
    if input.shape != target.shape:
        raise ValueError("input %s and target %s must have the same shape" % (tuple(input.shape), tuple(target.shape)))
    if input.shape[0] > 65535:
        raise ValueError("at most 65535 items per call, got %d" % input.shape[0])
    if isinstance(num_bins, bool) or not isinstance(num_bins, (int, np.integer)) or not 4 <= num_bins <= 64:
        raise ValueError("num_bins must be an integer in [4, 64], got %r" % (num_bins,))
    try:
        lo, hi = (float(v) for v in value_range)
    except (TypeError, ValueError):
        raise ValueError("value_range must be a pair (lo, hi) of numbers, got %r" % (value_range,)) from None
    with np.errstate(over="ignore"):
        lo32, hi32 = np.float32(lo), np.float32(hi)
        s = np.float32((int(num_bins) - 1) / (float(hi32) - float(lo32))) if hi32 > lo32 else np.float32(0)
    if not (np.isfinite(lo32) and np.isfinite(hi32) and lo32 < hi32 and np.isfinite(s) and s > 0):
        raise ValueError("value_range (%r, %r) must be finite in float32 with lo < hi and (num_bins - 1) / (hi - lo) a "
                         "finite positive float" % (lo, hi))
    return _Mi.apply(input, target, int(num_bins), float(lo32), float(hi32))



# --------------------------------------------------------------------------- validation metrics (not differentiable)
JACOBIAN_STATS = ("folding_count", "folding_abs_sum", "det_min", "det_max", "det_sum", "det_sum_sq", "nonfinite_count")


def _need_map(phi):
    """ValueError unless phi is a (B,3,D,H,W) tensor (shape only: the device and dtype are checked after it)."""
    if not isinstance(phi, torch.Tensor) or phi.dim() != 5 or phi.shape[1] != 3:
        raise ValueError("phi must be a (B,3,D,H,W) tensor, got %s" % (tuple(phi.shape) if isinstance(phi, torch.Tensor) else type(phi).__name__,))


def jacobian_det(phi, boundary="linear", margin=0, want_map=False):
    """Jacobian determinant of a map phi (B,3,D,H,W) in [-1,1] (channel c addresses volume axis c) with the
    regulariser's central differences and face rule `boundary`, scaled so that the identity map has det 1.

    Returns (stats, det): stats is a (B,7) float64 CUDA tensor ordered as JACOBIAN_STATS, over the voxels at least
    `margin` from every face (sums and min / max over finite values only); det is the (B,D,H,W) float32 map when
    want_map, else None.  Parity with the reference's utils.py:20-55 is unpinned (include/liftreg_b200.h)."""
    _need_map(phi)
    code = _fd_boundary(boundary)
    phi = _need_cuda_f32(phi, "phi")
    B, _, D, H, W = phi.shape
    stats = torch.empty((B, 7), device=phi.device, dtype=torch.float64)
    det = torch.empty((B, D, H, W), device=phi.device, dtype=torch.float32) if want_map else None
    _call("lr_jacobian_det", phi.device, _ptr(phi), B, D, H, W, code, int(margin), _ptr(det), _ptr(stats))
    return stats, det


# --------------------------------------------------------------------------- folding penalty (training term)
class _FoldPenalty(torch.autograd.Function):
    @staticmethod
    def forward(ctx, phi, boundary):
        phi = _need_cuda_f32(phi, "phi")
        B, _, D, H, W = phi.shape
        stats = torch.empty((B, 7), device=phi.device, dtype=torch.float64)
        _call("lr_jacobian_det", phi.device, _ptr(phi), B, D, H, W, boundary, 0, None, _ptr(stats))
        ctx.save_for_backward(phi)
        ctx.boundary = boundary
        return (stats[:, 1].sum() / float(B * D * H * W)).to(torch.float32)

    @staticmethod
    def backward(ctx, grad_loss):
        phi, = ctx.saved_tensors
        B, _, D, H, W = phi.shape
        g = _grad_scalar(grad_loss, phi.device)
        gphi = torch.empty_like(phi)
        _call("lr_jacobian_fold_backward", phi.device, _ptr(phi), B, D, H, W, ctx.boundary, _ptr(g), _ptr(gphi))
        return gphi, None


def fold_penalty(phi, boundary="linear"):
    """Folding penalty of a map phi (B,3,D,H,W) in [-1,1]: the mean over (B, D, H, W) of max(0, -det J), with det the
    value jacobian_det computes (same boundary, every voxel, non-finite values skipped).  A float32 scalar on phi's
    device, computed without a host synchronisation; differentiable wrt phi (subgradient over the strict fold set
    det < 0).  The reference has no such term, so parity is unpinned (include/liftreg_b200.h,
    lr_jacobian_fold_backward)."""
    _need_map(phi)
    return _FoldPenalty.apply(phi, _fd_boundary(boundary))


def _label_map(t, name):
    if not isinstance(t, torch.Tensor):
        raise TypeError("%s must be a torch.Tensor, got %s" % (name, type(t).__name__))
    if not t.is_cuda:
        raise RuntimeError("%s must be a CUDA tensor: liftreg_b200 has no CPU path (got device %s)" % (name, t.device))
    if t.dtype in (torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64, torch.bool):
        t = t.float()
    return _need_cuda_f32(t, name)


def label_confusion(pred, target, num_labels):
    """Confusion matrix of two label maps with a leading batch axis (any trailing shape, equal for both):
    counts (B,L,L) int64 with counts[b,p,t] = #voxels where pred == p and target == t, and invalid (B,) int64 = #voxels
    where either value is not an integer in [0, L).  Float32 maps (what the nearest-mode warp returns) are read as they
    are, integer maps are converted with .float().  1 <= num_labels <= 128."""
    if pred.shape != target.shape or pred.dim() < 1:
        raise ValueError("pred %s and target %s must have the same shape (B, ...)" % (tuple(pred.shape), tuple(target.shape)))
    L = int(num_labels)
    if not 1 <= L <= 128:
        raise ValueError("num_labels must be in [1, 128], got %d" % L)
    pred, target = _label_map(pred, "pred"), _label_map(target, "target")
    if pred.device != target.device:
        raise ValueError("pred and target must be on the same device")
    B = pred.shape[0]
    N = pred.numel() // B if B else 0
    counts = torch.empty((B, L, L), device=pred.device, dtype=torch.int64)
    invalid = torch.empty((B,), device=pred.device, dtype=torch.int64)
    _call("lr_label_confusion", pred.device, _ptr(pred), _ptr(target), B, N, L, _ptr(counts), _ptr(invalid))
    return counts, invalid


def _label_volumes(pred, target):
    """Two label maps (B,1,D,H,W) or (B,D,H,W) of equal shape on one CUDA device -> contiguous float32 (B,D,H,W)."""
    out = []
    for t, name in ((pred, "pred"), (target, "target")):
        t = _label_map(t, name)
        _volume_shape(t, name)
        out.append((t[:, 0] if t.dim() == 5 else t).contiguous())
    if out[0].shape != out[1].shape:
        raise ValueError("pred %s and target %s must have the same shape" % (tuple(pred.shape), tuple(target.shape)))
    if out[0].device != out[1].device:
        raise ValueError("pred and target must be on the same device")
    return out


def label_surface_counts(pred, target, num_labels):
    """Surface sizes of every label in two label maps (B,1,D,H,W) or (B,D,H,W) (float32 as the nearest-mode warp returns
    them, or an integer dtype): counts (B,2,L) int64 = [|S_pred(l)|, |S_target(l)|] and invalid (B,) int64 = #voxels
    where either value is not an integer in [0, L).  S_M(l) is the set of voxels labelled l with a face neighbour outside
    the volume or labelled otherwise (include/liftreg_b200.h, lr_label_surface_counts).  1 <= num_labels <= 128."""
    L = int(num_labels)
    if not 1 <= L <= 128:
        raise ValueError("num_labels must be in [1, 128], got %d" % L)
    pred, target = _label_volumes(pred, target)
    B, D, H, W = pred.shape
    counts = torch.empty((B, 2, L), device=pred.device, dtype=torch.int64)
    invalid = torch.empty((B,), device=pred.device, dtype=torch.int64)
    _call("lr_label_surface_counts", pred.device, _ptr(pred), _ptr(target), B, D, H, W, L, _ptr(counts), _ptr(invalid))
    return counts, invalid


def surface_distances(from_map, to_map, label, spacing=(1.0, 1.0, 1.0), sizes=None):
    """Directed surface distances of one label: for every voxel of S_from(label), the distance in mm to the nearest voxel
    of S_to(label) with spacing (s_D, s_H, s_W), formed as scipy's distance_transform_edt forms it (include/liftreg_b200.h,
    lr_surface_distances; +inf where S_to is empty).  Maps as in label_surface_counts.

    sizes: |S_from(label)| per item (B,) on the host, e.g. label_surface_counts(...)[0][:, k, label] read back; None
    runs that count pass here (a host synchronisation).  Returns (dist, seg_offset, stats) on the maps' device: dist
    (sum(sizes),) float64 holds item b's distances, in no particular order, at [seg_offset[b], seg_offset[b+1]);
    seg_offset (B+1,) int64; stats (B,3) float64 = [count, sum, max]."""
    label = int(label)
    if not 1 <= label <= 127:
        raise ValueError("label must be in [1, 128), got %d" % label)
    sp = [float(s) for s in spacing]
    if len(sp) != 3 or not all(math.isfinite(s) and s > 0 for s in sp):
        raise ValueError("spacing must be 3 finite values > 0, got %r" % (spacing,))
    src, dst = _label_volumes(from_map, to_map)
    B, D, H, W = src.shape
    if sizes is None:
        sizes = label_surface_counts(src, dst, 128)[0][:, 0, label].cpu().numpy()
    sizes = np.asarray(sizes, dtype=np.int64).reshape(-1)
    if sizes.shape != (B,) or (sizes < 0).any():
        raise ValueError("sizes must hold B=%d counts >= 0, got %r" % (B, sizes))
    offsets = np.concatenate([[0], np.cumsum(sizes)])
    seg_offset = torch.from_numpy(offsets).to(src.device)
    dist = torch.empty((max(int(offsets[-1]), 1),), device=src.device, dtype=torch.float64)
    stats = torch.empty((B, 3), device=src.device, dtype=torch.float64)
    nbytes = _native.lib().lr_surface_distance_workspace_bytes(B, D, H, W)
    if nbytes == 0:
        raise ValueError("maps of shape %s are too large for lr_surface_distances (B*D*H*W < 2^31, B <= 65535, "
                         "H and W <= 65535)" % (tuple(src.shape),))
    ws = torch.empty((nbytes,), device=src.device, dtype=torch.uint8)
    _call("lr_surface_distances", src.device, _ptr(src), _ptr(dst), B, D, H, W, label, sp[0], sp[1], sp[2], _ptr(seg_offset),
          _ptr(dist), _ptr(stats), _ptr(ws), nbytes)
    return dist[:int(offsets[-1])], seg_offset, stats


# --------------------------------------------------------------------------- soft Dice of the warped labels (training term)
def _dice_loss_from_sums(sums):
    """1 - mean_b of the mean over S_b = {l >= 1 : P + T > 0} of 2 I / (P + T) (1 where S_b is empty), from sums
    (B,L,3) float64 = [I, P, T]; float64 on the sums' device, no host synchronisation"""
    I, P, T = sums.unbind(-1)
    den = P + T
    in_s = den > 0
    in_s[:, 0] = False
    n = in_s.sum(1)
    dice_l = torch.where(in_s, 2.0 * I / torch.where(in_s, den, 1.0), 0.0)
    dice = torch.where(n > 0, dice_l.sum(1) / n.clamp(min=1), 1.0)
    return 1.0 - dice.mean()


class _LabelDice(torch.autograd.Function):
    @staticmethod
    def forward(ctx, phi, src, tgt, num_labels):
        phi = _need_cuda_f32(phi, "phi")
        B, _, D, H, W = phi.shape
        sums = torch.empty((B, num_labels, 3), device=phi.device, dtype=torch.float64)
        _call("lr_label_dice_sums", phi.device, _ptr(phi), _ptr(src), _ptr(tgt), B, D, H, W, num_labels, _ptr(sums))
        ctx.save_for_backward(phi, src, tgt, sums)
        return _dice_loss_from_sums(sums).to(torch.float32)

    @staticmethod
    def backward(ctx, grad_loss):
        phi, src, tgt, sums = ctx.saved_tensors
        B, _, D, H, W = phi.shape
        g = _grad_scalar(grad_loss, phi.device)
        gphi = torch.empty_like(phi)
        _call("lr_label_dice_backward", phi.device, _ptr(phi), _ptr(src), _ptr(tgt), B, D, H, W, sums.shape[1], _ptr(sums),
              _ptr(g), _ptr(gphi))
        return gphi, None, None, None


def label_dice_loss(phi, source_labels, target_labels, num_labels):
    """Soft Dice loss of the moving label map warped trilinearly by phi, against the target labels: VoxelMorph's
    semi-supervised term (one-hot labels, trilinear warp with zeros padding, 1 - soft Dice) without materialising the
    one-hot channels.  1 - mean_b of the mean Dice over the labels 1..L-1 present in either map (definition:
    include/liftreg_b200.h, lr_label_dice_sums).

    phi (B,3,D,H,W) CUDA float32 in [-1,1] (channel c addresses volume axis c, as ops.warp); label maps (B,1,D,H,W) or
    (B,D,H,W), float32 or an integer dtype (converted with .float()); a value that is not an integer in
    [0, num_labels) counts as no label.  2 <= num_labels <= 128.  A float32 scalar on phi's device, computed without a
    host synchronisation; differentiable wrt phi (the labels are data).  The reference has no such term, so parity is
    unpinned."""
    _need_map(phi)
    L = int(num_labels)
    if not 2 <= L <= 128:
        raise ValueError("num_labels must be in [2, 128], got %d" % L)
    want = (phi.shape[0],) + tuple(phi.shape[2:])
    maps = []
    for t, name in ((source_labels, "source_labels"), (target_labels, "target_labels")):
        t = _label_map(t, name)
        _volume_shape(t, name, want)
        if t.device != phi.device:
            raise ValueError("%s must be on phi's device %s (got %s)" % (name, phi.device, t.device))
        maps.append((t[:, 0] if t.dim() == 5 else t).contiguous())
    return _LabelDice.apply(phi, maps[0], maps[1], L)
