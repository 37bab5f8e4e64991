"""ctypes binding of libliftreg_b200.so (the C-ABI declared in include/liftreg_b200.h).

There is NO CPU or PyTorch fallback: if the shared library is missing, or a call fails, this module raises.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LIFTREG_B200_LIB") or os.path.join(_HERE, "_lib", "libliftreg_b200.so")   # env: kernel experiments

c_float_p = ctypes.POINTER(ctypes.c_float)
c_double_p = ctypes.POINTER(ctypes.c_double)
_i, _i64, _f, _vp, _sz = ctypes.c_int, ctypes.c_int64, ctypes.c_float, ctypes.c_void_p, ctypes.c_size_t

# name -> (restype, argtypes); must list every LR_API symbol of include/liftreg_b200.h
# (tests/test_abi_symbols.py cross-checks this table against the header and the built library).
SIGNATURES = {
    "lr_abi_version": (_i, []),
    "lr_last_error": (ctypes.c_char_p, []),
    "lr_device_count": (_i, []),
    "lr_set_numerics": (_i, [_i]),
    "lr_get_numerics": (_i, []),
    "lr_launch_count": (ctypes.c_longlong, []),
    "lr_launch_count_reset": (None, []),
    "lr_drr_forward": (_i, [_vp, _i, _i, _i, _i, c_double_p, _i, _i, _i, _i, c_float_p, _i, _f, _vp, _vp]),
    "lr_drr_backward": (_i, [_vp, _i, _i, _i, _i, c_double_p, _i, _i, _i, _i, c_float_p, _i, _f, _vp, _vp]),
    "lr_project_grid": (_i, [c_double_p, _i, _i, _i, _i, _i, _i, c_float_p, _i, _i, _vp, _vp, _vp]),
    "lr_drr_forward_peers": (_i, [_vp, _i, _i, _i, _i, c_double_p, _i, _i, _i, _i, c_float_p, _i, _f, _vp, _i, _i, _vp]),
    "lr_peer_alloc": (_i, [_sz, _vp, _vp]),
    "lr_peer_open": (_i, [_vp, _vp]),
    "lr_peer_close": (_i, [_vp]),
    "lr_peer_free": (_i, [_vp]),
    "lr_drr_forward_host_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i]),
    "lr_drr_forward_host": (_i, [_vp, _i, _i, _i, _i, c_double_p, _i, _i, _i, _i, c_float_p, _i, _f, _vp, _vp, _sz, _vp]),
    "lr_backproject_forward": (_i, [_vp, c_float_p, _i, _i, _i, _i, _i, _i, _i, _vp, _i64, _i64, _vp]),
    "lr_backproject_forward_slab": (_i, [_vp, c_float_p, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _i64, _i64, _vp]),
    "lr_backproject_backward": (_i, [_vp, _i64, _i64, c_float_p, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "lr_backproj_grid": (_i, [c_float_p, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "lr_backproject_forward_host_workspace_bytes": (_sz, [_i, _i, _i, _i, _i, _i, _i]),
    "lr_backproject_forward_host": (_i, [_vp, c_float_p, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "lr_backproject_forward_host_async": (_i, [_vp, c_float_p, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "lr_stream_synchronize": (_i, [_vp]),
    "lr_warp_forward_host_async": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "lr_warp_forward": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "lr_warp_backward": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "lr_warp_forward_slab": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "lr_warp_backward_slab": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "lr_identity_map": (_i, [_i, _i, _i, _vp, _vp]),
    "lr_warp_forward_host_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "lr_warp_forward_host": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _sz, _vp]),
    "lr_pca_decode": (_i, [_vp, _vp, _vp, _i, _i, _i64, _i, _i, _i, _i, _vp, _vp]),
    "lr_pca_decode_backward": (_i, [_vp, _vp, _i, _i, _i64, _vp, _vp]),
    "lr_atten_coef": (_i, [_vp, _i64, _vp, _vp]),
    "lr_warp_forward_plan": (_i, [_i, _i, _i, _i, _i, ctypes.POINTER(ctypes.c_int)]),
    "lr_backproject_forward_plan": (_i, [_i, _i, _i, _i, _i, _i, _i, ctypes.POINTER(ctypes.c_int)]),
    "lr_probe_l1_gather": (_i, [_vp, _i64, _i, _i, _i, _vp, _vp]),
    "lr_probe_issue": (_i, [_i, _i, _vp, _vp]),
    "lr_probe_issue_packed": (_i, [_i, _i, _vp, _vp]),
    "lr_ncc_sums": (_i, [_vp, _vp, _i, _i64, _vp, _vp]),
    "lr_ncc_backward": (_i, [_vp, _vp, _i, _i64, _vp, _vp, _vp, _vp]),
    "lr_diffusion_reg_sum": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "lr_diffusion_reg_backward": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "lr_jacobian_det": (_i, [_vp, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "lr_jacobian_fold_backward": (_i, [_vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "lr_label_confusion": (_i, [_vp, _vp, _i, _i64, _i, _vp, _vp, _vp]),
    "lr_label_surface_counts": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp]),
    "lr_surface_distance_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "lr_surface_distances": (_i, [_vp, _vp, _i, _i, _i, _i, _i, ctypes.c_double, ctypes.c_double, ctypes.c_double, _vp, _vp,
                                  _vp, _vp, _sz, _vp]),
    "lr_local_ncc_sum": (_i, [_vp, _vp, _i, _i, _i, _i, _i, ctypes.c_double, _vp, _vp]),
    "lr_local_ncc_workspace_bytes": (_sz, [_i, _i, _i, _i, _i]),
    "lr_local_ncc_backward": (_i, [_vp, _vp, _i, _i, _i, _i, _i, ctypes.c_double, _vp, _vp, _vp, _sz, _vp]),
    "lr_label_dice_sums": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "lr_label_dice_backward": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp]),
    "lr_ngf_sum": (_i, [_vp, _vp, _i, _i, _i, _i, _i, ctypes.c_double, _vp, _vp]),
    "lr_ngf_backward": (_i, [_vp, _vp, _i, _i, _i, _i, _i, ctypes.c_double, _vp, _vp, _vp]),
    "lr_mi_hist": (_i, [_vp, _vp, _i, _i64, _i, _f, _f, _vp, _vp]),
    "lr_mi_backward": (_i, [_vp, _vp, _i, _i64, _i, _f, _f, _vp, _vp, _vp, _vp]),
}

_lib = None


class NativeLibraryError(RuntimeError):
    pass


def lib():
    """Load libliftreg_b200.so (once). Raises NativeLibraryError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryError(
                "libliftreg_b200.so is not built (%s). Run `python -m liftreg_b200.build` "
                "(or __graft_entry__.build()); there is no CPU/PyTorch fallback." % LIB_PATH)
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)     # AttributeError here = header / library mismatch
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


def check(status, what):
    """Turn a negative lr_status into RuntimeError(lr_last_error())."""
    if status != 0:
        msg = lib().lr_last_error()
        raise RuntimeError("%s failed (status %d): %s" % (what, status, msg.decode() if msg else "?"))


NUMERICS = {"fast": 0, "exact": 1}


def set_numerics(mode):
    """'fast' (default: blends as fused lerps, <= 1e-6 rel-L2 from ATen) or 'exact' (ATen's operation order, bit-identical
    values).  Indices and weights are bit-exact in both.  Returns the previous mode name."""
    prev = get_numerics()
    check(lib().lr_set_numerics(NUMERICS[mode] if isinstance(mode, str) else int(mode)), "lr_set_numerics")
    return prev


def get_numerics():
    return "exact" if lib().lr_get_numerics() == 1 else "fast"


def launch_count():
    return int(lib().lr_launch_count())


def launch_count_reset():
    lib().lr_launch_count_reset()
