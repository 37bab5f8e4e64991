"""liftreg_b200 -- B200-native geometric resampling for LiftReg (DRR projection, backprojection, warp).

Host-side mirror of the reference's operator interface over a C-ABI CUDA library (sm_100a):
    liftreg_b200.sdct_projection_utils   <-> reference src/liftreg/utils/sdct_projection_utils.py
    liftreg_b200.net_utils               <-> reference src/liftreg/utils/net_utils.py (Bilinear, identity maps)
    liftreg_b200.layers                  <-> reference src/liftreg/layers/layers.py (proj_layer)
    liftreg_b200.ops                     functional autograd ops over include/liftreg_b200.h
    liftreg_b200.dropin                  makes an installed reference use the above
    liftreg_b200.sharding                multi-GPU partitioning (view-sharded DRR, slab-sharded backprojection/warp)
    liftreg_b200.metrics                 validation metrics on the GPU (Jacobian folding, per-label overlap; parity unpinned)
"""
__version__ = "0.1.0"
