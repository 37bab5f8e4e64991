#!/usr/bin/env python
"""Quick per-kernel timing loop for kernel development (not the contract benchmark -- that is bench.py).

    python tools/kbench.py [warp] [backproject] [drr] [--iters N] [--labels L]

Times each kernel at the cfg2 / cfg1 sizes with rotating buffers (cold L2) under a CUDA graph and prints us per launch."""
import ctypes
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

from liftreg_b200 import _native, ops, synthetic  # noqa: E402

VOL, DET, P, R = (160, 160, 160), (256, 256), 4, 8


def main():
    iters = 2000
    args = list(sys.argv[1:])
    if "--iters" in args:
        k = args.index("--iters")
        iters = int(args[k + 1])
        del args[k:k + 2]
    batch = 1
    if "--batch" in args:        # batch items per launch for warp / backproject (BASELINE configs[2] uses 8)
        k = args.index("--batch")
        batch = int(args[k + 1])
        del args[k:k + 2]
    n_labels = 2
    if "--labels" in args:       # labels of the dice entries: 2 or 6
        k = args.index("--labels")
        n_labels = int(args[k + 1])
        del args[k:k + 2]
    which = args or ["warp", "backproject", "drr"]
    dev = torch.device("cuda:0")
    lib = _native.lib()
    stream = torch.cuda.Stream()
    rs = np.random.RandomState(0)
    nv = VOL[0] * VOL[1] * VOL[2]
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    poses = synthetic.wrapper_poses(60.0, P, VOL[1])
    poses32 = np.ascontiguousarray(poses.astype(np.float32))
    phi = torch.from_numpy((synthetic.smooth_displacement(VOL) + synthetic.identity_map_np(VOL))[None]).to(dev).repeat(batch, 1, 1, 1, 1)
    moving = torch.from_numpy(rs.uniform(-1, 1, (1, 1) + VOL).astype(np.float32)).to(dev).repeat(batch, 1, 1, 1, 1)
    proj = torch.from_numpy(rs.uniform(-1, 1, (1, P) + DET).astype(np.float32)).to(dev).repeat(batch, 1, 1, 1)
    mu = torch.from_numpy(rs.uniform(0, 0.3, (1,) + VOL).astype(np.float32)).to(dev)
    sets = [dict(phi=phi.clone(), moving=moving.clone(), proj=proj.clone(), mu=mu.clone(),
                 warped=torch.empty((batch, 1) + VOL, device=dev), lifted=torch.empty((batch, P) + VOL, device=dev),
                 drr=torch.empty((1, P, 240, 240), device=dev), drr256=torch.empty((1, P, 256, 256), device=dev)) for _ in range(R)]
    sp3 = np.array([2.2, 2.2, 2.2], np.float32)
    p64 = np.ascontiguousarray(poses, np.float64)

    def k_warp(s, st):
        _native.check(lib.lr_warp_forward(vp(s["moving"]), vp(s["phi"]), batch, 1, *VOL, 0, 0, 1, 0, vp(s["warped"]), st), "warp")

    def k_backproject(s, st):
        _native.check(lib.lr_backproject_forward(vp(s["proj"]), ops._fp(poses32), batch, P, DET[0], DET[1], *VOL, vp(s["lifted"]),
                                                 P * nv, nv, st), "backproject")

    def k_drr(s, st):
        _native.check(lib.lr_drr_forward(vp(s["mu"]), 1, *VOL, ops._dp(p64), 1, P, 240, 240, ops._fp(sp3), 0,
                                         ctypes.c_float(0.1), vp(s["drr"]), st), "drr")

    def k_drr256(s, st):
        _native.check(lib.lr_drr_forward(vp(s["mu"]), 1, *VOL, ops._dp(p64), 1, P, 256, 256, ops._fp(sp3), 0,
                                         ctypes.c_float(0.1), vp(s["drr256"]), st), "drr256")

    gout = torch.from_numpy(rs.standard_normal((1, 1) + VOL).astype(np.float32)).to(dev)
    gphi = [torch.empty((1, 3) + VOL, device=dev) for _ in range(R)]
    gdrr = torch.from_numpy(rs.standard_normal((1, P, 240, 240)).astype(np.float32)).to(dev)
    gvol = [torch.zeros((1,) + VOL, device=dev) for _ in range(R)]
    for i, s_ in enumerate(sets):
        s_["gphi"], s_["gvol"] = gphi[i], gvol[i]

    def k_warp_bwd(s, st):     # d/dphi only (what training needs: LiftRegDeformSubspaceBackproj.py:69 with moving as data)
        _native.check(lib.lr_warp_backward(vp(gout), vp(s["moving"]), vp(s["phi"]), 1, 1, *VOL, 0, 0, 1, 0, None, vp(s["gphi"]), st), "warp_bwd")

    def k_drr_bwd(s, st):
        _native.check(lib.lr_drr_backward(vp(gdrr), 1, *VOL, ops._dp(p64), 1, P, 240, 240, ops._fp(sp3), 0,
                                          ctypes.c_float(0.1), vp(s["gvol"]), st), "drr_bwd")

    if "pca" in which or "pca_bwd" in which:
        K = 56
        basis = torch.empty((3 * nv, K), device=dev).normal_(0, 1e-3)       # 2.75 GB, as the model holds it
        pmean = torch.zeros(3 * nv, device=dev)
        coefs = torch.randn(1, K, device=dev)
        pout = [torch.empty((1, 3 * nv), device=dev) for _ in range(R)]
        for i, s_ in enumerate(sets):
            s_["pout"] = pout[i]

    if "pca_bwd" in which:
        pgout = torch.randn(1, 3 * nv, device=dev)
        pgc = torch.zeros(1, 56, device=dev)

    def k_pca_bwd(s, st):
        _native.check(lib.lr_pca_decode_backward(vp(pgout), vp(basis), 1, 56, 3 * nv, vp(pgc), st), "pca_bwd")

    def k_pca(s, st):
        _native.check(lib.lr_pca_decode(vp(coefs), vp(basis), vp(pmean), 1, K, 3 * nv, 1, *VOL, vp(s["pout"]), st), "pca")

    ncc_sums = torch.zeros((1, 7), device=dev, dtype=torch.float64)
    ncc_g = torch.ones(1, device=dev)

    def k_ncc(s, st):          # forward of the similarity loss: one pass over warped + target (+ memset and a B-thread finalisation)
        _native.check(lib.lr_ncc_sums(vp(s["warped"]), vp(s["moving"]), 1, nv, vp(ncc_sums), st), "ncc")

    def k_ncc_bwd(s, st):
        _native.check(lib.lr_ncc_backward(vp(s["warped"]), vp(s["moving"]), 1, nv, vp(ncc_sums), vp(ncc_g), vp(s["gvol"]), st), "ncc_bwd")

    reg_sum = torch.zeros(1, device=dev, dtype=torch.float64)

    def k_reg(s, st):          # displacement regulariser (SubspaceLoss.py:51-67): one pass over the 3-channel field
        _native.check(lib.lr_diffusion_reg_sum(vp(s["phi"]), 1, *VOL, 0, vp(reg_sum), st), "reg")

    def k_reg_bwd(s, st):
        _native.check(lib.lr_diffusion_reg_backward(vp(s["phi"]), 1, *VOL, 0, vp(ncc_g), vp(s["gphi"]), st), "reg_bwd")

    jac_stats = torch.zeros((1, 7), device=dev, dtype=torch.float64)

    def k_jac(s, st):          # Jacobian-determinant statistics of the map (validation folding metric): one pass over phi
        _native.check(lib.lr_jacobian_det(vp(s["phi"]), 1, *VOL, 0, 0, None, vp(jac_stats), st), "jac")

    def k_jac_map(s, st):      # ... and the determinant map written out
        _native.check(lib.lr_jacobian_det(vp(s["phi"]), 1, *VOL, 0, 0, vp(s["warped"]), vp(jac_stats), st), "jac_map")

    def k_fold_bwd(s, st):     # d fold / d phi (folding penalty adjoint): reads phi, writes grad_phi
        _native.check(lib.lr_jacobian_fold_backward(vp(s["phi"]), 1, *VOL, 0, vp(ncc_g), vp(s["gphi"]), st), "fold_bwd")

    if "fold_bwd8" in which or "dice_bwd8" in which:
        phi8 = [torch.from_numpy((synthetic.smooth_displacement(VOL, seed=b) + synthetic.identity_map_np(VOL))[None]).to(dev)
                for b in range(8)]
        for i, s_ in enumerate(sets):
            s_["phi8"] = torch.cat(phi8, 0) + 1e-3 * i
            s_["gphi8"] = torch.empty((8, 3) + VOL, device=dev)

    def k_fold_bwd8(s, st):
        _native.check(lib.lr_jacobian_fold_backward(vp(s["phi8"]), 8, *VOL, 0, vp(ncc_g), vp(s["gphi8"]), st), "fold_bwd8")

    lncc_sum = torch.zeros(8, device=dev, dtype=torch.float64)
    lncc_ws = torch.empty(lib.lr_local_ncc_workspace_bytes(8 if "lncc_bwd8" in which else 1, *VOL, 9), device=dev, dtype=torch.uint8)

    def k_lncc(s, st):         # local NCC forward, w = 9: one pass over two volumes
        _native.check(lib.lr_local_ncc_sum(vp(s["moving"]), vp(s["mu"]), 1, *VOL, 9, 1e-5, vp(lncc_sum), st), "lncc")

    def k_lncc_bwd(s, st):     # local NCC adjoint, w = 9: coefficient pass (x, y -> 12 B workspace) + box-sum pass
        _native.check(lib.lr_local_ncc_backward(vp(s["moving"]), vp(s["mu"]), 1, *VOL, 9, 1e-5, vp(ncc_g), vp(s["gvol"]),
                                                vp(lncc_ws), lncc_ws.numel(), st), "lncc_bwd")

    if "lncc_bwd8" in which:
        for i, s_ in enumerate(sets):
            s_["x8"] = torch.from_numpy(rs.uniform(-1, 1, (8, 1) + VOL).astype(np.float32)).to(dev)
            s_["y8"] = torch.from_numpy(rs.uniform(-1, 1, (8, 1) + VOL).astype(np.float32)).to(dev)
            s_["g8"] = torch.empty((8, 1) + VOL, device=dev)

    def k_lncc_bwd8(s, st):
        _native.check(lib.lr_local_ncc_backward(vp(s["x8"]), vp(s["y8"]), 8, *VOL, 9, 1e-5, vp(ncc_g), vp(s["g8"]),
                                                vp(lncc_ws), lncc_ws.numel(), st), "lncc_bwd8")

    ngf_sum = torch.zeros(8, device=dev, dtype=torch.float64)

    def k_ngf(s, st):          # NGF forward: one pass over two volumes (8 B per voxel)
        _native.check(lib.lr_ngf_sum(vp(s["moving"]), vp(s["mu"]), 1, *VOL, 0, 1.0, vp(ngf_sum), st), "ngf")

    def k_ngf_bwd(s, st):      # NGF adjoint: reads x and y, writes grad_x (12 B per voxel)
        _native.check(lib.lr_ngf_backward(vp(s["moving"]), vp(s["mu"]), 1, *VOL, 0, 1.0, vp(ncc_g), vp(s["gvol"]), st), "ngf_bwd")

    if "ngf_bwd8" in which and "x8" not in sets[0]:
        for i, s_ in enumerate(sets):
            s_["x8"] = torch.from_numpy(rs.uniform(-1, 1, (8, 1) + VOL).astype(np.float32)).to(dev)
            s_["y8"] = torch.from_numpy(rs.uniform(-1, 1, (8, 1) + VOL).astype(np.float32)).to(dev)
            s_["g8"] = torch.empty((8, 1) + VOL, device=dev)

    def k_ngf_bwd8(s, st):
        _native.check(lib.lr_ngf_backward(vp(s["x8"]), vp(s["y8"]), 8, *VOL, 0, 1.0, vp(ncc_g), vp(s["g8"]), st), "ngf_bwd8")

    mi_names = ("mi", "mi_bwd", "mi_bwd8")
    if any(n in which for n in mi_names):
        # the unit-normalised CT phantom pair: the histogram's contention depends on the image content (air and bone
        # saturate the range), so uniform noise would time a different kernel
        mi_y = torch.from_numpy(synthetic.hu_to_unit(synthetic.ct_phantom(VOL, seed=0))[None, None]).to(dev)
        mi_x = ops.warp(mi_y, torch.from_numpy(synthetic.smooth_displacement(VOL, seed=1, max_disp=0.05, coarse=4)).to(dev)[None]
                        + ops.identity_map(VOL, dev))
        mi_hist = torch.zeros((8, 32, 34), device=dev, dtype=torch.float64)
        _native.check(lib.lr_mi_hist(vp(mi_x), vp(mi_y), 1, nv, 32, -1.0, 1.0, vp(mi_hist), None), "mi")
        for s_ in sets:
            s_["mi_x"], s_["mi_y"], s_["mi_g"] = mi_x.clone(), mi_y.clone(), torch.empty_like(mi_x)
        if "mi_bwd8" in which:
            _native.check(lib.lr_mi_hist(vp(mi_x.repeat(8, 1, 1, 1, 1)), vp(mi_y.repeat(8, 1, 1, 1, 1)), 8, nv, 32, -1.0, 1.0,
                                         vp(mi_hist), None), "mi8")
            for s_ in sets:
                s_["mi_x8"], s_["mi_y8"] = mi_x.repeat(8, 1, 1, 1, 1), mi_y.repeat(8, 1, 1, 1, 1)
                s_["mi_g8"] = torch.empty_like(s_["mi_x8"])
        torch.cuda.synchronize()

    def k_mi(s, st):           # MI forward: the joint histogram of warped + target (8 B per voxel), nb = 32
        _native.check(lib.lr_mi_hist(vp(s["mi_x"]), vp(s["mi_y"]), 1, nv, 32, -1.0, 1.0, vp(mi_hist), st), "mi")

    def k_mi_bwd(s, st):       # MI adjoint: reads x and y, writes grad_x (12 B per voxel)
        _native.check(lib.lr_mi_backward(vp(s["mi_x"]), vp(s["mi_y"]), 1, nv, 32, -1.0, 1.0, vp(mi_hist), vp(ncc_g),
                                         vp(s["mi_g"]), st), "mi_bwd")

    def k_mi_bwd8(s, st):
        _native.check(lib.lr_mi_backward(vp(s["mi_x8"]), vp(s["mi_y8"]), 8, nv, 32, -1.0, 1.0, vp(mi_hist), vp(ncc_g),
                                         vp(s["mi_g8"]), st), "mi_bwd8")

    dice_names = ("dice", "dice_bwd", "dice_bwd8")
    if "labels2" in which or "labels6" in which or any(n in which for n in dice_names):
        # label maps as a validation item has them: mostly background, a few organ-sized blobs, target = shifted pred
        zz, yy, xx = np.meshgrid(*[np.arange(n) for n in VOL], indexing="ij")
        for i, s_ in enumerate(sets):
            for L in (2, 6):
                lab = np.zeros(VOL, np.float32)
                for k in range(1, L):
                    c = rs.randint(40, 120, 3)
                    lab[(zz - c[0]) ** 2 + (yy - c[1]) ** 2 + (xx - c[2]) ** 2 < 30 ** 2] = k
                s_["pred%d" % L] = torch.from_numpy(lab).to(dev)
                s_["target%d" % L] = torch.from_numpy(np.roll(lab, 3, axis=0)).to(dev)
    if "dice_bwd8" in which:
        for s_ in sets:
            s_["src8"] = torch.stack([torch.roll(s_["pred%d" % n_labels], b, 0) for b in range(8)])
            s_["tgt8"] = torch.stack([torch.roll(s_["target%d" % n_labels], b, 0) for b in range(8)])
    dice_sums = torch.zeros((8, n_labels, 3), device=dev, dtype=torch.float64)
    L_ = n_labels

    def k_dice(s, st):         # soft Dice sums of the warped labels: phi, target labels and 8 moving-label taps per voxel
        _native.check(lib.lr_label_dice_sums(vp(s["phi"]), vp(s["pred%d" % L_]), vp(s["target%d" % L_]), 1, *VOL, L_,
                                             vp(dice_sums), st), "dice")

    def k_dice_bwd(s, st):     # its adjoint: the same reads, grad_phi written
        _native.check(lib.lr_label_dice_backward(vp(s["phi"]), vp(s["pred%d" % L_]), vp(s["target%d" % L_]), 1, *VOL, L_,
                                                 vp(dice_sums), vp(ncc_g), vp(s["gphi"]), st), "dice_bwd")

    def k_dice_bwd8(s, st):
        _native.check(lib.lr_label_dice_backward(vp(s["phi8"]), vp(s["src8"]), vp(s["tgt8"]), 8, *VOL, L_, vp(dice_sums), vp(ncc_g),
                                                 vp(s["gphi8"]), st), "dice_bwd8")

    conf_counts, conf_invalid = torch.zeros((1, 36), device=dev, dtype=torch.int64), torch.zeros(1, device=dev, dtype=torch.int64)

    def k_labels(L):           # confusion matrix of two label maps (validation overlap metrics)
        def k(s, st):
            _native.check(lib.lr_label_confusion(vp(s["pred%d" % L]), vp(s["target%d" % L]), 1, nv, L, vp(conf_counts),
                                                 vp(conf_invalid), st), "labels%d" % L)
        return k

    if "sdist" in which or "sdist8" in which:
        # the phantom's two lungs (labels 1, 2) as target, the same map warped (nearest) by a smooth displacement as
        # pred; B = 8 stacks 8 displacements.  One map pair and one workspace serve every set: the 16 B/voxel workspace
        # is larger than L2 at B = 8 and about half of it at B = 1.
        zz, yy, xx = np.meshgrid(*[np.linspace(-1, 1, n) for n in VOL], indexing="ij")
        lung = np.zeros(VOL, np.float32)
        for l, cx in ((1, -0.38), (2, 0.38)):
            lung[(zz / 0.62) ** 2 + (yy / 0.45) ** 2 + ((xx - cx) / 0.30) ** 2 <= 1.0] = l
        disp8 = torch.from_numpy(np.stack([synthetic.smooth_displacement(VOL, seed=b) for b in range(8)])).to(dev)
        tgt8 = torch.from_numpy(lung).to(dev)[None, None].repeat(8, 1, 1, 1, 1)
        pred8 = ops.warp(tgt8, disp8, zero_boundary=True, using_scale=False, mode="nearest", disp_plus_identity=True)
        sd = {}
        for nb in (1, 8):
            cnt = ops.label_surface_counts(pred8[:nb], tgt8[:nb], 3)[0][:, :, 1].cpu().numpy()     # label 1 (one lung)
            offs = [torch.from_numpy(np.concatenate([[0], np.cumsum(cnt[:, k])])).to(dev) for k in (0, 1)]
            nbytes = lib.lr_surface_distance_workspace_bytes(nb, *VOL)
            sd[nb] = (pred8[:nb].contiguous(), tgt8[:nb].contiguous(), offs,
                      torch.empty(int(cnt.sum(0).max()), device=dev, dtype=torch.float64),
                      torch.empty((nb, 3), device=dev, dtype=torch.float64), torch.empty(nbytes, device=dev, dtype=torch.uint8), nbytes)

    def k_sdist_b(nb):         # both directed surface distances of one lung label: pred -> target and target -> pred
        def k(s, st):
            p, t, offs, dist, stats, ws, nbytes = sd[nb]
            for a, b, off in ((p, t, offs[0]), (t, p, offs[1])):
                _native.check(lib.lr_surface_distances(vp(a), vp(b), nb, *VOL, 1, 2.2, 2.2, 2.2, vp(off), vp(dist), vp(stats),
                                                       vp(ws), nbytes, st), "sdist")
        return k

    def k_atten(s, st):        # HU -> attenuation (sdct:6-13), elementwise
        _native.check(lib.lr_atten_coef(vp(s["moving"]), nv, vp(s["warped"]), st), "atten")

    def k_idmap(s, st):        # identity map (net_utils.py:59-87), write-only
        _native.check(lib.lr_identity_map(*VOL, vp(s["gphi"]), st), "idmap")

    units = {"atten": (k_atten, nv, 8 * nv), "idmap": (k_idmap, nv, 12 * nv), "reg": (k_reg, nv, 12 * nv), "jac": (k_jac, nv, 12 * nv), "jac_map": (k_jac_map, nv, 16 * nv),
             "labels2": (k_labels(2), nv, 8 * nv), "labels6": (k_labels(6), nv, 8 * nv), "reg_bwd": (k_reg_bwd, nv, 24 * nv), "fold_bwd": (k_fold_bwd, nv, 24 * nv), "fold_bwd8": (k_fold_bwd8, 8 * nv, 8 * 24 * nv), "ncc": (k_ncc, nv, 8 * nv), "lncc": (k_lncc, nv, 8 * nv), "lncc_bwd": (k_lncc_bwd, nv, 44 * nv),
             "lncc_bwd8": (k_lncc_bwd8, 8 * nv, 8 * 44 * nv), "ngf": (k_ngf, nv, 8 * nv), "ngf_bwd": (k_ngf_bwd, nv, 12 * nv),
             "ngf_bwd8": (k_ngf_bwd8, 8 * nv, 8 * 12 * nv), "mi": (k_mi, nv, 8 * nv), "mi_bwd": (k_mi_bwd, nv, 12 * nv),
             "mi_bwd8": (k_mi_bwd8, 8 * nv, 8 * 12 * nv), "dice": (k_dice, nv, 20 * nv), "dice_bwd": (k_dice_bwd, nv, 32 * nv),
             "dice_bwd8": (k_dice_bwd8, 8 * nv, 8 * 32 * nv), "ncc_bwd": (k_ncc_bwd, nv, 12 * nv), "warp": (k_warp, batch * nv, batch * 20 * nv), "pca": (k_pca, 3 * nv, 4 * 3 * nv * 56 + 8 * 3 * nv),
             "pca_bwd": (k_pca_bwd, 3 * nv, 4 * 3 * nv * 56 + 4 * 3 * nv), "warp_bwd": (k_warp_bwd, nv, 32 * nv),
             "drr_bwd": (k_drr_bwd, P * 240 * 240 * VOL[1], 4 * nv + 4 * P * 240 * 240), "backproject": (k_backproject, batch * P * nv, batch * (4 * P * nv + 4 * P * DET[0] * DET[1])),
             "drr": (k_drr, P * 240 * 240 * VOL[1], 4 * nv + 4 * P * 240 * 240),
             "drr256": (k_drr256, P * 256 * 256 * VOL[1], 4 * nv + 4 * P * 256 * 256),
             # per direction: both maps read once, the two 4-byte intermediates written and read once (24 B per voxel)
             "sdist": (k_sdist_b(1), 2 * nv, 2 * 24 * nv), "sdist8": (k_sdist_b(8), 2 * 8 * nv, 2 * 8 * 24 * nv)}
    for name in which:
        fn, n_units, nbytes = units[name]
        g = torch.cuda.CUDAGraph()
        with torch.cuda.stream(stream):
            st = ctypes.c_void_p(stream.cuda_stream)
            fn(sets[0], st); stream.synchronize()
            with torch.cuda.graph(g, stream=stream):
                for r in range(R):
                    fn(sets[r], st)
            for _ in range(3):
                g.replay()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(iters // R):
                g.replay()
            e1.record(stream)
        torch.cuda.synchronize()
        us = 1e3 * e0.elapsed_time(e1) / (iters // R * R)
        print("%-19s %8.2f us  %8.1f G units/s  %7.1f GB/s (algorithmic)" % (name, us, n_units / us * 1e-3, nbytes / us * 1e-3))


if __name__ == "__main__":
    main()
