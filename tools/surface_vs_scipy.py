#!/usr/bin/env python
"""Surface-distance metrics (Hausdorff, HD95, ASSD of two labels) at 160^3 and 2.2 mm: metrics.surface_distance on the
GPU against the same metrics from scipy on the host, in the same run.

    python tools/surface_vs_scipy.py [--iters N]

The target is the phantom's two lungs (synthetic.ct_phantom's ellipsoids) as labels 1 and 2; pred is that map warped
(nearest, zeros outside) by synthetic.smooth_displacement, one seed per item.  Prints the wall time of
metrics.surface_distance including its readback (host clock around the call, which ends in a device synchronisation;
the median of N calls after a warm-up) at B = 1 and B = 8, scipy's time per item (binary_erosion, distance_transform_edt
twice per label, np.percentile), the largest difference between the two, and the card's name and power limit."""
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402
from scipy import ndimage as ndi  # noqa: E402

from liftreg_b200 import metrics, ops, synthetic  # noqa: E402

VOL = (160, 160, 160)
SPACING = (2.2, 2.2, 2.2)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def lungs():
    z, y, x = np.meshgrid(*(np.linspace(-1, 1, n, dtype=np.float32) for n in VOL), indexing="ij")
    out = np.zeros(VOL, np.float32)
    for l, cx in ((1, -0.38), (2, 0.38)):
        out[(z / 0.62) ** 2 + (y / 0.45) ** 2 + ((x - cx) / 0.30) ** 2 <= 1.0] = l
    return out


def scipy_metrics(pred, target, labels=(1, 2)):
    """hd, hd95, assd per label of one item, as metrics.surface_distance defines them"""
    faces = ndi.generate_binary_structure(3, 1)
    out = []
    for l in labels:
        sp, st = [m & ~ndi.binary_erosion(m, faces, border_value=0) for m in (pred == l, target == l)]
        a = ndi.distance_transform_edt(~st, sampling=SPACING)[sp]
        b = ndi.distance_transform_edt(~sp, sampling=SPACING)[st]
        out.append([max(a.max(), b.max()), max(np.percentile(a, 95), np.percentile(b, 95)), (a.mean() + b.mean()) / 2])
    return np.array(out)


def main():
    iters = 20
    if "--iters" in sys.argv:
        iters = int(sys.argv[sys.argv.index("--iters") + 1])
    dev = torch.device("cuda:0")
    print("card:", card())
    target = torch.from_numpy(lungs()).to(dev)[None, None].repeat(8, 1, 1, 1, 1)
    disp = torch.from_numpy(np.stack([synthetic.smooth_displacement(VOL, seed=b) for b in range(8)])).to(dev)
    pred = ops.warp(target, disp, zero_boundary=True, using_scale=False, mode="nearest", disp_plus_identity=True)
    pred_np, target_np = pred[:, 0].cpu().numpy(), target[:, 0].cpu().numpy()

    t0 = time.perf_counter()
    ref = np.stack([scipy_metrics(pred_np[b], target_np[b]) for b in range(8)])         # (8, 2 labels, 3)
    t_scipy = (time.perf_counter() - t0) / 8
    print("scipy (host, both lungs of one item): %.3f s per item (mean of 8)" % t_scipy)

    for B in (1, 8):
        p, t = pred[:B].contiguous(), target[:B].contiguous()
        for _ in range(3):
            res = metrics.surface_distance(p, t, SPACING, num_labels=3)
        times = []
        for _ in range(iters):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = metrics.surface_distance(p, t, SPACING, num_labels=3)
            times.append(time.perf_counter() - t0)
        got = np.stack([res["hd"][:, 1:], res["hd95"][:, 1:], res["assd"][:, 1:]], -1)   # (B, 2, 3)
        rel = np.abs(got - ref[:B]) / ref[:B]
        print("B=%d  metrics.surface_distance: median %.3f ms (min %.3f) per call, %.3f ms per item; speed-up vs scipy "
              "%.0fx per item; max rel diff hd %.2e hd95 %.2e assd %.2e"
              % (B, 1e3 * np.median(times), 1e3 * min(times), 1e3 * np.median(times) / B, t_scipy * B / np.median(times),
                 rel[..., 0].max(), rel[..., 1].max(), rel[..., 2].max()))
    print("B=8 item 0: hd %s hd95 %s assd %s (mm, labels 1 and 2)" % (res["hd"][0, 1:], res["hd95"][0, 1:], res["assd"][0, 1:]))


if __name__ == "__main__":
    main()
