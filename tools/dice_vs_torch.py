#!/usr/bin/env python
"""Soft Dice loss of the warped label map at 160^3: the library's fused pair (lr_label_dice_sums + lr_label_dice_backward)
against the stock-op composition VoxelMorph uses (one-hot labels -> ops.warp(zero_boundary=True, using_scale=False) ->
torch sums, autograd backward), on the same GPU in the same run, at L = 2, 6 and 14.

    python tools/dice_vs_torch.py [--iters N] [--batch B ...] [--labels L ...]

Prints, per batch size and label count, the time of forward + backward of each (CUDA events around N iterations after a
warm-up), the peak memory each allocates beyond its inputs, and how far the two agree (loss, gradient), with the card's
name and power limit."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from dice_reference import blob_labels, stock_dice_loss  # noqa: E402
from liftreg_b200 import ops, synthetic  # noqa: E402

VOL = (160, 160, 160)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def step_kernel(phi, src, tgt, L):
    p = phi.clone().requires_grad_(True)
    loss = ops.label_dice_loss(p, src, tgt, L)
    loss.backward()
    return loss, p.grad


def step_torch(phi, src, tgt, L):
    p = phi.clone().requires_grad_(True)
    loss = stock_dice_loss(p, src, tgt, L)
    loss.backward()
    return loss, p.grad


def timed(fn, args, iters):
    for _ in range(3):
        fn(*args)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn(*args)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, (torch.cuda.max_memory_allocated() - base) / 2 ** 20


def main():
    args = sys.argv[1:]
    iters = int(args[args.index("--iters") + 1]) if "--iters" in args else 20
    batches = [int(a) for i, a in enumerate(args) if i > 0 and args[i - 1] == "--batch"] or [1]
    label_counts = [int(a) for i, a in enumerate(args) if i > 0 and args[i - 1] == "--labels"] or [2, 6, 14]
    dev = torch.device("cuda:0")
    print("card: %s" % card())
    for B in batches:
        phi = np.stack([synthetic.identity_map_np(VOL) + synthetic.smooth_displacement(VOL, seed=b, max_disp=0.03)
                        for b in range(B)]).astype(np.float32)
        phi = torch.from_numpy(phi).to(dev)
        for L in label_counts:
            src, tgt = blob_labels(B, VOL, L, seed=L, shift=3)
            src, tgt = torch.from_numpy(src).to(dev), torch.from_numpy(tgt).to(dev)
            lk, gk = step_kernel(phi, src, tgt, L)
            lt, gt = step_torch(phi, src, tgt, L)
            rel = float((gk.double() - gt.double()).norm() / gt.double().norm())
            tk, mk = timed(step_kernel, (phi, src, tgt, L), iters)
            tt, mt = timed(step_torch, (phi, src, tgt, L), iters)
            print("B=%d %s L=%d: fused %.3f ms, %.0f MiB | stock ops %.3f ms, %.0f MiB | x%.1f | "
                  "loss %.8f vs %.8f (|diff| %.2e), gradient rel-L2 %.2e"
                  % (B, "x".join(map(str, VOL)), L, tk, mk, tt, mt, tt / tk, lk.item(), lt.item(), abs(lk.item() - lt.item()), rel))
            del src, tgt, gk, gt
            torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
