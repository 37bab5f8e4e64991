#!/usr/bin/env python
"""Local NCC (w = 9) at 160^3: the library's kernels against VoxelMorph's formulation in fp32 stock torch (five conv3d
with a ones kernel forward, autograd backward), on the same GPU in the same run.

    python tools/lncc_vs_torch.py [--iters N] [--batch B ...]

Prints, per batch size, the time of forward + backward of each (CUDA events around N iterations after a warm-up),
the peak memory each allocates beyond its inputs, and how far the two agree (loss, gradient), with the card's name
and power limit.  The torch convolutions run in full fp32 (TF32 off), as the comparison needs."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from lncc_reference import voxelmorph_ncc_torch  # noqa: E402
from liftreg_b200 import ops, synthetic  # noqa: E402

VOL, WIN, EPS = (160, 160, 160), 9, 1e-5


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def step_kernel(x, y):
    p = x.clone().requires_grad_(True)
    loss = ops.local_ncc_loss(p, y, WIN, EPS)
    loss.backward()
    return loss, p.grad


def step_torch(x, y):
    p = x.clone().requires_grad_(True)
    loss = voxelmorph_ncc_torch(p, y, WIN, EPS)[0]
    loss.backward()
    return loss, p.grad


def timed(fn, x, y, iters):
    for _ in range(3):
        fn(x, y)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn(x, y)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, (torch.cuda.max_memory_allocated() - base) / 2 ** 20


def main():
    args = sys.argv[1:]
    iters = int(args[args.index("--iters") + 1]) if "--iters" in args else 20
    batches = [int(a) for i, a in enumerate(args) if i > 0 and args[i - 1] == "--batch"] or [1, 8]
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    dev = torch.device("cuda:0")
    print("card: %s" % card())
    for B in batches:
        x = np.stack([synthetic.hu_to_unit(synthetic.ct_phantom(VOL, seed=b)) for b in range(B)])[:, None]
        y = np.stack([synthetic.hu_to_unit(synthetic.ct_phantom(VOL, seed=100 + b)) for b in range(B)])[:, None]
        x, y = torch.from_numpy(x).to(dev), torch.from_numpy(y).to(dev)
        lk, gk = step_kernel(x, y)
        lt, gt = step_torch(x, y)
        rel = float((gk.double() - gt.double()).norm() / gt.double().norm())
        tk, mk = timed(step_kernel, x, y, iters)
        tt, mt = timed(step_torch, x, y, iters)
        print("B=%d %s w=%d: kernels %.3f ms, %.0f MiB | stock torch fp32 conv3d %.3f ms, %.0f MiB | x%.1f | "
              "loss %.8f vs %.8f (|diff| %.2e), gradient rel-L2 %.2e"
              % (B, "x".join(map(str, VOL)), WIN, tk, mk, tt, mt, tt / tk, lk.item(), lt.item(), abs(lk.item() - lt.item()), rel))
        del x, y, gk, gt
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
