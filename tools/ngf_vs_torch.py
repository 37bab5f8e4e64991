#!/usr/bin/env python
"""NGF similarity (eps = 1, linear face rule) at 160^3: the library's kernels against the stock-op fp32 composition of
the same definition (tests/ngf_reference.ngf_torch: mermaid-style central differences by slicing, elementwise products,
a mean; autograd backward), on the same GPU in the same run.

    python tools/ngf_vs_torch.py [--iters N] [--batch B ...]

Prints, per batch size, the time of forward + backward of each (CUDA events around N iterations after a warm-up),
the peak memory each allocates beyond its inputs, and how far the two agree (loss, gradient), with the card's name
and power limit.  x is the CT phantom warped by a smooth displacement, y the phantom."""
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from ngf_reference import ngf_torch  # noqa: E402
from liftreg_b200 import ops, synthetic  # noqa: E402

VOL, EPS, BOUNDARY = (160, 160, 160), 1.0, "linear"


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def step_kernel(x, y):
    p = x.clone().requires_grad_(True)
    loss = ops.ngf_loss(p, y, EPS, BOUNDARY)
    loss.backward()
    return loss, p.grad


def step_torch(x, y):
    p = x.clone().requires_grad_(True)
    loss = ngf_torch(p, y, EPS, BOUNDARY)
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
    dev = torch.device("cuda:0")
    print("card: %s" % card())
    idm = ops.identity_map(VOL, dev)
    for B in batches:
        y = np.stack([synthetic.hu_to_unit(synthetic.ct_phantom(VOL, seed=b)) for b in range(B)])[:, None]
        disp = np.stack([synthetic.smooth_displacement(VOL, seed=10 + b, max_disp=0.05, coarse=4) for b in range(B)])
        y = torch.from_numpy(y).to(dev)
        x = ops.warp(y, torch.from_numpy(disp).to(dev) + idm)
        del disp
        lk, gk = step_kernel(x, y)
        lt, gt = step_torch(x, y)
        rel = float((gk.double() - gt.double()).norm() / gt.double().norm())
        tk, mk = timed(step_kernel, x, y, iters)
        tt, mt = timed(step_torch, x, y, iters)
        print("B=%d %s eps=%g %s: kernels %.3f ms, %.0f MiB | stock torch fp32 %.3f ms, %.0f MiB | x%.1f | "
              "loss %.8f vs %.8f (|diff| %.2e), gradient rel-L2 %.2e"
              % (B, "x".join(map(str, VOL)), EPS, BOUNDARY, tk, mk, tt, mt, tt / tk, lk.item(), lt.item(),
                 abs(lk.item() - lt.item()), rel))
        del x, y, gk, gt
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
