#!/usr/bin/env python
"""Mutual information similarity (32 bins over (-1, 1)) at 160^3: the library's kernels against the stock-op fp32
composition of the same definition (tests/mi_reference.mi_torch: clamp, cubic B-spline weights, scatter_add into the
joint histogram, MI; autograd backward), on the same GPU in the same run.

    python tools/mi_vs_torch.py [--iters N] [--batch B ...] [--bins NB]

Prints, per batch size, the time of forward + backward of each (CUDA events around N iterations after a warm-up),
the peak memory each allocates beyond its inputs, and how far the two agree (loss, gradient), with the card's name
and power limit.  x is the unit-normalised CT phantom warped by a smooth displacement, y the phantom.  It also
estimates the adjoint's per-block table build: lr_mi_backward on a 4-voxel item (one block: the table build and the
launch) against lr_ncc_backward on the same item (the launch alone), both as CUDA-graph replays."""
import ctypes
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from mi_reference import mi_torch  # noqa: E402
from liftreg_b200 import _native, ops, synthetic  # noqa: E402

VOL = (160, 160, 160)


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[torch.cuda.current_device()] if out else torch.cuda.get_device_name()
    except (OSError, subprocess.SubprocessError):
        return torch.cuda.get_device_name() + ", power limit unknown"


def step_kernel(x, y, nb):
    p = x.clone().requires_grad_(True)
    loss = ops.mi_loss(p, y, nb)
    loss.backward()
    return loss, p.grad


def step_torch(x, y, nb):
    p = x.clone().requires_grad_(True)
    loss = mi_torch(p, y, nb)
    loss.backward()
    return loss, p.grad


def timed(fn, x, y, nb, iters):
    for _ in range(3):
        fn(x, y, nb)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn(x, y, nb)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, (torch.cuda.max_memory_allocated() - base) / 2 ** 20


def graph_us(fn, reps=200, rounds=20):
    """us per call of fn(stream) from CUDA-graph replays of `reps` calls"""
    stream = torch.cuda.Stream()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        st = ctypes.c_void_p(stream.cuda_stream)
        fn(st)
        stream.synchronize()
        with torch.cuda.graph(g, stream=stream):
            for _ in range(reps):
                fn(st)
        g.replay()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(rounds):
            g.replay()
        e1.record(stream)
    torch.cuda.synchronize()
    return 1e3 * e0.elapsed_time(e1) / (reps * rounds)


def table_build(dev, nb):
    lib = _native.lib()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    x = torch.linspace(-1, 1, 4, device=dev)[None]
    y = x.flip(1).contiguous()
    g1, gx = torch.ones(1, device=dev), torch.empty_like(x)
    hist = torch.empty((1, nb, nb + 2), device=dev, dtype=torch.float64)
    sums = torch.empty((1, 7), device=dev, dtype=torch.float64)
    # a full histogram (every bin non-zero) so every table entry takes the log
    hist.fill_(1.0)
    _native.check(lib.lr_ncc_sums(vp(x), vp(y), 1, 4, vp(sums), None), "ncc")
    t_mi = graph_us(lambda st: _native.check(lib.lr_mi_backward(vp(x), vp(y), 1, 4, nb, -1.0, 1.0, vp(hist), vp(g1), vp(gx), st),
                                             "mi_bwd"))
    t_ncc = graph_us(lambda st: _native.check(lib.lr_ncc_backward(vp(x), vp(y), 1, 4, vp(sums), vp(g1), vp(gx), st), "ncc_bwd"))
    return t_mi, t_ncc


def main():
    args = sys.argv[1:]
    iters = int(args[args.index("--iters") + 1]) if "--iters" in args else 20
    nb = int(args[args.index("--bins") + 1]) if "--bins" in args else 32
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
        lk, gk = step_kernel(x, y, nb)
        lt, gt = step_torch(x, y, nb)
        rel = float((gk.double() - gt.double()).norm() / gt.double().norm())
        tk, mk = timed(step_kernel, x, y, nb, iters)
        tt, mt = timed(step_torch, x, y, nb, iters)
        print("B=%d %s bins=%d: kernels %.3f ms, %.0f MiB | stock torch fp32 %.3f ms, %.0f MiB | x%.1f | "
              "loss %.8f vs %.8f (|diff| %.2e), gradient rel-L2 %.2e"
              % (B, "x".join(map(str, VOL)), nb, tk, mk, tt, mt, tt / tk, lk.item(), lt.item(), abs(lk.item() - lt.item()), rel))
        del x, y, gk, gt
        torch.cuda.empty_cache()
    t_mi, t_ncc = table_build(dev, nb)
    print("adjoint table build (bins=%d): lr_mi_backward on 4 voxels %.2f us, lr_ncc_backward on 4 voxels %.2f us, "
          "difference %.2f us" % (nb, t_mi, t_ncc, t_mi - t_ncc))


if __name__ == "__main__":
    main()
