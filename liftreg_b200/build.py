"""Builds libliftreg_b200.so in-tree with nvcc for sm_100a (no torch headers, no JIT cache).

    python -m liftreg_b200.build [--force] [--verbose]

The .so lands in liftreg_b200/_lib/ (git-ignored; travels to the GPU box with the gpurun snapshot).
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB_DIR = os.path.join(HERE, "_lib")
LIB_PATH = os.path.join(LIB_DIR, "libliftreg_b200.so")
SOURCES = ["api.cu", "warp.cu", "backproject.cu", "drr.cu", "pca_decode.cu", "losses.cu", "surface.cu", "probe.cu"]
HEADERS = [os.path.join(CSRC, "common.cuh"), os.path.join(os.path.dirname(HERE), "include", "liftreg_b200.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    "--fmad=false",            # no implicit FMA contraction anywhere: every fused op in the kernels is explicit
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-O2",
    "-Xptxas", "-v",
    "--shared", "-cudart", "static",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.exists(cand) or not os.path.isabs(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, s) for s in SOURCES] + HEADERS + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_variant(name, defines):
    """Kernel experiments: compile with extra -D flags into _lib/variants/<name>.so (use via LIFTREG_B200_LIB)."""
    out = os.path.join(LIB_DIR, "variants", name + ".so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    env = dict(os.environ)
    env.pop("CC", None)
    env.pop("CXX", None)
    cmd = [_nvcc()] + NVCC_FLAGS + ["-D" + d for d in defines] + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", out]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + res.stdout + res.stderr)
    return out


def build(force=False, verbose=False):
    """Compile every CUDA source into one shared library. Returns the path."""
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    env = dict(os.environ)
    env.pop("CC", None)   # this image exports CC=/opt/gcc/bin/gcc; let nvcc pick the system g++
    env.pop("CXX", None)
    cmd = [_nvcc()] + NVCC_FLAGS + [os.path.join(CSRC, s) for s in SOURCES] + ["-o", LIB_PATH + ".tmp"]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    log = res.stdout + res.stderr
    with open(os.path.join(LIB_DIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log)
    os.replace(LIB_PATH + ".tmp", LIB_PATH)
    if verbose:
        print(log)
    return LIB_PATH


if __name__ == "__main__":
    if "--variant" in sys.argv:          # python -m liftreg_b200.build --variant NAME [DEFINE=VALUE ...]
        k = sys.argv.index("--variant")
        print(build_variant(sys.argv[k + 1], sys.argv[k + 2:]))
        sys.exit(0)
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
