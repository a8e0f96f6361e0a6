"""Builds eggshell_b200/libeggshell_b200.so for sm_100a with nvcc (in-tree, no JIT cache).

egg_collide.cu is compiled with -fmad=false: its threshold comparisons must see the same FP64
values as the CPU arithmetic (see the file header); the solver kernels keep FMA contraction.
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libeggshell_b200.so")
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = (["-DEGG_STREAM_CHECKS"] if os.environ.get("EGG_STREAM_CHECKS") else []) + (["-DEGG_DENSE_TIMING"] if os.environ.get("EGG_DENSE_TIMING") else []) + ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "--expt-relaxed-constexpr"]
UNITS = [
    ("egg_collide.cu", ["-fmad=false"]),
    ("egg_solve.cu", []),
    ("egg_pgs.cu", []),
    ("egg_iter.cu", []),
    ("egg_pgs_stream.cu", []),
    ("egg_pgs_runs.cu", []),
    ("egg_dense.cu", ["-fmad=false"]),
    ("egg_mppi.cu", []),
    ("egg_capi.cu", []),
]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    hdrs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    hdrs.append(os.path.join(HERE, "..", "include", "egg_cuda.h"))
    hdrs.append(os.path.abspath(__file__))
    objs = []
    os.makedirs(os.path.join(HERE, "build"), exist_ok=True)
    for src, extra in UNITS:
        s = os.path.join(CSRC, src)
        o = os.path.join(HERE, "build", src.replace(".cu", ".o"))
        if force or _stale(o, [s] + hdrs):
            cmd = [nvcc] + ARCH + COMMON + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd), flush=True)
            subprocess.check_call(cmd)
        objs.append(o)
    if force or _stale(OUT, objs):
        cmd = [nvcc] + ARCH + ["-shared", "-o", OUT] + objs + ["-lcudart"]
        subprocess.check_call(cmd)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
