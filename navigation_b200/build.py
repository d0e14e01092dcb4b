"""Builds navigation_b200/libnavgpu.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
import glob
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libnavgpu.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-O3", "-lineinfo", "-std=c++17",
    # fp64 geometry and cost sums must round exactly like the reference's x86-64 code: no FMA contraction
    "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared",
]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = (sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.inc")) +
            glob.glob(os.path.join(HERE, "..", "include", "*.h")))
    return any(os.path.getmtime(p) > t for p in deps)


def build(force=False, verbose=False, out=LIB):
    """Compiles the library to `out` (in-tree by default, where it is only rebuilt when a source is newer)."""
    if out == LIB and not force and not needs_build():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", out] + sources()
    subprocess.check_call(cmd)
    return out


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
