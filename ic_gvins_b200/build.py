"""Build libicgvins_b200.so (all CUDA kernels + the C ABI) in-tree with nvcc for sm_100a.

Usage:  python -m ic_gvins_b200.build   (or __graft_entry__.build())
nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the gpurun snapshot.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libicgvins_b200.so")

ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-lineinfo", "-std=c++17", "-Xcompiler", "-fPIC", "-Xcompiler", "-Wall", "-Xcompiler", "-Wno-unused-function"]
# per-file extra flags: the image-path kernels must reproduce the reference library's float sequence (no FMA contraction)
LINK_LIBS: list[str] = ["-ldl", "-lpthread"]  # cudart is linked statically (nvcc default) and needs both
SOURCES = {
    "common.cu": [],
    "klt.cu": ["-fmad=false"],
    "detect.cu": ["-fmad=false"],
    "clahe.cu": ["-fmad=false"],
    "camera.cu": ["-fmad=false"],
    "fundamental.cu": ["-fmad=false"],  # host code; no contraction of the reference's double sequence
    "geom.cu": ["-fmad=false"],         # device versions of the camera model / RANSAC gate / triangulation / IMU propagation (same cores)
    "ba.cu": [],
    "ba_cull.cu": ["-fmad=false"],      # post-solve outlier culling: the float cast in cam2pixel makes its decisions sensitive to contraction
}


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.isabs(c) and os.path.exists(c) or not os.path.isabs(c)):
            return c
    raise RuntimeError("nvcc not found")


def _stale(out: str, deps: list[str]) -> bool:
    if not os.path.exists(out):
        return True
    t = os.path.getmtime(out)
    return any(os.path.getmtime(d) > t for d in deps)


def build(verbose: bool = False, force: bool = False, prof: bool = False) -> str:
    """prof=True builds libicgvins_b200_prof.so beside the product library: same sources with -DICG_BA_PHASE_CLOCKS (in-kernel phase clocks of
    ba_solve / ba_lin_cam; the instrumentation perturbs register allocation, so it never goes into the product build)."""
    nvcc = _nvcc()
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".hpp"))]
    headers.append(os.path.join(HERE, "..", "include", "icgvins_b200.h"))
    objs = []
    lib = LIB.replace(".so", "_prof.so") if prof else LIB
    for src, extra in SOURCES.items():
        path = os.path.join(CSRC, src)
        if not os.path.exists(path):
            continue
        obj = os.path.join(CSRC, src.replace(".cu", "_prof.o" if prof else ".o"))
        if force or _stale(obj, [path] + headers):
            cmd = [nvcc] + ARCH + COMMON + extra + (["-DICG_BA_PHASE_CLOCKS"] if prof else []) + (["-Xptxas", "-v"] if verbose else []) + ["-c", path, "-o", obj]
            if verbose:
                print(" ".join(cmd))
            subprocess.run(cmd, check=True)
        objs.append(obj)
    if force or _stale(lib, objs):
        cmd = [nvcc] + ARCH + ["-shared", "-o", lib] + objs + LINK_LIBS
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
    return lib


if __name__ == "__main__":
    print(build(verbose="-v" in sys.argv, force="-f" in sys.argv, prof="--prof" in sys.argv))
