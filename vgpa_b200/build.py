"""
Build libvgpa_b200.so (the sm_100a CUDA kernels + the C ABI) in-tree with nvcc.

    python -m vgpa_b200.build [--force] [--verbose]

The shared library lands next to this file so that it travels with the repo
snapshot to the GPU box (it is git-ignored, not gpurun-ignored).
"""
import os
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
LIB = PKG / "libvgpa_b200.so"
SOURCES = ["api.cu", "small_dim.cu", "l63_lanes.cu", "l96_sweeps.cu", "l96_energy.cu", "vecops.cu", "hyper.cu", "init.cu",
           "datagen.cu", "l96_dyn.cu"]
HEADERS = ["common.cuh", "ptx.cuh", "l63_grad.cuh", "../../include/vgpa_b200.h"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O2"]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.sep not in cand or os.path.exists(cand)):
            return cand
    raise RuntimeError("nvcc not found")


def _stale(target, deps):
    if not target.exists():
        return True
    t = target.stat().st_mtime
    return any((CSRC / d).resolve().stat().st_mtime > t for d in deps)


def build_library(force=False, verbose=False):
    """Compile every .cu for sm_100a and link the shared library."""
    objdir = PKG / "build"
    objdir.mkdir(exist_ok=True)
    nvcc = _nvcc()
    objs = []
    procs = []
    for src in SOURCES:
        obj = objdir / (src.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, [src] + HEADERS):
            cmd = [nvcc, *NVCC_FLAGS, "-c", str(CSRC / src), "-o", str(obj)]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
                print(" ".join(cmd), flush=True)
            procs.append((src, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    failed = False
    for src, pr in procs:
        out, _ = pr.communicate()
        if pr.returncode != 0 or verbose:
            print(f"--- {src} ---\n{out}", flush=True)
        failed |= pr.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    if force or procs or not LIB.exists():
        cmd = [nvcc, "-shared", "-o", str(LIB), *map(str, objs), "-gencode", "arch=compute_100a,code=sm_100a"]
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    build_library(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(LIB)
