"""Builds libdigb200.so (the sm_100a kernels + C ABI) in-tree with nvcc.

Run as ``python -m digdriver_b200.build`` or through ``__graft_entry__.build()``.
nvcc cross-compiles without a GPU, so this works in the CPU-only build container; the
resulting .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
import glob
import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_PATH = os.path.join(PKG_DIR, "libdigb200.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC",
    "-shared",
]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(
        os.path.join(PKG_DIR, "..", "include", "*.h"))
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force=False, verbose=False, extra_flags=(), out_path=None):
    """extra_flags / out_path: developer builds beside the product library (e.g. -DDIG_LB_TIMING)."""
    if out_path is not None:
        nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
        cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + ["-o", out_path] + sources()
        res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
        if res.returncode != 0:
            sys.stderr.write(res.stdout)
            raise RuntimeError("nvcc failed (%d)" % res.returncode)
        return out_path
    if not force and not needs_build():
        return LIB_PATH
    nvcc = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found; libdigb200.so cannot be built")
    cmd = [nvcc] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB_PATH] + sources()
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed (%d)" % res.returncode)
    return LIB_PATH


if __name__ == "__main__":
    if "--timing" in sys.argv:
        print(build_library(extra_flags=["-DDIG_LB_TIMING"], out_path=os.path.join(PKG_DIR, "libdigb200_timing.so")))
    else:
        print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
