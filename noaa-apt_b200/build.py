"""Builds libaptb200.so (CUDA kernels + C ABI) in-tree with nvcc for sm_100a.

The library is the product: every compute entry point lives in it and there is
no CPU fallback.  nvcc cross-compiles without a GPU, so this also runs on the
CPU-only build container.
"""
import glob
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libaptb200.so")

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "-Xcompiler", "-fPIC,-ffp-contract=off,-fno-fast-math,-Wall",
    "-cudart", "static",
    "-shared",
    # compress the sm_100a image (14 -> 3 MB of library); without this nvcc leaves an 8 MB image uncompressed
    "-Xfatbin", "-compress-all",
]


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")) + glob.glob(os.path.join(CSRC, "*.cpp")))


def _deps():
    return sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + glob.glob(os.path.join(CSRC, "*.hpp")) + \
        glob.glob(os.path.join(ROOT, "include", "*.h"))


def up_to_date():
    if not os.path.exists(LIB):
        return False
    t = os.path.getmtime(LIB)
    return all(os.path.getmtime(f) <= t for f in _deps())


def build_library(force=False, verbose=False, extra_flags=(), out=None):
    """out: build an experimental variant next to the product library (select it with APTB200_LIB=<path>)."""
    if out is None and not force and up_to_date():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + list(extra_flags) + ["-I", os.path.join(ROOT, "include"), "-I", CSRC, "-o", out or LIB] + sources()
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return out or LIB


if __name__ == "__main__":
    import sys
    build_library(force="-f" in sys.argv, verbose=True,
                  extra_flags=["-Xptxas", "-v"] if "-v" in sys.argv else [])
    print(LIB)
