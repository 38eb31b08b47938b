"""Compile csrc/dvc_b200.cu into libdvc_b200.so (in-tree, next to this file) with nvcc for sm_100a."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "csrc", "dvc_b200.cu")
LIB = os.path.join(HERE, "libdvc_b200.so")
DEPS = [os.path.join(HERE, "csrc", f) for f in os.listdir(os.path.join(HERE, "csrc"))] + [
    os.path.join(os.path.dirname(HERE), "include", "dvc_b200.h")]

# -ffp-contract=off: host-side constants (the Farneback taps and Gram inverse) must round each operation as OpenCV does,
# also on hosts whose compiler would otherwise fuse multiply-adds.
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC,-ffp-contract=off", "--threads", "2"]


def find_nvcc() -> str:
    nvcc = shutil.which("nvcc") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "nvcc")
    if not os.path.exists(nvcc):
        raise RuntimeError("nvcc not found: cannot build libdvc_b200.so")
    return nvcc


def is_stale(lib: str = LIB) -> bool:
    if not os.path.exists(lib):
        return True
    t = os.path.getmtime(lib)
    return any(os.path.getmtime(d) > t for d in DEPS if os.path.exists(d))


LIB_MEASURE = os.path.join(HERE, "libdvc_b200_measure.so")


def build(force: bool = False, verbose: bool = False, measure: bool = False) -> str:
    """measure=True builds the -DDVC_MEASURE flavour (environment switches for A/B runs: tools/ and the gray-variant test)
    next to the product."""
    lib = LIB_MEASURE if measure else LIB
    if not force and not is_stale(lib):
        return lib
    cmd = [find_nvcc()] + NVCC_FLAGS + (["-DDVC_MEASURE"] if measure else []) + (["-Xptxas", "-v"] if verbose else []) + ["-o", lib, SRC]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + r.stdout + r.stderr)
    if verbose:
        sys.stderr.write(r.stderr)
    return lib


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv, measure="--measure" in sys.argv))
