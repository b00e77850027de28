"""Builds the C-ABI CUDA library in-tree (diffsinger_b200/lib/libdsx.so) with nvcc for sm_100a.

    python diffsinger_b200/build.py            # incremental (skips when sources are older than the .so)
    python diffsinger_b200/build.py --force
"""
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = [os.path.join(HERE, "csrc", f) for f in ("dsx_api.cu", "dsx_simt.cu", "dsx_tc.cu", "dsx_stack.cu", "dsx_selftest.cu")]
HDR = [os.path.join(HERE, "csrc", f) for f in ("dsx_internal.h", "dsx_ptx.cuh", "dsx_rng.cuh", "dsx_tc_common.cuh",
                                                  "dsx_update.cuh")] + \
      [os.path.join(os.path.dirname(HERE), "include", "dsx.h")]
LIB = os.path.join(HERE, "lib", "libdsx.so")
NVCC_FLAGS = ["-std=c++17", "-O3", "-lineinfo", "-gencode", "arch=compute_100a,code=sm_100a",
              "-Xcompiler", "-fPIC", "-shared"]


def nvcc_path():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if c and (os.path.sep not in c or os.path.exists(c)):
            return c
    return "nvcc"


def up_to_date():
    if not os.path.exists(LIB):
        return False
    t = os.path.getmtime(LIB)
    return all(os.path.getmtime(f) <= t for f in SRC + HDR)


def build(force=False, verbose=False):
    if not force and up_to_date():
        return LIB
    os.makedirs(os.path.dirname(LIB), exist_ok=True)
    cmd = [nvcc_path()] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-o", LIB] + SRC
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + " ".join(cmd) + "\n" + r.stdout + r.stderr)
    if verbose:
        print(r.stderr)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
