"""Builds liboz_b200.so (hand-written sm_100a CUDA + the C-ABI) in-tree with nvcc."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
SO = os.path.join(HERE, "liboz_b200.so")
SOURCES = ["oz_rules.cu", "oz_tree.cu", "oz_net.cu", "oz_capi.cu", "oz_dist.cu", "oz_solve.cu"]


def nvcc_path() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def stale() -> bool:
    if os.environ.get("OZ_B200_LIB"):
        return False  # an explicitly selected prebuilt library is used as is
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".h"))]
    deps.append(os.path.join(HERE, "..", "include", "oz_b200.h"))
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not stale():
        return SO
    cmd = [nvcc_path(), "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
           "-Xcompiler", "-fPIC", "-shared", "-cudart", "static", "-o", SO] + SOURCES + ["-ldl"]
    if verbose:
        cmd[1:1] = ["-Xptxas", "-v"]
    subprocess.check_call(cmd, cwd=CSRC)
    return SO


if __name__ == "__main__":
    import sys
    print(build(force=True, verbose="-v" in sys.argv))
