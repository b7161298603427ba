"""Compile librtgrff_b200.so for sm_100a with nvcc (in-tree; the .so travels to the GPU box).

    python -m raytracinggrff_b200.build [--force]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys
from pathlib import Path

PKG = Path(__file__).resolve().parent
CSRC = PKG / "csrc"
OUT = PKG / "librtgrff_b200.so"

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-shared"]


def cuda_tool(name):
    """A CUDA toolkit program (nvcc, cuobjdump): from PATH, else from $CUDA_HOME/bin (default /usr/local/cuda),
    so that a shell whose PATH lacks the toolkit still builds."""
    return shutil.which(name) or str(Path(os.environ.get("CUDA_HOME") or "/usr/local/cuda") / "bin" / name)


def build_library(force=False, verbose=False):
    srcs = sorted(CSRC.glob("*.cu")) + sorted(CSRC.glob("*.cuh")) + [PKG.parent / "include" / "rtgrff.h"]
    if not force and OUT.exists() and all(s.stat().st_mtime <= OUT.stat().st_mtime for s in srcs):
        return OUT
    cmd = [cuda_tool("nvcc"), *NVCC_FLAGS, "-o", str(OUT), str(CSRC / "rtgrff_api.cu")]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    res = subprocess.run(cmd, capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed:\n{' '.join(cmd)}\n{res.stdout}\n{res.stderr}")
    if verbose:
        print(res.stderr)
    return OUT


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
