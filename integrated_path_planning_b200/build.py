"""In-tree build of libfot.so for sm_100a (nvcc cross-compiles without a GPU)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
SRC = os.path.join(HERE, "csrc", "fot_api.cu")
DEPS = [SRC, os.path.join(HERE, "csrc", "fot_kernels.cuh"), os.path.join(HERE, "csrc", "fot_device.cuh"),
        os.path.join(HERE, "csrc", "fot_sweep_items.cuh"), os.path.join(HERE, "csrc", "fot_sweep_pairs.cuh"),
        os.path.join(HERE, "csrc", "fot_sweep_math.cuh"),
        os.path.join(HERE, "csrc", "fot_predict.cuh"), os.path.join(HERE, "csrc", "fot_frenet.cuh"),
        os.path.join(HERE, "csrc", "fot_rank.cuh"), os.path.join(HERE, "csrc", "fot_weights.cuh"),
        os.path.join(HERE, "csrc", "fot_assess.cuh"), os.path.join(HERE, "csrc", "fot_assess_cand.cuh"),
        os.path.join(ROOT, "include", "fot.h")]
OUT = os.path.join(HERE, "libfot.so")

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    # reference-order fp64: no implicit FMA contraction; fused ops are written out as fma()
    "-fmad=false",
    "-Xcompiler", "-fPIC", "-shared",
]


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and os.path.exists(OUT) and all(os.path.getmtime(OUT) >= os.path.getmtime(d) for d in DEPS):
        return OUT
    nvcc = os.environ.get("NVCC", "nvcc")
    cmd = [nvcc, *NVCC_FLAGS, "-I", os.path.join(ROOT, "include"), "-o", OUT, SRC]
    if verbose:
        cmd.insert(1, "-Xptxas=-v")
    proc = subprocess.run(cmd, capture_output=True, text=True)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + proc.stdout + proc.stderr)
    if verbose:
        print(proc.stderr)
    return OUT


if __name__ == "__main__":
    print(build_library(force="--force" in sys.argv, verbose="-v" in sys.argv))
