"""Build recipe for libacsolver_b200.so (hand-written CUDA for sm_100a behind a C ABI).

``python -m ac_solver_b200.build`` or ``build()``; nvcc cross-compiles without a GPU.  The
library is built IN-TREE (ac_solver_b200/libacsolver_b200.so, git-ignored) so that it
travels with the repo snapshot to the GPU box.
"""

from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libacsolver_b200.so")
SOURCES = ["capi.cu", "moves_kernel.cu", "generic_kernel.cu", "greedy.cu", "sbfs.cu", "pbfs.cu", "mbfs.cu", "beam.cu", "goalset.cu", "sym.cu", "ball.cu", "ppo_kernels.cu"]
NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared",
]


def _nvcc() -> str:
    for cand in (shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found: cannot build libacsolver_b200.so")


def is_stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [
        os.path.join(HERE, "..", "include", "acsolver_b200.h")
    ]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not is_stale():
        return LIB
    srcs = [os.path.join(CSRC, s) for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]
    extra = os.environ.get("ACS_NVCC_EXTRA", "").split()  # e.g. -DPB_UNROLL=1 for kernel experiments
    cmd = [_nvcc(), *NVCC_FLAGS, *extra, "-o", LIB, *srcs]
    if verbose:
        cmd.insert(1, "-Xptxas")
        cmd.insert(2, "-v")
        print(" ".join(cmd))
    env = dict(os.environ)
    env.pop("CC", None)  # the image exports a gcc wrapper that nvcc must not pick up
    env.pop("CXX", None)
    subprocess.check_call(cmd, env=env)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
