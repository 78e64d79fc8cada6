"""Builds libmpcb200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python mpc-rl_for_avs_b200/build.py [--force] [--verbose]

mpc_prepare.cu is compiled with -fmad=false (its FP64 predicates must round exactly like the numpy
oracle), mpc_sens.cu too (its FP64 linear algebra stays within rounding of the host build's); everything else
with default FMA contraction.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, os.environ.get("MPC_LIB_NAME", "libmpcb200.so"))      # MPC_LIB_NAME / MPC_BUILD_DEFS: A/B experiment builds only
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC", "-Xcompiler", "-fvisibility=hidden",
          "--expt-relaxed-constexpr"]
UNITS = [("mpc_solve.cu", []), ("mpc_prepare.cu", ["-fmad=false"]), ("mpc_capi.cu", []), ("mpc_env.cu", []), ("mpc_kkt.cu", []),
         ("mpc_sens.cu", ["-fmad=false"])]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libmpcb200.so for sm_100a)")


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(HERE, "..", "include", "mpc_b200.h"), __file__]
    return any(os.path.getmtime(d) > t for d in deps if os.path.exists(d))


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    nvcc = _nvcc()
    objdir = os.path.join(HERE, "build", os.path.basename(LIB))
    os.makedirs(objdir, exist_ok=True)
    objs = []
    for src, extra in UNITS:
        obj = os.path.join(objdir, src.replace(".cu", ".o"))
        cmd = [nvcc, *ARCH, *COMMON, *extra, *os.environ.get("MPC_BUILD_DEFS", "").split(), "-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            cmd.insert(1, "-Xptxas")
            cmd.insert(2, "-v")
            print(" ".join(cmd), flush=True)
        subprocess.check_call(cmd)
        objs.append(obj)
    cmd = [nvcc, *ARCH, "-shared", "-o", LIB, *objs]
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
