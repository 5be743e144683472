"""Builds libgpp_b200.so (sm_100a only) in-tree with nvcc.  No JIT cache: the built library sits next to
this file so it travels with the repo snapshot to the GPU box."""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, "libgpp_b200.so")

# (source, extra flags).  gram.cu / gn.cu: no FMA contraction, the oracle's multiply/add order is kept.
SOURCES = [
    ("gemm_dmma.cu", []),
    ("chol.cu", []),
    ("gram.cu", ["-fmad=false"]),
    ("gn.cu", ["-fmad=false"]),
    ("capi.cu", []),
    ("dist.cu", []),
    ("predvar.cu", []),
]
ARCH = ["-gencode", "arch=compute_100a,code=sm_100a"]
COMMON = ["-O3", "-std=c++17", "-lineinfo", "-Xcompiler", "-fPIC"]


def _nvcc():
    nv = shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"
    if not os.path.exists(nv):
        raise RuntimeError("nvcc not found")
    return nv


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nv = _nvcc()
    objdir = os.path.join(HERE, "build")
    os.makedirs(objdir, exist_ok=True)
    headers = [os.path.join(CSRC, "gpp_internal.cuh"), os.path.join(HERE, "..", "include", "gpp.h"), __file__]
    objs = []
    for src, extra in SOURCES:
        s = os.path.join(CSRC, src)
        if not os.path.exists(s):
            continue
        o = os.path.join(objdir, src.replace(".cu", ".o"))
        objs.append(o)
        if force or _stale(o, [s] + headers):
            cmd = [nv] + ARCH + COMMON + extra + ["-c", s, "-o", o]
            if verbose:
                print(" ".join(cmd))
            subprocess.run(cmd, check=True)
    if force or _stale(LIB, objs):
        cmd = [nv] + ARCH + ["-shared", "-o", LIB] + objs + (["-lnccl"] if any(o.endswith("dist.o") for o in objs) else [])
        if verbose:
            print(" ".join(cmd))
        subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
