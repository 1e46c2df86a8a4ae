"""Build csrc/libnnmpc.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

    python -m industrial_nnmpc_2021_b200.build [--force] [--verbose]
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(CSRC, "libnnmpc.so")
SOURCES = ["qp.cu", "ts.cu", "sim.cu", "mlp.cu", "gemm_bench.cu", "lp.cu", "oz.cu", "online.cu", "ipm.cu"]
HEADERS = ["gemm_f64.cuh", "nnmpc_common.cuh", "qp.cuh", "ts.cuh", "lp.cuh", "lp_gemm.cuh", "lp_iter.cuh", "oz.cuh", "oz_gemm.cuh", "mlp_tc.cuh", os.path.join("..", "..", "include", "nnmpc.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC", "-Xcompiler", "-O3", "--use_fast_math=false"]


def find_nvcc():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (needed to build libnnmpc.so)")


def _stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, s) for s in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False, out=None, defines=()):
    """Default: csrc/libnnmpc.so.  `out` + `defines` build an experimental variant next to it (e.g.
    defines=("NNMPC_EPI_WARPS=16",), out="libnnmpc_e16.so"), loaded when NNMPC_LIB_PATH points at it."""
    variant = out is not None
    lib = os.path.join(CSRC, out) if variant else LIB
    if not variant and not force and not _stale():
        return LIB
    nvcc = find_nvcc()
    flags = [f for f in NVCC_FLAGS if not f.startswith("--use_fast_math")] + [f"-D{d}" for d in defines]
    if verbose:
        flags += ["-Xptxas", "-v"]
    objs = []
    procs = []
    tag = ("." + os.path.splitext(out)[0]) if variant else ""
    for s in SOURCES:
        o = os.path.join(CSRC, s.replace(".cu", tag + ".o"))
        objs.append(o)
        cmd = [nvcc] + flags + ["-c", os.path.join(CSRC, s), "-o", o]
        procs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
    for cmd, p in procs:
        out, _ = p.communicate()
        if verbose or p.returncode:
            print(" ".join(cmd))
            print(out)
        if p.returncode:
            raise RuntimeError("nvcc failed")
    cmd = [nvcc, "-shared", "-o", lib] + objs + ["-gencode", "arch=compute_100a,code=sm_100a", "-lcudart"]
    subprocess.run(cmd, check=True)
    return lib


if __name__ == "__main__":
    kw = {}
    if "--out" in sys.argv:
        kw["out"] = sys.argv[sys.argv.index("--out") + 1]
        kw["defines"] = tuple(a[2:] for a in sys.argv if a.startswith("-D"))
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv, **kw))
