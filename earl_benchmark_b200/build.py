"""Compile the CUDA library IN-TREE for sm_100a:  earl_benchmark_b200/libearl_b200.so

    python -m earl_benchmark_b200.build [--force] [--verbose]

Translation units: the tabletop step and its three-object variant (bit-exact fp64 arithmetic, so no FMA contraction), the articulated-body engine
of the Sawyer tasks (fp32, FMA on) once per compile-time capacity set: the primary set that exports the earl_mj_* entry
points (earl_mj.cu) and the extra-large set of its redo pass (earl_mj_xl.cu); the kitchen engine likewise
(earl_mj_kitchen.cu, earl_mj_kitchen_xl.cu).  The .so is git-ignored but travels to the GPU box with the repo snapshot.
"""
import os
import subprocess
import sys

PKG = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG, "csrc")
INCLUDE = os.path.join(os.path.dirname(PKG), "include")
LIB = os.path.join(PKG, "libearl_b200.so")
OBJDIR = os.path.join(PKG, "build")
# (source, extra flags)
MJ_EXTRA = os.environ.get("EARL_MJ_EXTRA_FLAGS", "").split()  # profiling / trace builds (-DMJ_PHASE_TIMING, -DMJ_TRACE_DEVICE)
UNITS = [("earl_b200.cu", ["--fmad=false"]), ("earl_tt3.cu", ["--fmad=false"]), ("earl_mj.cu", MJ_EXTRA), ("earl_mj_xl.cu", MJ_EXTRA),
         ("earl_mj_kitchen.cu", MJ_EXTRA), ("earl_mj_kitchen_xl.cu", MJ_EXTRA)]
SOURCES = [os.path.join(CSRC, u[0]) for u in UNITS]
DEPS = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(INCLUDE, f) for f in os.listdir(INCLUDE)]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-O2,-fvisibility=hidden",
]


def stale():
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force=False, verbose=False):
    if not force and not stale():
        return LIB
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    os.makedirs(OBJDIR, exist_ok=True)
    objs, procs = [], []
    for src, extra in UNITS:
        obj = os.path.join(OBJDIR, src.replace(".cu", ".o"))
        cmd = [nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, os.path.join(CSRC, src)]
        if verbose:
            print(" ".join(cmd))
        procs.append((cmd, subprocess.Popen(cmd)))
        objs.append(obj)
    for cmd, p in procs:
        if p.wait() != 0:
            raise subprocess.CalledProcessError(p.returncode, cmd)
    cmd = [nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-o", LIB] + objs
    if verbose:
        print(" ".join(cmd))
    subprocess.check_call(cmd)
    return LIB


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose="--verbose" in sys.argv)
    print(LIB)
