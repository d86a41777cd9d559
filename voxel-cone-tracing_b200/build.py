"""Builds lib/libvct_b200.so from csrc/*.cu with nvcc for sm_100a (in-tree; the .so travels to the GPU box).

    python voxel-cone-tracing_b200/build.py [--force] [--verbose]

--fmad=false is deliberate: coverage, depth-slice and shadow-compare decisions must be bit-identical
to the CPU oracle, so no float expression may be contracted into an FMA (DESIGN.md "Defined semantics").
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIBDIR = os.path.join(HERE, "lib")
LIB = os.path.join(LIBDIR, "libvct_b200.so")
SOURCES = ["vct_api.cu", "vct_shadow.cu", "vct_voxelize.cu", "vct_mip.cu", "vct_cone.cu", "vct_comm.cu", "vct_view.cu"]
HEADERS = ["vct_internal.h", "vct_raster.cuh", os.path.join("..", "..", "include", "vct_c_api.h")]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "--fmad=false", "-std=c++17",
              "-Xcompiler", "-fPIC,-O2", "--expt-relaxed-constexpr", "-cudart", "static"]


def nvcc():
    return shutil.which("nvcc") or "/usr/local/cuda/bin/nvcc"


def up_to_date():
    if not os.path.exists(LIB):
        return False
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return all(os.path.getmtime(d) <= t for d in deps)


def build(force=False, verbose=False):
    if not force and up_to_date():
        return LIB
    os.makedirs(LIBDIR, exist_ok=True)
    objs = []
    procs = []
    for s in SOURCES:
        o = os.path.join(LIBDIR, s.replace(".cu", ".o"))
        cmd = [nvcc(), *NVCC_FLAGS, "-c", os.path.join(CSRC, s), "-o", o]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
            print(" ".join(cmd))
        procs.append((s, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(o)
    failed = False
    for s, p in procs:
        out, _ = p.communicate()
        if p.returncode != 0 or verbose:
            print(f"--- {s}\n{out}")
        failed |= p.returncode != 0
    if failed:
        raise RuntimeError("nvcc failed")
    cmd = [nvcc(), "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static",
           "-Xcompiler", "-fPIC", "-Xlinker", "--version-script=" + os.path.join(CSRC, "exports.map"),
           "-o", LIB, *objs]
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
