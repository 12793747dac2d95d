"""Builds libb200rt.so (the C-ABI library of include/b200rt.h) in-tree with nvcc for sm_100a.

    python sycl-ray-tracing_b200/build.py [--force] [--verbose]

-fmad=false: the device code is written so that every float expression is evaluated as written (see
csrc/pt_device.cuh); fused multiply-adds are requested explicitly where they are wanted.
"""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
LIB = os.path.join(HERE, os.environ.get("B200RT_BUILD_LIB", "libb200rt.so"))
SOURCES = ["capi.cu", "kernels.cu", "wavefront.cu", "persist.cu", "env_tables.cu", "denoise.cu", "bvh_build_gpu.cu", "refit.cu", "bvh_build.cpp", "obj_ingest.cpp", "hdr_ingest.cpp"]
HEADERS = ["bvh_build.h", "bvh_emit.cuh", "device_types.h", "kernels.h", "pt_device.cuh", "wf_device.cuh", "obj_ingest.h", os.path.join("..", "..", "include", "b200rt.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-lineinfo",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-fmad=false",
] + (["-DB200RT_PREFETCH"] if os.environ.get("B200RT_BUILD_PREFETCH") else []) + os.environ.get("B200RT_BUILD_DEFS", "").split() + [
    "-Xcompiler", "-fPIC,-fopenmp,-O3",
    "-ccbin", "/usr/bin/g++",
]


def _stale() -> bool:
    if not os.path.exists(LIB):
        return True
    t = os.path.getmtime(LIB)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not _stale():
        return LIB
    objs = []
    objdir = os.path.join(CSRC, "_obj_" + os.path.splitext(os.path.basename(LIB))[0])
    os.makedirs(objdir, exist_ok=True)
    for src in SOURCES:
        obj = os.path.join(objdir, os.path.splitext(src)[0] + ".o")
        cmd = ["nvcc"] + NVCC_FLAGS + (["-Xptxas", "-v"] if verbose else []) + ["-c", os.path.join(CSRC, src), "-o", obj]
        if verbose:
            print(" ".join(cmd), flush=True)
        subprocess.run(cmd, check=True)
        objs.append(obj)
    cmd = ["nvcc", "-shared", "-ccbin", "/usr/bin/g++", "-Xcompiler", "-fopenmp", "-o", LIB] + objs + ["-lgomp"]
    if verbose:
        print(" ".join(cmd), flush=True)
    subprocess.run(cmd, check=True)
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
