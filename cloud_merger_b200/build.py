"""Builds cloud_merger_b200/libcloud_merger_gpu.so (sm_100a only) with nvcc. In-tree, so the .so travels with the repo."""
from __future__ import annotations

import concurrent.futures as cf
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
LIB = os.path.join(HERE, "libcloud_merger_gpu.so")
SOURCES = ["cm_transform_crop.cu", "cm_voxel.cu", "cm_radix_sort.cu", "cm_zones.cu", "cm_outlier.cu", "cm_route.cu", "cm_plane.cu", "cm_statistical.cu", "cm_api.cu"]
HEADERS = ["cm_common.cuh", "cm_kernels.h", os.path.join("..", "..", "include", "cloud_merger_gpu.h")]

NVCC_FLAGS = [
    "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo",
    "--fmad=false",  # parity: PCL's CPU build has no FMA; the kernels also use __fmul_rn/__fadd_rn explicitly
    "-Xcompiler", "-fPIC", "-Xcompiler", "-ffp-contract=off",  # host side of the plane refit: no FMA either
     "-Xcompiler", "-fvisibility=hidden", "-Xptxas", "-v", "-Xcudafe", "--diag_suppress=177",
]


def _nvcc() -> str:
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def _stale(target: str, deps) -> bool:
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    os.makedirs(OBJ, exist_ok=True)
    nvcc = _nvcc()
    hdrs = [os.path.join(CSRC, h) for h in HEADERS] + [os.path.abspath(__file__)]
    jobs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s.replace(".cu", ".o"))
        if force or _stale(obj, [src] + hdrs):
            jobs.append((src, obj))

    def compile_one(job):
        src, obj = job
        cmd = [nvcc] + NVCC_FLAGS + ["-c", src, "-o", obj]
        r = subprocess.run(cmd, capture_output=True, text=True)
        with open(obj + ".log", "w") as f:
            f.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
        if r.returncode != 0:
            raise RuntimeError("nvcc failed for %s:\n%s%s" % (src, r.stdout, r.stderr))
        return r.stderr

    with cf.ThreadPoolExecutor(max_workers=4) as ex:
        for log in ex.map(compile_one, jobs):
            if verbose:
                print(log)
    objs = [os.path.join(OBJ, s.replace(".cu", ".o")) for s in SOURCES]
    if force or jobs or _stale(LIB, objs):
        cmd = [nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-cudart", "static", "-o", LIB] + objs + ["-ldl"]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("link failed:\n%s%s" % (r.stdout, r.stderr))
    return LIB


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
