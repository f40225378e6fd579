"""Builds libraytrace_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU)."""
from __future__ import annotations

import os
import shutil
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OUT = os.path.join(HERE, "libraytrace_b200.so")
SOURCES = ["rt_api.cu"]
HEADERS = ["rt_device.cuh", "rt_kernels.cuh", "rt_cull_tc.cuh", "rt_bvh_build.cuh", "rt_scene_build.cuh", os.path.join("..", "..", "include", "raytrace_b200.h")]

NVCC_FLAGS = (["-DRT_TAIL_DIAG"] if os.environ.get("RT_TAIL_DIAG") else []) + [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC", "-shared", "-Xptxas", "-v",
]


def _nvcc():
    for c in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if c and os.path.exists(c):
            return c
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(OUT):
        return True
    t = os.path.getmtime(OUT)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.abspath(__file__)]
    return any(os.path.getmtime(d) > t for d in deps)


def build_library(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return OUT
    cmd = [_nvcc()] + NVCC_FLAGS + ["-ccbin", "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"]
    cmd += ["-o", OUT] + [os.path.join(CSRC, f) for f in SOURCES] + ["-ldl"]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    log = os.path.join(HERE, "csrc", "build.log")
    with open(log, "w") as f:
        f.write(" ".join(cmd) + "\n" + res.stdout)
    if verbose or res.returncode != 0:
        print(res.stdout)
    if res.returncode != 0:
        raise RuntimeError(f"nvcc failed ({res.returncode}); see {log}")
    return OUT


if __name__ == "__main__":
    print(build_library(force=True, verbose=True))
