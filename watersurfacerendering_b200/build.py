"""Build libwsocean.so (the C-ABI CUDA library) in-tree with nvcc for sm_100a.

    python -m watersurfacerendering_b200.build [--force] [--verbose]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels with the repo snapshot.
"""
from __future__ import annotations

import os
import shutil
import subprocess
import sys

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(PKG_DIR)
CSRC = os.path.join(PKG_DIR, "csrc")
INCLUDE = os.path.join(ROOT, "include")
LIB_PATH = os.path.join(PKG_DIR, "libwsocean.so")

SOURCES = ["wso_kernels.cu", "wso_kernels2.cu", "wso_slab_kernels.cu", "wso_prepare_kernels.cu", "wso_query_kernels.cu",
           "wso_api.cu", "wso_slab.cu", "wso_host_prepare.cpp"]
HEADERS = ["wso_device.cuh", "wso_kernels.cuh", "wso_kernels2.cuh", "wso_simt.cuh", "wso_launch.h", "wso_host_prepare.h",
           "wso_query.cuh"]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo", "-O3", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden,-ffp-contract=off,-O2",
    "-Xptxas", "-v",
    "--shared", "-cudart", "static", "--threads", "0",
]


def _nvcc() -> str:
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", shutil.which("nvcc")):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found")


def needs_build() -> bool:
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(INCLUDE, "wsocean.h")]
    return any(os.path.exists(d) and os.path.getmtime(d) > t for d in deps)


def build(force: bool = False, verbose: bool = False) -> str:
    if not force and not needs_build():
        return LIB_PATH
    srcs = [os.path.join(CSRC, s) for s in SOURCES]
    if not all(os.path.exists(s) for s in srcs):
        if os.path.exists(LIB_PATH):
            return LIB_PATH
        raise RuntimeError("CUDA sources missing and no prebuilt libwsocean.so")
    cmd = [_nvcc(), *NVCC_FLAGS, "-ccbin", "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++",
           "-I", CSRC, "-I", INCLUDE, "-o", LIB_PATH, *srcs]
    res = subprocess.run(cmd, capture_output=True, text=True)
    log = res.stdout + res.stderr
    with open(os.path.join(PKG_DIR, "build.log"), "w") as f:
        f.write(" ".join(cmd) + "\n" + log)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed:\n" + log[-6000:])
    if verbose:
        print(log)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="--verbose" in sys.argv))
