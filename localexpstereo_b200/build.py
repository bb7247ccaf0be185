"""Builds the CUDA extension in-tree: localexpstereo_b200/liblexp_cuda.so (sm_100a only)."""
from __future__ import annotations

import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "liblexp_cuda.so")
SRCS = [os.path.join(HERE, "csrc", "lexp_capi.cu")]
DEPS = SRCS + [os.path.join(HERE, "csrc", "lexp_kernels.cuh"), os.path.join(HERE, "csrc", "lexp_gc.cuh"), os.path.join(HERE, "..", "include", "lexp_cuda.h")]

NVCC_FLAGS = [
    "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
    "-Xcompiler", "-fPIC,-fvisibility=hidden", "-shared", "-Xptxas=-v",
]


def needs_build():
    if not os.path.exists(SO):
        return True
    t = os.path.getmtime(SO)
    return any(os.path.getmtime(d) > t for d in DEPS)


def build(force=False, verbose=False):
    # LEXP_NVCC_DEFS: extra -D flags for build-time kernel variants (diagnosis only, e.g. "-DLEXP_TRACE=1"); a variant build is
    # always forced and the next plain build() restores the default kernel because the .so is older than this marker
    extra = os.environ.get("LEXP_NVCC_DEFS", "").split()
    marker = SO + ".variant"
    if extra:
        force = True
    elif os.path.exists(marker):
        force = True
    if not force and not needs_build():
        return SO
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    cmd = [nvcc] + NVCC_FLAGS + extra + ["-o", SO] + SRCS
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        sys.stderr.write(res.stdout + res.stderr)
    if res.returncode != 0:
        raise RuntimeError("nvcc failed building liblexp_cuda.so")
    with open(os.path.join(HERE, "build_ptxas.log"), "w") as f:
        f.write(res.stdout + res.stderr)
    if extra:
        with open(marker, "w") as f:
            f.write(" ".join(extra))
    elif os.path.exists(marker):
        os.remove(marker)
    return SO


if __name__ == "__main__":
    build(force="--force" in sys.argv, verbose=True)
    print(SO)
