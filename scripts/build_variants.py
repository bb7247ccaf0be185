#!/usr/bin/env python
"""Builds the diagnosis build of lexp_kernels.cuh (-DLEXP_TRACE=1) next to the product library, as
variants/liblexp_cuda_trace.so (git-ignored), and prints the ptxas resource lines.  scripts/gpu_trace.sh runs it on the GPU."""
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from localexpstereo_b200 import build as B  # noqa: E402

VARIANTS = {
    "trace": ["-DLEXP_TRACE=1"],                    # diagnosis: per-team wait / busy cycles of every launch (scripts/gpu_trace.sh)
}


def main(names):
    out_dir = os.path.join(ROOT, "variants")
    os.makedirs(out_dir, exist_ok=True)
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    for name in names or VARIANTS:
        so = os.path.join(out_dir, f"liblexp_cuda_{name}.so")
        r = subprocess.run([nvcc] + B.NVCC_FLAGS + VARIANTS[name] + ["-o", so] + B.SRCS, capture_output=True, text=True)
        if r.returncode:
            print(r.stderr[-3000:])
            raise SystemExit(f"variant {name} failed to build")
        txt = r.stdout + r.stderr
        res = []
        for m in re.finditer(r"Function properties for (\S+)\n\s+(\d+) bytes stack frame, (\d+) bytes spill stores, (\d+) bytes spill loads\nptxas info\s+: Used (\d+) registers", txt):
            if "lexp_fused_kernel" in m.group(1):
                tag = re.search(r"ILi(\d+)ELb(\d)", m.group(1))
                res.append(f"R{tag.group(1)}{'n' if tag.group(2) == '1' else ''}: {m.group(5)} regs, spill {m.group(3)}/{m.group(4)} B")
        print(f"{name:10s} {' '.join(VARIANTS[name]):28s} | " + " | ".join(res))


if __name__ == "__main__":
    main(sys.argv[1:])
