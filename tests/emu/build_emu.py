"""TEST INFRASTRUCTURE ONLY.  Builds tests/emu/liblexp_emu.so: the product's own sources (csrc/lexp_capi.cu + lexp_kernels.cuh)
compiled by g++ with -DLEXP_EMU against tests/emu/cuda_runtime.h, a host emulation of the CUDA execution model (fibers +
named barriers).  Same C-ABI as liblexp_cuda.so; loaded only by tests/test_emu_*.py, never by the package."""
import os
import subprocess

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SRC = os.path.join(ROOT, "localexpstereo_b200", "csrc", "lexp_capi.cu")
DEPS = [SRC, os.path.join(ROOT, "localexpstereo_b200", "csrc", "lexp_kernels.cuh"), os.path.join(ROOT, "localexpstereo_b200", "csrc", "lexp_gc.cuh"), os.path.join(ROOT, "include", "lexp_cuda.h"),
        os.path.join(HERE, "cuda_runtime.h"), os.path.abspath(__file__)]
SO = os.path.join(HERE, "liblexp_emu.so")


def build(force=False, defs=(), tag=""):
    """`defs`: extra -D flags selecting a build-time kernel variant (e.g. ("-DLEXP_TRACE=1",)), `tag` names its library."""
    so = SO if not tag else os.path.join(HERE, f"liblexp_emu_{tag}.so")
    if os.environ.get("LEXP_EMU_NO_REBUILD") and os.path.exists(so):  # worker processes of a test: the parent has built it
        return so
    if not force and os.path.exists(so) and os.path.getmtime(so) >= max(os.path.getmtime(d) for d in DEPS):
        return so
    return _compile(so, list(defs))


def _compile(SO, defs):
    # -ffp-contract=off: only the explicit fmaf() calls fuse.  nvcc also contracts plain a*b+c expressions, so the emulated
    # results differ from the GPU's in the last bits, but they are identical across build-time variants of the kernel, which is
    # what the A/B equivalence tests need.  -mfma only makes fmaf() a single instruction.
    fma = ["-mfma"] if "fma" in open("/proc/cpuinfo").read() else []
    cmd = ["/usr/bin/g++", "-std=c++17", "-O2", "-g", "-DLEXP_EMU", "-fPIC", "-shared", "-ffp-contract=off",
           "-fvisibility=hidden", "-fvisibility-inlines-hidden", "-fno-gnu-unique"] + defs + fma + [
        "-I", HERE, "-x", "c++", SRC, "-o", SO + ".tmp"]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("building the emulator failed:\n" + r.stderr[-8000:])
    os.replace(SO + ".tmp", SO)
    return SO


if __name__ == "__main__":
    print(build(force=True))
