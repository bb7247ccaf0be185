#!/usr/bin/env python
"""TEST INFRASTRUCTURE ONLY (manual tool, not part of the default suite).  Memory-checks the kernel source on the CPU emulator:
builds the emulator library with AddressSanitizer -- "device" buffers and the dynamic shared memory are then exact-size heap
blocks, so the first byte the kernel reads or writes out of bounds is reported -- and drives the fuzz tests through it.

    python tests/emu/asan_fuzz.py [first_seed last_seed]       (re-executes itself with libasan preloaded)
    LEXP_ASAN_DEFS="-DLEXP_TRACE=1" python tests/emu/asan_fuzz.py 0 40      (the diagnosis build)
"""
import ctypes as C
import os
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
SO = os.path.join(HERE, "liblexp_emu_asan.so")


def build():
    src = os.path.join(ROOT, "localexpstereo_b200", "csrc", "lexp_capi.cu")
    cmd = ["/usr/bin/g++", "-std=c++17", "-O1", "-g", "-DLEXP_EMU", "-fPIC", "-shared", "-ffp-contract=off", "-fvisibility=hidden",
           "-fvisibility-inlines-hidden", "-fno-gnu-unique", "-mfma", "-fsanitize=address", "-fno-omit-frame-pointer",
           "-I", HERE, "-x", "c++", src, "-o", SO] + os.environ.get("LEXP_ASAN_DEFS", "").split()
    subprocess.check_call(cmd)


def main():
    if "libasan" not in os.environ.get("LD_PRELOAD", ""):
        build()
        asan = subprocess.check_output(["/usr/bin/gcc", "-print-file-name=libasan.so"], text=True).strip()
        env = dict(os.environ, LD_PRELOAD=os.path.realpath(asan), ASAN_OPTIONS="detect_leaks=0:detect_stack_use_after_return=0")
        raise SystemExit(subprocess.call([sys.executable, os.path.abspath(__file__)] + sys.argv[1:], env=env))
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from localexpstereo_b200 import _capi
    lib = C.CDLL(SO)
    for name, (res, args) in _capi.SYMBOLS.items():
        f = getattr(lib, name)
        f.restype, f.argtypes = res, args
    _capi._lib = lib
    import test_emu_fuzz as T

    class Env:
        @staticmethod
        def setenv(k, v):
            os.environ[k] = v

    lo, hi = (int(sys.argv[1]), int(sys.argv[2])) if len(sys.argv) > 2 else (0, 20)
    for seed in range(lo, hi):
        T.test_random_rects_and_planes_match_the_oracle(seed)
    for seed in range(4):
        T.test_random_batches_with_forced_tilings(seed, Env)
    os.environ.pop("LEXP_TILE_OH", None)
    T.test_one_large_cell_is_cut_into_many_work_items()
    print(f"asan fuzz: seeds {lo}..{hi - 1}, forced tilings (both energies) and the large cell ran clean")


if __name__ == "__main__":
    main()
