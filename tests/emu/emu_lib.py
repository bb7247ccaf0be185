"""TEST INFRASTRUCTURE ONLY.  Loads tests/emu/liblexp_emu.so (the product's CUDA sources compiled for the host emulator, see
cuda_runtime.h in this directory) and swaps it in as the library behind localexpstereo_b200._capi for the duration of a test
module.  The package itself never does this: without liblexp_cuda.so and a GPU it raises."""
import contextlib
import ctypes as C
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
if HERE not in sys.path:
    sys.path.insert(0, HERE)

_emu = {}

VARIANTS = {"": (), "trace": ("-DLEXP_TRACE=1",)}  # build-time kernel variants (lexp_kernels.cuh), "" = the shipped kernel


def load(variant=""):
    if variant not in _emu:
        import build_emu
        from localexpstereo_b200 import _capi
        L = C.CDLL(build_emu.build(defs=VARIANTS[variant], tag=variant))
        for name, (res, args) in _capi.SYMBOLS.items():
            f = getattr(L, name)
            f.restype, f.argtypes = res, args
        _emu[variant] = L
    return _emu[variant]


@contextlib.contextmanager
def emulated(order=None, variant=""):
    """`order`: LEXP_EMU_ORDER for the fiber scheduler (0 forward, 1 reverse, 2 shuffled every pass)."""
    from localexpstereo_b200 import _capi
    prev_lib, prev_env = _capi._lib, os.environ.get("LEXP_EMU_ORDER")
    _capi._lib = load(variant)
    if order is not None:
        os.environ["LEXP_EMU_ORDER"] = str(order)
    try:
        yield _capi._lib
    finally:
        _capi._lib = prev_lib
        if prev_env is None:
            os.environ.pop("LEXP_EMU_ORDER", None)
        else:
            os.environ["LEXP_EMU_ORDER"] = prev_env
