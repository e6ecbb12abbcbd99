"""ctypes loader for libomvg_b200.so.  Fails loudly: there is no CPU fallback."""
from __future__ import annotations

import ctypes
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libomvg_b200.so")
_lib = None


class OmvgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"omvg_b200 error {code}: {msg}")
        self.code = code


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a).  openmvg_b200 has no CPU fallback.")
        L = ctypes.CDLL(LIB_PATH)
        L.omvg_last_error.restype = ctypes.c_char_p
        L.omvg_match_launch_count.restype = ctypes.c_uint64
        L.omvg_match_launch_count.argtypes = [ctypes.c_void_p]
        L.omvg_match_kernel_variant.restype = ctypes.c_int
        L.omvg_match_kernel_variant.argtypes = [ctypes.c_void_p]
        _lib = L
    return _lib


def check(rc: int) -> None:
    if rc != 0:
        raise OmvgError(rc, lib().omvg_last_error().decode(errors="replace"))
