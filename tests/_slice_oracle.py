"""TEST INFRASTRUCTURE -- the CPU restatement of svr_render_slices (tests/slice_oracle.cpp, on the CPU oracle's texture
filter), compiled on first use (tests/_cpp_oracle.py)."""
import ctypes as C

import numpy as np

from oracle import binding as B
from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _cpp_oracle as O

_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = O.load("slice_oracle", {"svr_oracle_slices": [C.POINTER(B.OracleScene), C.POINTER(L.SliceParams), C.c_void_p, C.c_void_p]})
    return _lib


def oracle(voxels, fmt, dims, volume):
    """A CpuOracle scene for slices (no transfer function or camera is used: a zero table and a default camera stand in)."""
    return B.CpuOracle(voxels, fmt, dims, volume, np.zeros((2, 4), np.float32), S.default_camera(dims, 8, 8))


def slices(orc, params):
    """(value (count, H, W) float32, u8 (count, H, W, 4))."""
    shape = (params.count, params.imageH, params.imageW)
    value = np.zeros(shape, np.float32)
    u8 = np.zeros(shape + (4,), np.uint8)
    lib().svr_oracle_slices(C.byref(orc.scene), C.byref(params), value.ctypes.data, u8.ctypes.data)
    return value, u8
