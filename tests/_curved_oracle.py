"""TEST INFRASTRUCTURE -- the CPU restatement of svr_render_curved (tests/curved_oracle.cpp, on the CPU oracle's texture
filter), compiled on first use (tests/_cpp_oracle.py).  Its frame table comes from svr_curve_frames."""
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
        _lib = O.load("curved_oracle", {"svr_oracle_curved": [C.POINTER(B.OracleScene), C.POINTER(L.CurvedParams), C.c_void_p, C.c_void_p,
                                                              C.c_void_p]})
    return _lib


def oracle(voxels, fmt, dims, volume):
    """A CpuOracle scene for curved reformation (no transfer function or camera is used)."""
    return B.CpuOracle(voxels, fmt, dims, volume, np.zeros((2, 4), np.float32), S.default_camera(dims, 8, 8))


def stations(params):
    return params.count if params.layout == L.CURVED_CROSS else params.imageH


def curved(orc, params, points):
    """(value (count, H, W) float32, u8 (count, H, W, 4))."""
    frames = S.curve_frames(points, list(params.up), params.stationSpacing, stations(params))
    shape = (params.count, params.imageH, params.imageW)
    value = np.zeros(shape, np.float32)
    u8 = np.zeros(shape + (4,), np.uint8)
    lib().svr_oracle_curved(C.byref(orc.scene), C.byref(params), frames.ctypes.data, value.ctypes.data, u8.ctypes.data)
    return value, u8
