"""TEST INFRASTRUCTURE -- the CPU restatement of svr_render_isosurface (tests/isosurface_oracle.cpp, on the CPU oracle's ray
generation, texture filter and gradient), compiled on first use (tests/_cpp_oracle.py)."""
import ctypes as C

import numpy as np

from oracle import binding as B

import _cpp_oracle as O

_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = O.load("isosurface_oracle", {"svr_oracle_isosurface": [C.POINTER(B.OracleScene), C.c_float, C.c_float, C.POINTER(C.c_float),
                                                                      C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]})
    return _lib


def oracle(voxels, fmt, dims, volume, camera):
    """A CpuOracle scene for isosurfaces (no transfer function is used: a zero table stands in)."""
    return B.CpuOracle(voxels, fmt, dims, volume, np.zeros((2, 4), np.float32), camera)


def isosurface(orc, iso, step, color=(1.0, 1.0, 1.0), rows=None):
    """(surface (H, W, 4) float32, u8 (H, W, 4)) of the rows [y0, y1) (default: all); the other rows stay 0."""
    s = orc.scene
    W, H = s.camera.imageW, s.camera.imageH
    y0, y1 = rows if rows else (0, H)
    surface = np.zeros((H, W, 4), np.float32)
    u8 = np.zeros((H, W, 4), np.uint8)
    lib().svr_oracle_isosurface(C.byref(s), iso, step, (C.c_float * 3)(*color), W, y0, y1, surface.ctypes.data, u8.ctypes.data)
    return surface, u8
