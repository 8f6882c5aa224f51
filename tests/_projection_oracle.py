"""TEST INFRASTRUCTURE -- the CPU restatement of svr_render_projection (tests/projection_oracle.cpp, on the CPU oracle's ray
generation and texture filter), compiled on first use (tests/_cpp_oracle.py)."""
import ctypes as C

import numpy as np

from oracle import binding as B

import _cpp_oracle as O

MODES = {"max": 0, "min": 1, "mean": 2}
_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = O.load("projection_oracle", {"svr_oracle_project": [C.POINTER(B.OracleScene), C.c_int, C.c_float, C.c_float, C.c_float, C.c_uint32,
                                                                   C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]})
    return _lib


def oracle(voxels, fmt, dims, volume, camera):
    """A CpuOracle scene for projections (no transfer function is used: a zero table stands in)."""
    return B.CpuOracle(voxels, fmt, dims, volume, np.zeros((2, 4), np.float32), camera)


def project(orc, mode, step, window=(0.5, 1.0), rows=None):
    """(value (H, W) float32, u8 (H, W, 4)) of the rows [y0, y1) (default: all); the other rows stay 0."""
    s = orc.scene
    W, H = s.camera.imageW, s.camera.imageH
    y0, y1 = rows if rows else (0, H)
    value = np.zeros((H, W), np.float32)
    u8 = np.zeros((H, W, 4), np.uint8)
    lib().svr_oracle_project(C.byref(s), MODES[mode], step, window[0], window[1], W, y0, y1, value.ctypes.data, u8.ctypes.data)
    return value, u8
