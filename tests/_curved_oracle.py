"""TEST INFRASTRUCTURE -- the CPU restatement of svr_render_curved (tests/curved_oracle.cpp, on the CPU oracle's texture
filter), compiled on first use into a temporary directory.  Its frame table comes from svr_curve_frames."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from oracle import binding as B
from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "curved_oracle.cpp")
_lib = None


def lib():
    global _lib
    if _lib is None:
        out = os.path.join(tempfile.mkdtemp(prefix="svr_curved_oracle_"), "libsvr_curved_oracle.so")
        # the flags of oracle/Makefile's cpu target (the distro compiler: it has libgomp)
        subprocess.check_call(["/usr/bin/g++", "-O3", "-fopenmp", "-fno-fast-math", "-shared", "-fPIC", "-o", out, SRC])
        lib_ = C.CDLL(out)
        lib_.svr_oracle_curved.argtypes = [C.POINTER(B.OracleScene), C.POINTER(L.CurvedParams), C.c_void_p, C.c_void_p, C.c_void_p]
        _lib = lib_
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
