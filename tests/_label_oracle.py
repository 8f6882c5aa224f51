"""TEST INFRASTRUCTURE -- the CPU restatement of svr_render_labels and svr_render_label_slices (tests/label_oracle.cpp, on the
CPU oracle's rays), compiled on first use (tests/_cpp_oracle.py)."""
import ctypes as C
import os

import numpy as np

from oracle import binding as B
from sunvolumerender_b200 import _lib as L

import _cpp_oracle as O

_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = O.load("label_oracle", {
            "svr_oracle_labels": [C.POINTER(B.OracleScene), C.c_void_p, C.c_float, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                  C.c_void_p],
            "svr_oracle_label_slices": [C.POINTER(B.OracleScene), C.POINTER(L.SliceParams), C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]})
    return _lib


def oracle(labels, volume, camera):
    """A CpuOracle scene over u8 labels shaped (nz, ny, nx) (no transfer function is used: a zero table stands in)."""
    labels = np.ascontiguousarray(labels, dtype=np.uint8)
    nz, ny, nx = labels.shape
    return B.CpuOracle(labels, L.VOXEL_U8, (nx, ny, nz), volume, np.zeros((2, 4), np.float32), camera)


def _table(table):
    return np.ascontiguousarray(np.ctypeslib.as_array(table.color), dtype=np.float32)


def labels(orc, table, step, rows=None):
    """(surface (H, W, 4) float32, u8 (H, W, 4), label (H, W) u8) of the rows [y0, y1) (default: all); the other rows stay 0."""
    s = orc.scene
    W, H = s.camera.imageW, s.camera.imageH
    y0, y1 = rows if rows else (0, H)
    surface = np.zeros((H, W, 4), np.float32)
    u8 = np.zeros((H, W, 4), np.uint8)
    lab = np.zeros((H, W), np.uint8)
    t = _table(table)
    lib().svr_oracle_labels(C.byref(s), t.ctypes.data, step, W, y0, y1, surface.ctypes.data, u8.ctypes.data, lab.ctypes.data)
    return surface, u8, lab


def label_slices(orc, params, table, img=None, outline=False):
    """(label (count, H, W) u8, img composited in place (a copy; None when img is None))."""
    shape = (params.count, params.imageH, params.imageW)
    lab = np.zeros(shape, np.uint8)
    out = None if img is None else np.ascontiguousarray(img, dtype=np.uint8).copy()
    t = _table(table)
    lib().svr_oracle_label_slices(C.byref(orc.scene), C.byref(params), t.ctypes.data, 1 if outline else 0,
                                  None if out is None else out.ctypes.data, lab.ctypes.data)
    return lab, out


def write_metaimage(path, arr, etype, channels=1, compressed=False, msb=False, detached=False):
    """A .mha (LOCAL data) or, with detached, a .mhd and its .raw; arr shaped (nz, ny, nx[, channels])."""
    import zlib

    nz, ny, nx = arr.shape[:3]
    raw = np.ascontiguousarray(arr).astype(arr.dtype.newbyteorder(">") if msb else arr.dtype).tobytes()
    if compressed:
        raw = zlib.compress(raw)
    lines = ["ObjectType = Image", "NDims = 3", f"DimSize = {nx} {ny} {nz}", "ElementSpacing = 1.5 1 2", f"ElementType = {etype}",
             f"BinaryDataByteOrderMSB = {'True' if msb else 'False'}"]
    if channels != 1:
        lines.append(f"ElementNumberOfChannels = {channels}")
    if compressed:
        lines += ["CompressedData = True", f"CompressedDataSize = {len(raw)}"]
    path = str(path)
    if detached:
        rawname = os.path.basename(path) + ".raw"
        with open(os.path.join(os.path.dirname(path), rawname), "wb") as f:
            f.write(raw)
        lines.append(f"ElementDataFile = {rawname}")
        with open(path, "w") as f:
            f.write("\n".join(lines) + "\n")
    else:
        lines.append("ElementDataFile = LOCAL")
        with open(path, "wb") as f:
            f.write(("\n".join(lines) + "\n").encode() + raw)
    return path
