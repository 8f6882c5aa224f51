"""Intensity projection (svr_render_projection) without a GPU: the parameter struct's layout, the argument checks (all made
before any CUDA call), and closed forms on the CPU restatement (tests/projection_oracle.cpp) that the GPU tests hold the
kernel to."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _projection_oracle as PO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEP = S.raycast_step_size()


def test_projection_params_layout_matches_header(tmp_path):
    probe = tmp_path / "probe.c"
    probe.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "svr_render.h"\n'
        "int main(void){printf(\"%zu %zu %zu %zu %zu %d %d %d\\n\", sizeof(svr_projection_params), offsetof(svr_projection_params, mode),"
        " offsetof(svr_projection_params, stepSize), offsetof(svr_projection_params, windowCenter), offsetof(svr_projection_params, windowWidth),"
        " SVR_PROJECT_MAX, SVR_PROJECT_MIN, SVR_PROJECT_MEAN);return 0;}\n"
    )
    exe = tmp_path / "probe"
    subprocess.check_call(["/usr/bin/gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    P = L.ProjectionParams
    assert got == [C.sizeof(P), P.mode.offset, P.stepSize.offset, P.windowCenter.offset, P.windowWidth.offset, L.PROJECT_MAX, L.PROJECT_MIN, L.PROJECT_MEAN]


def test_argument_errors_are_reported_before_any_cuda_call():
    lib = L.load()
    vol, cam = S.host_volume_struct((8, 8, 8)), S.default_camera((8, 8, 8), 16, 16)
    out = C.c_void_p(16)  # never dereferenced: every call below fails its checks first

    def call(img=out, value=out, volume=vol, camera=cam, mode=L.PROJECT_MAX, step=0.5, center=0.5, width=1.0, phase=0, stride=1, params=True):
        p = L.ProjectionParams(mode, step, center, width)
        rows = C.c_uint32(0)
        rc = lib.svr_render_projection(img, value, C.byref(volume) if volume is not None else None, C.byref(camera) if camera is not None else None,
                                       C.byref(p) if params else None, phase, stride, C.byref(rows))
        return rc, lib.svr_last_error().decode()

    bad = [dict(volume=None), dict(camera=None), dict(params=False), dict(img=None, value=None), dict(mode=-1), dict(mode=3),
           dict(step=0.0), dict(step=-1.0), dict(step=float("inf")), dict(step=float("nan")), dict(width=0.0), dict(width=-2.0),
           dict(width=float("inf")), dict(width=float("nan")), dict(center=float("nan")), dict(phase=1, stride=1), dict(phase=0, stride=0),
           dict(phase=5, stride=3)]
    for kw in bad:
        rc, msg = call(**kw)
        assert rc != 0, kw
        assert "svr_render_projection" in msg, (kw, msg)


def _scene(voxels, fmt, n, w=64, h=48, camera=None):
    vol = S.host_volume_struct((n, n, n))
    cam = camera or S.default_camera((n, n, n), w, h)
    return vol, cam, PO.oracle(voxels, fmt, (n, n, n), vol, cam)


def test_constant_slab_gives_the_constant_in_every_mode():
    n, c = 32, np.float32(0.37)
    vox = np.full((n, n, n), c, np.float32)
    vol, cam, _ = _scene(vox, L.VOXEL_F32, n)
    inset = 2.0 * 2.0 / n  # two voxels, in units of the half extent
    vol.x_clip = L.Vec2(-1.0 + inset, 1.0 - inset)
    vol.y_clip = L.Vec2(-1.0 + inset, 1.0 - inset)
    vol.z_clip = L.Vec2(-1.0 + inset, 0.5)
    orc = PO.oracle(vox, L.VOXEL_F32, (n, n, n), vol, cam)
    got = {m: PO.project(orc, m, STEP)[0] for m in ("max", "min", "mean")}
    crossing = got["max"] != 0
    assert crossing.mean() > 0.2
    for m, v in got.items():
        assert np.abs(v[crossing] - c).max() <= 1e-6, m
        assert np.all(v[~crossing] == 0), m


def test_min_mean_max_are_ordered():
    n = 48
    vox = S.sphere_volume(n, L.VOXEL_U16)
    _, _, orc = _scene(vox, L.VOXEL_U16, n)
    lo, mean, hi = (PO.project(orc, m, STEP)[0] for m in ("min", "mean", "max"))
    assert hi.max() > 0.5
    assert np.all(lo <= mean + 1e-6) and np.all(mean <= hi + 1e-6)


def test_rays_that_miss_the_box_give_zero():
    n = 32
    vox = np.full((n, n, n), 200, np.uint8)
    cam = S.make_camera((0.0, 0.0, 4.0 * n), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0, 64, 48)
    _, _, orc = _scene(vox, L.VOXEL_U8, n, camera=cam)
    # the box spans +-n/2; from z = 4n it covers a small disc around the image centre: the border rows and columns miss it
    for m in ("max", "min", "mean"):
        v = PO.project(orc, m, STEP)[0]
        assert v[24, 32] > 0.3, m  # min: the samples next to the faces blend in the border value 0
        border = np.concatenate([v[:4].ravel(), v[-4:].ravel(), v[:, :4].ravel(), v[:, -4:].ravel()])
        assert np.all(border == 0), m


def test_density_scale_two_doubles_the_value_exactly():
    n = 40
    vox = S.sphere_volume(n, L.VOXEL_U8)
    vol, cam, orc1 = _scene(vox, L.VOXEL_U8, n)
    vol2 = L.Volume.from_buffer_copy(vol)
    vol2.densityScale = 2.0
    orc2 = PO.oracle(vox, L.VOXEL_U8, (n, n, n), vol2, cam)
    for m in ("max", "min", "mean"):
        a, b = PO.project(orc1, m, STEP)[0], PO.project(orc2, m, STEP)[0]
        assert np.array_equal(b, np.float32(2) * a), m


def test_window_mapping_follows_the_formula():
    n = 40
    vox = S.sphere_volume(n, L.VOXEL_U16)
    _, _, orc = _scene(vox, L.VOXEL_U16, n)
    for center, width in ((0.5, 1.0), (0.3, 0.2), (0.9, 0.05), (-1.0, 3.5)):
        value, u8 = PO.project(orc, "max", STEP, (center, width))
        c, w = np.float32(center), np.float32(width)
        g = np.clip((value - (c - np.float32(0.5) * w)) / w, np.float32(0), np.float32(1)).astype(np.float32)
        q = (np.float32(255) * g).astype(np.int32).astype(np.uint8)
        assert np.array_equal(u8[..., 0], q) and np.array_equal(u8[..., 1], q) and np.array_equal(u8[..., 2], q)
        assert np.all(u8[..., 3] == 255)
    assert len(np.unique(u8[..., 0])) > 2
