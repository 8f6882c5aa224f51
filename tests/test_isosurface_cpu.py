"""Isosurface (svr_render_isosurface) without a GPU: the parameter struct's layout, the argument checks (all made before any CUDA
call), and closed forms on the CPU restatement (tests/isosurface_oracle.cpp) that the GPU tests hold the kernel to."""
import ctypes as C
import math
import os
import subprocess

import numpy as np

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _isosurface_oracle as IO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEP = S.raycast_step_size()
H_STEP = 0.5 * STEP


def test_isosurface_params_layout_matches_header(tmp_path):
    probe = tmp_path / "probe.c"
    probe.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "svr_render.h"\n'
        "int main(void){printf(\"%zu %zu %zu %zu\\n\", sizeof(svr_isosurface_params), offsetof(svr_isosurface_params, isoValue),"
        " offsetof(svr_isosurface_params, stepSize), offsetof(svr_isosurface_params, color));return 0;}\n"
    )
    exe = tmp_path / "probe"
    subprocess.check_call(["/usr/bin/gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    P = L.IsosurfaceParams
    assert got == [C.sizeof(P), P.isoValue.offset, P.stepSize.offset, P.color.offset]


def test_argument_errors_are_reported_before_any_cuda_call():
    lib = L.load()
    vol, cam = S.host_volume_struct((8, 8, 8)), S.default_camera((8, 8, 8), 16, 16)
    out = C.c_void_p(16)  # never dereferenced: every call below fails its checks first

    def call(img=out, surface=out, volume=vol, camera=cam, iso=0.5, step=0.5, color=(1.0, 0.5, 0.0), phase=0, stride=1, params=True):
        p = L.IsosurfaceParams(iso, step, (C.c_float * 3)(*color))
        rows = C.c_uint32(0)
        rc = lib.svr_render_isosurface(img, surface, C.byref(volume) if volume is not None else None, C.byref(camera) if camera is not None else None,
                                       C.byref(p) if params else None, phase, stride, C.byref(rows))
        return rc, lib.svr_last_error().decode()

    nan, inf = float("nan"), float("inf")
    bad = [dict(volume=None), dict(camera=None), dict(params=False), dict(img=None, surface=None),
           dict(step=0.0), dict(step=-1.0), dict(step=inf), dict(step=nan), dict(iso=nan), dict(iso=inf), dict(iso=-inf),
           dict(color=(nan, 0.0, 0.0)), dict(color=(0.0, inf, 0.0)), dict(color=(0.0, 0.0, -0.01)), dict(color=(1.01, 0.0, 0.0)),
           dict(phase=1, stride=1), dict(phase=0, stride=0), dict(phase=5, stride=3)]
    for kw in bad:
        rc, msg = call(**kw)
        assert rc != 0, kw
        assert "svr_render_isosurface" in msg, (kw, msg)


def _rays(cam):
    """Pixel-centre ray directions of camera_ray_center (float64), (H, W, 3)."""
    W, H = cam.imageW, cam.imageH
    x = np.arange(W, dtype=np.float64)
    y = np.arange(H, dtype=np.float64)
    nx = (2.0 * ((x + 0.5) / (W - 1.0)) - 1.0) * cam.aspectRatio * cam.tanFovxOverTwo
    ny = (2.0 * ((y + 0.5) / (H - 1.0)) - 1.0) * cam.tanFovxOverTwo
    u, v, w = (np.array(cam.u.tuple()), np.array(cam.v.tuple()), np.array(cam.w.tuple()))
    d = nx[None, :, None] * u + ny[:, None, None] * v - w
    return d / np.linalg.norm(d, axis=2, keepdims=True)


def _hit_points(cam, surface):
    """World hit points from the depth: x = pos + dir z / (dir . -w)."""
    d = _rays(cam)
    back = -np.array(cam.w.tuple())
    z = np.where(np.isfinite(surface[..., 3:4]), surface[..., 3:4], 0).astype(np.float64)
    return np.array(cam.pos.tuple()) + d * (z / (d @ back)[..., None])


def _ramp_scene(n, ds):
    """f32 ramp along x, voxel i = (i + 1/2) / n, so tex3D = x / n + 1/2 in world x; y and z clipped two voxels in so that no sample
    reads the border.  The camera on -x looks along +x: every ray enters where the value is about 0."""
    vox = np.ascontiguousarray(np.broadcast_to(((np.arange(n) + 0.5) / n).astype(np.float32), (n, n, n)))
    vol = S.host_volume_struct((n, n, n))
    vol.densityScale = ds
    inset = 2.0 * 2.0 / n
    vol.y_clip = L.Vec2(-1.0 + inset, 1.0 - inset)
    vol.z_clip = L.Vec2(-1.0 + inset, 1.0 - inset)
    D = 2.0 * n
    cam = S.look_at_camera((-D, 0.0, 0.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), fovx=30.0, image_w=64, image_h=48)
    return vox, vol, cam, D


def test_linear_ramp_gives_a_plane():
    """tex3D of a linear ramp is linear up to the filter's 8-bit weights.  The filter rounds the texel coordinate to 1/256 voxel
    (at most 1/512 off) and each texel's weight to 1/256; along a ramp in x only the summed weight of the x + 1 texels matters,
    and it equals the rounded fraction, or one unit more where two roundings tie.  So the value crosses iso within 3/512 voxel of
    the plane x = n (iso / ds - 1/2), and the linear interpolation that ends the refinement keeps that bound (the interpolant of
    a function within e of a line crosses iso within e / slope of it).  The plane is perpendicular to the view direction, so
    every hit has the depth D + x_plane (1e-4 for fp32 arithmetic at depths of about 2n), and the normal is -x (the gradient, +x,
    turned to the camera)."""
    n = 32
    for ds, iso in ((1.0, 0.5), (1.0, 0.3), (2.0, 0.5), (2.0, 1.4)):
        vox, vol, cam, D = _ramp_scene(n, ds)
        surface, u8 = IO.isosurface(IO.oracle(vox, L.VOXEL_F32, (n, n, n), vol, cam), iso, STEP, color=(1.0, 0.5, 0.25))
        hit = np.isfinite(surface[..., 3])
        assert hit.mean() > 0.3, (ds, iso)
        plane = n * (iso / ds - 0.5)
        z = surface[..., 3][hit]
        assert np.abs(z - (D + plane)).max() <= 3.0 / 512 + 1e-4, (ds, iso, float(np.abs(z - (D + plane)).max()))
        nrm = surface[..., :3][hit]
        assert np.abs(nrm - np.array([-1.0, 0.0, 0.0], np.float32)).max() <= 1e-3, (ds, iso)
        assert np.all(u8[..., 3][hit] == 255) and np.all(u8[~hit] == 0)
        # the hit points lie on the plane
        x = _hit_points(cam, surface)[hit]
        assert np.abs(x[:, 0] - plane).max() <= 3.0 / 512 + 1e-4


def test_constant_slab_hits_at_the_first_sample():
    """A constant above the threshold with the clip planes inset: every ray that crosses the slab hits sample 0 (t_0 = max(tNear, 0)
    + h / 2, no refinement), its gradient is 0 (the six taps read the same constant), so n = 0, cos = 1, spec = 0 and
    rgb = 0.8 color; the depth follows from the box entry."""
    n, c = 32, np.float32(0.37)
    vox = np.full((n, n, n), c, np.float32)
    vol = S.host_volume_struct((n, n, n))
    inset = 2.0 * 2.0 / n
    lo, hi = -1.0 + inset, 1.0 - inset
    vol.x_clip, vol.y_clip, vol.z_clip = L.Vec2(lo, hi), L.Vec2(lo, hi), L.Vec2(lo, 0.5)
    cam = S.default_camera((n, n, n), 64, 48)
    color = (1.0, 0.5, 0.2)
    surface, u8 = IO.isosurface(IO.oracle(vox, L.VOXEL_F32, (n, n, n), vol, cam), 0.3, STEP, color=color)
    # the expected entry, in float64: slab [n/2 lo, n/2 hi] per axis (z up to n/2 0.5)
    d = _rays(cam)
    o = np.array(cam.pos.tuple())
    bmin = np.array([n / 2 * lo] * 3)
    bmax = np.array([n / 2 * hi, n / 2 * hi, n / 2 * 0.5])
    with np.errstate(divide="ignore"):
        t1, t2 = (bmin - o) / d, (bmax - o) / d
    tnear, tfar = np.minimum(t1, t2).max(axis=2), np.maximum(t1, t2).min(axis=2)
    t0 = np.maximum(tnear, 0.0)
    crossing = (tfar > tnear) & (np.floor((tfar - t0) / H_STEP + 0.5) >= 1)
    hit = np.isfinite(surface[..., 3])
    assert hit.mean() > 0.2
    edge = np.abs((tfar - t0) / H_STEP + 0.5 - np.round((tfar - t0) / H_STEP + 0.5)) < 1e-3  # K decided by rounding
    assert np.array_equal(hit[~edge], crossing[~edge])
    back = -np.array(cam.w.tuple())
    depth = (t0 + 0.5 * H_STEP) * (d @ back)
    assert np.abs(surface[..., 3][hit] - depth[hit]).max() <= 1e-3
    assert np.all(surface[..., :3][hit] == 0)
    want = [int(np.float32(255) * np.float32(np.float32(x) * np.float32(0.8))) for x in color]
    assert np.all(u8[hit] == np.array(want + [255], np.uint8))
    assert np.all(u8[~hit] == 0)


def test_rays_that_miss_give_the_miss_values():
    n = 32
    vox = np.full((n, n, n), 200, np.uint8)
    cam = S.make_camera((0.0, 0.0, 4.0 * n), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0, 64, 48)
    vol = S.host_volume_struct((n, n, n))
    surface, u8 = IO.isosurface(IO.oracle(vox, L.VOXEL_U8, (n, n, n), vol, cam), 0.5, STEP)
    # the box spans +-n/2; from z = 4n it covers a small disc around the image centre: the border rows and columns miss it
    assert np.isfinite(surface[24, 32, 3]) and u8[24, 32, 3] == 255
    for sl in (np.s_[:4], np.s_[-4:], np.s_[:, :4], np.s_[:, -4:]):
        s, i = surface[sl].reshape(-1, 4), u8[sl].reshape(-1, 4)
        assert np.all(s[:, :3] == 0) and np.all(s[:, 3] == np.inf) and np.all(i == 0)
    # a threshold above every value: every ray misses
    surface, u8 = IO.isosurface(IO.oracle(vox, L.VOXEL_U8, (n, n, n), vol, cam), 0.9, STEP)
    assert np.all(surface[..., 3] == np.inf) and np.all(surface[..., :3] == 0) and np.all(u8 == 0)


def test_sphere_hits_lie_on_the_radius():
    """C1's sphere (rho = 1 - r / (0.45 n), u8) at iso 0.5: the hit points lie at radius 0.225 n within
        0.45 n / 510    the u8 rounding of the voxels (half an LSB of rho),
      + 1 / (4 r)       trilinear interpolation of r (the trace of its Hessian is 2 / r, the error at most 1/8 of it per voxel^2),
      + sqrt(3) / 256   the filter's 8-bit weights (1/256 voxel per axis),
      + h / 16          the final bracket after four bisections, where the ray grazes the surface,
    voxels.  The normals are radial."""
    n = 64
    vox = S.sphere_volume(n, L.VOXEL_U8)
    vol = S.host_volume_struct((n, n, n))
    for cam in (S.default_camera((n, n, n), 96, 80),
                S.look_at_camera((0.9 * n, 0.7 * n, 1.1 * n), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), fovx=45.0, image_w=96, image_h=80)):
        surface, u8 = IO.isosurface(IO.oracle(vox, L.VOXEL_U8, (n, n, n), vol, cam), 0.5, STEP)
        hit = np.isfinite(surface[..., 3])
        assert hit.mean() > 0.05
        r0 = 0.225 * n
        tol = 0.45 * n / 510 + 1 / (4 * r0) + math.sqrt(3) / 256 + H_STEP / 16
        x = _hit_points(cam, surface)[hit]
        r = np.linalg.norm(x, axis=1)
        assert np.abs(r - r0).max() <= tol, (float(np.abs(r - r0).max()), tol)
        # the normal is radial; it faces the ray's origin, so a grazing ray that crosses just past the tangent point sees it inwards
        nrm = surface[..., :3][hit]
        assert np.abs(np.sum(nrm * x / r[:, None], axis=1)).min() > 0.99
        assert np.sum(nrm * _rays(cam)[hit], axis=1).max() <= 0
        assert u8[..., 0][hit].max() > 200
