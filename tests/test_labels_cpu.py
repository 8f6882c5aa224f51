"""Label maps (svr_render_labels, svr_render_label_slices, svr_labels_create, svr_labels_load_metaimage) without a GPU: the
table's layout, the argument checks (all made before any CUDA call), and closed forms on the CPU restatement
(tests/label_oracle.cpp) that the GPU tests hold the kernels to."""
import ctypes as C
import math
import os
import subprocess

import numpy as np

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _label_oracle as LO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEP = S.raycast_step_size()
H_STEP = 0.5 * STEP


def test_label_params_layout_matches_header(tmp_path):
    probe = tmp_path / "probe.c"
    probe.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "svr_render.h"\n'
        'int main(void){printf("%zu %zu\\n", sizeof(svr_label_params), offsetof(svr_label_params, color[3][2]));return 0;}\n'
    )
    exe = tmp_path / "probe"
    subprocess.check_call(["/usr/bin/gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert got == [4096, (3 * 4 + 2) * 4] and C.sizeof(L.LabelParams) == 4096


def _errors(call, bad, who):
    for kw in bad:
        rc, msg = call(**kw)
        assert rc != 0, kw
        assert who in msg, (kw, msg)


def test_render_labels_argument_errors_are_reported_before_any_cuda_call():
    lib = L.load()
    vol, cam = S.host_volume_struct((8, 8, 8)), S.default_camera((8, 8, 8), 16, 16)
    good = S.label_table({1: (1.0, 0.0, 0.0, 1.0)})
    out = C.c_void_p(16)  # never dereferenced: every call below fails its checks first

    def call(img=out, surface=out, label=out, volume=vol, camera=cam, table=good, step=0.5, phase=0, stride=1):
        rows = C.c_uint32(0)
        rc = lib.svr_render_labels(img, surface, label, C.byref(volume) if volume is not None else None,
                                   C.byref(camera) if camera is not None else None, C.byref(table) if table is not None else None, step,
                                   phase, stride, C.byref(rows))
        return rc, lib.svr_last_error().decode()

    nan, inf = float("nan"), float("inf")
    bad = [dict(volume=None), dict(camera=None), dict(table=None), dict(img=None, surface=None, label=None),
           dict(step=0.0), dict(step=-1.0), dict(step=inf), dict(step=nan), dict(phase=1, stride=1), dict(phase=0, stride=0),
           dict(phase=5, stride=3), dict()]  # the last: a volume without a texture is not a label volume
    for lab, c, x in ((1, 0, nan), (0, 3, -0.5), (255, 3, 1.5), (7, 1, inf)):
        t = S.label_table({1: (1.0, 0.0, 0.0, 1.0)})
        t.color[lab][c] = x
        bad.append(dict(table=t))
    _errors(call, bad, "svr_render_labels")
    rc, msg = call()
    assert "not a label volume" in msg


def test_render_label_slices_argument_errors_are_reported_before_any_cuda_call():
    lib = L.load()
    vol = S.host_volume_struct((8, 8, 8))
    good = S.label_table({1: (1.0, 0.0, 0.0, 0.5)})
    out = C.c_void_p(16)

    def call(img=out, label=out, volume=vol, params=True, table=good, outline=0, **kw):
        p = S.axis_slice((8, 8, 8), (1.0, 1.0, 1.0), "z", 4)
        for k, v in kw.items():
            setattr(p, k, v) if not isinstance(v, tuple) else getattr(p, k).__setitem__(slice(None), v)
        rc = lib.svr_render_label_slices(img, label, C.byref(volume) if volume is not None else None, C.byref(p) if params else None,
                                         C.byref(table) if table is not None else None, outline)
        return rc, lib.svr_last_error().decode()

    nan = float("nan")
    t = S.label_table({1: (1.0, 0.0, 0.0, 0.5)})
    t.color[2][0] = nan
    bad = [dict(volume=None), dict(params=False), dict(table=None), dict(img=None, label=None), dict(table=t),
           dict(outline=2), dict(outline=-1), dict(imageW=0), dict(count=0), dict(mode=3), dict(thickness=-1.0),
           dict(axisU=(nan, 0.0, 0.0)), dict(axisV=(1.0, 0.0, 0.0)), dict(windowWidth=0.0), dict()]
    _errors(call, bad, "svr_render_label_slices")


def test_labels_create_argument_errors():
    lib = L.load()
    v = L.Volume()
    data = np.zeros(8, np.uint8)
    for args in ((None, data.ctypes.data, 0, 2, 2, 2, 1.0, 1.0, 1.0), (C.byref(v), None, 0, 2, 2, 2, 1.0, 1.0, 1.0),
                 (C.byref(v), data.ctypes.data, 0, 0, 2, 2, 1.0, 1.0, 1.0), (C.byref(v), data.ctypes.data, 0, 2, 2, 16385, 1.0, 1.0, 1.0),
                 (C.byref(v), data.ctypes.data, 0, 2, 2, 2, 0.0, 1.0, 1.0), (C.byref(v), data.ctypes.data, 0, 2, 2, 2, 1.0, float("inf"), 1.0)):
        assert lib.svr_labels_create(*args) != 0
        assert "svr_labels_create" in lib.svr_last_error().decode()


def test_label_metaimage_errors_are_reported_before_any_cuda_call(tmp_path):
    lib = L.load()
    cases = [("float.mha", np.zeros((2, 2, 2), np.float32), "MET_FLOAT", 1, "integers"),
             ("double.mha", np.zeros((2, 2, 2), np.float64), "MET_DOUBLE", 1, "integers"),
             ("v256.mha", np.array([0, 1, 256, 2, 0, 0, 0, 0], np.uint16).reshape(2, 2, 2), "MET_USHORT", 1, "256"),
             ("neg.mha", np.array([0, 1, 2, -1, 0, 0, 0, 0], np.int16).reshape(2, 2, 2), "MET_SHORT", 1, "-1"),
             ("big.mhd", np.array([0, 70000, 0, 0, 0, 0, 0, 0], np.int32).reshape(2, 2, 2), "MET_INT", 1, "70000"),
             ("two.mha", np.zeros((2, 2, 2, 2), np.uint8), "MET_UCHAR", 2, "one channel")]
    for name, arr, etype, ch, what in cases:
        path = LO.write_metaimage(tmp_path / name, arr, etype, channels=ch, detached=name.endswith(".mhd"))
        v, m = L.Volume(), C.c_uint32(0)
        assert lib.svr_labels_load_metaimage(path.encode(), C.byref(v), C.byref(m)) != 0, name
        msg = lib.svr_last_error().decode()
        assert "svr_labels_load_metaimage" in msg and what in msg, (name, msg)
    v = L.Volume()
    assert lib.svr_labels_load_metaimage(str(tmp_path / "missing.mha").encode(), C.byref(v), None) != 0


# ---- closed forms on the restatement

def _axis_camera(n, W=16, H=16, D=None):
    """On -x looking along +x; the ray of pixel (W/2 - 1, H/2 - 1) is exactly +x through the volume's centre line."""
    D = 2.0 * n if D is None else D
    return S.make_camera((-D, 0.0, 0.0), (0, 0, 1), (0, 1, 0), (-1, 0, 0), 30.0, 0.0, 1.0, 1.0, W, H), D


def _inset(vol, n, axes="yz", voxels=2):
    inset = 2.0 * voxels / n
    for a in axes:
        setattr(vol, a + "_clip", L.Vec2(-1.0 + inset, 1.0 - inset))


def _rays(cam):
    W, H = cam.imageW, cam.imageH
    x = np.arange(W, dtype=np.float64)
    y = np.arange(H, dtype=np.float64)
    nx = (2.0 * ((x + 0.5) / (W - 1.0)) - 1.0) * cam.aspectRatio * cam.tanFovxOverTwo
    ny = (2.0 * ((y + 0.5) / (H - 1.0)) - 1.0) * cam.tanFovxOverTwo
    u, v, w = (np.array(cam.u.tuple()), np.array(cam.v.tuple()), np.array(cam.w.tuple()))
    d = nx[None, :, None] * u + ny[:, None, None] * v - w
    return d / np.linalg.norm(d, axis=2, keepdims=True)


def _hit_points(cam, surface):
    d = _rays(cam)
    back = -np.array(cam.w.tuple())
    z = np.where(np.isfinite(surface[..., 3:4]), surface[..., 3:4], 0).astype(np.float64)
    return np.array(cam.pos.tuple()) + d * (z / (d @ back)[..., None])


def test_half_space_puts_the_surface_on_the_voxel_face():
    """Label 1 in voxels x >= 8 of 16: along x, m is (1 - f) vis(i) + f vis(i + 1), which is 1/2 exactly at u = 7.5, the face
    between voxels 7 and 8 (world x = 0).  m is linear across that cell, so the linear interpolation of the refinement lands on
    it up to fp32 rounding (1e-4 voxel).  The gradient is +x; the normal faces the camera, -x."""
    n = 16
    lab = np.zeros((n, n, n), np.uint8)
    lab[:, :, 8:] = 1
    vol = S.host_volume_struct((n, n, n))
    _inset(vol, n)
    cam = S.look_at_camera((-2.0 * n, 0.0, 0.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), fovx=30.0, image_w=48, image_h=40)
    surface, u8, got = LO.labels(LO.oracle(lab, vol, cam), S.label_table({1: (1.0, 0.5, 0.25, 1.0)}), STEP)
    hit = np.isfinite(surface[..., 3])
    assert hit.mean() > 0.3
    x = _hit_points(cam, surface)[hit]
    assert np.abs(x[:, 0]).max() <= 1e-4 * 2 * n
    assert np.abs(surface[..., :3][hit] - np.array([-1.0, 0.0, 0.0], np.float32)).max() <= 1e-6
    assert np.all(got[hit] == 1) and np.all(got[~hit] == 0)
    assert np.all(u8[..., 3][hit] == 255) and np.all(u8[~hit] == 0)


def test_hiding_the_front_slab_reveals_the_back_one():
    n = 16
    lab = np.zeros((n, n, n), np.uint8)
    lab[:, :, 3:6] = 1
    lab[:, :, 10:13] = 2
    vol = S.host_volume_struct((n, n, n))
    _inset(vol, n)
    cam = S.look_at_camera((-2.0 * n, 0.0, 0.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), fovx=30.0, image_w=48, image_h=40)
    orc = LO.oracle(lab, vol, cam)
    both = S.label_table({1: (1.0, 0.0, 0.0, 1.0), 2: (0.0, 1.0, 0.0, 1.0)})
    back = S.label_table({1: (1.0, 0.0, 0.0, 0.0), 2: (0.0, 1.0, 0.0, 1.0)})
    for table, want, face in ((both, 1, 3), (back, 2, 10)):
        surface, u8, got = LO.labels(orc, table, STEP)
        hit = np.isfinite(surface[..., 3])
        assert hit.mean() > 0.3
        assert np.all(got[hit] == want)
        x = _hit_points(cam, surface)[hit]
        assert np.abs(x[:, 0] - (face - n / 2)).max() <= 1e-4 * 2 * n
        own, other = (1, 0) if want == 2 else (0, 1)  # the label's colour channel; the other holds the specular term alone
        assert np.all(u8[..., own][hit] > u8[..., other][hit] + 100)


def test_ball_hits_lie_at_its_radius():
    """A ball of label 3, the voxels whose centres lie within R of the centre.  Every corner of the cell around x lies within
    sqrt(3) voxels of x, so m(x) = 0 where |x| > R + sqrt(3) and m(x) = 1 where |x| < R - sqrt(3): the level 1/2 lies in that shell.
    The refined hit lies within the final bracket (h / 16) of points with m < 1/2 and m >= 1/2, so |r - R| <= sqrt(3) + h / 16."""
    n, R = 32, 9.0
    c = np.arange(n) + 0.5 - n / 2
    lab = ((c[:, None, None] ** 2 + c[None, :, None] ** 2 + c[None, None, :] ** 2) <= R * R).astype(np.uint8) * 3
    vol = S.host_volume_struct((n, n, n))
    table = S.label_table({3: (0.2, 0.4, 1.0, 1.0)})
    for cam in (S.default_camera((n, n, n), 64, 48),
                S.look_at_camera((0.9 * n, 0.7 * n, 1.1 * n), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), fovx=45.0, image_w=64, image_h=48)):
        surface, u8, got = LO.labels(LO.oracle(lab, vol, cam), table, STEP)
        hit = np.isfinite(surface[..., 3])
        assert hit.mean() > 0.05
        r = np.linalg.norm(_hit_points(cam, surface)[hit], axis=1)
        assert np.abs(r - R).max() <= math.sqrt(3) + H_STEP / 16
        assert np.all(got[hit] == 3)
        assert np.sum(surface[..., :3][hit] * _rays(cam)[hit], axis=1).max() <= 0


def test_a_clip_plane_through_a_block_caps_it_at_the_first_sample():
    """A block of label 1 filling the volume, clipped at x = -n/4: every ray through the clipped box has m(t_0) = 1 at its first
    sample, so t_hit = t_0 = max(tNear, 0) + h / 2 with no refinement."""
    n = 16
    lab = np.ones((n, n, n), np.uint8)
    vol = S.host_volume_struct((n, n, n))
    _inset(vol, n)
    vol.x_clip = L.Vec2(-0.5, 1.0)
    cam, D = _axis_camera(n, 32, 24)
    surface, u8, got = LO.labels(LO.oracle(lab, vol, cam), S.label_table({1: (1.0, 1.0, 1.0, 1.0)}), STEP)
    d = _rays(cam)
    o = np.array(cam.pos.tuple())
    bmin, bmax = np.array([-n / 4, -n / 2 + 2, -n / 2 + 2]), np.array([n / 2, n / 2 - 2, n / 2 - 2])
    with np.errstate(divide="ignore"):
        t1, t2 = (bmin - o) / d, (bmax - o) / d
    tnear, tfar = np.minimum(t1, t2).max(axis=2), np.maximum(t1, t2).min(axis=2)
    hit = np.isfinite(surface[..., 3])
    assert hit.mean() > 0.2 and np.all(tfar[hit] > tnear[hit])
    depth = (np.maximum(tnear, 0.0) + 0.5 * H_STEP) * (d @ -np.array(cam.w.tuple()))
    assert np.abs(surface[..., 3][hit] - depth[hit]).max() <= 1e-3
    assert np.all(got[hit] == 1)


def test_equally_weighted_labels_go_to_the_smaller_id():
    """Label a in the half y < 8 and label b in y >= 8 of the block x >= 8.  The centre ray (pixel (7, 7) of 16 x 16) runs along
    +x at y = z = 0: u.y = 7.5, f.y = 1/2, so the corners of both labels weigh the same wherever it hits.  The smaller id wins
    either way round."""
    n = 16
    for a, b in ((1, 2), (2, 1), (9, 4)):
        lab = np.zeros((n, n, n), np.uint8)
        lab[:, :8, 8:] = a
        lab[:, 8:, 8:] = b
        vol = S.host_volume_struct((n, n, n))
        cam, D = _axis_camera(n)
        surface, u8, got = LO.labels(LO.oracle(lab, vol, cam), S.label_table({a: (1.0, 0.0, 0.0, 1.0), b: (0.0, 1.0, 0.0, 1.0)}), STEP)
        assert np.isfinite(surface[7, 7, 3])
        assert abs(surface[7, 7, 3] - D) <= 1e-4 * D
        assert got[7, 7] == min(a, b), (a, b, int(got[7, 7]))
