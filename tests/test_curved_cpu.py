"""Curved planar reformation (svr_render_curved, svr_curve_frames) without a GPU: the parameter struct's layout, the argument
checks (all made before any CUDA call), the frame rule against an independent float64 restatement and against closed forms
(straight line, planar arc, helix), and closed forms on the CPU restatement of the pixel rule (tests/curved_oracle.cpp)."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _curved_oracle as CO
import _slice_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("up", "layout", "imageW", "imageH", "count", "mode", "pixelSpacing", "stationSpacing", "angle0", "angleStep", "thickness",
          "sampleSpacing", "windowCenter", "windowWidth")


def test_curved_params_layout_matches_header(tmp_path):
    probe = tmp_path / "probe.c"
    offs = ", ".join(f"offsetof(svr_curved_params, {f})" for f in FIELDS)
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "svr_render.h"\n'
                     f'int main(void){{printf("{"%zu " * (len(FIELDS) + 3)}\\n", sizeof(svr_curved_params), {offs}, '
                     '(size_t)SVR_CURVED_STRAIGHTENED, (size_t)SVR_CURVED_CROSS);return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["/usr/bin/gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    P = L.CurvedParams
    assert got == [C.sizeof(P)] + [getattr(P, f).offset for f in FIELDS] + [L.CURVED_STRAIGHTENED, L.CURVED_CROSS]


LINE = np.array([[0.0, -4.0, 0.0], [0.0, 4.0, 0.0]], np.float32)


def test_argument_errors_are_reported_before_any_cuda_call():
    lib = L.load()
    vol = S.host_volume_struct((8, 8, 8))
    out = C.c_void_p(16)  # never dereferenced: every call below fails its checks first
    inf, nan = float("inf"), float("nan")

    def call(img=out, value=out, volume=vol, params=True, points=LINE, n=None, **kw):
        p = S.straightened_curve(8, 8, 1.0, up=(1.0, 0.0, 0.0), thickness=4.0)
        for k, v in kw.items():
            if k == "up":
                p.up[:] = v
            else:
                setattr(p, k, v)
        pts = None if points is None else np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1, 3))
        rc = lib.svr_render_curved(img, value, C.byref(volume) if volume is not None else None, C.byref(p) if params else None,
                                   None if pts is None else pts.ctypes.data, len(pts) if n is None else n)
        return rc, lib.svr_last_error().decode()

    assert call(img=None, value=None)[0] != 0
    bad = [dict(volume=None), dict(params=False), dict(points=None, n=2), dict(img=None, value=None),
           dict(points=LINE[:1]), dict(points=LINE, n=1), dict(points=np.zeros(((1 << 20) + 1, 3), np.float32)),
           dict(points=[[0, 0, 0], [nan, 1, 0]]), dict(points=[[0, 0, 0], [inf, 1, 0]]), dict(points=[[1, 2, 3]] * 5),
           dict(up=(nan, 0, 0)), dict(up=(0, inf, 0)), dict(up=(0, 0, 0)), dict(up=(0, 1, 0)), dict(up=(1e-8, -3, 0)),
           dict(points=[[0, 0, 0], [0, 0.4, 0]]),  # L = 0.4 < half a station
           dict(layout=-1), dict(layout=2), dict(imageW=0), dict(imageH=0), dict(imageW=16385), dict(imageH=16385),
           dict(count=0), dict(count=65536), dict(mode=-1), dict(mode=3),
           dict(pixelSpacing=0.0), dict(pixelSpacing=-1.0), dict(pixelSpacing=inf), dict(pixelSpacing=nan),
           dict(stationSpacing=0.0), dict(stationSpacing=-1.0), dict(stationSpacing=inf), dict(stationSpacing=nan),
           dict(angle0=inf), dict(angle0=nan), dict(angleStep=inf), dict(angleStep=nan),
           dict(thickness=-1.0), dict(thickness=inf), dict(thickness=nan), dict(sampleSpacing=0.0), dict(sampleSpacing=-1.0),
           dict(sampleSpacing=inf), dict(sampleSpacing=nan), dict(thickness=65537.0, sampleSpacing=1.0),
           dict(windowWidth=0.0), dict(windowWidth=-1.0), dict(windowWidth=inf), dict(windowWidth=nan), dict(windowCenter=nan),
           dict(layout=L.CURVED_CROSS, count=0), dict(layout=L.CURVED_CROSS, up=(0, 1, 0))]
    for kw in bad:
        rc, msg = call(**kw)
        assert rc != 0, kw
        assert "svr_render_curved" in msg, (kw, msg)


def test_curve_frames_argument_errors():
    lib = L.load()
    up = np.array([1, 0, 0], np.float32)
    outbuf = np.zeros((4, 4, 4), np.float32)

    def call(points=LINE, n=None, upv=up, spacing=1.0, stations=4, out=outbuf):
        pts = None if points is None else np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1, 3))
        rc = lib.svr_curve_frames(None if pts is None else pts.ctypes.data, len(pts) if n is None else n,
                                  None if upv is None else np.ascontiguousarray(upv, np.float32).ctypes.data, C.c_float(spacing), stations,
                                  None if out is None else out.ctypes.data)
        return rc, lib.svr_last_error().decode()

    assert call()[0] == 0
    nan = float("nan")
    bad = [dict(points=None, n=2), dict(upv=None), dict(out=None), dict(n=1), dict(points=[[0, 0, 0], [nan, 0, 0]]),
           dict(points=[[0, 0, 0]] * 3), dict(upv=[0, 0, 0]), dict(upv=[0, 2, 0]), dict(upv=[nan, 0, 0]), dict(spacing=0.0),
           dict(spacing=nan), dict(spacing=100.0), dict(stations=0)]
    for kw in bad:
        rc, msg = call(**kw)
        assert rc != 0, kw
        assert "svr_curve_frames" in msg, (kw, msg)


def frames_f64(points, up, spacing, n):
    """The frame rule of include/svr_render.h restated in float64 numpy: (n, 4, 4)."""
    P = np.asarray(points, np.float32).astype(np.float64).reshape(-1, 3)
    keep = np.ones(len(P), bool)
    keep[1:] = np.any(P[1:] != P[:-1], axis=1)
    P = P[keep]
    S_ = np.concatenate([[0.0], np.cumsum(np.sqrt(((P[1:] - P[:-1]) ** 2).sum(1)))])
    L_, D, M = S_[-1], float(np.float32(spacing)), len(P)

    def seg(s):
        return min(max(int(np.searchsorted(S_, s, side="right")) - 1, 0), M - 2)

    def c(s):
        m = seg(s)
        return P[m] + ((s - S_[m]) / (S_[m + 1] - S_[m])) * (P[m + 1] - P[m])

    out = np.zeros((n, 4, 4))
    r = None
    for i in range(n):
        s = (i + 0.5) * D
        if s > L_:
            break
        ci = c(s)
        d = c(min(s + D, L_)) - c(max(s - D, 0.0))
        if not d.any():
            m = seg(s)
            d = P[m + 1] - P[m]
        ti = d / np.linalg.norm(d)
        if r is None:
            u = np.asarray(up, np.float32).astype(np.float64)
            r = u - u.dot(ti) * ti
            r /= np.linalg.norm(r)
        else:
            v1 = ci - cp
            rl, tl = r, tp
            if v1.dot(v1) != 0:
                rl = r - 2 / v1.dot(v1) * v1.dot(r) * v1
                tl = tp - 2 / v1.dot(v1) * v1.dot(tp) * v1
            v2 = ti - tl
            if v2.dot(v2) != 0:
                rl = rl - 2 / v2.dot(v2) * v2.dot(rl) * v2
            r = rl - rl.dot(ti) * ti
            r /= np.linalg.norm(r)
        out[i, 0, :3], out[i, 0, 3] = ci, 1
        out[i, 1, :3], out[i, 2, :3], out[i, 3, :3] = ti, r, np.cross(ti, r)
        cp, tp = ci, ti
    return out


def random_polyline(rng, n):
    steps = rng.normal(size=(n - 1, 3)) * 0.6 + np.array([0.5, 0.2, 0.1])
    return np.concatenate([np.zeros((1, 3)), np.cumsum(steps, axis=0)]).astype(np.float32)


@pytest.mark.parametrize("seed", range(6))
def test_curve_frames_match_a_float64_restatement(seed):
    rng = np.random.default_rng(seed)
    pts = random_polyline(rng, 40)
    if seed % 2:  # repeated points
        idx = np.sort(rng.integers(0, len(pts), 12))
        pts = np.insert(pts, idx, pts[idx], axis=0)
    up = (0.3, -0.2, 1.0)
    spacing = float(rng.uniform(0.2, 1.5))
    n = int(S.polyline_length(pts) / spacing) + 5  # a few stations past the end
    got = S.curve_frames(pts, up, spacing, n)
    want = frames_f64(pts, up, spacing, n)
    assert np.abs(got - want).max() <= 1e-6 * max(1.0, np.abs(want).max())
    assert got[-1, 0, 3] == 0 and got[0, 0, 3] == 1


def test_a_curve_that_doubles_back():
    """Out along x and back: at the turn the central difference is zero and the segment's direction is used."""
    pts = np.array([[0, 0, 0], [2, 0, 0], [4, 0, 0], [4, 0, 0], [2, 0, 0], [0, 0, 0]], np.float32)
    got = S.curve_frames(pts, (0, 0, 1), 1.0, 9)
    want = frames_f64(pts, (0, 0, 1), 1.0, 9)
    assert np.abs(got - want).max() <= 1e-6
    assert np.all(got[:8, 0, 3] == 1) and got[8, 0, 3] == 0
    assert np.allclose(got[:4, 1, :3], [1, 0, 0]) and np.allclose(got[4:8, 1, :3], [-1, 0, 0])
    pts2 = np.array([[0, 0, 0], [1, 0, 0], [0, 0, 0]], np.float32)  # station at the turn: c(2) - c(0) = 0
    f = S.curve_frames(pts2, (0, 0, 1), 1.0, 2)
    assert np.abs(f - frames_f64(pts2, (0, 0, 1), 1.0, 2)).max() <= 1e-6
    assert np.allclose(f[1, 1, :3], [-1, 0, 0])  # the segment of s = 1.5, the second one


def test_straight_line_gives_a_constant_frame():
    a, d = np.array([1.0, -2.0, 0.5]), np.array([2.0, 3.0, -1.0]) / np.sqrt(14.0)
    pts = np.array([a, a + 10 * d, a + 30 * d], np.float32)
    f = S.curve_frames(pts, (0, 0, 1), 0.7, 50)
    L_ = S.polyline_length(pts)
    valid = (np.arange(50) + 0.5) * np.float64(np.float32(0.7)) <= L_
    assert np.array_equal(f[:, 0, 3] == 1, valid)
    s = (np.arange(50)[valid] + 0.5) * np.float64(np.float32(0.7))
    cs = pts[0].astype(np.float64) + s[:, None] * (pts[2].astype(np.float64) - pts[0]) / np.linalg.norm(pts[2].astype(np.float64) - pts[0])
    assert np.abs(f[valid, 0, :3] - cs).max() <= 1e-5
    for k in (1, 2, 3):
        assert np.abs(f[valid, k, :3] - f[0, k, :3]).max() <= 1e-6
    assert np.all(f[~valid] == 0)


def test_frames_are_orthonormal():
    pts = random_polyline(np.random.default_rng(5), 200)
    f = S.curve_frames(pts, (0, 1, 0), 0.3, 400)
    v = f[f[:, 0, 3] == 1][:, 1:, :3].astype(np.float64)
    gram = np.einsum("nij,nkj->nik", v, v)
    assert np.abs(gram - np.eye(3)).max() <= 1e-6
    assert np.abs(np.cross(v[:, 0], v[:, 1]) - v[:, 2]).max() <= 1e-6


def test_planar_arc_has_no_twist():
    u = np.linspace(0, 1.5 * np.pi, 2000)
    pts = np.stack([10 * np.cos(u), 10 * np.sin(u), np.full_like(u, 3.0)], 1).astype(np.float32)
    f = S.curve_frames(pts, (0, 0, 1), 0.5, 100)
    v = f[:, 0, 3] == 1
    assert v.sum() == 94
    assert np.abs(f[v, 2, :3] - [0, 0, 1]).max() <= 1e-6


def test_helix_frame_turns_at_the_torsion_rate():
    """On a helix (radius R, pitch 2 pi k) the rotation-minimising frame turns against the Frenet frame at d(phi)/ds = -tau,
    tau = k / (R^2 + k^2).  Bound: the polyline has V vertices per turn, so its arc length per radian of u is the chord
    sqrt((2R sin(du/2))^2 + (k du)^2) / du rather than sqrt(R^2 + k^2): the rate in the polyline's arc length differs from tau by
    the relative amount R^2 du^2 / (24 (R^2 + k^2)) (8e-8 here).  The frames are those of the polyline, which turns only at its
    vertices: double reflection over a station step D follows the true RMF with an error of order (kappa D)^4 per step
    (Wang et al. 2008), 1e-7 here, and the least-squares slope over the many stations adds rounding only.  1e-4 relative
    leaves three orders of margin for both."""
    R, k, turns, V = 12.0, 3.0, 3, 4096
    u = np.linspace(0, 2 * np.pi * turns, V * turns + 1)
    pts = np.stack([R * np.cos(u), R * np.sin(u), k * u], 1).astype(np.float32)
    D = 0.25
    f = S.curve_frames(pts, (0, 0, 1), D, 2000)
    v = f[:, 0, 3] == 1
    c, t, r = f[v, 0, :3].astype(np.float64), f[v, 1, :3].astype(np.float64), f[v, 2, :3].astype(np.float64)
    N = -np.stack([c[:, 0], c[:, 1], np.zeros(len(c))], 1)
    N /= np.linalg.norm(N, axis=1, keepdims=True)
    B = np.cross(t, N)
    phi = np.unwrap(np.arctan2((r * B).sum(1), (r * N).sum(1)))
    s = (np.arange(len(phi)) + 0.5) * D
    slope = np.polyfit(s, phi, 1)[0]
    tau = k / (R * R + k * k)
    assert abs(slope + tau) <= 1e-4 * tau, (slope, -tau)


def test_stations_past_the_end_are_invalid():
    f = S.curve_frames(LINE, (1, 0, 0), 1.0, 12)
    assert np.all(f[:8, 0, 3] == 1) and np.all(f[8:] == 0)


N_VOL = 24


def _ct_orc(fmt=L.VOXEL_F32, vol=None, seed=3):
    rng = np.random.default_rng(seed)
    d = rng.random((N_VOL,) * 3, dtype=np.float32)
    vox = S.encode_voxels(d, fmt)
    vol = vol or S.host_volume_struct((N_VOL,) * 3)
    return vox, vol


def test_straight_centerline_equals_the_slice_restatement():
    """A straightened CPR along y with up = +x equals the axial slice through the same voxel plane (slab along -z: MAX and MIN
    exactly, MEAN sums in reverse order); cross-sections along z with up = +x equal the axial stack, for every mode."""
    n = N_VOL
    vox, vol = _ct_orc()
    sorc = SO.oracle(vox, L.VOXEL_F32, (n, n, n), vol)
    corc = CO.oracle(vox, L.VOXEL_F32, (n, n, n), vol)
    iz = 9
    z0 = iz + 0.5 - n / 2
    line_y = np.array([[0, -n / 2, z0], [0, n / 2, z0]], np.float32)
    line_z = np.array([[0, 0, -n / 2], [0, 0, n / 2]], np.float32)
    for thick in (0, 6):
        for mode in ("max", "min", "mean"):
            want = SO.slices(sorc, S.axis_slice((n, n, n), (1, 1, 1), "z", iz, thickness_voxels=thick, mode=mode))[0]
            p = S.straightened_curve(n, n, 1.0, up=(1, 0, 0), thickness=thick, sample_spacing=1.0, mode=mode)
            got = CO.curved(corc, p, line_y)[0]
            if mode == "mean":
                assert np.abs(got - want).max() <= 4 * np.spacing(np.float32(1)), mode
            else:
                assert np.array_equal(got, want), (thick, mode)
            want = SO.slices(sorc, S.axis_slice((n, n, n), (1, 1, 1), "z", 0, thickness_voxels=thick, count=n, mode=mode))[0]
            p = S.curve_cross_sections(n, n, n, 1.0, 1.0, up=(1, 0, 0), thickness=thick, sample_spacing=1.0, mode=mode)
            assert np.array_equal(CO.curved(corc, p, line_z)[0], want), (thick, mode)


def test_outside_pixels_and_invalid_stations_have_alpha_zero():
    n = N_VOL
    vox, vol = _ct_orc(L.VOXEL_U8)
    orc = CO.oracle(vox, L.VOXEL_U8, (n, n, n), vol)
    line = np.array([[0, -n / 2, 0], [0, n / 2, 0]], np.float32)
    for thick in (0, 4):
        p = S.straightened_curve(2 * n, n + 6, 1.0, up=(1, 0, 0), thickness=thick, window=(0.5, 1.0))
        value, u8 = CO.curved(orc, p, line)
        x = np.arange(2 * n) + 0.5 - n
        inside = np.abs(x) <= n / 2
        assert np.all(u8[0, :n, inside, 3] == 255) and np.all(u8[0, :n, ~inside] == 0) and np.all(value[0, :n, ~inside] == 0)
        assert np.all(u8[0, n:] == 0) and np.all(value[0, n:] == 0)  # stations past the end
