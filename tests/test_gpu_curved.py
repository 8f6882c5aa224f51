"""GPU tests of curved planar reformation (svr_render_curved): parity with the CPU restatement (tests/curved_oracle.cpp),
straight centerlines against slices bit for bit, a tube about a helix, the mirror at angle + pi, bit-exact macrocell skipping,
new voxels, the staging of the frame table across calls, no effect on the other renderers and the headless driver.  Every
option a test changes is restored (the session's renderer is shared)."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _curved_oracle as CO
from _gpu_common import setup, small_config
from test_gpu_projection import _tie_volume, check_vs_oracle

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODES = ("max", "min", "mean")
STEP = S.raycast_step_size()


@pytest.fixture(autouse=True)
def restore_options(renderer):
    saved = {k: renderer.get_option(k) for k in range(L.OPT_PT_DENOISE + 1)}
    yield
    for k, v in saved.items():
        renderer.set_option(k, v)


def render(r, points, params):
    value, img = r.render_curved(points, params)
    torch.cuda.synchronize()
    return value, img


def s_curve(n, m=400, phase=0.0):
    """A smooth curve through an n^3 volume (spacing 1, centred on the origin), m points."""
    u = np.linspace(0.0, 1.0, m)
    return np.stack([0.22 * n * np.sin(2 * np.pi * u + phase), (u - 0.5) * 0.8 * n, 0.15 * n * np.cos(np.pi * u + phase)], 1).astype(np.float32)


def straight(n, mode="max", thickness=0.0, count=1, h=None, window=(0.4, 0.7)):
    return S.straightened_curve(80, h or int(0.9 * n), 0.9, station_spacing=1.0, up=(0, 0, 1), count=count, angle0=0.3,
                                angle_step=0.8, thickness=thickness, sample_spacing=0.55, mode=mode, window=window)


def cross(n, mode="max", thickness=0.0, count=5):
    return S.curve_cross_sections(48, 40, count, 0.7, 0.17 * n, up=(0, 0, 1), angle=0.4, thickness=thickness, sample_spacing=0.55,
                                  mode=mode, window=(0.4, 0.7))


@pytest.mark.parametrize("gen,fmt", [(L.GEN_SPHERE, L.VOXEL_U16), (L.GEN_CT, L.VOXEL_U8)])
@pytest.mark.parametrize("mode", MODES)
def test_matches_cpu_restatement(renderer, gen, fmt, mode):
    cfg = small_config(gen=gen, fmt=fmt)
    vox = setup(renderer, cfg)
    n = cfg.n
    orc = CO.oracle(vox, fmt, (n, n, n), renderer.volume)
    pts = s_curve(n)
    for p in (straight(n, mode, 0.0, 2), straight(n, mode, 0.3 * n, 2), cross(n, mode, 0.0), cross(n, mode, 0.3 * n)):
        value, img = render(renderer, pts, p)
        ref_value, ref_u8 = CO.curved(orc, p, pts)
        assert ref_value.max() > 0.1 and (ref_u8[..., 3] == 255).mean() > 0.2
        check_vs_oracle(value, img, ref_value, ref_u8)
        # inclusion can flip only for a sample on the box's surface, where fp32 contraction moves it by an ulp
        assert (img[..., 3].cpu().numpy() != ref_u8[..., 3]).mean() <= 1e-3


DIMS = (40, 28, 20)


def _random_volume(fmt, seed=11):
    rng = np.random.default_rng(seed)
    nx, ny, nz = DIMS
    d = rng.random((nz, ny, nx), dtype=np.float32)
    return S.encode_voxels(d, fmt)


@pytest.mark.parametrize("fmt", [L.VOXEL_U8, L.VOXEL_F32])
def test_straight_centerlines_equal_slices_bit_for_bit(renderer, fmt):
    """Spacing 1, centerlines through voxel centres: a straightened CPR along y with up = +x is the axial slice (its slab runs
    along -z: MAX and MIN exactly, MEAN sums in reverse order), and cross-sections along z with up = +x are the axial stack."""
    setup(renderer, small_config())
    renderer.load_volume(_random_volume(fmt), fmt, DIMS)
    nx, ny, nz = DIMS
    iz = 7
    z0 = iz + 0.5 - nz / 2
    line_y = np.array([[0, -ny / 2, z0], [0, ny / 2, z0]], np.float32)
    line_z = np.array([[0, 0, -nz / 2], [0, 0, nz / 2]], np.float32)
    for skip in (0, 1):
        renderer.set_option(L.OPT_RC_SKIP, skip)
        for thick in (0, 6):
            for mode in MODES:
                want, want_u8 = renderer.render_slices(S.axis_slice(DIMS, (1, 1, 1), "z", iz, thickness_voxels=thick, mode=mode))
                got, got_u8 = render(renderer, line_y, S.straightened_curve(nx, ny, 1.0, up=(1, 0, 0), thickness=thick, sample_spacing=1.0,
                                                                         mode=mode))
                if mode == "mean":
                    assert torch.allclose(got, want, rtol=4e-7, atol=0), (skip, thick)
                else:
                    assert torch.equal(got, want) and torch.equal(got_u8, want_u8), (skip, thick, mode)
                want, want_u8 = renderer.render_slices(S.axis_slice(DIMS, (1, 1, 1), "z", 0, thickness_voxels=thick, count=nz, mode=mode))
                got, got_u8 = render(renderer, line_z, S.curve_cross_sections(nx, ny, nz, 1.0, 1.0, up=(1, 0, 0), thickness=thick,
                                                                           sample_spacing=1.0, mode=mode))
                assert torch.equal(got, want) and torch.equal(got_u8, want_u8), (skip, thick, mode)


HELIX_R, HELIX_K, TUBE_R = 14.0, 4.0, 3.0


def _helix(u):
    return np.stack([HELIX_R * np.cos(u), HELIX_R * np.sin(u), HELIX_K * u], 1)


def test_tube_about_a_helix(renderer):
    """A bright tube of radius R about a helix: in every straightened row its bright columns are one run centred on W/2 of
    half-width R / pixelSpacing +- 2 px, and every cross-section shows a centred disc of radius R +- 1 px."""
    from scipy.spatial import cKDTree

    n = 64
    setup(renderer, small_config())
    ax = np.arange(n) + 0.5 - n / 2
    zz, yy, xx = np.meshgrid(ax, ax, ax, indexing="ij")
    u_all = np.linspace(-4.0, 4.0, 20000)  # the tube runs past the CPR's centerline at both ends
    dist = cKDTree(_helix(u_all)).query(np.stack([xx.ravel(), yy.ravel(), zz.ravel()], 1))[0].reshape(n, n, n)
    vox = np.clip(0.5 + (TUBE_R - dist), 0.0, 1.0).astype(np.float32)  # 0.5 on the tube's surface
    renderer.load_volume(vox, L.VOXEL_F32, (n, n, n))
    pts = _helix(np.linspace(-3.0, 3.0, 3000)).astype(np.float32)
    ps = 0.5
    W = 48
    L_ = S.polyline_length(pts)
    H = int(L_ / 1.0)
    value = render(renderer, pts, S.straightened_curve(W, H, ps, station_spacing=1.0, up=(0, 0, 1), count=4, angle_step=0.7))[0].cpu().numpy()
    for j in range(4):
        for y in range(H):
            cols = np.nonzero(value[j, y] >= 0.5)[0]
            assert len(cols) and np.all(np.diff(cols) == 1), (j, y)
            centre, half = (cols[0] + cols[-1] + 1) / 2.0, (cols[-1] + 1 - cols[0]) / 2.0
            assert abs(centre - W / 2) <= 1.0 and abs(half - TUBE_R / ps) <= 2.0, (j, y, centre, half)
    count = 40
    p = S.curve_cross_sections(24, 24, count, 1.0, L_ / count, up=(0, 0, 1))
    value = render(renderer, pts, p)[0].cpu().numpy()
    x = np.arange(24) + 0.5 - 12
    rad = np.hypot(x[None, :], x[:, None])
    for j in range(count):
        bright = value[j] >= 0.5
        assert np.all(bright[rad <= TUBE_R - 1]) and not np.any(bright[rad >= TUBE_R + 1]), j


def test_the_image_at_angle_plus_pi_is_the_mirror(renderer):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16)
    setup(renderer, cfg)
    pts = s_curve(cfg.n)
    p = S.straightened_curve(96, 50, 0.6, station_spacing=1.0, up=(0, 0, 1), count=2, angle0=0.4, angle_step=math.pi)
    value, img = render(renderer, pts, p)
    a, b = value[0].cpu().numpy(), value[1].cpu().numpy()[:, ::-1]
    assert a.max() > 0.1
    d = np.abs(a - b)
    assert d.mean() < 5e-5 and (d < 1e-4).mean() >= 0.99


VOLUMES = [("ct", L.VOXEL_U8), ("ct", L.VOXEL_U16), ("ct", L.VOXEL_F16), ("ct", L.VOXEL_F32), ("ties", L.VOXEL_U8), ("ties", L.VOXEL_U16)]


@pytest.mark.parametrize("kind,fmt", VOLUMES)
def test_skipping_is_bit_exact(renderer, kind, fmt):
    n = 64
    setup(renderer, small_config(gen=L.GEN_CT, fmt=fmt))
    if kind == "ties":
        renderer.load_volume(_tie_volume(n, fmt), fmt, (n, n, n))
    pts = s_curve(n)
    for clip in ((-1.0, 1.0), (-0.3, 0.3)):
        renderer.set_volume_params(x_clip=clip, y_clip=clip, z_clip=clip)
        for mode in MODES:
            for p in (straight(n, mode, 0.45 * n, 2), cross(n, mode, 0.45 * n)):
                renderer.set_option(L.OPT_RC_SKIP, 0)
                ref, ref_u8 = render(renderer, pts, p)
                assert mode == "min" or clip[0] > -1.0 or float(ref.max()) > 0.05
                renderer.set_option(L.OPT_RC_SKIP, 1)
                for cell in (4, 8, 16, 32):
                    renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
                    got, got_u8 = render(renderer, pts, p)
                    assert torch.equal(got, ref), (clip, mode, p.layout, cell, int((got != ref).sum()))
                    assert torch.equal(got_u8, ref_u8), (clip, mode, p.layout, cell)


def test_skipping_skips(renderer):
    """Skipping leaves the step count alone and drops a share of the taps of MIP and AIP slabs on the small CT."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_COUNTERS, 1)
    n = cfg.n
    pts = s_curve(n)
    counts = {}
    for mode in MODES:
        p = straight(n, mode, 0.6 * n)
        for skip in (0, 1):
            renderer.set_option(L.OPT_RC_SKIP, skip)
            renderer.reset_counters()
            render(renderer, pts, p)
            counts[mode, skip] = renderer.counters()
    print({f"{m} skip={k}": {c_: c[c_] for c_ in ("paths", "steps", "skipped", "shade_taps", "cells")} for (m, k), c in counts.items()})
    for mode in MODES:
        off, on = counts[mode, 0], counts[mode, 1]
        assert off["steps"] == on["steps"] > 0 and off["paths"] == on["paths"] == p.imageW * p.imageH
        assert off["skipped"] == 0 and off["cells"] == 0 and off["shade_taps"] == off["steps"]
        assert on["shade_taps"] + on["skipped"] == on["steps"] and on["cells"] > 0
    for mode in ("max", "mean"):
        on = counts[mode, 1]
        assert on["skipped"] > 0.1 * on["steps"], (mode, on)
    # a slab of fewer than 32 samples does not walk (include/svr_render.h)
    renderer.set_option(L.OPT_RC_SKIP, 1)
    renderer.reset_counters()
    render(renderer, pts, straight(n, "max", 16 * 0.55))
    c = renderer.counters()
    assert c["cells"] == 0 and c["skipped"] == 0 and c["shade_taps"] == c["steps"] > 0, c


@pytest.mark.parametrize("on_device", [0, 1])
def test_new_voxels_are_seen(renderer, on_device):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    n = cfg.n
    pts = s_curve(n)
    for mode in MODES:
        render(renderer, pts, straight(n, mode, 0.4 * n))  # ranges of the CT
    sphere = S.sphere_volume(n, L.VOXEL_U8)
    renderer.upload_volume(torch.from_numpy(sphere.reshape(-1).copy()).cuda() if on_device else sphere)
    orc = CO.oracle(sphere, cfg.fmt, (n, n, n), renderer.volume)
    for mode in MODES:
        p = straight(n, mode, 0.4 * n)
        value, img = render(renderer, pts, p)
        check_vs_oracle(value, img, *CO.curved(orc, p, pts))
        renderer.set_option(L.OPT_RC_SKIP, 0)
        assert torch.equal(render(renderer, pts, p)[0], value)
        renderer.set_option(L.OPT_RC_SKIP, 1)


def test_calls_without_a_synchronise_between_them_keep_their_curves(renderer):
    """Each call stages its own frame table; a second call behind a long one must not overwrite what the first still reads."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16)
    setup(renderer, cfg)
    n = cfg.n
    a, b = s_curve(n), s_curve(n, 250, phase=1.3)
    slow = S.straightened_curve(512, 512, 0.1, station_spacing=0.08, up=(0, 0, 1), count=8, thickness=0.5 * n, sample_spacing=0.25)
    pa, pb = straight(n, "max", 0.2 * n, 3), cross(n, "mean", 0.2 * n, 7)
    ref_a, ref_b = render(renderer, a, pa), render(renderer, b, pb)
    for _ in range(2):
        renderer.render_curved(b, slow)  # keeps the stream busy behind the copies below
        got_a = renderer.render_curved(a, pa)
        got_b = renderer.render_curved(b, pb)
        got_a2 = renderer.render_curved(b, pa)
        torch.cuda.synchronize()
        assert torch.equal(got_a[0], ref_a[0]) and torch.equal(got_a[1], ref_a[1])
        assert torch.equal(got_b[0], ref_b[0]) and torch.equal(got_b[1], ref_b[1])
        assert not torch.equal(got_a2[0], ref_a[0])


def _grid_cell(r):
    dims, cell = (C.c_int32 * 3)(), C.c_int32(0)
    L.check(r.lib.svr_grid_info(dims, C.byref(cell)), "svr_grid_info")
    return int(cell.value)


def test_other_renderers_are_unchanged(renderer):
    """CPR calls between setup and render change neither a path-traced nor a ray-cast image, and keep the macrocell edge the
    path tracer chose (automatic size)."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_MACROCELL_SIZE, 0)
    pts = s_curve(cfg.n)

    def pathtrace():
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(8, 2)
        torch.cuda.synchronize()
        return renderer.hdr.clone(), renderer.img.clone()

    def raycast():
        out = torch.zeros(cfg.width * cfg.height * 4, dtype=torch.float32, device="cuda")
        renderer.render_raycasting_f32(out, STEP, img=renderer.img)
        torch.cuda.synchronize()
        return out, renderer.img.clone()

    hdr0, img0 = pathtrace()
    cell0 = _grid_cell(renderer)
    rc0, rc_u80 = raycast()
    for p in (straight(cfg.n, "max", 0.5 * cfg.n), straight(cfg.n), cross(cfg.n, "mean", 8.0)):
        setup(renderer, cfg)
        renderer.set_option(L.OPT_MACROCELL_SIZE, 0)
        render(renderer, pts, p)
        hdr, img = pathtrace()
        assert torch.equal(hdr, hdr0) and torch.equal(img, img0)
        render(renderer, pts, p)
        assert _grid_cell(renderer) == cell0
        hdr, img = pathtrace()
        assert torch.equal(hdr, hdr0) and torch.equal(img, img0)
        render(renderer, pts, p)
        rc, rc_u8 = raycast()
        assert torch.equal(rc, rc0) and torch.equal(rc_u8, rc_u80)


@pytest.mark.parametrize("slab", [0, 9])
def test_headless_driver_writes_the_python_image(renderer, tmp_path, slab):
    exe = os.path.join(ROOT, "tools", "svr_headless")
    if not os.path.exists(exe):
        pytest.skip("tools/svr_headless was not built (make tools)")
    n, W, H = 64, 96, 80
    pts = s_curve(n, 300)
    curve = tmp_path / "curve.txt"
    curve.write_text("\n".join(" ".join(repr(float(v)) for v in q) for q in pts))
    out = str(tmp_path / "cpr")
    subprocess.check_call([exe, "--config", "C1", "--n", str(n), "--w", str(W), "--h", str(H), "--mode", "cpr", "--curve", str(curve),
                           "--up", "0.2,0,1", "--slab", str(slab), "--window", "0.4,0.6", "--reps", "1", "--out", out], cwd=str(tmp_path))
    with open(out + ".ppm", "rb") as f:
        data = f.read()
    ppm = np.frombuffer(data[-W * H * 3:], np.uint8).reshape(H, W, 3)[::-1]
    # the driver's volume: C1's generator at n = 64, spacing 1 (svr_headless.cpp)
    setup(renderer, small_config(n=n, w=W, h=H, gen=L.GEN_SPHERE, fmt=L.VOXEL_U8))
    renderer.load_volume(renderer.generate_volume(L.GEN_SPHERE, L.VOXEL_U8, n, 1234), L.VOXEL_U8, (n, n, n))
    p = S.straightened_curve(W, H, 1.0, up=(0.2, 0, 1), thickness=float(slab), sample_spacing=1.0, window=(0.4, 0.6))
    mine = render(renderer, pts, p)[1][0].cpu().numpy()[..., :3]
    assert mine.max() > 100
    assert np.array_equal(ppm, mine)
