"""GPU tests of the intensity projections (svr_render_projection): parity with the CPU restatement
(tests/projection_oracle.cpp, the CPU oracle's rays and texture filter), bit-exact macrocell skipping, band splits, scene
changes, no effect on the other renderers, the canvas's projection mode and the headless driver.  The reference has no
projection mode, so the CPU restatement and closed forms are the only checkers.  Every option a test changes is restored
(the session's renderer is shared)."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S
from sunvolumerender_b200.canvas import Canvas

import _projection_oracle as PO
from _gpu_common import setup, small_config

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEP = S.raycast_step_size()
MODES = ("max", "min", "mean")
SLAB = (-0.3, 0.3)


@pytest.fixture(autouse=True)
def restore_options(renderer):
    saved = {k: renderer.get_option(k) for k in range(L.OPT_PT_DENOISE + 1)}
    yield
    for k, v in saved.items():
        renderer.set_option(k, v)


def project(r, mode, window=(0.5, 1.0), phase=0, stride=1, img_fill=0, value_fill=0.0):
    H, W = r.camera.imageH, r.camera.imageW
    out = torch.full((H * W,), value_fill, dtype=torch.float32, device="cuda")
    r.img.fill_(img_fill)
    rows = r.render_projection(mode, window, STEP, out=out, phase=phase, stride=stride)
    torch.cuda.synchronize()
    return out.view(H, W).clone(), r.ldr_image().clone(), rows


def oracle_of(r, fmt, vox, dims=None):
    n = vox.shape[0]
    return PO.oracle(vox, fmt, dims or (n, n, n), r.volume, r.camera)


def check_vs_oracle(value, u8, ref_value, ref_u8):
    d = np.abs(value.cpu().numpy() - ref_value)
    assert d.mean() < 5e-5 and (d < 1e-4).mean() >= 0.99, (float(d.mean()), float((d < 1e-4).mean()))
    du8 = np.abs(u8.cpu().numpy().astype(int) - ref_u8.astype(int)).max()
    assert du8 <= 2, int(du8)


def oblique_camera(n, w, h):
    return S.look_at_camera((0.9 * n, 0.7 * n, 1.1 * n), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), fovx=45.0, image_w=w, image_h=h)


@pytest.mark.parametrize("gen,fmt", [(L.GEN_SPHERE, L.VOXEL_U16), (L.GEN_CT, L.VOXEL_U8)])
@pytest.mark.parametrize("mode", MODES)
def test_matches_cpu_restatement(renderer, gen, fmt, mode):
    cfg = small_config(gen=gen, fmt=fmt)
    vox = setup(renderer, cfg)
    if mode == "min":  # every ray through the whole box meets air (0): a slab inside the body
        renderer.set_volume_params(x_clip=SLAB, y_clip=SLAB, z_clip=SLAB)
    window = (0.4, 0.7)
    value, u8, _ = project(renderer, mode, window)
    ref_value, ref_u8 = PO.project(oracle_of(renderer, fmt, vox), mode, STEP, window)
    assert ref_value.max() > (0.01 if mode == "min" else 0.1)
    check_vs_oracle(value, u8, ref_value, ref_u8)


def _tie_volume(n, fmt, seed=7):
    """Blocks of 5 voxels holding one of four integer levels: the running maximum / minimum often equals a cell's bound."""
    rng = np.random.default_rng(seed)
    levels = np.array([0, 60, 61, 200], np.int64) * (257 if fmt == L.VOXEL_U16 else 1)
    b = (n + 4) // 5
    blocks = levels[rng.integers(0, 4, size=(b, b, b))]
    vox = np.repeat(np.repeat(np.repeat(blocks, 5, 0), 5, 1), 5, 2)[:n, :n, :n]
    return np.ascontiguousarray(vox.astype(np.uint8 if fmt == L.VOXEL_U8 else np.uint16))


VOLUMES = [("ct", L.VOXEL_U8), ("ct", L.VOXEL_U16), ("ct", L.VOXEL_F16), ("ct", L.VOXEL_F32), ("ties", L.VOXEL_U8), ("ties", L.VOXEL_U16)]


@pytest.mark.parametrize("kind,fmt", VOLUMES)
def test_skipping_is_bit_exact(renderer, kind, fmt):
    n, w, h = 64, 96, 80
    setup(renderer, small_config(gen=L.GEN_CT, fmt=fmt, w=w, h=h))
    if kind == "ties":
        renderer.load_volume(_tie_volume(n, fmt), fmt, (n, n, n))
    for cam, clip in ((S.default_camera((n, n, n), w, h), (-1.0, 1.0)), (oblique_camera(n, w, h), (-1.0, 1.0)), (oblique_camera(n, w, h), SLAB)):
        renderer.set_camera(cam)
        renderer.set_volume_params(x_clip=clip, y_clip=clip, z_clip=clip)
        for mode in MODES:
            renderer.set_option(L.OPT_RC_SKIP, 0)
            ref, ref_u8, _ = project(renderer, mode)
            assert mode == "min" or float(ref.max()) > 0.05
            renderer.set_option(L.OPT_RC_SKIP, 1)
            for cell in (4, 8, 16, 32):
                renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
                got, got_u8, _ = project(renderer, mode)
                assert torch.equal(got, ref), (mode, cell, int((got != ref).sum()))
                assert torch.equal(got_u8, ref_u8), (mode, cell)


def test_skipping_skips(renderer):
    """Skipping leaves the step count alone and removes a substantial share of the taps of MIP and AIP on the small CT.  The
    first B200 run skipped 0.44 of the steps for MIP, 0.52 for AIP and 0.82 for MinIP (air is 0: once a ray has met it, every
    cell is skippable); the bounds leave room for the generator's other seeds."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_COUNTERS, 1)
    counts = {}
    for mode in MODES:
        for skip in (0, 1):
            renderer.set_option(L.OPT_RC_SKIP, skip)
            renderer.reset_counters()
            project(renderer, mode)
            counts[mode, skip] = renderer.counters()
    print({f"{m} skip={k}": {n: c[n] for n in ("steps", "skipped", "shade_taps", "cells")} for (m, k), c in counts.items()})
    for mode in MODES:
        off, on = counts[mode, 0], counts[mode, 1]
        assert off["steps"] == on["steps"] and off["paths"] == on["paths"] == cfg.width * cfg.height
        assert off["skipped"] == 0 and off["shade_taps"] == off["steps"]
        assert on["shade_taps"] + on["skipped"] == on["steps"]
    for mode in ("max", "mean"):
        on, off = counts[mode, 1], counts[mode, 0]
        assert on["skipped"] > 0.3 * on["steps"], (mode, on)
        assert on["shade_taps"] < 0.7 * off["shade_taps"], (mode, on, off)


@pytest.mark.parametrize("stride", [3, 4])
def test_bands_tile_the_frame(renderer, stride):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, w=150, h=101)
    setup(renderer, cfg)
    for mode in MODES:
        full, full_u8, rows = project(renderer, mode, (0.3, 0.5))
        assert rows == renderer.get_option(L.OPT_RC_BLOCK) // 16
        value = torch.full_like(full, -7.0)
        img = torch.zeros_like(full_u8)
        covered = torch.zeros(full.shape, dtype=torch.int32, device="cuda")
        for phase in range(stride):
            part, part_u8, rows = project(renderer, mode, (0.3, 0.5), phase, stride, img_fill=0, value_fill=-7.0)
            assert rows == renderer.get_option(L.OPT_RC_BLOCK) // 16
            written = part_u8[..., 3] == 255
            assert torch.equal(written, part != -7.0)
            covered += written.int()
            value[written] = part[written]
            img[written] = part_u8[written]
        assert int(covered.min()) == 1 and int(covered.max()) == 1
        assert torch.equal(value, full) and torch.equal(img, full_u8)


def test_camera_inside_the_volume(renderer):
    """No samples behind the camera: t0 = max(tNear, 0)."""
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8)
    vox = setup(renderer, cfg)
    renderer.set_camera(S.make_camera((3.0, -2.0, 10.0), (1, 0, 0), (0, 1, 0), (0, 0, 1), 60.0, 0.0, 1.0, 1.0, cfg.width, cfg.height))
    orc = oracle_of(renderer, cfg.fmt, vox)
    for mode in MODES:
        value, u8, _ = project(renderer, mode)
        ref_value, ref_u8 = PO.project(orc, mode, STEP)
        check_vs_oracle(value, u8, ref_value, ref_u8)


@pytest.mark.parametrize("on_device", [0, 1])
def test_new_voxels_are_seen(renderer, on_device):
    """svr_volume_upload of other voxels (host copy, or the fused device path that reduces the ranges in the same pass): the
    projection follows the new voxels, with skipping on."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    for mode in MODES:
        project(renderer, mode)  # ranges of the CT
    sphere = S.sphere_volume(cfg.n, L.VOXEL_U8)
    renderer.upload_volume(torch.from_numpy(sphere.reshape(-1).copy()).cuda() if on_device else sphere)
    orc = oracle_of(renderer, cfg.fmt, sphere)
    for mode in MODES:
        value, u8, _ = project(renderer, mode)
        ref_value, ref_u8 = PO.project(orc, mode, STEP)
        check_vs_oracle(value, u8, ref_value, ref_u8)
        renderer.set_option(L.OPT_RC_SKIP, 0)
        assert torch.equal(project(renderer, mode)[0], value)
        renderer.set_option(L.OPT_RC_SKIP, 1)


def test_clip_planes_and_density_scale(renderer):
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8)
    vox = setup(renderer, cfg)
    renderer.set_volume_params(x_clip=(-0.5, 0.9), z_clip=(-1.0, 0.2))
    one = {m: project(renderer, m)[0] for m in MODES}
    orc = oracle_of(renderer, cfg.fmt, vox)
    for mode in MODES:
        value, u8, _ = project(renderer, mode)
        check_vs_oracle(value, u8, *PO.project(orc, mode, STEP))
    renderer.set_volume_params(density_scale=2.0)
    for mode in MODES:
        assert torch.equal(project(renderer, mode)[0], 2.0 * one[mode]), mode
    # constant slab, clip planes inset by two voxels: every crossing ray projects to the constant in every mode
    n, c = cfg.n, np.float32(0.37)
    renderer.load_volume(np.full((n, n, n), c, np.float32), L.VOXEL_F32, (n, n, n))
    inset = 4.0 / n
    renderer.set_volume_params(x_clip=(-1 + inset, 1 - inset), y_clip=(-1 + inset, 1 - inset), z_clip=(-1 + inset, 0.5))
    got = {m: project(renderer, m)[0].cpu().numpy() for m in MODES}
    crossing = got["max"] != 0
    assert crossing.mean() > 0.2
    for m in MODES:
        assert np.abs(got[m][crossing] - c).max() <= 1e-6 and np.all(got[m][~crossing] == 0), m


def _grid_cell(r):
    dims, cell = (C.c_int32 * 3)(), C.c_int32(0)
    L.check(r.lib.svr_grid_info(dims, C.byref(cell)), "svr_grid_info")
    return int(cell.value)


def test_other_renderers_are_unchanged(renderer):
    """A projection between setup and render changes neither a path-traced nor a ray-cast image, and keeps the macrocell
    edge the path tracer chose (automatic size)."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_MACROCELL_SIZE, 0)

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
    for mode in MODES:
        setup(renderer, cfg)
        renderer.set_option(L.OPT_MACROCELL_SIZE, 0)
        project(renderer, mode)
        hdr, img = pathtrace()
        assert torch.equal(hdr, hdr0) and torch.equal(img, img0), mode
        project(renderer, mode)
        assert _grid_cell(renderer) == cell0
        hdr, img = pathtrace()
        assert torch.equal(hdr, hdr0) and torch.equal(img, img0), mode
        project(renderer, mode)
        rc, rc_u8 = raycast()
        assert torch.equal(rc, rc0) and torch.equal(rc_u8, rc_u80), mode


def test_canvas_projection_mode(renderer):
    W = H = 128
    cfg = small_config(n=64, w=W, h=H, gen=L.GEN_CT, fmt=L.VOXEL_U16)
    setup(renderer, cfg)
    canvas = Canvas(W, H)
    try:
        canvas.set_volume(renderer.volume, cfg.extent, STEP)  # no transfer function: projection mode does not need one
        assert canvas.lib.svr_canvas_set_render_mode(canvas.c, 3) != 0
        assert b"svr_canvas_set_render_mode" in canvas.lib.svr_last_error()
        before = canvas.paint_count
        canvas.set(render_mode=L.RENDER_MODE_PROJECTION)
        assert canvas.paint_count == before + 1 and canvas.frame_no == 0
        before = canvas.paint_count
        canvas.set_projection("mean", (0.2, 0.3))
        assert canvas.paint_count == before + 1 and canvas.frame_no == 0  # one repaint, then the restart
        canvas.mouse_press(10, 10, L.BUTTON_LEFT)
        canvas.mouse_move(30, 20, L.BUTTON_LEFT)
        canvas.paint()
        assert canvas.frame_no == 1
        for mode, window in (("mean", (0.2, 0.3)), ("max", (0.5, 1.0)), ("min", (0.1, 0.4))):
            if mode != "mean":
                canvas.set_projection(mode, window)
                canvas.paint()
            mine = canvas.image()
            renderer.set_camera(canvas.camera())
            value, u8, _ = project(renderer, mode, window)
            assert mode == "min" or float(value.max()) > 0.05
            assert np.array_equal(mine, u8.cpu().numpy()), mode
        with pytest.raises(L.SvrError):
            canvas.set_projection("max", (0.5, 0.0))
    finally:
        canvas.close()


def test_headless_driver_writes_the_python_image(renderer, tmp_path):
    exe = os.path.join(ROOT, "tools", "svr_headless")
    if not os.path.exists(exe):
        pytest.skip("tools/svr_headless was not built (make tools)")
    n, W, H = 64, 96, 80
    out = str(tmp_path / "mip")
    subprocess.check_call([exe, "--config", "C1", "--n", str(n), "--w", str(W), "--h", str(H), "--mode", "mip", "--window", "0.4,0.6",
                           "--reps", "1", "--out", out], cwd=str(tmp_path))
    with open(out + ".ppm", "rb") as f:
        data = f.read()
    ppm = np.frombuffer(data[-W * H * 3:], np.uint8).reshape(H, W, 3)[::-1]
    # the driver's scene: C1's generator at n = 64, spacing 1, and its camera (svr_headless.cpp), in the same float arithmetic
    setup(renderer, small_config(n=n, w=W, h=H, gen=L.GEN_SPHERE, fmt=L.VOXEL_U8))
    renderer.load_volume(renderer.generate_volume(L.GEN_SPHERE, L.VOXEL_U8, n, 1234), L.VOXEL_U8, (n, n, n))
    libm = C.CDLL("libm.so.6")
    libm.tanf.restype, libm.tanf.argtypes = C.c_float, [C.c_float]
    cam = L.Camera()
    cam.imageW, cam.imageH, cam.exposure, cam.apeture, cam.focalLength = W, H, 1.0, 0.0, 1.0
    cam.aspectRatio = float(np.float32(W) / np.float32(H))
    cam.tanFovxOverTwo = libm.tanf(float(np.float32(float(np.float32(45.0) * np.float32(0.5)) * math.pi / float(np.float32(180.0)))))
    cam.pos = L.Vec3(0.0, 0.0, float(np.float32(1.5 * n / (2.0 * math.tan(45.0 * 0.5 * math.pi / 180.0)))))
    cam.u, cam.v, cam.w = L.Vec3(1, 0, 0), L.Vec3(0, 1, 0), L.Vec3(0, 0, 1)
    renderer.set_camera(cam)
    step = float(np.float32(0.5) * np.sqrt(np.float32(3.0)))
    renderer.img.zero_()
    renderer.render_projection("max", (0.4, 0.6), step)
    torch.cuda.synchronize()
    mine = renderer.ldr_image().cpu().numpy()[..., :3]
    assert mine.max() > 100
    assert np.array_equal(ppm, mine)
