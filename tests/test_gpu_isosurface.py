"""GPU tests of the isosurface (svr_render_isosurface): parity with the CPU restatement (tests/isosurface_oracle.cpp, the CPU
oracle's rays, texture filter and gradient), bit-exact macrocell skipping, band splits, scene changes, no effect on the other
renderers and the headless driver.  The reference has no isosurface mode, so the CPU restatement and its closed forms
(tests/test_isosurface_cpu.py) are the only checkers.  Every option a test changes is restored (the session's renderer is
shared)."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _isosurface_oracle as IO
from _gpu_common import setup, small_config

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEP = S.raycast_step_size()
H_STEP = 0.5 * STEP
SLAB = (-0.3, 0.3)
SKIN, BONE = 0.15, 0.7
COLOR = (0.9, 0.8, 0.6)


@pytest.fixture(autouse=True)
def restore_options(renderer):
    saved = {k: renderer.get_option(k) for k in range(L.OPT_PT_DENOISE + 1)}
    yield
    for k, v in saved.items():
        renderer.set_option(k, v)


def iso(r, value, phase=0, stride=1, img_fill=0, surface_fill=0.0):
    H, W = r.camera.imageH, r.camera.imageW
    surface = torch.full((H * W * 4,), surface_fill, dtype=torch.float32, device="cuda")
    r.img.fill_(img_fill)
    rows = r.render_isosurface(value, STEP, COLOR, surface=surface, phase=phase, stride=stride)
    torch.cuda.synchronize()
    return surface.view(H, W, 4).clone(), r.ldr_image().clone(), rows


def oracle_of(r, fmt, vox):
    n = vox.shape[0]
    return IO.oracle(vox, fmt, (n, n, n), r.volume, r.camera)


def check_vs_oracle(surface, u8, ref_surface, ref_u8):
    """The hit / miss mask agrees on >= 99 % of the pixels.  Where both hit, the depth is within h (one sample: a 1-ulp
    difference of a texture coordinate can flip an 8-bit weight and so the sample that first reaches iso) and u8 within 2 LSB
    (the ray caster's bound: fast-math powf and normalisation) on >= 99 % of them.  Misses are (0, 0, 0, +inf) and a zero image
    on both sides."""
    s, u = surface.cpu().numpy(), u8.cpu().numpy().astype(int)
    hit, ref_hit = np.isfinite(s[..., 3]), np.isfinite(ref_surface[..., 3])
    assert ref_hit.mean() > 0.01
    assert (hit == ref_hit).mean() >= 0.99, float((hit == ref_hit).mean())
    both = hit & ref_hit
    dz = np.abs(s[..., 3][both] - ref_surface[..., 3][both])
    assert (dz <= H_STEP).mean() >= 0.99, float((dz <= H_STEP).mean())
    du = np.abs(u[both] - ref_u8[both].astype(int)).max(axis=1)
    assert (du <= 2).mean() >= 0.99, float((du <= 2).mean())
    miss = ~hit
    assert np.all(s[miss][:, :3] == 0) and np.all(s[miss][:, 3] == np.inf) and np.all(u[miss] == 0)


def oblique_camera(n, w, h):
    return S.look_at_camera((0.9 * n, 0.7 * n, 1.1 * n), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), fovx=45.0, image_w=w, image_h=h)


@pytest.mark.parametrize("gen,fmt", [(L.GEN_SPHERE, L.VOXEL_U16), (L.GEN_CT, L.VOXEL_U8)])
@pytest.mark.parametrize("value", [SKIN, BONE])
def test_matches_cpu_restatement(renderer, gen, fmt, value):
    cfg = small_config(gen=gen, fmt=fmt)
    vox = setup(renderer, cfg)
    for cam in (S.default_camera(cfg.extent, cfg.width, cfg.height), oblique_camera(cfg.n, cfg.width, cfg.height)):
        renderer.set_camera(cam)
        surface, u8, _ = iso(renderer, value)
        ref_surface, ref_u8 = IO.isosurface(oracle_of(renderer, fmt, vox), value, STEP, COLOR)
        check_vs_oracle(surface, u8, ref_surface, ref_u8)


def _tie_volume(n, fmt, seed=7):
    """Blocks of 5 voxels holding one of four integer levels: a cell's maximum often equals the threshold exactly."""
    rng = np.random.default_rng(seed)
    levels = np.array([0, 60, 61, 200], np.int64) * (257 if fmt == L.VOXEL_U16 else 1)
    b = (n + 4) // 5
    blocks = levels[rng.integers(0, 4, size=(b, b, b))]
    vox = np.repeat(np.repeat(np.repeat(blocks, 5, 0), 5, 1), 5, 2)[:n, :n, :n]
    return np.ascontiguousarray(vox.astype(np.uint8 if fmt == L.VOXEL_U8 else np.uint16))


# (volume, format, thresholds); the ties volume's 61 / 255 is one of its levels (u16: 61 * 257 / 65535, the same value)
VOLUMES = [("ct", L.VOXEL_U8, (SKIN, BONE)), ("ct", L.VOXEL_U16, (SKIN, BONE)), ("ct", L.VOXEL_F16, (SKIN, BONE)),
           ("ct", L.VOXEL_F32, (SKIN, BONE)), ("ties", L.VOXEL_U8, (61 / 255,)), ("ties", L.VOXEL_U16, (61 / 255,))]


@pytest.mark.parametrize("kind,fmt,values", VOLUMES)
def test_skipping_is_bit_exact(renderer, kind, fmt, values):
    n, w, h = 64, 96, 80
    setup(renderer, small_config(gen=L.GEN_CT, fmt=fmt, w=w, h=h))
    if kind == "ties":
        renderer.load_volume(_tie_volume(n, fmt), fmt, (n, n, n))
    for cam, clip in ((S.default_camera((n, n, n), w, h), (-1.0, 1.0)), (oblique_camera(n, w, h), (-1.0, 1.0)), (oblique_camera(n, w, h), SLAB)):
        renderer.set_camera(cam)
        renderer.set_volume_params(x_clip=clip, y_clip=clip, z_clip=clip)
        for value in values:
            renderer.set_option(L.OPT_RC_SKIP, 0)
            ref, ref_u8, _ = iso(renderer, value)
            assert float(torch.isfinite(ref[..., 3]).float().mean()) > 0.01, (value, clip)
            renderer.set_option(L.OPT_RC_SKIP, 1)
            for cell in (4, 8, 16, 32):
                renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
                got, got_u8, _ = iso(renderer, value)
                assert torch.equal(got, ref), (value, cell, int((got != ref).any(dim=2).sum()))
                assert torch.equal(got_u8, ref_u8), (value, cell)


def test_skipping_skips(renderer):
    """Skipping leaves the step count alone and drops a large share of the bone threshold's steps on the small CT (air and soft
    tissue lie below it).  The first B200 run skipped 0.91 of the steps at 0.7 (bone) and 0.70 at 0.15 (skin: only the air
    around the body lies below it); the bound leaves room for the generator's other seeds."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_COUNTERS, 1)
    counts = {}
    for value in (SKIN, BONE):
        for skip in (0, 1):
            renderer.set_option(L.OPT_RC_SKIP, skip)
            renderer.reset_counters()
            surface, _, _ = iso(renderer, value)
            counts[value, skip] = renderer.counters()
            counts[value, skip]["hits"] = int(torch.isfinite(surface[..., 3]).sum())
    print({f"iso={v} skip={k}": {n: c[n] for n in ("steps", "skipped", "shade_taps", "cells", "hits")} for (v, k), c in counts.items()})
    for value in (SKIN, BONE):
        off, on = counts[value, 0], counts[value, 1]
        assert off["steps"] == on["steps"] and off["paths"] == on["paths"] == cfg.width * cfg.height
        assert off["hits"] == on["hits"] > 0
        assert off["skipped"] == 0 and off["cells"] == 0 and off["shade_taps"] == off["steps"]
        assert on["shade_taps"] + on["skipped"] == on["steps"]
    on = counts[BONE, 1]
    assert on["skipped"] > 0.6 * on["steps"], on


@pytest.mark.parametrize("stride", [3, 4])
def test_bands_tile_the_frame(renderer, stride):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, w=150, h=101)
    setup(renderer, cfg)
    for value in (SKIN, BONE):
        full, full_u8, rows = iso(renderer, value)
        assert rows == renderer.get_option(L.OPT_RC_BLOCK) // 16
        surface = torch.full_like(full, -7.0)
        img = torch.zeros_like(full_u8)
        covered = torch.zeros(full.shape[:2], dtype=torch.int32, device="cuda")
        for phase in range(stride):
            part, part_u8, rows = iso(renderer, value, phase, stride, img_fill=0x11, surface_fill=-7.0)
            assert rows == renderer.get_option(L.OPT_RC_BLOCK) // 16
            # a written pixel has alpha 255 (hit) or 0 (miss) and a surface value that is never -7 (a unit normal or 0, depth)
            written = part_u8[..., 3] != 0x11
            assert torch.equal((part != -7.0).all(dim=2), written) and torch.equal((part == -7.0).all(dim=2), ~written)
            covered += written.int()
            surface[written] = part[written]
            img[written] = part_u8[written]
        assert int(covered.min()) == 1 and int(covered.max()) == 1
        assert torch.equal(surface, full) and torch.equal(img, full_u8)


def test_camera_inside_the_volume(renderer):
    """No samples behind the camera: t0 = max(tNear, 0).  From (3, -2, 10) (rho 0.63) the rays meet the 0.7 surface ahead; from
    (1, 2, 4) (rho 0.84) the camera sits inside the 0.5 solid and every ray hits at its first sample (the cap)."""
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8)
    vox = setup(renderer, cfg)
    for pos, value in (((3.0, -2.0, 10.0), 0.7), ((1.0, 2.0, 4.0), 0.5)):
        renderer.set_camera(S.make_camera(pos, (1, 0, 0), (0, 1, 0), (0, 0, 1), 60.0, 0.0, 1.0, 1.0, cfg.width, cfg.height))
        surface, u8, _ = iso(renderer, value)
        ref_surface, ref_u8 = IO.isosurface(oracle_of(renderer, cfg.fmt, vox), value, STEP, COLOR)
        check_vs_oracle(surface, u8, ref_surface, ref_u8)
    # (1, 2, 4) lies where rho > 0.5: every ray hits at its first sample, half a step from the camera
    renderer.set_camera(S.make_camera((1.0, 2.0, 4.0), (1, 0, 0), (0, 1, 0), (0, 0, 1), 60.0, 0.0, 1.0, 1.0, cfg.width, cfg.height))
    surface = iso(renderer, 0.5)[0].cpu().numpy()
    assert np.all(np.isfinite(surface[..., 3])) and surface[..., 3].max() <= 0.5 * H_STEP + 1e-5


@pytest.mark.parametrize("on_device", [0, 1])
def test_new_voxels_are_seen(renderer, on_device):
    """svr_volume_upload of other voxels (host copy, or the fused device path that reduces the ranges in the same pass): the
    isosurface follows the new voxels, with skipping on."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    for value in (SKIN, BONE):
        iso(renderer, value)  # ranges of the CT
    sphere = S.sphere_volume(cfg.n, L.VOXEL_U8)
    renderer.upload_volume(torch.from_numpy(sphere.reshape(-1).copy()).cuda() if on_device else sphere)
    orc = oracle_of(renderer, cfg.fmt, sphere)
    for value in (SKIN, BONE):
        surface, u8, _ = iso(renderer, value)
        check_vs_oracle(surface, u8, *IO.isosurface(orc, value, STEP, COLOR))
        renderer.set_option(L.OPT_RC_SKIP, 0)
        assert torch.equal(iso(renderer, value)[0], surface)
        renderer.set_option(L.OPT_RC_SKIP, 1)


def _grid_cell(r):
    dims, cell = (C.c_int32 * 3)(), C.c_int32(0)
    L.check(r.lib.svr_grid_info(dims, C.byref(cell)), "svr_grid_info")
    return int(cell.value)


def test_other_renderers_are_unchanged(renderer):
    """An isosurface between setup and render changes neither a path-traced nor a ray-cast image, and keeps the macrocell edge
    the path tracer chose (automatic size)."""
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
    for value in (SKIN, BONE):
        setup(renderer, cfg)
        renderer.set_option(L.OPT_MACROCELL_SIZE, 0)
        iso(renderer, value)
        hdr, img = pathtrace()
        assert torch.equal(hdr, hdr0) and torch.equal(img, img0), value
        iso(renderer, value)
        assert _grid_cell(renderer) == cell0
        hdr, img = pathtrace()
        assert torch.equal(hdr, hdr0) and torch.equal(img, img0), value
        iso(renderer, value)
        rc, rc_u8 = raycast()
        assert torch.equal(rc, rc0) and torch.equal(rc_u8, rc_u80), value


def test_headless_driver_writes_the_python_image(renderer, tmp_path):
    exe = os.path.join(ROOT, "tools", "svr_headless")
    if not os.path.exists(exe):
        pytest.skip("tools/svr_headless was not built (make tools)")
    n, W, H = 64, 96, 80
    out = str(tmp_path / "iso")
    subprocess.check_call([exe, "--config", "C1", "--n", str(n), "--w", str(W), "--h", str(H), "--mode", "iso", "--iso", "0.4",
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
    renderer.render_isosurface(0.4, step)
    torch.cuda.synchronize()
    mine = renderer.ldr_image().cpu().numpy()[..., :3]
    assert mine.max() > 100
    assert np.array_equal(ppm, mine)
