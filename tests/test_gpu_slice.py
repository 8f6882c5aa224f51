"""GPU tests of slices and slabs (svr_render_slices): parity with the CPU restatement (tests/slice_oracle.cpp, the CPU oracle's
texture filter), closed forms on axis slices and slabs, bit-exact macrocell skipping, new voxels, no effect on the other
renderers and the headless driver.  Every option a test changes is restored (the session's renderer is shared)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _slice_oracle as SO
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


def render(r, params):
    value, img = r.render_slices(params)
    torch.cuda.synchronize()
    return value, img


def oblique(n, mode="max", thickness=0.0, count=1, window=(0.4, 0.7), size=96):
    """An oblique stack through the middle of an n^3 volume (spacing 1)."""
    return S.oblique_slice((0.07 * n, -0.05 * n, 0.03 * n), (0.6, 0.45, 1.0), (0.1, 1.0, 0.2), 1.1 * n / size, size, size - 16,
                           count=count, slice_step=0.13 * n, thickness=thickness, sample_spacing=0.55, mode=mode, window=window)


@pytest.mark.parametrize("gen,fmt", [(L.GEN_SPHERE, L.VOXEL_U16), (L.GEN_CT, L.VOXEL_U8)])
@pytest.mark.parametrize("mode", MODES)
def test_matches_cpu_restatement(renderer, gen, fmt, mode):
    cfg = small_config(gen=gen, fmt=fmt)
    vox = setup(renderer, cfg)
    n = cfg.n
    orc = SO.oracle(vox, fmt, (n, n, n), renderer.volume)
    for thickness, count in ((0.0, 3), (0.3 * n, 2)):
        p = oblique(n, mode, thickness, count)
        value, img = render(renderer, p)
        ref_value, ref_u8 = SO.slices(orc, p)
        assert ref_value.max() > 0.1 and 0.2 < (ref_u8[..., 3] == 255).mean() < 1.0
        check_vs_oracle(value, img, ref_value, ref_u8)
        assert np.array_equal(img[..., 3].cpu().numpy(), ref_u8[..., 3])


DIMS, SPACING = (40, 28, 20), (0.8, 1.0, 1.3)  # non-cubic, anisotropic


def _random_volume(fmt, seed=11):
    rng = np.random.default_rng(seed)
    nx, ny, nz = DIMS
    d = rng.random((nz, ny, nx), dtype=np.float32)
    vox = S.encode_voxels(d, fmt)
    norm = {L.VOXEL_U8: 255.0, L.VOXEL_U16: 65535.0}.get(fmt, 1.0)
    return vox, (vox.astype(np.float32) / np.float32(norm)).astype(np.float32)


def _plane(ref, axis, index):
    return {"z": lambda: ref[index], "y": lambda: ref[:, index, :], "x": lambda: ref[:, :, index]}[axis]()


@pytest.mark.parametrize("fmt", [L.VOXEL_U8, L.VOXEL_U16, L.VOXEL_F16, L.VOXEL_F32])
def test_axis_slices_are_the_voxels(renderer, fmt):
    """A fetch at a texel centre has 8-bit weights 0 and 1: the voxel itself, up to the texture unit's normalisation of
    integer formats (1 ulp); exactly for f32."""
    setup(renderer, small_config())
    vox, ref = _random_volume(fmt)
    renderer.load_volume(vox, fmt, DIMS, SPACING)
    for axis, index in (("z", 7), ("y", 20), ("x", 33)):
        value = render(renderer, S.axis_slice(DIMS, SPACING, axis, index))[0][0].cpu().numpy()
        want = _plane(ref, axis, index)
        assert value.shape == want.shape
        if fmt == L.VOXEL_F32:
            assert np.array_equal(value, want), axis
        else:
            assert np.all(np.abs(value - want) <= np.spacing(want)), (axis, float(np.abs(value - want).max()))


def test_stack_of_every_axial_slice_is_the_volume(renderer):
    setup(renderer, small_config())
    vox, ref = _random_volume(L.VOXEL_F32)
    renderer.load_volume(vox, L.VOXEL_F32, DIMS, SPACING)
    value, img = render(renderer, S.axis_slice(DIMS, SPACING, "z", 0, count=DIMS[2]))
    assert torch.equal(value.cpu(), torch.from_numpy(ref))
    assert bool((img[..., 3] == 255).all())


def test_whole_depth_slab_is_the_column_max_and_min(renderer):
    setup(renderer, small_config())
    vox, ref = _random_volume(L.VOXEL_F32)
    renderer.load_volume(vox, L.VOXEL_F32, DIMS, SPACING)
    for skip in (0, 1):
        renderer.set_option(L.OPT_RC_SKIP, skip)
        for mode, want in (("max", ref.max(axis=0)), ("min", ref.min(axis=0))):
            p = S.axis_slice(DIMS, SPACING, "z", 0, thickness_voxels=DIMS[2], mode=mode)
            p.center[2] = 0.0  # the volume's middle: the samples lie on the voxel centres of each column
            assert np.array_equal(render(renderer, p)[0][0].cpu().numpy(), want), (mode, skip)


VOLUMES = [("ct", L.VOXEL_U8), ("ct", L.VOXEL_U16), ("ct", L.VOXEL_F16), ("ct", L.VOXEL_F32), ("ties", L.VOXEL_U8), ("ties", L.VOXEL_U16)]


@pytest.mark.parametrize("kind,fmt", VOLUMES)
def test_skipping_is_bit_exact(renderer, kind, fmt):
    n = 64
    setup(renderer, small_config(gen=L.GEN_CT, fmt=fmt))
    if kind == "ties":
        renderer.load_volume(_tie_volume(n, fmt), fmt, (n, n, n))
    views = [("axis", (-1.0, 1.0)), ("oblique", (-1.0, 1.0)), ("oblique", (-0.3, 0.3))]
    for view, clip in views:
        renderer.set_volume_params(x_clip=clip, y_clip=clip, z_clip=clip)
        for mode in MODES:
            if view == "axis":
                p = S.axis_slice((n, n, n), (1, 1, 1), "y", 30, thickness_voxels=24, count=3, mode=mode)
            else:
                p = oblique(n, mode, 0.45 * n, 2)
            renderer.set_option(L.OPT_RC_SKIP, 0)
            ref, ref_u8 = render(renderer, p)
            assert mode == "min" or float(ref.max()) > 0.05
            renderer.set_option(L.OPT_RC_SKIP, 1)
            for cell in (4, 8, 16, 32):
                renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
                got, got_u8 = render(renderer, p)
                assert torch.equal(got, ref), (view, clip, mode, cell, int((got != ref).sum()))
                assert torch.equal(got_u8, ref_u8), (view, clip, mode, cell)


def test_skipping_skips(renderer):
    """Skipping leaves the step count alone and removes a share of the taps of MIP and AIP slabs on the small CT.  The first
    B200 run skipped 0.30 of the steps for MIP, 0.31 for AIP and 0.62 for MinIP on this oblique slab; the bound leaves room for
    the generator's other seeds."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_COUNTERS, 1)
    n = cfg.n
    counts = {}
    for mode in MODES:
        p = oblique(n, mode, 0.6 * n, 1)
        for skip in (0, 1):
            renderer.set_option(L.OPT_RC_SKIP, skip)
            renderer.reset_counters()
            render(renderer, p)
            counts[mode, skip] = renderer.counters()
    print({f"{m} skip={k}": {c_: c[c_] for c_ in ("paths", "steps", "skipped", "shade_taps", "cells")} for (m, k), c in counts.items()})
    for mode in MODES:
        off, on = counts[mode, 0], counts[mode, 1]
        assert off["steps"] == on["steps"] > 0 and off["paths"] == on["paths"] == p.imageW * p.imageH
        assert off["skipped"] == 0 and off["cells"] == 0 and off["shade_taps"] == off["steps"]
        assert on["shade_taps"] + on["skipped"] == on["steps"] and on["cells"] > 0
    for mode in ("max", "mean"):
        on = counts[mode, 1]
        assert on["skipped"] > 0.2 * on["steps"], (mode, on)


@pytest.mark.parametrize("on_device", [0, 1])
def test_new_voxels_are_seen(renderer, on_device):
    """svr_volume_upload of other voxels (host copy, or the fused device path): slab results follow them with skipping on."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    n = cfg.n
    for mode in MODES:
        render(renderer, oblique(n, mode, 0.4 * n))  # ranges of the CT
    sphere = S.sphere_volume(n, L.VOXEL_U8)
    renderer.upload_volume(torch.from_numpy(sphere.reshape(-1).copy()).cuda() if on_device else sphere)
    orc = SO.oracle(sphere, cfg.fmt, (n, n, n), renderer.volume)
    for mode in MODES:
        p = oblique(n, mode, 0.4 * n)
        value, img = render(renderer, p)
        check_vs_oracle(value, img, *SO.slices(orc, p))
        renderer.set_option(L.OPT_RC_SKIP, 0)
        assert torch.equal(render(renderer, p)[0], value)
        renderer.set_option(L.OPT_RC_SKIP, 1)


def _grid_cell(r):
    dims, cell = (C.c_int32 * 3)(), C.c_int32(0)
    L.check(r.lib.svr_grid_info(dims, C.byref(cell)), "svr_grid_info")
    return int(cell.value)


def test_other_renderers_are_unchanged(renderer):
    """Slices between setup and render change neither a path-traced nor a ray-cast image, and keep the macrocell edge the path
    tracer chose (automatic size)."""
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
    for p in (oblique(cfg.n, "max", 0.5 * cfg.n), oblique(cfg.n), S.axis_slice((cfg.n,) * 3, (1, 1, 1), "x", 10, 8, mode="mean")):
        setup(renderer, cfg)
        renderer.set_option(L.OPT_MACROCELL_SIZE, 0)
        render(renderer, p)
        hdr, img = pathtrace()
        assert torch.equal(hdr, hdr0) and torch.equal(img, img0)
        render(renderer, p)
        assert _grid_cell(renderer) == cell0
        hdr, img = pathtrace()
        assert torch.equal(hdr, hdr0) and torch.equal(img, img0)
        render(renderer, p)
        rc, rc_u8 = raycast()
        assert torch.equal(rc, rc0) and torch.equal(rc_u8, rc_u80)


@pytest.mark.parametrize("axis,slab", [("z", 0), ("y", 9)])
def test_headless_driver_writes_the_python_image(renderer, tmp_path, axis, slab):
    exe = os.path.join(ROOT, "tools", "svr_headless")
    if not os.path.exists(exe):
        pytest.skip("tools/svr_headless was not built (make tools)")
    n, W, H = 64, 96, 80
    out = str(tmp_path / "slice")
    subprocess.check_call([exe, "--config", "C1", "--n", str(n), "--w", str(W), "--h", str(H), "--mode", "slice", "--axis", axis,
                           "--index", "27", "--slab", str(slab), "--window", "0.4,0.6", "--reps", "1", "--out", out], cwd=str(tmp_path))
    with open(out + ".ppm", "rb") as f:
        data = f.read()
    ppm = np.frombuffer(data[-W * H * 3:], np.uint8).reshape(H, W, 3)[::-1]
    # the driver's volume: C1's generator at n = 64, spacing 1 (svr_headless.cpp)
    setup(renderer, small_config(n=n, w=W, h=H, gen=L.GEN_SPHERE, fmt=L.VOXEL_U8))
    renderer.load_volume(renderer.generate_volume(L.GEN_SPHERE, L.VOXEL_U8, n, 1234), L.VOXEL_U8, (n, n, n))
    p = S.axis_slice((n, n, n), (1, 1, 1), axis, 27, thickness_voxels=slab, window=(0.4, 0.6))
    p.imageW, p.imageH = W, H
    mine = render(renderer, p)[1][0].cpu().numpy()[..., :3]
    assert mine.max() > 100
    assert np.array_equal(ppm, mine)
