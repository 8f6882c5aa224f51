"""GPU parity of the ray caster (render_raycasting, raycasting.h:8) through the C ABI.

Checkers: the reference's own unmodified kernel_raycasting (oracle/_ref; u8 output, and its float
twin for the 1e-4 bound north_star states) and the CPU oracle.  Tolerances:
  * vs the reference's float twin: 1e-4 per channel on the pre-quantisation RGBA (north_star);
  * vs the reference's u8 image: 1 LSB;
  * vs the CPU oracle (IEEE libm, no FMA contraction): the images agree to ~1e-6 except where a
    1-ulp difference in a texture coordinate flips one 8-bit filter weight; checked as mean abs
    difference < 5e-5 and 99% of the pixels within 1e-4.
"""
import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

from _gpu_common import check_rgba, check_u8, cpu_oracle, oracle_reference, raycast_f32, setup, small_config

pytestmark = pytest.mark.gpu
STEP = S.raycast_step_size()


def _check_vs_reference(r, cfg):
    setup(r, cfg)
    mine = raycast_f32(r)
    mine_u8 = r.ldr_image().cpu().numpy()
    ref = oracle_reference(r, cfg)
    ref.render_raycasting(STEP)
    check_u8(mine_u8, ref)
    twin = oracle_reference(r, cfg, f32=True)
    twin.render_raycasting(STEP)
    check_rgba(mine.cpu().numpy(), twin)
    assert mine.cpu().numpy()[..., 3].max() > 0.5  # the volume is actually visible
    return mine


@pytest.mark.parametrize("fmt", [L.VOXEL_U8, L.VOXEL_U16, L.VOXEL_F16, L.VOXEL_F32])
def test_small_sphere_all_voxel_formats(renderer, fmt):
    _check_vs_reference(renderer, small_config(fmt=fmt))


@pytest.mark.parametrize("tf", ["default", "thin", "cloud"])
def test_small_ct_all_transfer_functions(renderer, tf):
    _check_vs_reference(renderer, small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, tf=tf))


def test_config_c1_full_size(renderer):
    _check_vs_reference(renderer, S.CONFIGS["C1"])


@pytest.mark.parametrize("tf", ["thin", "default"])
def test_config_c2_full_size(renderer, tf):
    cfg = S.Config("C2", 256, L.VOXEL_U8, L.GEN_CT, 1024, 1024, tf)
    _check_vs_reference(renderer, cfg)


def test_against_cpu_oracle(renderer):
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U16)
    vox = setup(renderer, cfg)
    mine = raycast_f32(renderer).cpu().numpy()
    rgba, u8, _ = cpu_oracle(renderer, cfg, vox).raycast(STEP)
    d = np.abs(mine - rgba)
    assert d.mean() < 5e-5
    assert (d.max(axis=2) < 1e-4).mean() > 0.99
    assert np.abs(renderer.ldr_image().cpu().numpy().astype(int) - u8.astype(int)).max() <= 2


def test_skipping_is_bit_exact(renderer):
    """Empty-space skipping and leaping only remove zero contributions (svr_raycast.cu header)."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8, tf="thin", w=128, h=128)
    setup(renderer, cfg)
    imgs = []
    for skip, leap, cell in ((0, 1, 8), (1, 0, 8), (1, 1, 8), (1, 1, 4), (1, 1, 16)):
        renderer.set_option(L.OPT_RC_SKIP, skip)
        renderer.set_option(L.OPT_LEAP, leap)
        renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
        imgs.append(raycast_f32(renderer).clone())
    for im in imgs[1:]:
        assert torch.equal(im, imgs[0])
    renderer.set_option(L.OPT_MACROCELL_SIZE, 8)


def test_skipping_actually_skips(renderer):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8, tf="thin")
    setup(renderer, cfg)
    renderer.set_option(L.OPT_COUNTERS, 1)
    counts = {}
    for skip in (0, 1):
        renderer.set_option(L.OPT_RC_SKIP, skip)
        renderer.reset_counters()
        renderer.render_raycasting()
        counts[skip] = renderer.counters()
    renderer.set_option(L.OPT_COUNTERS, 0)
    assert counts[0]["steps"] == counts[1]["steps"]  # every sample position is still enumerated
    assert counts[1]["skipped"] > 0.3 * counts[1]["steps"]
    assert counts[1]["shade_taps"] < 0.8 * counts[0]["shade_taps"]
    assert counts[0]["paths"] == cfg.width * cfg.height


def test_rows_partition_equals_full_frame(renderer):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16)
    setup(renderer, cfg)
    full = raycast_f32(renderer).clone()
    parts = torch.zeros_like(full).view(-1)
    for y0, y1 in S.split_rows(cfg.height, 3):
        renderer.render_raycasting_f32(parts, rows=(y0, y1))
    torch.cuda.synchronize()
    assert torch.equal(parts.view_as(full), full)


def test_transfer_function_edit_is_seen(renderer):
    """The TF content can change behind the same volume (gui/transferfunction.cpp:128-151): the
    majorant grid must follow, or skipping would drop visible samples."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8, tf="thin")
    setup(renderer, cfg)
    a = raycast_f32(renderer).clone()
    renderer.set_transfer_function(S.tf_table("default"))
    b = raycast_f32(renderer).clone()
    renderer.set_option(L.OPT_RC_SKIP, 0)
    b_noskip = raycast_f32(renderer).clone()
    assert not torch.equal(a, b)
    assert torch.equal(b, b_noskip)


def test_clip_planes_and_density_scale(renderer):
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    renderer.set_volume_params(density_scale=0.6, x_clip=(-0.5, 0.9), z_clip=(-1.0, 0.2))
    mine = raycast_f32(renderer).cpu().numpy()
    twin = oracle_reference(renderer, cfg, f32=True)
    twin.render_raycasting(STEP)
    check_rgba(mine, twin)
    renderer.set_option(L.OPT_RC_SKIP, 0)
    assert np.array_equal(raycast_f32(renderer).cpu().numpy(), mine)


def test_camera_inside_the_volume(renderer):
    """tNear < 0: the reference marches from behind the eye (raycasting.cu:29); reproduced."""
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    renderer.set_camera(S.make_camera((3.0, -2.0, 10.0), (1, 0, 0), (0, 1, 0), (0, 0, 1), 60.0, 0.0, 1.0, 1.0, cfg.width, cfg.height))
    mine = raycast_f32(renderer).cpu().numpy()
    twin = oracle_reference(renderer, cfg, f32=True)
    twin.render_raycasting(STEP)
    check_rgba(mine, twin)


def test_empty_volume_and_ragged_image_size(renderer):
    """Image sizes the reference cannot render (not a multiple of 16; it has no bounds guard)."""
    cfg = small_config(n=32, w=100, h=70, gen=L.GEN_SPHERE, fmt=L.VOXEL_U8)
    vox = setup(renderer, cfg)
    mine = raycast_f32(renderer).cpu().numpy()
    rgba, _, _ = cpu_oracle(renderer, cfg, vox).raycast(STEP)
    assert np.abs(mine - rgba).mean() < 5e-5
    empty = np.zeros((32, 32, 32), np.uint8)
    renderer.load_volume(empty, L.VOXEL_U8, (32, 32, 32), max_grad_mag=1.0)
    out = raycast_f32(renderer)
    assert float(out.abs().max()) == 0.0
    assert int(renderer.ldr_image().max()) == 0


def test_interleaved_bands_tile_the_image(renderer):
    """svr_render_raycasting_bands: the bands of phases 0..stride-1 are disjoint and together are the frame."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, w=150, h=101)
    setup(renderer, cfg)
    renderer.render_raycasting(STEP)
    torch.cuda.synchronize()
    full = renderer.ldr_image().clone()
    assert int(full[..., 3].max()) > 100
    for stride, block in ((3, 64), (8, 64), (2, 256), (1, 128)):
        renderer.set_option(L.OPT_RC_BLOCK, block)
        total = torch.zeros_like(full, dtype=torch.int32)
        for phase in range(stride):
            renderer.img.zero_()
            rows = renderer.render_raycasting_bands(phase, stride, STEP)
            torch.cuda.synchronize()
            assert rows == block // 16
            part = renderer.ldr_image()
            # bands are counted from the middle of the image outwards: k = 0 is the middle band, 1 the one below, ...
            n_bands = (cfg.height + rows - 1) // rows
            mid = n_bands // 2
            k_of_band = torch.tensor([2 * (b - mid) if b >= mid else 2 * (mid - b) - 1 for b in range(n_bands)], device="cuda")
            k = k_of_band[torch.arange(cfg.height, device="cuda") // rows]
            assert int(part[k % stride != phase].abs().sum()) == 0     # nothing outside this phase's bands
            total += part.int()
        assert torch.equal(total, full.int())
    renderer.set_option(L.OPT_RC_BLOCK, 64)
    assert renderer.lib.svr_render_raycasting_bands(None, None, None, None, None, STEP, 0, 1, None) != 0
