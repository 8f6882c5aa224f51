"""Kernel shape 4 (svr_pathtrace.cu: camera rays tracked against a per-pixel majorant profile the warp builds once per
pixel; SVR_OPT_PT_PROFILE = 1, opt-in: it makes a quarter of shape 2's cell visits but measured slower, DESIGN.md 3.1).

The profile is a different -- equally valid -- majorant than the per-cell one, so samples make other random walks than in
shapes 1-3: parity with the reference's kernel_pathtracer (oracle/_ref) is statistical, as for every Philox mode
(tests/test_gpu_pathtrace.py::_statistical_parity: RMSE at equal spp <= 1.15 x the reference-vs-reference noise floor,
Welch statistic per 16x16 tile <= 4.5 for >= 99.5 % of the tiles, image means within 1-3 %).  What stays exact: the image
is a deterministic function of (seed, scene, sample range); launch geometry and the refill threshold only change the
order of float additions; counted paths are exact; the profile is conservative (checked against brute-force fetches).

Where oracle/_ref is not built, the reference arm of the statistical comparisons is the product's reference-twin
mode (tests/test_gpu_pathtrace.py::_statistical_parity)."""
import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

from _gpu_common import setup, small_config
from test_gpu_pathtrace import _statistical_parity

pytestmark = pytest.mark.gpu


def _setup(r, cfg):
    setup(r, cfg)
    r.set_option(L.OPT_PT_PROFILE, 1)


def _render(r, spp, depth, first=0):
    r.frame_no = first
    r.render_pathtracer_spp(spp, depth)
    torch.cuda.synchronize()
    return r.hdr_image().clone()


@pytest.mark.parametrize("gen,fmt,tf,depth,estimator,res", [
    (L.GEN_CT, L.VOXEL_U16, "default", 1, 0, (128, 128)),      # opaque body, single scattering (C3's regime)
    (L.GEN_CT, L.VOXEL_U16, "default", 6, 1, (128, 128)),      # deeper paths, ratio-tracked shadows
    (L.GEN_CLOUD, L.VOXEL_F16, "cloud", 32, 0, (128, 128)),    # high-albedo cloud (C4's regime)
    (L.GEN_SPHERE, L.VOXEL_U8, "thin", 8, 0, (128, 128)),      # thin medium: large cells, most rays cross without colliding
    (L.GEN_CT, L.VOXEL_U16, "default", 3, 0, (64, 64)),        # few, large pixels: the rays of a pixel spread over > 1 voxel
])
def test_profile_kernel_is_statistically_the_reference(renderer, gen, fmt, tf, depth, estimator, res):
    cfg = small_config(n=64, w=res[0], h=res[1], gen=gen, fmt=fmt, tf=tf, depth=depth)
    _setup(renderer, cfg)
    renderer.set_option(L.OPT_MACROCELL_SIZE, 0)   # the automatic cell size, as the product runs
    renderer.set_option(L.OPT_SHADOW_ESTIMATOR, estimator)

    def configure():
        renderer.set_option(L.OPT_PT_MODE, 2)
        renderer.set_option(L.OPT_PT_KERNEL, 2)
        renderer.set_option(L.OPT_PT_PROFILE, 1)

    _statistical_parity(renderer, cfg, depth, 16, 16, configure, mean_tol=0.02)


@pytest.mark.parametrize("cell", [2, 4, 16, 32])
def test_profile_kernel_parity_at_every_cell_size(renderer, cell):
    """Cell sizes from finer than a pixel's ray spread to a few cells across the volume (slabs several cells thick never
    occur at this size; the 4K / 2048^3 test covers them)."""
    depth = 2
    cfg = small_config(n=64, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=depth)
    _setup(renderer, cfg)
    renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
    _statistical_parity(renderer, cfg, depth, 16, 16, lambda: None, mean_tol=0.02)


@pytest.mark.parametrize("variant", ["clip_planes", "camera_inside", "density_and_gradient", "anisotropic_spacing", "wide_image"])
def test_profile_kernel_scene_variants(renderer, variant):
    depth = 2
    w, h = (200, 72) if variant == "wide_image" else (128, 128)
    cfg = small_config(n=64, w=w, h=h, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=depth)
    _setup(renderer, cfg)
    if variant == "clip_planes":
        renderer.set_volume_params(x_clip=(-0.6, 0.35), y_clip=(-1.0, 0.5), z_clip=(-0.2, 1.0))
    elif variant == "camera_inside":
        renderer.set_camera(S.look_at_camera((3.0, -2.0, 10.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), image_w=w, image_h=h))
    elif variant == "density_and_gradient":
        renderer.set_volume_params(density_scale=0.6, gradient_factor=1.0)
    elif variant == "anisotropic_spacing":
        vox = renderer.generate_volume(L.GEN_CT, L.VOXEL_U16, cfg.n, 1234)
        renderer.load_volume(vox, cfg.fmt, (cfg.n,) * 3, spacing=(1.0, 0.7, 1.6))
        ext = (cfg.n * 1.0, cfg.n * 0.7, cfg.n * 1.6)
        renderer.set_camera(S.look_at_camera((90.0, 60.0, 150.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), image_w=w, image_h=h))
        renderer.set_area_lights([S.default_area_light(ext)])
    if variant != "wide_image":
        _statistical_parity(renderer, cfg, depth, 16, 16, lambda: None, mean_tol=0.02)
    else:
        # no reference library of this size: shape 4 against shape 2 of this library (itself held to the reference)
        a = torch.stack([_render(renderer, 64, depth, first=j * 64) for j in range(8)]).mean(0)
        renderer.set_option(L.OPT_PT_PROFILE, 0)
        b = torch.stack([_render(renderer, 64, depth, first=j * 64) for j in range(8)]).mean(0)
        assert abs(float(a.mean()) - float(b.mean())) < 0.02 * float(b.mean())


def test_profile_kernel_is_deterministic_and_launch_geometry_only_reorders_additions(renderer):
    cfg = small_config(n=96, w=150, h=101, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=3)
    _setup(renderer, cfg)
    renderer.set_option(L.OPT_PT_WARP_MIN_SPP, 1)
    for spp in (64, 40, 7):
        base = _render(renderer, spp, 3)
        assert float(base.max()) > 0
        assert torch.equal(_render(renderer, spp, 3), base)       # run to run: bit for bit
        for wp, blk in ((1, 64), (7, 64), (3, 128)):
            renderer.set_option(L.OPT_PT_WARP_PIXELS, wp)
            renderer.set_option(L.OPT_PT_BLOCK, blk)
            assert torch.equal(_render(renderer, spp, 3), base)   # which warp renders a pixel does not matter at all
        renderer.set_option(L.OPT_PT_WARP_PIXELS, 4)
        renderer.set_option(L.OPT_PT_BLOCK, 128)
        for refill in (1, 16, 32):                                  # when lanes take new samples: other order of additions
            renderer.set_option(L.OPT_PT_REFILL, refill)
            assert torch.allclose(_render(renderer, spp, 3), base, rtol=5e-5, atol=2e-6)
        renderer.set_option(L.OPT_PT_REFILL, 0)
    # a batch split in two adds up to the batch (the multi-GPU split), up to float summation order
    W, H = cfg.width, cfg.height
    whole = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    renderer.accumulate(whole, 3, 0, 96, clear=True)
    parts = torch.zeros_like(whole)
    renderer.accumulate(parts, 3, 0, 40, clear=True)
    renderer.accumulate(parts, 3, 40, 56, clear=False)
    torch.cuda.synchronize()
    assert torch.allclose(parts, whole, rtol=5e-5, atol=2e-5)
    assert float(whole.view(H, W, 4)[..., 3].min()) == 96.0
    # seeds matter
    renderer.set_option(L.OPT_SEED, 77)
    assert not torch.equal(_render(renderer, 64, 3), base)


def test_profile_kernel_counts_every_path_and_makes_fewer_cell_visits(renderer):
    cfg = small_config(n=96, w=128, h=96, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=1)
    _setup(renderer, cfg)
    renderer.set_option(L.OPT_MACROCELL_SIZE, 4)
    counts = {}
    for prof in (0, 1):
        renderer.set_option(L.OPT_PT_PROFILE, prof)
        renderer.set_option(L.OPT_COUNTERS, 1)
        renderer.reset_counters()
        _render(renderer, 64, 1)
        counts[prof] = renderer.counters()
        renderer.set_option(L.OPT_COUNTERS, 0)
    assert counts[0]["paths"] == counts[1]["paths"] == cfg.width * cfg.height * 64
    # the same medium, the same estimator: scatter events agree within Monte Carlo noise ...
    assert abs(counts[0]["scatters"] - counts[1]["scatters"]) < 0.01 * counts[0]["scatters"]
    # ... and the camera-ray walk is gone: cells are visited once per pixel instead of once per sample
    assert counts[1]["cells"] < 0.5 * counts[0]["cells"]


def test_profile_is_conservative_against_brute_force(renderer):
    """Delta tracking is unbiased only if sigma <= M(t) at every tentative collision.  With the accept test `u * M < sigma`
    a violation cannot be seen in the image statistics of a small test, so it is counted: SVR_CNT_SKIPPED counts the
    tentative collisions of camera rays with sigma > M(t) when counters are on.  It must be zero -- thin, coarse, fine,
    anisotropic and close-up scenes, where a pixel's rays spread over several voxels."""
    for n, w, h, cell, tf, cam in ((64, 128, 128, 4, "default", None), (64, 48, 48, 2, "default", None), (64, 32, 32, 2, "thin", None),
                                   (96, 160, 90, 8, "default", (20.0, 30.0, 70.0)), (64, 16, 16, 2, "default", None)):
        cfg = small_config(n=n, w=w, h=h, gen=L.GEN_CT, fmt=L.VOXEL_U16, tf=tf, depth=1)
        _setup(renderer, cfg)
        renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
        if cam:
            renderer.set_camera(S.look_at_camera(cam, (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), image_w=w, image_h=h))
        renderer.set_option(L.OPT_COUNTERS, 1)
        renderer.reset_counters()
        _render(renderer, 256, 1)
        c = renderer.counters()
        renderer.set_option(L.OPT_COUNTERS, 0)
        assert c["track_taps"] > 0
        assert c["skipped"] == 0, (n, w, h, cell, tf, c["skipped"], c["track_taps"])
