"""Kernel shape 5 (svr_pathtrace.cu: rays and scatter events are work items in per-warp queues, lanes take them as they
become free, a warp renders a run of pixels whose rays share the pool; SVR_OPT_PT_KERNEL = 5).

Same estimator as the reference's kernel_pathtracer; the shadow ray draws from a stream of its own, so samples make other
random walks than in shapes 1-3: parity with the reference (oracle/_ref) is statistical (tests/test_gpu_pathtrace.py::
_statistical_parity).  Exact properties: every path is counted once; radiance is summed per pixel in fixed point, so the
image does not depend on how lanes were scheduled -- bit-identical across re-fill thresholds, run lengths and block sizes.

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
    r.set_option(L.OPT_PT_KERNEL, 5)
    r.set_option(L.OPT_PT_POOL_PIXELS, 0)


def _render(r, spp, depth, first=0):
    r.frame_no = first
    r.render_pathtracer_spp(spp, depth)
    torch.cuda.synchronize()
    return r.hdr_image().clone()


@pytest.mark.parametrize("gen,fmt,tf,depth,estimator,env", [
    (L.GEN_CT, L.VOXEL_U16, "default", 1, 0, False),      # opaque body, single scattering
    (L.GEN_CT, L.VOXEL_U16, "default", 6, 1, False),      # deeper paths, ratio-tracked shadows
    (L.GEN_CLOUD, L.VOXEL_F16, "cloud", 32, 0, True),     # high-albedo cloud under a sky (C4's regime)
    (L.GEN_CLOUD, L.VOXEL_F16, "cloud", 32, 1, False),
    (L.GEN_SPHERE, L.VOXEL_U8, "thin", 8, 0, False),      # thin medium: long flights (chunks go back into the pool)
])
def test_pool_kernel_is_statistically_the_reference(renderer, gen, fmt, tf, depth, estimator, env):
    cfg = small_config(n=64, gen=gen, fmt=fmt, tf=tf, depth=depth, env=env)
    _setup(renderer, cfg)
    renderer.set_option(L.OPT_MACROCELL_SIZE, 0)   # the automatic cell size, as the product runs
    renderer.set_option(L.OPT_SHADOW_ESTIMATOR, estimator)
    _statistical_parity(renderer, cfg, depth, 16, 32, lambda: None, mean_tol=0.02, env=env)


@pytest.mark.parametrize("variant", ["clip_planes", "camera_inside", "thin_lens", "two_lights", "light_in_view"])
def test_pool_kernel_scene_variants(renderer, variant):
    depth = 3
    cfg = small_config(n=64, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=depth)
    _setup(renderer, cfg)
    if variant == "clip_planes":
        renderer.set_volume_params(x_clip=(-0.6, 0.35), y_clip=(-1.0, 0.5), z_clip=(-0.2, 1.0))
    elif variant == "camera_inside":
        renderer.set_camera(S.look_at_camera((3.0, -2.0, 10.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), image_w=cfg.width, image_h=cfg.height))
    elif variant == "thin_lens":
        renderer.set_camera(S.default_camera(cfg.extent, cfg.width, cfg.height, apeture=1.5, focal_length=60.0))
    elif variant == "two_lights":
        l2 = S.default_area_light(cfg.extent)
        l2.disk.center = L.Vec3(70.0, 20.0, 40.0)
        n = -np.array([70.0, 20.0, 40.0]) / np.linalg.norm([70.0, 20.0, 40.0])
        l2.disk.normal = L.Vec3(*[float(x) for x in n])
        l2.color = L.Vec3(0.4, 0.7, 1.0)
        renderer.set_area_lights([S.default_area_light(cfg.extent), l2])
    elif variant == "light_in_view":
        from test_gpu_lights_in_view import SCENES

        renderer.set_area_lights(SCENES["inside_volume"])
    _statistical_parity(renderer, cfg, depth, 16, 16, lambda: None, mean_tol=0.02)


def test_pool_kernel_image_does_not_depend_on_scheduling(renderer):
    """Fixed-point sums: the order in which lanes finish rays does not reach the image."""
    cfg = small_config(n=80, w=150, h=101, gen=L.GEN_CLOUD, fmt=L.VOXEL_F16, tf="cloud", depth=16, env=True)
    _setup(renderer, cfg)
    renderer.set_option(L.OPT_PT_WARP_MIN_SPP, 1)
    for spp in (64, 40, 7):
        base = _render(renderer, spp, 16)
        assert float(base.max()) > 0
        assert torch.equal(_render(renderer, spp, 16), base)
        for refill, pixels, blk in ((1, 16, 128), (32, 16, 128), (8, 5, 64), (16, 1, 128), (4, 16, 64)):
            renderer.set_option(L.OPT_PT_REFILL, refill)
            renderer.set_option(L.OPT_PT_POOL_PIXELS, pixels)
            renderer.set_option(L.OPT_PT_BLOCK, blk)
            assert torch.equal(_render(renderer, spp, 16), base), (spp, refill, pixels, blk)
        renderer.set_option(L.OPT_PT_REFILL, 0)
        renderer.set_option(L.OPT_PT_POOL_PIXELS, 0)
        renderer.set_option(L.OPT_PT_BLOCK, 128)
    # a batch split in two adds up to the batch (the multi-GPU sample split), up to float rounding of the two partial sums
    W, H = cfg.width, cfg.height
    whole = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    renderer.accumulate(whole, 16, 0, 96, clear=True)
    parts = torch.zeros_like(whole)
    renderer.accumulate(parts, 16, 0, 40, clear=True)
    renderer.accumulate(parts, 16, 40, 56, clear=False)
    torch.cuda.synchronize()
    assert torch.allclose(parts, whole, rtol=2e-6, atol=1e-6)
    assert float(whole.view(H, W, 4)[..., 3].min()) == 96.0
    renderer.set_option(L.OPT_SEED, 77)
    assert not torch.equal(_render(renderer, 64, 16), base)


def test_pool_kernel_counts(renderer):
    """Every path is handed out exactly once; the medium scatters as often as in shape 2 (within Monte Carlo noise)."""
    cfg = small_config(n=64, w=128, h=96, gen=L.GEN_CLOUD, fmt=L.VOXEL_F16, tf="cloud", depth=32)
    setup(renderer, cfg)
    counts = {}
    for shape in (2, 5):
        renderer.set_option(L.OPT_PT_KERNEL, shape)
        renderer.set_option(L.OPT_COUNTERS, 1)
        renderer.reset_counters()
        _render(renderer, 64, 32)
        counts[shape] = renderer.counters()
        renderer.set_option(L.OPT_COUNTERS, 0)
    assert counts[2]["paths"] == counts[5]["paths"] == cfg.width * cfg.height * 64
    assert counts[5]["scatters"] > 0
    assert abs(counts[2]["scatters"] - counts[5]["scatters"]) < 0.01 * counts[2]["scatters"]
    assert counts[5]["shade_taps"] == 7 * counts[5]["scatters"]


def test_pool_kernel_depth_zero_and_no_lights(renderer):
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8)
    _setup(renderer, cfg)
    assert float(_render(renderer, 32, 0).max()) == 0.0       # traceDepth 0: the bounce loop never runs
    renderer.set_area_lights([])
    assert float(_render(renderer, 32, 3).max()) == 0.0       # nothing emits
    renderer.set_env_light(S.constant_env_light(), enabled=True)
    img = _render(renderer, 32, 3)
    assert img[0, 0, 0].item() == pytest.approx(0.5)          # a corner ray sees the constant sky
