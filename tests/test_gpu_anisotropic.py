"""GPU parity on a volume shaped like real CT data: dimensions that are neither equal nor multiples of the
macrocell edge (70 x 52 x 37 voxels) and anisotropic spacing (0.7, 1.0, 1.9) -- what VolumeReader hands over
for a MetaImage file (core/VolumeReader.cpp:174-201: bbox = +-dim*spacing/2, step size from the spacing).
Ray caster against the reference's float twin (1e-4), path tracer against the reference path for path (twin
mode) -- against the CPU oracle where the reference's kernels are not built -- and statistically (product mode, see
_statistical_parity for its reference arm), acceleration toggles bit-exact."""
import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

from _gpu_common import check_paths, check_rgba, check_u8, oracle_reference, raycast_f32
from test_gpu_pathtrace import _frames, _statistical_parity

pytestmark = pytest.mark.gpu

DIMS = (70, 52, 37)          # x, y, z
SPACING = (0.7, 1.0, 1.9)
W, H = 128, 128   # a canvas size the reference is compiled for (WIDTH/HEIGHT are compile-time, common.h:8-9)


class _Cfg:  # what reference() and the helpers read from a Config
    width, height, name, fmt, dims = W, H, "aniso", L.VOXEL_U16, DIMS


def _voxels(dims=DIMS):
    """Two overlapping ellipsoids with a dense core, u16, indexed (z, y, x); air is exactly 0."""
    nx, ny, nz = dims
    z, y, x = np.meshgrid(np.arange(nz), np.arange(ny), np.arange(nx), indexing="ij")
    fx, fy, fz = (x + 0.5) / nx - 0.5, (y + 0.5) / ny - 0.5, (z + 0.5) / nz - 0.5
    body = 1.0 - np.sqrt((fx / 0.42) ** 2 + (fy / 0.36) ** 2 + (fz / 0.40) ** 2)
    core = 1.0 - np.sqrt(((fx - 0.1) / 0.15) ** 2 + ((fy + 0.05) / 0.2) ** 2 + (fz / 0.18) ** 2)
    d = np.clip(body * 2.0, 0, 0.35) + np.clip(core * 3.0, 0, 0.6)
    return (np.clip(d, 0, 1) * 65535.0 + 0.5).astype(np.uint16)


def _setup(r, depth=2, tf="default", cell=8):
    r.set_option(L.OPT_PT_MODE, 2)
    r.set_option(L.OPT_PT_KERNEL, 2)
    r.set_option(L.OPT_PT_WARP_PIXELS, 4)
    r.set_option(L.OPT_PT_WARP_MIN_SPP, 32)
    r.set_option(L.OPT_SHADOW_ESTIMATOR, 0)
    r.set_option(L.OPT_RC_SKIP, 1)
    r.set_option(L.OPT_LEAP, 1)
    r.set_option(L.OPT_PT_ENTRY_CACHE, 1)
    r.set_option(L.OPT_MACROCELL_SIZE, cell)
    r.set_option(L.OPT_COUNTERS, 0)
    r.set_option(L.OPT_SEED, 0x5EED)
    vox = _voxels()
    r.load_volume(vox, L.VOXEL_U16, DIMS, spacing=SPACING)
    extent = tuple(d * s for d, s in zip(DIMS, SPACING))
    r.set_transfer_function(S.tf_table(tf))
    # off-axis camera: no ray is parallel to a grid axis
    eye = (0.9 * extent[0], 0.55 * extent[1], 1.6 * extent[2])
    wv = np.array(eye) / np.linalg.norm(eye)
    uv = np.cross((0.0, 1.0, 0.0), wv)
    uv /= np.linalg.norm(uv)
    vv = np.cross(wv, uv)
    r.set_camera(S.make_camera(eye, tuple(uv), tuple(vv), tuple(wv), 45.0, 0.0, 1.0, 1.0, W, H))
    light = S.default_area_light(extent)
    r.set_area_lights([light])
    r.set_env_light(S.constant_env_light(), enabled=False)
    return vox


def test_volume_struct_follows_the_reader(renderer):
    _setup(renderer)
    v = renderer.volume
    for a, d, s in zip("xyz", DIMS, SPACING):
        assert getattr(v.bbox.vmax, a) == pytest.approx(0.5 * d * s) and getattr(v.bbox.vmin, a) == pytest.approx(-0.5 * d * s)
        assert getattr(v.spacing, a) == np.float32(s) and getattr(v.invSpacing, a) == pytest.approx(1.0 / s)


@pytest.mark.parametrize("tf", ["default", "thin"])
def test_raycaster_matches_reference(renderer, tf):
    _setup(renderer, tf=tf)
    step = S.raycast_step_size(SPACING)
    imgs = []
    for skip, leap, cell in ((1, 1, 8), (0, 1, 8), (1, 0, 4), (1, 1, 16)):
        renderer.set_option(L.OPT_RC_SKIP, skip)
        renderer.set_option(L.OPT_LEAP, leap)
        renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
        imgs.append(raycast_f32(renderer).clone())
    for im in imgs[1:]:
        assert torch.equal(im, imgs[0])  # skipping removes zero contributions only
    mine = imgs[0].cpu().numpy()
    assert mine[..., 3].max() > 0.5
    twin = oracle_reference(renderer, _Cfg, f32=True)
    twin.render_raycasting(step)
    check_rgba(mine, twin)
    ref = oracle_reference(renderer, _Cfg)
    ref.render_raycasting(step)
    check_u8(renderer.ldr_image().cpu().numpy(), ref)


def test_path_tracer_twin_mode_matches_reference(renderer):
    depth = 3
    _setup(renderer, depth)
    renderer.set_option(L.OPT_PT_MODE, 0)
    renderer.set_option(L.OPT_PT_KERNEL, 1)
    ref = oracle_reference(renderer, _Cfg)
    mine = _frames(renderer, 4, depth)
    ref.frame_no = 0
    ref.render_pathtracer(4, depth)
    theirs = ref.hdr_image().cpu().numpy()
    assert theirs.max() > 0
    check_paths(mine, theirs, ref, frac=0.999, mean_rel=1e-3)


def test_path_tracer_product_mode_is_statistically_the_reference(renderer):
    depth = 3
    _setup(renderer, depth)
    _statistical_parity(renderer, _Cfg, depth, 8, 64, lambda: None)


def test_path_tracer_acceleration_toggles_are_bit_exact(renderer):
    depth = 3
    _setup(renderer, depth)
    imgs = []
    for shape, leap, cache, cell in ((2, 1, 1, 8), (2, 0, 0, 8), (1, 1, 0, 8)):
        renderer.set_option(L.OPT_PT_KERNEL, shape)
        renderer.set_option(L.OPT_LEAP, leap)
        renderer.set_option(L.OPT_PT_ENTRY_CACHE, cache)
        renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(64, depth)
        torch.cuda.synchronize()
        imgs.append(renderer.hdr_image().clone())
    assert float(imgs[0].max()) > 0
    assert torch.equal(imgs[0], imgs[1])
    assert torch.allclose(imgs[2], imgs[0], rtol=2e-5, atol=1e-6)  # megakernel: summation order only
