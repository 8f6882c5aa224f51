"""Area lights INSIDE the view frustum: the camera ray's own light hit (pathtracer.cu:214-229 ->
get_nearest_light_sample, core/lights/light_sample.h:23-49 -> cudaDisk::Intersect, core/geometry/cuda_disk.h:32-51)
and the conservative per-pixel light cull this library puts in front of it (classify_pixel).

Checker: the reference's own unmodified kernel_pathtracer (oracle/_ref) on the same texture objects and seeds; where
it is not built, the CPU oracle (tests/_gpu_common.py::check_paths gives its bounds).
  * reference-twin mode: the same walk path for path -- every channel within 1e-4 * max(1, |reference|) (the radiance
    of a small disk is in the hundreds, where 1e-4 absolute is below one float ulp) on >= 99.9 % of the pixels;
  * product mode (local majorants + Philox): statistical parity as tests/test_gpu_pathtrace.py defines it;
  * the light cull on and off: bit-identical images, every kernel shape.
"""
import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

from _gpu_common import OracleRef, check_paths, check_u8, oracle_reference, setup, small_config
from test_gpu_pathtrace import _statistical_parity

pytestmark = pytest.mark.gpu

N = 64                      # volume edge; the camera sits at z = 1.5 N / (2 tan 22.5 deg) = 115.9 looking down -z
EYE = S.eye_distance((N, N, N))


def _light(center, normal, radius, intensity=2.0, color=(1.0, 0.9, 0.7)):
    l = L.AreaLight()
    l.disk.radius = radius
    l.disk.center = L.Vec3(*[float(x) for x in center])
    n = np.asarray(normal, np.float64)
    n = n / np.linalg.norm(n)
    l.disk.normal = L.Vec3(*[float(x) for x in n])
    l.color = L.Vec3(*color)
    l.intensity = intensity
    return l


def _half_width(z):
    """Half extent of the view frustum (45 deg fov, square image) at depth z."""
    return (EYE - z) * np.tan(np.radians(22.5))


# name -> lights.  Every scene keeps the default light above the volume (out of view: 35.7 deg off axis) so that the
# volume itself is lit, and adds disks the camera can see.
def _scenes():
    above = S.default_area_light((N, N, N))
    edge_x = _half_width(60.0)
    ring = [_light((26 * np.cos(a), 26 * np.sin(a), 50.0), (0.1 * np.cos(a), 0.1 * np.sin(a), 1.0), 1.5, intensity=0.1) for a in np.linspace(0, 2 * np.pi, 7, endpoint=False)]
    return {
        # in front of the volume, facing the camera: the camera ray stops on the disk and adds its radiance
        "front_facing": [above, _light((10.0, 8.0, 60.0), (0, 0, 1), 6.0)],
        # in front, facing away: the reference adds 0 and breaks (pathtracer.cu:223-228): a black disk over the volume
        "front_facing_away": [above, _light((-8.0, 5.0, 60.0), (0, 0, -1), 7.0)],
        # behind the volume: seen only by camera rays that cross the box without colliding (ls.t > t otherwise)
        "behind_volume": [above, _light((0.0, 0.0, -60.0), (0, 0, 1), 40.0)],
        # cut by the right image edge
        "clipped_by_image_edge": [above, _light((edge_x, -4.0, 60.0), (-0.3, 0, 1), 5.0)],
        # inside the medium: some camera rays collide before the disk, some after
        "inside_volume": [above, _light((0.0, 0.0, 0.0), (0.2, 0.1, 1), 14.0)],
        # tilted almost edge-on, default (large) intensity: radiance in the hundreds
        "grazing_bright": [above, _light((-14.0, -10.0, 45.0), (1.0, 0.0, 0.08), 8.0, intensity=500.0)],
        # seven small disks around the volume + the one above: eight lights, many disk-edge pixels for the cull (dim: radiance
        # 2.25, so that the few hundred disk-edge pixels do not carry the whole image RMSE)
        "ring_of_small_disks": [above] + ring,
        # only lights in view, nothing above
        "only_in_view": [_light((0.0, 20.0, 70.0), (0, -0.5, 1), 4.0), _light((-20.0, -15.0, 40.0), (0.5, 0.5, 1), 3.0)],
    }


SCENES = _scenes()


def _close(mine, theirs):
    d = np.abs(mine - theirs)
    return (d <= 1e-4 * np.maximum(1.0, np.abs(theirs))).all(axis=2)


def _setup(renderer, name, depth, lens):
    cfg = small_config(n=N, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=depth)
    setup(renderer, cfg)
    if lens:
        renderer.set_camera(S.default_camera(cfg.extent, cfg.width, cfg.height, apeture=1.5, focal_length=60.0))
    renderer.set_area_lights(SCENES[name])
    return cfg


def _lit_by_camera_rays(renderer, cfg, name):
    """Pixels whose centre ray hits one of the in-view disks (host restatement of cuda_disk.h:32-51): the test scenes
    must really put lights in view."""
    cam = renderer.camera
    W, H = cfg.width, cfg.height
    x = (np.arange(W) + 0.5) / (W - 1.0) * 2 - 1
    y = (np.arange(H) + 0.5) / (H - 1.0) * 2 - 1
    nx, ny = np.meshgrid(x * cam.aspectRatio * cam.tanFovxOverTwo, y * cam.tanFovxOverTwo)
    d = np.stack([nx, ny, -np.ones_like(nx)], axis=-1)
    d /= np.linalg.norm(d, axis=-1, keepdims=True)
    o = np.array([cam.pos.x, cam.pos.y, cam.pos.z])
    hit = np.zeros((H, W), bool)
    for l in SCENES[name]:
        c = np.array([l.disk.center.x, l.disk.center.y, l.disk.center.z])
        n = np.array([l.disk.normal.x, l.disk.normal.y, l.disk.normal.z])
        den = d @ n
        with np.errstate(divide="ignore", invalid="ignore"):
            t = ((c - o) @ n) / den
            p = o + t[..., None] * d
        hit |= (np.abs(den) > 1e-6) & (t >= 0) & (np.linalg.norm(p - c, axis=-1) <= l.disk.radius)
    return hit


@pytest.mark.parametrize("lens", [False, True], ids=["pinhole", "thin_lens"])
@pytest.mark.parametrize("name", sorted(SCENES))
def test_twin_mode_with_lights_in_view_is_the_reference_path_for_path(renderer, name, lens):
    depth = 3
    cfg = _setup(renderer, name, depth, lens)
    seen = _lit_by_camera_rays(renderer, cfg, name)
    assert seen.sum() >= 12, "the scene does not put a light in view"
    renderer.set_option(L.OPT_PT_MODE, 0)
    ref = oracle_reference(renderer, cfg)
    # kernel shape 1 (lane per pixel) frame by frame; shape 2 (sample-parallel warp) in one 33-sample batch
    for shape, frames in ((1, 3), (2, 33)):
        renderer.set_option(L.OPT_PT_KERNEL, shape)
        renderer.set_option(L.OPT_PT_WARP_MIN_SPP, 1)
        renderer.frame_no = 0
        if shape == 1:
            for _ in range(frames):
                renderer.render_pathtracer(depth)
        else:
            renderer.render_pathtracer_spp(frames, depth)
        torch.cuda.synchronize()
        mine = renderer.hdr_image().cpu().numpy()
        ref.frame_no = 0
        ref.render_pathtracer(frames, depth)
        theirs = ref.hdr_image().cpu().numpy()
        if isinstance(ref, OracleRef):
            check_paths(mine, theirs, ref, scaled=True)
        else:
            ok = _close(mine, theirs)
            assert ok.mean() >= 0.999, (name, shape, float(ok.mean()), float(np.abs(mine - theirs).max()))
            assert abs(mine.mean() - theirs.mean()) <= 2e-3 * theirs.mean()
        if not lens and name not in ("front_facing_away",):
            # the disk is visible in the image: pixels whose centre ray hits it carry (some of) its radiance or its shadow
            assert np.isfinite(mine).all()
        if name == "front_facing" and not lens:
            lit = mine[seen].mean(axis=-1)
            assert np.median(lit) > 10 * np.median(mine[~seen].mean(axis=-1) + 1e-6)
        if name == "front_facing_away" and not lens and shape == 1:
            inner = _lit_by_camera_rays_shrunk(renderer, cfg, name)
            assert inner.sum() > 0 and float(mine[inner].max()) == 0.0   # 0 added, path ended (pathtracer.cu:225-227)
        # the tone-mapped image as well (hdr_to_ldr)
        if isinstance(ref, OracleRef):
            check_u8(renderer.ldr_image().cpu().numpy(), ref)
        else:
            du8 = np.abs(renderer.ldr_image().cpu().numpy().astype(int) - ref.ldr_image().cpu().numpy().astype(int)).max(axis=2)
            assert (du8 <= 1).mean() >= 0.999


def _lit_by_camera_rays_shrunk(renderer, cfg, name):
    """Pixels all of whose jittered rays hit the in-view disk: 3x3 erosion of the centre-ray mask."""
    m = _lit_by_camera_rays(renderer, cfg, name)
    # the default light above is out of view, so the mask is the in-view disk alone
    e = m.copy()
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            e &= np.roll(np.roll(m, dy, axis=0), dx, axis=1)
    return e


@pytest.mark.parametrize("name", ["front_facing", "behind_volume", "inside_volume", "ring_of_small_disks", "clipped_by_image_edge"])
def test_product_mode_with_lights_in_view_is_statistically_the_reference(renderer, name):
    depth = 3
    cfg = _setup(renderer, name, depth, False)
    # 16 batches of 16 spp: the Welch statistic's tails depend on the number of batches the standard errors come from
    _statistical_parity(renderer, cfg, depth, 16, 16, lambda: renderer.set_option(L.OPT_PT_MODE, 2), mean_tol=0.02)


@pytest.mark.parametrize("name", sorted(SCENES))
def test_light_cull_is_bit_exact(renderer, name):
    """classify_pixel only rules out disks no camera ray of the pixel can hit: with the cull off every camera ray tests
    every disk, as the reference does, and the image must not change in a single bit."""
    depth = 2
    cfg = _setup(renderer, name, depth, False)
    for mode, shape, spp in ((2, 5, 40), (2, 4, 40), (2, 2, 40), (2, 1, 5), (2, 3, 40), (1, 2, 33), (0, 1, 2)):
        renderer.set_option(L.OPT_PT_MODE, mode)
        renderer.set_option(L.OPT_PT_KERNEL, shape)
        renderer.set_option(L.OPT_PT_WARP_MIN_SPP, 1)
        renderer.set_option(L.OPT_PT_QUEUE_MIN_DEPTH, 0)
        renderer.set_option(L.OPT_PT_PROFILE, 1 if shape == 4 else 0)
        imgs = []
        for cull in (1, 0):
            renderer.set_option(L.OPT_PT_LIGHT_CULL, cull)
            renderer.frame_no = 0
            renderer.render_pathtracer_spp(spp, depth)
            torch.cuda.synchronize()
            imgs.append(renderer.hdr_image().clone())
        renderer.set_option(L.OPT_PT_LIGHT_CULL, 1)
        assert float(imgs[0].max()) > 0
        assert torch.equal(imgs[0], imgs[1]), (name, mode, shape)


def test_light_cull_with_camera_close_to_a_large_light(renderer):
    """The cull's reach must hold when the disk is nearer than its own radius (angles are no longer small)."""
    cfg = small_config(n=N, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    setup(renderer, cfg)
    cam = S.look_at_camera((40.0, 30.0, 70.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), image_w=cfg.width, image_h=cfg.height)
    renderer.set_camera(cam)
    near = _light((36.0, 27.0, 62.0), (0.2, 0.3, 1.0), 25.0)   # 9 units from the eye, radius 25, partly behind it
    side = _light((-30.0, 0.0, 20.0), (1.0, 0.0, 0.3), 10.0)
    renderer.set_area_lights([near, side])
    renderer.set_option(L.OPT_PT_MODE, 0)
    ref = oracle_reference(renderer, cfg)
    renderer.frame_no = 0
    for _ in range(2):
        renderer.render_pathtracer(2)
    torch.cuda.synchronize()
    mine = renderer.hdr_image().cpu().numpy()
    ref.render_pathtracer(2, 2)
    theirs = ref.hdr_image().cpu().numpy()
    assert theirs.max() > 0
    if isinstance(ref, OracleRef):
        check_paths(mine, theirs, ref, scaled=True)
    else:
        assert _close(mine, theirs).mean() >= 0.999
    renderer.set_option(L.OPT_PT_MODE, 2)
    imgs = []
    for cull in (1, 0):
        renderer.set_option(L.OPT_PT_LIGHT_CULL, cull)
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(33, 2)
        torch.cuda.synchronize()
        imgs.append(renderer.hdr_image().clone())
    renderer.set_option(L.OPT_PT_LIGHT_CULL, 1)
    assert torch.equal(imgs[0], imgs[1])
