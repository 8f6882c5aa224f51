"""Denoising (svr_pathtracer_guides, svr_pathtracer_denoise, Renderer.guides / Renderer.denoise).

The filter is held to a float64 numpy restatement of the formulas in include/svr_render.h on synthetic inputs, to its
identities (iterations = 0 is svr_pathtracer_resolve bit for bit; a constant demodulated image and a zero-variance pixel
come back unchanged) and to the edges its guides must keep.  The guides are held to a Python restatement of the march on
the CPU oracle's texture sampler (oracle/binding.py: bit-exact to the texture hardware) and to an analytic sphere.  Image
quality is measured against a 32768-spp render.  The layout and argument tests at the end run without a GPU."""
import ctypes as C
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LUM = np.array([0.2126, 0.7152, 0.0722])
HK = np.array([1.0, 4.0, 6.0, 4.0, 1.0]) / 16.0
FLT_MIN = 1.1754944e-38  # the device flushes denormal weights to zero
DEFAULTS = dict(iterations=5, sigma_luminance=4.0, sigma_normal=128.0, sigma_depth=1.0, sigma_coverage=0.1)


# ---------------------------------------------------------------------------------------------------------------------
# numpy restatement of the filter (float64)
# ---------------------------------------------------------------------------------------------------------------------
def _modulation(ac):
    a = ac[..., 3:4]
    return np.maximum(a * ac[..., :3] + (1.0 - a), 1e-3)


def np_denoise(s, h, ac, nd, tan_fov, iterations, sigma_luminance, sigma_normal, sigma_depth, sigma_coverage):
    """hdr (H, W, 3) of svr_pathtracer_denoise for float4 images s, h, ac, nd of shape (H, W, 4)."""
    s, h, ac, nd = (np.asarray(x, np.float64) for x in (s, h, ac, nd))
    H, W = s.shape[:2]
    w = s[..., 3:4]
    with np.errstate(divide="ignore", invalid="ignore"):
        c = s[..., :3] * np.where(w > 0, 1.0 / w, 0.0)
        if iterations == 0:
            return c
        m = _modulation(ac)
        e = c / m
        hw, we = h[..., 3:4], w - h[..., 3:4]
        even = (s[..., :3] - h[..., :3]) / we / m
        odd = h[..., :3] / hw / m
        var = np.where(((hw > 0) & (we > 0))[..., 0], ((even - odd) @ LUM) ** 2 / 4.0, np.inf)
    p = np.pad(var, 1, mode="edge")
    b = [0.25, 0.5, 0.25]
    var = sum(b[j] * b[i] * p[j:j + H, i:i + W] for j in range(3) for i in range(3))
    n, z, a = nd[..., :3], nd[..., 3], ac[..., 3]
    n0 = (n == 0).all(axis=-1)
    pix = 2.0 * tan_fov / (H - 1.0)
    for it in range(iterations):
        st = 1 << it
        lp = e @ LUM
        lum_den = sigma_luminance * np.sqrt(var) + 1e-10
        z_den = sigma_depth * st * z * pix + 1e-10
        sw = np.zeros((H, W))
        acc = np.zeros((H, W, 3))
        sv = np.zeros((H, W))
        for dy in range(-2, 3):
            for dx in range(-2, 3):
                yy, xx = np.arange(H) + st * dy, np.arange(W) + st * dx
                vy, vx = (yy >= 0) & (yy < H), (xx >= 0) & (xx < W)
                valid = vy[:, None] & vx[None, :]
                Y, X = np.clip(yy, 0, H - 1)[:, None], np.clip(xx, 0, W - 1)[None, :]
                eq, vq, nq, zq, aq = e[Y, X], var[Y, X], n[Y, X], z[Y, X], a[Y, X]
                if sigma_normal > 0:
                    nq0 = n0[Y, X]
                    d = np.maximum((n * nq).sum(axis=-1), 0.0)
                    with np.errstate(divide="ignore"):
                        wn = np.where(n0 & nq0, 1.0, np.where(n0 | nq0, 0.0, d ** sigma_normal))
                else:
                    wn = np.ones((H, W))
                with np.errstate(invalid="ignore"):
                    ex = np.exp(-(np.abs(lp - eq @ LUM) / lum_den + np.abs(z - zq) / z_den + np.abs(a - aq) / sigma_coverage))
                ex = np.where(ex < FLT_MIN, 0.0, ex)
                wgt = np.where(valid, HK[dy + 2] * HK[dx + 2] * wn * ex, 0.0)
                wgt = np.where(wgt < FLT_MIN, 0.0, wgt)
                sw += wgt
                acc += wgt[..., None] * eq
                with np.errstate(invalid="ignore"):
                    sv += np.where(wgt > 0, wgt * wgt * vq, 0.0)
        e = acc / sw[..., None]
        var = sv / sw ** 2
    return m * e


def np_tone_map(x, exposure):
    return (1.0 - np.exp(-np.asarray(x, np.float64) * 16.0 * exposure)) ** 2.2


# ---------------------------------------------------------------------------------------------------------------------
# synthetic inputs
# ---------------------------------------------------------------------------------------------------------------------
def synthetic(H=37, W=53, seed=1):
    """sum, halfSum and guides: three coverage bands (0, 1, fractional), sample counts 32..256, some pixels with an empty
    odd half, a depth step, smooth normals (0 where the ray misses, and a few covered pixels without a gradient)."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:H, 0:W].astype(np.float64)
    alpha = np.where(xx < W // 3, 0.0, np.where(xx < 2 * W // 3, 1.0, rng.uniform(0.2, 0.9, (H, W))))
    albedo = np.clip(0.5 + 0.3 * np.sin(0.2 * xx[..., None] + np.array([0.0, 1.0, 2.0])) + 0.1 * rng.standard_normal((H, W, 3)), 0.05, 1.0)
    ac = np.concatenate([np.where(alpha[..., None] > 0, albedo, 0.0), alpha[..., None]], axis=-1)
    n = np.stack([0.3 * np.sin(0.1 * xx), 0.3 * np.cos(0.13 * yy), np.ones_like(xx)], axis=-1)
    n /= np.linalg.norm(n, axis=-1, keepdims=True)
    z = 200.0 + 0.5 * xx + np.where(yy > H // 2, 30.0, 0.0)
    nd = np.concatenate([n, z[..., None]], axis=-1)
    nd[alpha == 0] = 0.0
    nd[(alpha > 0) & (rng.uniform(size=(H, W)) < 0.03), :3] = 0.0
    w = rng.choice([32.0, 64.0, 96.0, 256.0], size=(H, W))
    base = 0.2 + 0.6 * (np.sin(0.15 * xx) * np.cos(0.1 * yy))[..., None] ** 2 + 0.05 * np.array([1.0, 0.5, 0.2])
    rad = base * _modulation(ac)
    sd = 0.3 * rad / np.sqrt(w[..., None] / 64.0)
    even = rad + sd * rng.standard_normal((H, W, 3))
    odd = rad + sd * rng.standard_normal((H, W, 3))
    s = np.concatenate([(even + odd) * (w[..., None] / 2.0), w[..., None]], axis=-1)
    h = np.concatenate([odd * (w[..., None] / 2.0), w[..., None] / 2.0], axis=-1)
    h[rng.uniform(size=(H, W)) < 0.04] = 0.0
    return [np.ascontiguousarray(x, np.float32) for x in (s, h, ac, nd)]


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
def _dev(a):
    import torch

    return torch.from_numpy(np.ascontiguousarray(a, np.float32).reshape(-1)).cuda()


def _scene(r, n=128, w=192, h=128, gen=L.GEN_CT, env=True):
    from _gpu_common import setup, small_config

    cfg = small_config(n=n, w=w, h=h, gen=gen, fmt=L.VOXEL_U16, env=env)
    vox = setup(r, cfg)
    return cfg, vox


def _camera_for(r, W, H):
    """A camera of W x H pixels (the filter reads only the image size, tanFovxOverTwo and exposure from it)."""
    r.set_camera(S.default_camera((64.0,) * 3, W, H))


def _run_filter(r, s, h, ac, nd, want_hdr=True, **kw):
    import torch

    H, W = s.shape[:2]
    bufs = [_dev(x) for x in (s, h, ac, nd)]
    r.denoise(bufs[0], bufs[1], (bufs[2], bufs[3]), want_hdr=want_hdr, **kw)
    torch.cuda.synchronize()
    return r.hdr_image().cpu().numpy().copy(), r.ldr_image().cpu().numpy().copy()


def _resolve(r, s):
    import torch

    r.resolve(_dev(s))
    torch.cuda.synchronize()
    return r.hdr_image().cpu().numpy().copy(), r.ldr_image().cpu().numpy().copy()


def _u8(hdr, exposure):
    return (np_tone_map(hdr, exposure) * 255.0).astype(np.float32).astype(np.int64)


@pytest.fixture
def scene(renderer):
    yield renderer
    renderer.set_option(L.OPT_PT_MODE, 2)
    renderer.set_option(L.OPT_ENV_NEE, 0)
    renderer.set_option(L.OPT_COUNTERS, 0)


# ---- 1. the filter against its numpy restatement
PARAM_SETS = {
    "defaults": {},
    "tight": dict(sigma_luminance=1.0, sigma_normal=16.0, sigma_depth=4.0, sigma_coverage=0.5),
    "loose_no_normal": dict(sigma_luminance=8.0, sigma_normal=0.0, sigma_depth=0.25, sigma_coverage=0.05),
}


@pytest.mark.gpu
@pytest.mark.parametrize("iterations", [1, 5])
@pytest.mark.parametrize("params", list(PARAM_SETS))
def test_filter_matches_numpy(scene, params, iterations):
    """53 x 37 (a multiple of no block size).  Tolerance: |gpu - numpy| <= 1e-4 max(1, |numpy|) on HDR.  The device computes
    in fp32 with fast math: __expf and __powf carry a relative error of a few 1e-7 (times the exponent, at most ~20 where a
    weight still matters), division is approximate (2 ulp), and the weighted sums of 25 taps over 5 iterations add a few ulp
    each; together they stay below 1e-5 relative, and 1e-4 leaves a margin for weights whose exponent is large.  u8: the tone
    map of the two HDR images differs by at most 1 LSB (a value near a quantisation step may round either way)."""
    r = scene
    _scene(r)
    s, h, ac, nd = synthetic()
    H, W = s.shape[:2]
    _camera_for(r, W, H)
    kw = dict(DEFAULTS, **PARAM_SETS[params], iterations=iterations)
    hdr, img = _run_filter(r, s, h, ac, nd, **kw)
    ref = np_denoise(s, h, ac, nd, r.camera.tanFovxOverTwo, **kw)
    assert np.isfinite(ref).all()
    err = np.abs(hdr.reshape(H, W, 3) - ref) / np.maximum(1.0, np.abs(ref))
    assert err.max() <= 1e-4, float(err.max())
    d = np.abs(img.reshape(H, W, 4)[..., :3].astype(np.int64) - _u8(ref, r.camera.exposure))
    assert d.max() <= 1, int(d.max())
    assert (img.reshape(H, W, 4)[..., 3] == 255).all()
    # the filter did something: the result is not the raw mean
    raw = s[..., :3] / s[..., 3:4]
    assert np.abs(ref - raw).max() > 1e-2


# ---- 2. identities
@pytest.mark.gpu
def test_zero_iterations_is_resolve_bit_for_bit(scene):
    import torch

    r = scene
    _scene(r, w=96, h=64)
    H, W = r.camera.imageH, r.camera.imageW
    s = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    h = torch.zeros_like(s)
    r.accumulate_adaptive(s, h, 1, 0, 64, 64, 32, 0.0)
    g = r.guides()
    r.resolve(s)
    torch.cuda.synchronize()
    ref_hdr, ref_img = r.hdr.clone(), r.img.clone()
    r.hdr.fill_(-1.0)
    r.img.fill_(7)
    r.denoise(s, h, g, iterations=0)
    torch.cuda.synchronize()
    assert torch.equal(r.hdr.view(torch.int32), ref_hdr.view(torch.int32))
    assert torch.equal(r.img, ref_img)
    # img alone (hdr untouched)
    r.hdr.fill_(-1.0)
    r.img.fill_(7)
    r.denoise(s, h, g, iterations=0, want_hdr=False)
    torch.cuda.synchronize()
    assert torch.equal(r.img, ref_img) and (r.hdr == -1.0).all()


@pytest.mark.gpu
def test_constant_demodulated_image_is_unchanged(scene):
    r = scene
    _scene(r)
    rng = np.random.default_rng(3)
    s, h, ac, nd = synthetic(seed=3)
    H, W = s.shape[:2]
    _camera_for(r, W, H)
    # any guides: random coverage, albedo, normals and depths
    ac = np.concatenate([rng.uniform(0.05, 1.0, (H, W, 3)), rng.choice([0.0, 1.0, 0.5], (H, W))[..., None]], axis=-1).astype(np.float32)
    n = rng.standard_normal((H, W, 3))
    nd = np.concatenate([n / np.linalg.norm(n, axis=-1, keepdims=True), rng.uniform(10, 300, (H, W, 1))], axis=-1).astype(np.float32)
    m = _modulation(ac.astype(np.float64))
    s[..., 3] = 64.0
    s[..., :3] = (0.7 * m * 64.0).astype(np.float32)  # c / m = 0.7 everywhere
    c, _ = _resolve(r, s)
    hdr, _ = _run_filter(r, s, h, ac, nd)
    rel = np.abs(hdr - c) / np.abs(c)
    assert rel.max() <= 1e-6, float(rel.max())


@pytest.mark.gpu
def test_zero_variance_pixel_is_unchanged(scene):
    r = scene
    _scene(r)
    s, h, ac, nd = synthetic(seed=4)
    H, W = s.shape[:2]
    _camera_for(r, W, H)
    h[s[..., 3] == 0] = 0.0
    pts = [(5, 7), (18, 26), (30, 45), (12, 40)]
    for y, x in pts:  # identical halves over the 3 x 3 window: Var = 0 after the prefilter
        h[y - 1:y + 2, x - 1:x + 2] = s[y - 1:y + 2, x - 1:x + 2] / 2.0
    c, _ = _resolve(r, s)
    hdr, _ = _run_filter(r, s, h, ac, nd)
    c, hdr = c.reshape(H, W, 3), hdr.reshape(H, W, 3)
    for y, x in pts:
        rel = np.abs(hdr[y, x] - c[y, x]) / np.abs(c[y, x])
        assert rel.max() <= 1e-6, (y, x, rel)
    # and pixels that are not: the filter moved them
    assert np.abs(hdr - c).max() > 1e-2


@pytest.mark.gpu
def test_sky_is_unchanged(scene):
    """All-sky pixels of a render (the constant environment: identical halves, Var = 0) away from the volume."""
    import torch

    r = scene
    _scene(r, n=64, w=96, h=64)
    H, W = r.camera.imageH, r.camera.imageW
    s = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    h = torch.zeros_like(s)
    r.accumulate_adaptive(s, h, 1, 0, 64, 64, 32, 0.0)
    g = r.guides()
    r.resolve(s)
    torch.cuda.synchronize()
    raw = r.hdr_image().cpu().numpy().copy()
    r.denoise(s, h, g)
    torch.cuda.synchronize()
    den = r.hdr_image().cpu().numpy()
    sky = np.all(raw == raw[0, 0], axis=-1)
    assert sky.mean() > 0.2
    core = sky.copy()
    for dy in (-1, 0, 1):
        for dx in (-1, 0, 1):
            core &= np.roll(np.roll(sky, dy, 0), dx, 1)
    rel = np.abs(den[core] - raw[core]) / raw[core]
    assert rel.max() <= 1e-6, float(rel.max())


# ---- 3. edges the guides keep
def _two_regions(H=40, W=24, seed=5):
    """Left and right halves, flat, mean radiance 1.00 and 1.02 against a per-pixel standard error of 0.035."""
    rng = np.random.default_rng(seed)
    mu = np.where(np.arange(W) < W // 2, 1.0, 1.02)[None, :, None] * np.ones((H, W, 3))
    even = mu + 0.05 * rng.standard_normal((H, W, 3))
    odd = mu + 0.05 * rng.standard_normal((H, W, 3))
    s = np.concatenate([(even + odd) * 32.0, np.full((H, W, 1), 64.0)], axis=-1)
    h = np.concatenate([odd * 32.0, np.full((H, W, 1), 32.0)], axis=-1)
    ac = np.concatenate([np.ones((H, W, 3)), np.ones((H, W, 1))], axis=-1)
    nd = np.concatenate([np.zeros((H, W, 2)), np.ones((H, W, 1)), np.full((H, W, 1), 100.0)], axis=-1)
    return [np.ascontiguousarray(x, np.float32) for x in (s, h, ac, nd)]


def _separate(kind, s, h, ac, nd, tan_fov):
    H, W = s.shape[:2]
    right = np.arange(W) >= W // 2
    if kind == "depth":
        f = 2.0 * 100.0 * tan_fov / (H - 1.0)
        nd[:, right, 3] = 100.0 + 100.0 * f  # 100 pixel footprints behind
    elif kind == "normal":
        nd[:, right, 2] = -1.0
    else:
        ac[:, ~right, 3] = 0.0  # coverage 0 against 1 (albedo 1: the same modulation, m = 1)
    return s, h, ac, nd


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["depth", "normal", "coverage"])
def test_edges_are_kept(scene, kind):
    """Each region's own mean is the mean of that region filtered as an image of its own (taps across the step dropped:
    what a perfect edge stop gives); the pixels two or more pixels from the step are compared.  Without the guide step the
    two regions blend (the luminance stop alone does not keep them apart): their means move toward each other."""
    r = scene
    _scene(r)
    s, h, ac, nd = _two_regions()
    H, W = s.shape[:2]
    half = W // 2

    def means(s, h, ac, nd):
        _camera_for(r, W, H)
        full, _ = _run_filter(r, s, h, ac, nd)
        full = full.reshape(H, W, 3)
        _camera_for(r, half, H)
        alone_l, _ = _run_filter(r, *[np.ascontiguousarray(x[:, :half]) for x in (s, h, ac, nd)])
        alone_r, _ = _run_filter(r, *[np.ascontiguousarray(x[:, half:]) for x in (s, h, ac, nd)])
        own_l, own_r = alone_l.reshape(H, half, 3)[:, : half - 2].mean(), alone_r.reshape(H, half, 3)[:, 2:].mean()
        return (full[:, : half - 2].mean() - own_l) / own_l, (full[:, half + 2:].mean() - own_r) / own_r

    blend_l, blend_r = means(s, h, ac, nd)
    sep_l, sep_r = means(*_separate(kind, s, h, ac, nd, S.default_camera((64.0,) * 3, W, H).tanFovxOverTwo))
    assert abs(sep_l) <= 1e-3 and abs(sep_r) <= 1e-3, (sep_l, sep_r)
    # the control: left (darker) pulled up, right pulled down, far more than with the guide step
    assert blend_l > 10 * abs(sep_l) and -blend_r > 10 * abs(sep_r), (blend_l, blend_r, sep_l, sep_r)


# ---- 4. guides against a restatement of the march on the CPU oracle's sampler
def _cam_ray(cam, x, y, jx, jy):
    f32 = np.float32
    u, v, w = (np.array([c.x, c.y, c.z], np.float32) for c in (cam.u, cam.v, cam.w))
    pos = np.array([cam.pos.x, cam.pos.y, cam.pos.z], np.float32)
    nx = f32(2.0) * ((f32(x) + f32(jx)) / (f32(cam.imageW) - f32(1))) - f32(1)
    ny = f32(2.0) * ((f32(y) + f32(jy)) / (f32(cam.imageH) - f32(1))) - f32(1)
    nx = nx * f32(cam.aspectRatio) * f32(cam.tanFovxOverTwo) * f32(cam.focalLength)
    ny = ny * f32(cam.tanFovxOverTwo) * f32(cam.focalLength)
    ax = ay = 0.0
    if cam.apeture != 0.0:
        ox, oy = 2.0 * jx - 1.0, 2.0 * jy - 1.0
        if ox == 0.0 and oy == 0.0:
            dx = dy = 0.0
        elif abs(ox) > abs(oy):
            rr, th = ox, 0.25 * math.pi * (oy / ox)
            dx, dy = rr * math.cos(th), rr * math.sin(th)
        else:
            rr, th = oy, 0.5 * math.pi - 0.25 * math.pi * (ox / oy)
            dx, dy = rr * math.cos(th), rr * math.sin(th)
        ax, ay = f32(dx * cam.apeture), f32(dy * cam.apeture)
    orig = pos + f32(ax) * u + f32(ay) * v
    d = (nx - f32(ax)) * u + (ny - f32(ay)) * v - f32(cam.focalLength) * w
    return orig.astype(np.float64), (d / np.linalg.norm(d)).astype(np.float64)


def _light_t(lights, o, d):
    best = np.inf
    for l in lights:
        c = np.array([l.disk.center.x, l.disk.center.y, l.disk.center.z])
        n = np.array([l.disk.normal.x, l.disk.normal.y, l.disk.normal.z])
        den = d @ n
        if abs(den) > 1e-6:
            t = ((c - o) @ n) / den
            if t >= 0 and np.linalg.norm(o + t * d - c) <= l.disk.radius and t < best:
                best = t
    return best


def _guides_np(r, k):
    import torch

    ac, nd = r.guides(rays_per_pixel=k)
    torch.cuda.synchronize()
    H, W = r.camera.imageH, r.camera.imageW
    return ac.view(H, W, 4).cpu().numpy(), nd.view(H, W, 4).cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 4])
def test_guides_match_restatement(scene, oracle_cpu, k):
    r = scene
    cfg, vox = _scene(r, n=32, w=24, h=16)
    r.set_camera(S.default_camera(cfg.extent, 24, 16, apeture=1.0, focal_length=50.0))
    from _gpu_common import OracleRef

    ref = OracleRef(r, cfg.fmt, (cfg.n,) * 3)
    ref.setup(r.volume, r.tf, r.camera, r.lights, r.env)
    mine_ac, mine_nd = _guides_np(r, k)
    theirs_ac, theirs_nd = restated_guides(ref.oracle, r.volume, r.camera, r.lights, k)
    cov = theirs_ac[..., 3]
    assert (cov > 0.05).mean() > 0.1 and (cov == 0).any()
    assert np.abs(mine_ac[..., 3] - cov).max() <= 1e-3
    sel = cov > 0.05
    assert np.abs(mine_ac[..., :3] - theirs_ac[..., :3])[sel].max() <= 1e-3
    assert (np.abs(mine_nd[..., 3] - theirs_nd[..., 3]) / theirs_nd[..., 3])[sel].max() <= 1e-3
    assert ((mine_nd[..., :3] * theirs_nd[..., :3]).sum(axis=-1)[sel] >= 0.999).all()
    miss = mine_ac[..., 3] == 0
    assert miss.any() and (mine_ac[miss] == 0).all() and (mine_nd[miss] == 0).all()


def restated_guides(oracle, vol, cam, lights, k):
    """The march of svr_pathtracer_guides in Python, one ray at a time, on the CPU oracle's tex3d and TF look-up."""
    from oracle import binding as B

    lib = B.cpu()
    scene_struct = oracle.scene
    H, W = cam.imageH, cam.imageW
    vmin = np.array([vol.bbox.vmin.x, vol.bbox.vmin.y, vol.bbox.vmin.z])
    vmax = np.array([vol.bbox.vmax.x, vol.bbox.vmax.y, vol.bbox.vmax.z])
    inv_size = np.array([vol.bbox.invSize.x, vol.bbox.invSize.y, vol.bbox.invSize.z])
    sp = np.array([vol.spacing.x, vol.spacing.y, vol.spacing.z])
    ds = vol.densityScale
    hstep = 0.5 * sp.min()
    back = -np.array([cam.w.x, cam.w.y, cam.w.z])
    pos = np.array([cam.pos.x, cam.pos.y, cam.pos.z])
    rgba = (C.c_float * 4)()
    out_ac, out_nd = np.zeros((H, W, 4)), np.zeros((H, W, 4))
    side = int(round(math.sqrt(k)))

    def inten(p):
        tc = (p - vmin) * inv_size
        return lib.svr_oracle_tex3d(C.byref(scene_struct), float(tc[0]), float(tc[1]), float(tc[2])) * ds

    for y in range(H):
        for x in range(W):
            alpha, A, Z, N = 0.0, np.zeros(3), 0.0, np.zeros(3)
            for j in range(side):
                for i in range(side):
                    o, d = _cam_ray(cam, x, y, (i + 0.5) / side, (j + 0.5) / side)
                    with np.errstate(divide="ignore", invalid="ignore"):
                        t1, t2 = (vmin - o) / d, (vmax - o) / d
                    tn, tf = np.minimum(t1, t2).max(), np.maximum(t1, t2).min()
                    if not tf > tn:
                        continue
                    t_end = min(tf, _light_t(lights, o, d))
                    t0, T, kk = max(tn, 0.0), 1.0, 0
                    while True:
                        t = t0 + (kk + 0.5) * hstep
                        kk += 1
                        if not t < t_end:
                            break
                        p = o + t * d
                        lib.svr_oracle_tf(C.byref(scene_struct), float(inten(p)), rgba)
                        sig = rgba[3]
                        if not sig > 0:
                            continue
                        em = math.expm1(-sig * hstep)
                        pw = -T * em
                        alpha += pw
                        A += pw * np.array(rgba[:3])
                        Z += pw * ((p - pos) @ back)
                        g = np.array([inten(p + e * sp) - inten(p - e * sp) for e in np.eye(3)]) * 0.5 / sp
                        if g @ g > 0:
                            nn = g / np.linalg.norm(g)
                            N += pw * (-nn if nn @ d > 0 else nn)
                        T += T * em
                        if T < 1e-3:
                            break
            if alpha > 0:
                nrm = np.linalg.norm(N)
                out_ac[y, x] = [*(A / alpha), alpha / k]
                out_nd[y, x] = [*(N / nrm if nrm > 0 else N), Z / alpha]
    return out_ac, out_nd


# ---- 5. guides, analytically: the isosurface of a sphere under a step transfer function
def _centre_rays(cam):
    W, H = cam.imageW, cam.imageH
    x = (np.arange(W) + 0.5) / (W - 1.0) * 2 - 1
    y = (np.arange(H) + 0.5) / (H - 1.0) * 2 - 1
    nx, ny = np.meshgrid(x * cam.aspectRatio * cam.tanFovxOverTwo, y * cam.tanFovxOverTwo)
    d = np.stack([nx, ny, -np.ones_like(nx)], axis=-1)
    return d / np.linalg.norm(d, axis=-1, keepdims=True)


@pytest.mark.gpu
def test_guides_of_a_sphere(scene):
    r = scene
    n, tau, sigma = 64, 0.5, 20.0
    _scene(r, n=n, w=96, h=96, gen=L.GEN_SPHERE, env=False)
    table = S.tf_table("default")
    table[:, 3] = np.where(np.linspace(0.0, 1.0, table.shape[0]) >= tau, sigma, 0.0)
    r.set_transfer_function(table)
    ac, nd = _guides_np(r, 1)
    cam = r.camera
    d = _centre_rays(cam)
    o = np.array([cam.pos.x, cam.pos.y, cam.pos.z])
    b = np.linalg.norm(np.cross(o, d), axis=-1)  # distance of the ray from the sphere's centre
    R = 0.45 * n * (1.0 - tau)
    miss = b > 0.45 * n + 1.5  # (trilinear filtering reaches one voxel beyond the support)
    assert miss.sum() > 100 and (ac[miss, 3] == 0).all() and (nd[miss] == 0).all()
    inside = b < 0.8 * R
    assert inside.sum() > 100
    t_hit = -(d @ o) - np.sqrt(np.maximum(R * R - b * b, 0.0))
    x_hit = o + t_hit[..., None] * d
    depth_hit = o[2] - x_hit[..., 2]  # view-space depth: the camera looks down -z
    assert (ac[inside, 3] > 0.99).all(), float(ac[inside, 3].min())
    assert (np.abs(nd[inside, 3] - depth_hit[inside]) <= 1.0 + 1.0 / sigma).all(), float(np.abs(nd[inside, 3] - depth_hit[inside]).max())
    radial = x_hit / np.linalg.norm(x_hit, axis=-1, keepdims=True)
    assert ((nd[..., :3] * radial).sum(axis=-1)[inside] >= 0.98).all()


@pytest.mark.gpu
def test_guides_stop_at_a_light_in_view(scene):
    from _gpu_common import setup, small_config
    from test_gpu_lights_in_view import SCENES, _lit_by_camera_rays

    r = scene
    cfg = small_config(n=64, gen=L.GEN_CT, fmt=L.VOXEL_U16)
    setup(r, cfg)
    hit = _lit_by_camera_rays(r, cfg, "front_facing")
    before, _ = _guides_np(r, 1)  # the disk is not bound yet: the volume behind it is seen
    r.set_area_lights(SCENES["front_facing"])
    ac, nd = _guides_np(r, 1)
    assert hit.sum() > 50 and (before[hit, 3] > 0.5).sum() > 50
    assert (ac[hit, 3] == 0).all() and (nd[hit] == 0).all()


# ---- 6. quality against a 32768-spp render
def _display(hdr, exposure):
    return np_tone_map(hdr, exposure)


def _rmse(a, b):
    return float(np.sqrt(((a - b) ** 2).mean()))


def _render(r, mn, mx, batch, threshold):
    import torch

    H, W = r.camera.imageH, r.camera.imageW
    s = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    h = torch.zeros_like(s)
    r.accumulate_adaptive(s, h, 1, 0, mn, mx, batch, threshold)
    return s, h


def _raw_and_denoised(r, s, h, g):
    import torch

    r.resolve(s)
    torch.cuda.synchronize()
    raw = r.hdr_image().cpu().numpy().copy()
    r.denoise(s, h, g)
    torch.cuda.synchronize()
    return raw, r.hdr_image().cpu().numpy().copy()


@pytest.mark.gpu
def test_quality(scene):
    """Display RMSE against 32768 spp, guides at 16 rays per pixel.  Measured on a B200 with 4-ray guides the filter misses two
    of these bounds (DESIGN.md section 7f): denoised 4096 spp at 1.16 x raw, adaptive + denoise at 1.04 x adaptive alone; a
    converged image needs guides whose sub-pixel average matches the samples' (16 rays: 1.06 x and 0.99 x)."""
    import torch

    r = scene
    _scene(r)
    H, W = r.camera.imageH, r.camera.imageW
    ex = r.camera.exposure
    ref = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    for b in range(32):
        r.accumulate(ref, 1, (1 << 24) + b * 1024, 1024, clear=b == 0)
    torch.cuda.synchronize()
    v = ref.view(H, W, 4).cpu().numpy().astype(np.float64)
    ref_disp = _display(v[..., :3] / v[..., 3:4], ex)
    g = r.guides(rays_per_pixel=16)
    out = {}
    for name, args in (("u64", (64, 64, 32, 0.0)), ("u4096", (4096, 4096, 32, 0.0)), ("adaptive", (64, 1024, 64, 2.0 / 255.0))):
        raw, den = _raw_and_denoised(r, *_render(r, *args), g)
        out[name] = (_rmse(_display(raw, ex), ref_disp), _rmse(_display(den, ex), ref_disp))
    assert out["u64"][1] <= 0.75 * out["u64"][0], out
    assert out["u4096"][1] <= 1.10 * out["u4096"][0], out
    assert out["adaptive"][1] < out["adaptive"][0], out


@pytest.mark.gpu
def test_light_in_view_does_not_bleed(scene):
    """A bright disk in front of the volume (display value near 1 against about 0.3 around it) must not leak into the pixels 3
    to 12 pixels outside it: their mean change (denoised - raw, 4096 spp, display units) stays within 0.25 / 255; leaking even
    a few per cent of the disk's weight would brighten them by several / 255.  (Per pixel they do not all stay within 1/255 of
    the raw image: measured on a B200, 15 % of the pixels 3 to 5 pixels out move by more, and 12 % do without the light --
    the filter's ordinary smoothing at 4096 spp, DESIGN.md section 7f.)"""
    from _gpu_common import setup, small_config
    from test_gpu_lights_in_view import SCENES, _lit_by_camera_rays

    r = scene
    cfg = small_config(n=64, gen=L.GEN_CT, fmt=L.VOXEL_U16)
    setup(r, cfg)
    r.set_area_lights(SCENES["front_facing"])
    hit = _lit_by_camera_rays(r, cfg, "front_facing")

    def grown(m, d):
        out = m.copy()
        for dy in range(-d, d + 1):
            for dx in range(-d, d + 1):
                out |= np.roll(np.roll(m, dy, 0), dx, 1)
        return out

    ring = grown(hit, 12) & ~grown(hit, 2)
    g = r.guides(rays_per_pixel=16)
    raw, den = _raw_and_denoised(r, *_render(r, 4096, 4096, 32, 0.0), g)
    ex = r.camera.exposure
    d = (_display(den, ex) - _display(raw, ex)).mean(axis=-1)
    assert hit.sum() > 50 and ring.sum() > 500
    assert _display(raw, ex)[hit].mean() > 0.8
    assert abs(d[ring].mean()) <= 0.25 / 255.0, float(d[ring].mean() * 255.0)


# ---- 7. errors
@pytest.mark.gpu
def test_rejected_arguments(scene):
    import torch

    r = scene
    _scene(r, n=64, w=32, h=32)
    H, W = r.camera.imageH, r.camera.imageW
    bufs = [torch.zeros(H * W * 4, dtype=torch.float32, device="cuda") for _ in range(4)]
    P = [C.c_void_p(b.data_ptr()) for b in bufs]
    img, hdr = C.c_void_p(r.img.data_ptr()), C.c_void_p(r.hdr.data_ptr())
    torch.cuda.synchronize()
    before = r.launch_count()

    def rejected(rc):
        assert rc != 0 and r.lib.svr_last_error()

    for ac, nd, k in ((None, P[3], 4), (P[2], None, 4), (P[2], P[3], 0), (P[2], P[3], 2), (P[2], P[3], 9)):
        rejected(r.lib.svr_pathtracer_guides(ac, nd, k))
    good = dict(iterations=5, sigmaLuminance=4.0, sigmaNormal=128.0, sigmaDepth=1.0, sigmaCoverage=0.1)
    bad_params = [dict(iterations=9)] + [{k: v} for k in ("sigmaLuminance", "sigmaDepth", "sigmaCoverage") for v in (0.0, -1.0, math.inf, math.nan)] + \
                 [dict(sigmaNormal=v) for v in (-1.0, math.inf, math.nan)]
    for bad in bad_params:
        p = L.DenoiseParams(**dict(good, **bad))
        rejected(r.lib.svr_pathtracer_denoise(img, hdr, P[0], P[1], P[2], P[3], C.byref(p)))
    for i in range(4):
        args = list(P)
        args[i] = None
        rejected(r.lib.svr_pathtracer_denoise(img, hdr, *args, None))
    rejected(r.lib.svr_pathtracer_denoise(None, None, *P, None))
    assert r.launch_count() == before
    with pytest.raises(L.SvrError):
        r.denoise(bufs[0], bufs[1], (bufs[2], bufs[3]), iterations=9)
    with pytest.raises(L.SvrError):
        r.denoise(bufs[0], bufs[1], (bufs[2], bufs[3]), sigma_luminance=0.0)
    with pytest.raises(L.SvrError):
        r.denoise(bufs[0], bufs[1], (None, bufs[3]))
    with pytest.raises(L.SvrError):
        r.guides(rays_per_pixel=3)
    assert r.launch_count() == before


# ---- 8. layout and argument checks without a GPU
def test_params_layout_and_defaults(tmp_path):
    probe = tmp_path / "probe.c"
    probe.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "svr_render.h"\n'
        "int main(void){printf(\"%zu %zu %zu\\n\", sizeof(svr_denoise_params), offsetof(svr_denoise_params, sigmaLuminance),"
        " offsetof(svr_denoise_params, sigmaCoverage));return 0;}\n"
    )
    exe = tmp_path / "probe"
    subprocess.check_call(["/usr/bin/gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    sizes = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    assert sizes == [C.sizeof(L.DenoiseParams), L.DenoiseParams.sigmaLuminance.offset, L.DenoiseParams.sigmaCoverage.offset]
    lib = L.load()
    p = L.DenoiseParams()
    assert lib.svr_denoise_defaults(C.byref(p)) == 0
    assert (p.iterations, p.sigmaLuminance, p.sigmaNormal, p.sigmaDepth, p.sigmaCoverage) == tuple(float(np.float32(v)) for v in DEFAULTS.values())
    assert lib.svr_denoise_defaults(None) != 0


def test_argument_errors_without_a_device():
    """Every argument check runs before any CUDA call.  (The pointers are never dereferenced: each call has a bad argument.)"""
    lib = L.load()
    f = [C.c_void_p(256 * (i + 1)) for i in range(6)]
    good = dict(iterations=5, sigmaLuminance=4.0, sigmaNormal=128.0, sigmaDepth=1.0, sigmaCoverage=0.1)
    cases = [(f[0], f[1], None, f[3], f[4], f[5], None), (f[0], f[1], f[2], None, f[4], f[5], None), (f[0], f[1], f[2], f[3], None, f[5], None),
             (f[0], f[1], f[2], f[3], f[4], None, None), (None, None, f[2], f[3], f[4], f[5], None)]
    for bad in [dict(iterations=9), dict(sigmaLuminance=0.0), dict(sigmaDepth=math.nan), dict(sigmaCoverage=-0.1), dict(sigmaNormal=-1.0),
                dict(sigmaLuminance=math.inf)]:
        cases.append((f[0], f[1], f[2], f[3], f[4], f[5], C.byref(L.DenoiseParams(**dict(good, **bad)))))
    for args in cases:
        assert lib.svr_pathtracer_denoise(*args) != 0
        assert lib.svr_last_error()
    assert lib.svr_pathtracer_guides(None, f[1], 4) != 0
    assert lib.svr_pathtracer_guides(f[0], f[1], 3) != 0
    assert b"raysPerPixel" in lib.svr_last_error()


def test_scene_checks_without_a_device():
    """A fresh process: no camera, no volume.  The denoiser reports the camera, the guide pass the volume, before any CUDA
    call (the pointers are never dereferenced)."""
    code = (
        "import ctypes as C, sys; sys.path.insert(0, %r)\n"
        "from sunvolumerender_b200 import _lib as L\n"
        "lib = L.load(); f = [C.c_void_p(256 * (i + 1)) for i in range(6)]\n"
        "assert lib.svr_pathtracer_denoise(*f, None) != 0 and b'setup_camera' in lib.svr_last_error(), lib.svr_last_error()\n"
        "assert lib.svr_pathtracer_guides(f[0], f[1], 4) != 0 and b'setup_volume' in lib.svr_last_error(), lib.svr_last_error()\n"
    ) % ROOT
    subprocess.check_call([sys.executable, "-c", code])
