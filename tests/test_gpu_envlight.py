"""Environment lighting (core/lights/cuda_environment_light.h:58-72; core/lights/lights.cpp:31-90) through
the C ABI.  The reference left its only call site commented out (pathtracer.cu:233); the checker is the
environment-light twin of the reference -- the same sources with that one line re-enabled at build time
(oracle/Makefile) -- so constant skies and HDR maps are compared path for path in the twin mode and
statistically in the product mode.  Where the twin is not built, constant skies are compared path for path with the CPU
oracle, and the statistical comparisons take the product's twin mode as their reference arm (see _statistical_parity)."""
import numpy as np
import pytest
import torch

from oracle import binding as B
from oracle import hdr_oracle as H
from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

from _gpu_common import OracleRef, check_paths, oracle_reference, reference, setup, small_config
from test_gpu_pathtrace import _frames, _statistical_parity

pytestmark = pytest.mark.gpu


def _sky_file(tmp_path, w=128, h=64):
    v, u = np.meshgrid(np.linspace(0, 1, h), np.linspace(0, 1, w), indexing="ij")
    img = np.stack([0.2 + 0.6 * u, 0.3 + 0.3 * np.sin(6.28 * u) ** 2, 0.9 - 0.7 * v], axis=2)
    img[h // 4: h // 4 + 4, w // 2: w // 2 + 6] = [60.0, 50.0, 30.0]
    return H.write_hdr(tmp_path / "sky.hdr", H.float_to_rgbe(img))


def _twin_check(renderer, cfg, depth, frames=3):
    """Path for path against the environment-light twin of the reference; where it is not built, against the CPU oracle,
    whose environment light is the constant sky: an HDR map is then compared only statistically (_statistical_parity)."""
    renderer.set_option(L.OPT_PT_MODE, 0)
    mine = _frames(renderer, frames, depth)
    if B.ref(cfg.width, cfg.height, env=True) is None and renderer.env.tex:
        return mine
    ref = oracle_reference(renderer, cfg, env=True)
    ref.render_pathtracer(frames, depth)
    theirs = ref.hdr_image().cpu().numpy()
    if isinstance(ref, OracleRef):
        check_paths(mine, theirs, ref, scaled=True)
    else:
        d = np.abs(mine - theirs).max(axis=2)
        tol = 1e-4 * np.maximum(1.0, theirs.max(axis=2))
        assert (d <= tol).mean() >= 0.998, (d.max(), (d <= tol).mean())
        assert abs(mine.mean() - theirs.mean()) <= 2e-3 * theirs.mean()
    return mine


def test_constant_sky_matches_the_reference_twin(renderer):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=3, env=True)
    setup(renderer, cfg)
    mine = _twin_check(renderer, cfg, 3)
    assert mine[0, 0] == pytest.approx([0.5, 0.5, 0.5])          # a corner ray sees the sky (gui/canvas.cpp:11-12)
    env = S.constant_env_light((0.1, 0.4, 0.9), intensity=2.0)
    renderer.set_env_light(env, enabled=True)
    mine = _twin_check(renderer, cfg, 3)
    assert mine[0, 0] == pytest.approx([0.2, 0.8, 1.8])
    _statistical_parity(renderer, cfg, 3, 8, 32, lambda: renderer.set_option(L.OPT_PT_MODE, 2), mean_tol=0.01, env=True)


def test_hdr_map_matches_the_reference_twin(renderer, tmp_path):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=3, env=True)
    setup(renderer, cfg)
    renderer.load_env_map(_sky_file(tmp_path), intensity=1.5, offset=(0.13, -0.04))
    mine = _twin_check(renderer, cfg, 3)
    assert np.ptp(mine[0, :, 2]) > 0.005                         # the map, not a constant, is what the corner rays see
    renderer.set_area_lights([])                                 # lit by the sky alone
    _twin_check(renderer, cfg, 2)
    _statistical_parity(renderer, cfg, 3, 8, 32, lambda: renderer.set_option(L.OPT_PT_MODE, 2), mean_tol=0.01, env=True)
    # offset wraps (cudaAddressModeWrap, lights.cpp:62-63): a whole turn changes nothing
    renderer.set_option(L.OPT_PT_MODE, 2)
    a = renderer.env
    renderer.frame_no = 0
    renderer.render_pathtracer_spp(4, 2)
    torch.cuda.synchronize()
    img0 = renderer.hdr_image().clone()
    a.offset = L.Vec2(a.offset.x + 1.0, a.offset.y)
    renderer.set_env_light(a, enabled=True)
    renderer.frame_no = 0
    renderer.render_pathtracer_spp(4, 2)
    torch.cuda.synchronize()
    assert torch.allclose(renderer.hdr_image(), img0, rtol=1e-3, atol=1e-4)


def _sun_file(tmp_path, w=256, h=128):
    """A dim sky with a small, very bright sun and a glowing horizon band: what importance sampling is for."""
    v, u = np.meshgrid(np.linspace(0, 1, h), np.linspace(0, 1, w), indexing="ij")
    img = np.stack([0.05 + 0.05 * u, 0.06 + 0.02 * v, 0.10 - 0.05 * v], axis=2)
    img[h // 3: h // 3 + 3, (3 * w) // 8: (3 * w) // 8 + 4] = [4000.0, 3600.0, 3000.0]   # 12 texels of 32768
    img[h // 2 - 1: h // 2 + 1, :] += 0.4
    return H.write_hdr(tmp_path / "sun.hdr", H.float_to_rgbe(img))


def _batches(renderer, K, per, depth):
    from test_gpu_pathtrace import _product_batches

    return _product_batches(renderer, K, per, depth)


def test_environment_sampler_tables_are_a_distribution_over_directions(renderer, tmp_path):
    import ctypes as C

    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2, env=True)
    setup(renderer, cfg)
    renderer.load_env_map(_sun_file(tmp_path), intensity=2.0, offset=(0.25, 0.0))
    w, h = C.c_uint32(), C.c_uint32()
    L.check(renderer.lib.svr_env_sampler_copy(None, None, C.byref(w), C.byref(h)))
    marg = np.zeros(h.value + 1, np.float32)
    cond = np.zeros((h.value, w.value + 1), np.float32)
    L.check(renderer.lib.svr_env_sampler_copy(C.c_void_p(marg.ctypes.data), C.c_void_p(cond.ctypes.data), C.byref(w), C.byref(h)))
    assert marg[0] == 0 and marg[-1] == 1 and (np.diff(marg) > 0).all()          # the floor: no row has probability 0
    assert (cond[:, 0] == 0).all() and (cond[:, -1] == 1).all() and (np.diff(cond, axis=1) > 0).all()
    # most of the probability sits on the sun: rows h/3 .. h/3 + 3 of the picture, columns shifted by the offset (u + 0.25)
    p = np.diff(marg)[:, None] * np.diff(cond, axis=1)
    rows = slice(int(h.value / 3) - 2, int(h.value / 3) + 6)
    assert p[rows].sum() > 0.5
    col = int(((3 / 8) - 0.25) * w.value)
    assert p[rows, col - 6: col + 14].sum() > 0.5


@pytest.mark.parametrize("sky,with_area_light,depth", [("soft", False, 3), ("soft", True, 2), ("sun", False, 3), ("sun", True, 2)])
def test_environment_next_event_estimation_has_the_same_mean_and_less_variance(renderer, tmp_path, sky, with_area_light, depth):
    """SVR_OPT_ENV_NEE against the environment-light twin of the reference (escaped paths look the map up): per-tile Welch
    statistic on the means, and the variance ratio brute force / next-event estimation at equal spp (reported).
    "soft": a sky whose brightest patch is 60 -- the reference's own estimate converges well enough for per-tile statistics;
    "sun": a 12-texel sun of radiance 4000 -- brute force is so noisy there (a tile's estimate is a handful of sun hits) that
    only the variance ratio and the image means are asserted."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=depth, env=True)
    setup(renderer, cfg)
    renderer.load_env_map(_sun_file(tmp_path) if sky == "sun" else _sky_file(tmp_path), intensity=1.0, offset=(0.1, 0.0))
    if not with_area_light:
        renderer.set_area_lights([])
    K, per = 16, 32
    ref = reference(renderer, cfg, env=True)
    from test_gpu_pathtrace import _reference_batches, _tile_means

    rb, ref_all = _reference_batches(ref, 4 * K, per, depth)
    del ref
    renderer.set_option(L.OPT_PT_MODE, 2)
    out = {}
    for nee in (0, 1):
        renderer.set_option(L.OPT_ENV_NEE, nee)
        out[nee] = _batches(renderer, K, per, depth)
    renderer.set_option(L.OPT_ENV_NEE, 0)
    lit = ref_all.mean(axis=2) > 0
    var = {k: v.var(axis=0, ddof=1)[lit].mean() for k, v in out.items()}
    ratio = var[0] / var[1]
    print(f"env NEE variance ratio (brute force / next-event), {sky} sky, area light {with_area_light}, depth {depth}: {ratio:.1f}")
    # (with an area light in the scene the pick is shared: the area light gets half the samples, which costs a soft sky more
    # than importance sampling it gains)
    assert ratio > (3.0 if sky == "sun" else 0.4), ratio
    # same mean as the reference twin: Welch per 16x16 tile (the brute-force side of the comparison is the noisy one)
    for nee in ((1, 0) if sky == "soft" else ()):
        mb = out[nee]
        tm = np.stack([_tile_means(b) for b in mb])
        tr = np.stack([_tile_means(b) for b in rb])
        se = np.sqrt(tm.var(axis=0, ddof=1) / tm.shape[0] + tr.var(axis=0, ddof=1) / tr.shape[0])
        num = np.abs(tm.mean(axis=0) - tr.mean(axis=0))
        z = num / np.maximum(se, 1e-30)
        # (tiles that see only the smooth sky have almost no variance: differences below the 1e-4 relative bound of the
        # deterministic outputs are not failures -- see _statistical_parity)
        ok = (z < 4.5) | (num <= 1e-4 * np.abs(tr.mean(axis=0)))
        assert ok.mean() >= 0.99, (nee, float(ok.mean()))
    # and the image means: next-event estimation within 2 % of the (much noisier) reference mean or 4.5 standard errors
    bm, br = out[1].mean(axis=(1, 2, 3)), rb.mean(axis=(1, 2, 3))
    se = np.sqrt(bm.var(ddof=1) / bm.size + br.var(ddof=1) / br.size)
    assert abs(bm.mean() - br.mean()) < max(0.02 * br.mean(), 4.5 * se), (bm.mean(), br.mean(), se)


def test_environment_next_event_estimation_with_a_constant_sky(renderer):
    """A constant sky is sampled uniformly over the sphere: still the reference twin's mean."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=3, env=True)
    setup(renderer, cfg)

    def configure():
        renderer.set_option(L.OPT_PT_MODE, 2)
        renderer.set_option(L.OPT_ENV_NEE, 1)

    # (sharing the pick with the sky halves the area light's samples: more noise at equal spp than the reference's own
    # estimator, so the RMSE bound is relaxed; the per-tile Welch statistic and the image means are held as everywhere)
    _statistical_parity(renderer, cfg, 3, 16, 16, configure, mean_tol=0.01, env=True, rmse_tol=2.0)
    renderer.set_option(L.OPT_ENV_NEE, 0)
