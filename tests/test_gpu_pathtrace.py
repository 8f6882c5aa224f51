"""GPU parity of the path tracer (render_pathtracer, pathtracer.h:17) through the C ABI.

Checkers: the reference's own unmodified kernel_pathtracer (oracle/_ref) on the same texture
objects and seeds, and the CPU oracle.  Where oracle/_ref is not built, the path-for-path comparisons take the CPU
oracle (bounds in tests/_gpu_common.py::check_paths) and the statistical ones the product's twin mode
(_statistical_parity).  Tolerances (BASELINE.json north_star; SURVEY.md section 8c):
  * reference-twin mode (global majorant, XORWOW, same draw order): path for path the same walk,
    so every pixel of every frame within 1e-4 of the reference's hdrBuffer;
  * Philox / local-majorant modes: same estimator, different random numbers.  The Monte Carlo noise
    floor is calibrated as RMSE(reference frames A, reference frames B) with disjoint seeds; the new
    image must satisfy RMSE(new, reference) <= 1.15 x that floor, and the converged means must agree
    per 16x16 tile within 4.5 sigma of the tile-mean estimates for >= 99.5% of the tiles.
"""
import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

from _gpu_common import OracleRef, check_paths, check_u8, cpu_oracle, oracle_reference, reference, rmse, rows_of, setup, small_config

pytestmark = pytest.mark.gpu


def _frames(r, n, depth):
    r.frame_no = 0
    for _ in range(n):
        r.render_pathtracer(depth)
    torch.cuda.synchronize()
    return r.hdr_image().cpu().numpy().copy()


@pytest.mark.parametrize("shape", [1, 0])
@pytest.mark.parametrize("depth", [1, 6])
def test_twin_mode_matches_reference_path_for_path(renderer, shape, depth):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=depth)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_PT_MODE, 0)
    renderer.set_option(L.OPT_PT_KERNEL, shape)
    ref = oracle_reference(renderer, cfg)
    for nframes in (1, 4):
        mine = _frames(renderer, nframes, depth)
        ref.frame_no = 0
        ref.render_pathtracer(nframes, depth)
        theirs = ref.hdr_image().cpu().numpy()
        assert theirs.max() > 0
        # FMA contraction may differ between the two compilations; over a long walk a last-bit
        # difference can flip one accept/reject and send that pixel down another path
        check_paths(mine, theirs, ref, frac=1.0 if depth == 1 else 0.999, mean_rel=1e-3)
    # the tone-mapped image too (hdr_to_ldr, pathtracer.cu:282-290)
    check_u8(renderer.ldr_image().cpu().numpy(), ref)


def test_twin_mode_matches_cpu_oracle(renderer):
    cfg = small_config(n=48, w=64, h=64, gen=L.GEN_SPHERE, fmt=L.VOXEL_U16, depth=3)
    vox = setup(renderer, cfg)
    renderer.set_option(L.OPT_PT_MODE, 0)
    mine = _frames(renderer, 2, 3)
    hdr, _ = cpu_oracle(renderer, cfg, vox).pathtrace(3, 0, 2)
    d = np.abs(mine - hdr).max(axis=2)
    # IEEE libm vs fast-math flips a few accept/reject decisions; those pixels walk a different path
    assert (d < 1e-3).mean() > 0.95
    assert abs(mine.mean() - hdr.mean()) < 0.03 * hdr.mean()


def test_twin_mode_batched_equals_frame_by_frame(renderer):
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8, depth=2)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_PT_MODE, 0)
    one_by_one = _frames(renderer, 6, 2)
    renderer.frame_no = 0
    renderer.render_pathtracer_spp(6, 2)
    torch.cuda.synchronize()
    batched = renderer.hdr_image().cpu().numpy()
    assert np.allclose(batched, one_by_one, rtol=1e-5, atol=1e-6)
    # and a batch continues a running mean started frame by frame (pathtracer.cu:81-84)
    _frames(renderer, 2, 2)
    renderer.render_pathtracer_spp(4, 2)
    torch.cuda.synchronize()
    assert np.allclose(renderer.hdr_image().cpu().numpy(), one_by_one, rtol=1e-5, atol=1e-6)


def _tile_means(img, tile=16):
    H, W, C = img.shape
    return img[: H // tile * tile, : W // tile * tile].reshape(H // tile, tile, W // tile, tile, C).mean(axis=(1, 3))


def _reference_batches(ref, batches, per_batch, depth):
    """Means of `batches` consecutive, disjoint blocks of `per_batch` reference frames, recovered from
    the running mean the reference keeps (pathtracer.cu:81-84): block j = (j+1) M_{j+1} - j M_j."""
    ref.frame_no = 0
    out, prev = [], None
    for j in range(batches):
        ref.render_pathtracer(per_batch, depth)
        cur = ref.hdr_image().cpu().numpy().astype(np.float64)
        out.append(cur.copy() if j == 0 else (j + 1) * cur - j * prev)
        prev = cur
    return np.stack(out), prev  # (batches, H, W, 3), mean of everything


def _product_batches(r, batches, per_batch, depth):
    W, H = r.camera.imageW, r.camera.imageH
    out = []
    for j in range(batches):
        part = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
        r.accumulate(part, depth, j * per_batch, per_batch, clear=True)
        torch.cuda.synchronize()
        v = part.view(H, W, 4).cpu().numpy().astype(np.float64)
        assert (v[..., 3] == per_batch).all()
        out.append(v[..., :3] / per_batch)
    return np.stack(out)


def _statistical_parity(renderer, cfg, depth, K, per, configure, mean_tol=0.01, env=False, rmse_tol=1.15):
    """Both sides render disjoint batches of `per` spp (reference 4K of them, product K).  Checks:
    (1) firefly-robust RMSE at equal spp (K*per) within 1.15x the reference-vs-reference noise floor --
    radiance is clamped at the 99.5th percentile of the lit reference pixels and medians over the four
    reference renders are compared, because a handful of firefly pixels carry most of the squared
    error and the plain RMSE of two reference renders varies 2x from pairing to pairing;
    (2) per 16x16 tile a Welch statistic on the batch means: |m_new - m_ref| <= 4.5 sqrt(se_new^2 +
    se_ref^2) for >= 99.5% of the tiles; (3) image means within `mean_tol` (or 4.5 standard errors).
    The reference arm is the reference's own kernel where oracle/_ref is built.  Elsewhere it is the PRODUCT's
    reference-twin mode (tests/_gpu_common.py::TwinRef: XORWOW, global majorant, megakernel), which
    tests/test_gpu_reference_golden.py holds to the reference's stored outputs and the twin tests here hold to the CPU
    oracle path for path; the CPU oracle itself is too slow for the thousands of frames these comparisons take."""
    ref = reference(renderer, cfg, env=env)
    rb, ref_all = _reference_batches(ref, 4 * K, per, depth)
    del ref
    halves = [rb[i * K:(i + 1) * K].mean(axis=0) for i in range(4)]
    cap = float(np.percentile(ref_all[ref_all > 0], 99.5))
    crmse = lambda a, b: rmse(np.minimum(a, cap), np.minimum(b, cap))
    floor = float(np.median([crmse(halves[i], halves[j]) for i in range(4) for j in range(i + 1, 4)]))

    configure()
    mb = _product_batches(renderer, K, per, depth)
    mine = mb.mean(axis=0)
    assert np.isfinite(mine).all()
    err = float(np.median([crmse(mine, h) for h in halves]))
    assert err <= rmse_tol * floor, (err, floor)

    tm = np.stack([_tile_means(b) for b in mb])           # (K, th, tw, 3)
    tr = np.stack([_tile_means(b) for b in rb])           # (4K, th, tw, 3)
    se_m = tm.std(axis=0, ddof=1) / np.sqrt(tm.shape[0])
    se_r = tr.std(axis=0, ddof=1) / np.sqrt(tr.shape[0])
    den = np.sqrt(se_m ** 2 + se_r ** 2)
    num = np.abs(tm.mean(axis=0) - tr.mean(axis=0))
    z = np.where(den > 0, num / np.maximum(den, 1e-30), np.where(num > 0, np.inf, 0.0))
    # Tiles that see only a smooth sky have almost no variance, and there the statistic resolves differences
    # of a few 1e-6 relative: the reference's XORWOW streams are seeded with consecutive integers
    # (curand_init(hash + pixel, 0, 0), pathtracer.cu:205-206) and its pixel jitter is measurably not uniform
    # (tools/gpu_env_debug.py: reference-vs-reference and product-vs-product agree, the two differ by 4e-6).
    # Differences below the 1e-4 relative bound used for deterministic outputs are not failures.
    ok = (z < 4.5) | (num <= 1e-4 * np.abs(tr.mean(axis=0)))
    assert ok.mean() >= 0.995, float(ok.mean())
    # image means: within `mean_tol`, or -- for scenes whose mean is carried by rare events -- within 4.5
    # standard errors of the difference as estimated from the batch-to-batch scatter
    bm, br = mb.mean(axis=(1, 2, 3)), rb.mean(axis=(1, 2, 3))
    se = np.sqrt(bm.var(ddof=1) / bm.size + br.var(ddof=1) / br.size)
    assert abs(mine.mean() - ref_all.mean()) < max(mean_tol * ref_all.mean(), 4.5 * se), (mine.mean(), ref_all.mean(), se)
    return mine, ref_all


@pytest.mark.parametrize("mode,estimator,shape", [(2, 0, 4), (2, 1, 4), (2, 0, 2), (2, 1, 2), (1, 0, 2), (1, 0, 1), (2, 0, 1), (2, 1, 1), (2, 0, 0), (1, 1, 0), (2, 0, 3), (2, 1, 3)])
def test_product_modes_are_statistically_the_reference(renderer, mode, estimator, shape):
    """Philox / local-majorant / ratio-tracking modes and all kernel shapes draw different random
    numbers from the same estimator as the reference's kernel_pathtracer."""
    depth = 4
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=depth)
    setup(renderer, cfg)

    def configure():
        renderer.set_option(L.OPT_PT_MODE, mode)
        renderer.set_option(L.OPT_SHADOW_ESTIMATOR, estimator)
        renderer.set_option(L.OPT_PT_KERNEL, shape)
        renderer.set_option(L.OPT_PT_PROFILE, 1 if shape == 4 else 0)

    _statistical_parity(renderer, cfg, depth, 8, 64, configure)


def test_acceleration_toggles_are_bit_exact(renderer):
    """Leaping, the camera-ray entry cache, the macrocell walk's kernel shape: none consumes a random
    number or changes a collision, so the images are identical bit for bit."""
    cfg = small_config(n=96, w=160, h=112, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=3)
    setup(renderer, cfg)
    imgs = []
    for shape, leap, cache in ((1, 0, 0), (1, 1, 0), (1, 1, 1), (0, 1, 1), (0, 0, 0)):
        renderer.set_option(L.OPT_PT_KERNEL, shape)
        renderer.set_option(L.OPT_LEAP, leap)
        renderer.set_option(L.OPT_PT_ENTRY_CACHE, cache)
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(8, 3)
        torch.cuda.synchronize()
        imgs.append(renderer.hdr_image().clone())
    assert float(imgs[0].max()) > 0
    for im in imgs[1:]:
        assert torch.equal(im, imgs[0])


def test_sample_parallel_shape_equals_megakernel_up_to_summation_order(renderer):
    """Kernel shape 2 hands the samples of a pixel to the lanes of a warp: every sample is the same
    pure function of (seed, pixel, sample), only the order of the float additions differs."""
    cfg = small_config(n=96, w=150, h=101, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=3)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_PT_PROFILE, 0)  # shape 2 proper: shape 4 makes other random walks (tested below)
    for mode, spp in ((2, 64), (2, 40), (0, 33), (1, 7)):
        renderer.set_option(L.OPT_PT_MODE, mode)
        renderer.set_option(L.OPT_PT_WARP_MIN_SPP, 1)
        imgs = {}
        for shape, wp, blk, cache in ((1, 4, 128, 1), (2, 4, 128, 1), (2, 1, 64, 0), (2, 7, 64, 1)):
            renderer.set_option(L.OPT_PT_KERNEL, shape)
            renderer.set_option(L.OPT_PT_WARP_PIXELS, wp)
            renderer.set_option(L.OPT_PT_BLOCK, blk)
            renderer.set_option(L.OPT_PT_ENTRY_CACHE, cache)
            renderer.frame_no = 0
            renderer.render_pathtracer_spp(spp, 3)
            torch.cuda.synchronize()
            imgs[(shape, wp, blk, cache)] = renderer.hdr_image().clone()
        base = imgs[(1, 4, 128, 1)]
        assert float(base.max()) > 0
        assert torch.allclose(imgs[(2, 4, 128, 1)], base, rtol=2e-5, atol=1e-6)
        # launch geometry and the entry cache do not enter the result at all
        assert torch.equal(imgs[(2, 1, 64, 0)], imgs[(2, 4, 128, 1)])
        assert torch.equal(imgs[(2, 7, 64, 1)], imgs[(2, 4, 128, 1)])
    renderer.set_option(L.OPT_PT_BLOCK, 128)


@pytest.mark.parametrize("gen,fmt,tf,depth,estimator", [(L.GEN_CT, L.VOXEL_U16, "default", 1, 0), (L.GEN_CT, L.VOXEL_U16, "default", 6, 1),
                                                     (L.GEN_CLOUD, L.VOXEL_F16, "cloud", 32, 0), (L.GEN_SPHERE, L.VOXEL_U8, "thin", 8, 0)])
def test_scatter_queue_shape_equals_sample_parallel_up_to_summation_order(renderer, gen, fmt, tf, depth, estimator):
    """Kernel shape 3 (camera rounds + a per-warp queue of scatter events in shared memory) serves every sample with
    the same random stream and the same sequence of draws as shape 2: identical paths, a different order of additions."""
    cfg = small_config(n=80, w=150, h=101, gen=gen, fmt=fmt, tf=tf, depth=depth, env=True)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_SHADOW_ESTIMATOR, estimator)
    renderer.set_option(L.OPT_PT_PROFILE, 0)          # shapes 2 and 3 proper
    renderer.set_option(L.OPT_PT_QUEUE_MIN_DEPTH, 0)  # shape 2 means shape 2 here, whatever the depth
    for spp in (96, 40):
        imgs = {}
        for shape, wp, blk in ((2, 4, 128), (3, 4, 128), (3, 3, 64)):
            renderer.set_option(L.OPT_PT_KERNEL, shape)
            renderer.set_option(L.OPT_PT_WARP_PIXELS, wp)
            renderer.set_option(L.OPT_PT_BLOCK, blk)
            renderer.frame_no = 0
            renderer.render_pathtracer_spp(spp, depth)
            torch.cuda.synchronize()
            imgs[(shape, wp, blk)] = renderer.hdr_image().clone()
        base = imgs[(2, 4, 128)]
        assert float(base.max()) > 0
        assert torch.allclose(imgs[(3, 4, 128)], base, rtol=5e-5, atol=2e-6), float((imgs[(3, 4, 128)] - base).abs().max())
        assert torch.equal(imgs[(3, 3, 64)], imgs[(3, 4, 128)])  # launch geometry does not enter the result
    # counted work is the same too: the same paths
    counts = {}
    for shape in (2, 3):
        renderer.set_option(L.OPT_PT_KERNEL, shape)
        renderer.set_option(L.OPT_COUNTERS, 1)
        renderer.reset_counters()
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(64, depth)
        torch.cuda.synchronize()
        counts[shape] = renderer.counters()
        renderer.set_option(L.OPT_COUNTERS, 0)
    # (the two kernels are compiled separately: a last-bit difference in a ray parameter can move a handful of
    # cell visits; collisions, scatter events and paths are the same)
    for k in counts[2]:
        if k == "cells":
            assert abs(counts[2][k] - counts[3][k]) <= 1e-4 * counts[2][k]
        else:
            assert counts[2][k] == counts[3][k], k
    assert counts[2]["scatters"] > 0
    # the default: shape 2 turns into shape 3 from traceDepth 8 on
    renderer.set_option(L.OPT_PT_KERNEL, 2)
    renderer.set_option(L.OPT_PT_BLOCK, 128)
    renderer.set_option(L.OPT_PT_WARP_PIXELS, 4)
    renderer.set_option(L.OPT_PT_QUEUE_MIN_DEPTH, 8)
    renderer.frame_no = 0
    renderer.render_pathtracer_spp(40, depth)
    torch.cuda.synchronize()
    auto = renderer.hdr_image().clone()
    assert torch.equal(auto, imgs[(3, 4, 128)] if depth >= 8 else imgs[(2, 4, 128)])


def test_deterministic_and_seeded(renderer):
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8, depth=2)
    setup(renderer, cfg)

    def render():
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(4, 2)
        torch.cuda.synchronize()
        return renderer.hdr_image().clone()

    a, b = render(), render()
    assert torch.equal(a, b)
    renderer.set_option(L.OPT_SEED, 1234)
    c = render()
    assert not torch.equal(a, c)
    # launch shape does not enter the random streams
    renderer.set_option(L.OPT_SEED, 0x5EED)
    renderer.set_option(L.OPT_PT_BLOCK, 64)
    assert torch.equal(render(), a)
    renderer.set_option(L.OPT_PT_BLOCK, 128)


def test_sample_split_and_resolve_equal_single_render(renderer):
    """The multi-GPU building blocks (SURVEY.md section 8e): partial sums over disjoint sample ranges add
    up to the image of the whole range, up to float summation order."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    setup(renderer, cfg)
    W, H = cfg.width, cfg.height
    renderer.frame_no = 0
    renderer.render_pathtracer_spp(12, 2)
    torch.cuda.synchronize()
    whole = renderer.hdr_image().clone()
    whole_ldr = renderer.ldr_image().clone()
    total = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    for first, count in S.split_samples(12, 3):
        part = torch.zeros_like(total)
        renderer.accumulate(part, 2, first, count, clear=True)
        total += part
    renderer.resolve(total)
    torch.cuda.synchronize()
    assert torch.allclose(renderer.hdr_image(), whole, rtol=1e-5, atol=1e-6)
    assert (renderer.ldr_image().int() - whole_ldr.int()).abs().max() <= 1
    assert float(total.view(H, W, 4)[..., 3].min()) == 12.0
    # accumulate without clear adds on top
    acc = torch.zeros_like(total)
    renderer.accumulate(acc, 2, 0, 5, clear=True)
    renderer.accumulate(acc, 2, 5, 7, clear=False)
    torch.cuda.synchronize()
    assert torch.allclose(acc, total, rtol=1e-5, atol=1e-5)


def test_environment_light(renderer):
    """The call the reference left commented out (pathtracer.cu:233), enabled by option."""
    cfg = small_config(n=48, w=64, h=64, gen=L.GEN_SPHERE, fmt=L.VOXEL_U16, depth=2, env=True)
    vox = setup(renderer, cfg)
    renderer.set_area_lights([])
    renderer.set_option(L.OPT_PT_MODE, 0)
    mine = _frames(renderer, 4, 2)
    assert mine[0, 0, 0] == pytest.approx(0.5)  # a corner ray misses the box and sees the constant sky
    oracle = cpu_oracle(renderer, cfg, vox, env_enabled=True)
    oracle.scene.numLights = 0
    hdr, _ = oracle.pathtrace(2, 0, 4)
    assert (np.abs(mine - hdr).max(axis=2) < 1e-3).mean() > 0.95
    # with the option off and no lights the image is black, as the reference ships
    renderer.set_option(L.OPT_ENV_ENABLED, 0)
    assert _frames(renderer, 1, 2).max() == 0.0


def test_no_lights_no_env_is_black_and_depth_zero_is_black(renderer):
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8)
    setup(renderer, cfg)
    renderer.set_area_lights([])
    for mode in (0, 1, 2):
        renderer.set_option(L.OPT_PT_MODE, mode)
        assert _frames(renderer, 1, 3).max() == 0.0
    renderer.set_area_lights([S.default_area_light(cfg.extent)])
    renderer.set_option(L.OPT_PT_MODE, 2)
    assert _frames(renderer, 1, 0).max() == 0.0  # traceDepth 0: the bounce loop never runs


def test_eight_lights_and_clamp(renderer):
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8, depth=2)
    setup(renderer, cfg)
    lights = []
    for i in range(9):  # one more than MAX_LIGHT_SOURCES: clamped to 8 (common.h:11)
        l = S.default_area_light(cfg.extent)
        ang = 2 * np.pi * i / 9
        l.disk.center = L.Vec3(80 * np.cos(ang), 90.0, 80 * np.sin(ang))
        lights.append(l)
    renderer.set_area_lights(lights)
    renderer.set_option(L.OPT_PT_MODE, 0)
    mine = _frames(renderer, 2, 2)
    ref = oracle_reference(renderer, cfg, lights=lights[:8])  # the reference itself would overrun its array with 9
    ref.render_pathtracer(2, 2)
    theirs = ref.hdr_image().cpu().numpy()
    # a last-bit difference can flip one accept/reject and send that pixel down another path
    check_paths(mine, theirs, ref, frac=0.999, mean_rel=2e-3)


def test_tone_map_matches_oracle(renderer, oracle_cpu):
    cfg = small_config(gen=L.GEN_SPHERE, fmt=L.VOXEL_U8, depth=2)
    vox = setup(renderer, cfg)
    renderer.frame_no = 0
    renderer.render_pathtracer_spp(8, 2)
    torch.cuda.synchronize()
    hdr = renderer.hdr_image().cpu().numpy()
    expect = cpu_oracle(renderer, cfg, vox).tonemap(hdr)
    got = renderer.ldr_image().cpu().numpy()
    assert np.abs(got.astype(int) - expect.astype(int)).max() <= 1
    assert (got[..., 3] == 255).all()


def test_majorants_are_conservative(renderer):
    """Every fetch the trackers can make inside a cell has opacity <= the cell's majorant; cells
    marked empty really are; leap distances never reach a non-empty cell."""
    import ctypes as C

    cfg = small_config(n=64, gen=L.GEN_CT, fmt=L.VOXEL_U16, tf="default")
    setup(renderer, cfg)
    renderer.set_volume_params(density_scale=0.8)
    renderer.frame_no = 0
    renderer.render_pathtracer_spp(1, 1)  # builds the grid
    dims = (C.c_int32 * 3)()
    cell = C.c_int32()
    L.check(renderer.lib.svr_grid_info(dims, C.byref(cell)))
    gx, gy, gz = dims
    maj = np.zeros((gz, gy, gx), np.float32)
    L.check(renderer.lib.svr_grid_copy(C.c_void_p(maj.ctypes.data), None))
    rng = np.random.default_rng(7)
    m = 400000
    uvw = rng.uniform(0, 1, (m, 3)).astype(np.float32)
    d_uvw = torch.from_numpy(uvw).cuda()
    d_i = torch.zeros(m, dtype=torch.float32, device="cuda")
    L.check(renderer.lib.svr_debug_sample_volume(C.byref(renderer.volume), C.c_void_p(d_uvw.data_ptr()), m, C.c_void_p(d_i.data_ptr())))
    d_x = (d_i * renderer.volume.densityScale).contiguous()
    d_tf = torch.zeros(m * 4, dtype=torch.float32, device="cuda")
    L.check(renderer.lib.svr_debug_sample_tf(C.byref(renderer.tf), C.c_void_p(d_x.data_ptr()), m, C.c_void_p(d_tf.data_ptr())))
    sigma = d_tf.view(m, 4)[:, 3].cpu().numpy()
    c = np.minimum((uvw * np.array([cfg.n / cell.value] * 3, np.float32)).astype(int), [gx - 1, gy - 1, gz - 1])
    mj = maj[c[:, 2], c[:, 1], c[:, 0]]
    assert (sigma <= np.maximum(mj, 0) + 1e-7).all()
    assert (sigma[mj <= 0] == 0).all()
    assert (mj > 0).any() and (mj < 0).any()
    # leap distance d: every cell within Chebyshev distance d-1 is empty
    occ = maj > 0
    zs, ys, xs = np.nonzero(maj < -1)
    for z, y, x in list(zip(zs, ys, xs))[:: max(1, len(zs) // 500)]:
        rad = int(-maj[z, y, x]) - 1
        sub = occ[max(z - rad, 0): z + rad + 1, max(y - rad, 0): y + rad + 1, max(x - rad, 0): x + rad + 1]
        assert not sub.any()


def test_config_c3_full_size_properties(renderer):
    """At BASELINE.json's full size (512^3 u16, 1920x1080): size-independent properties -- the
    acceleration structures change nothing, and the image agrees with the reference's own kernels
    within the calibrated noise floor at equal spp (the product's twin mode where oracle/_ref is not built, as in
    _statistical_parity)."""
    cfg = S.CONFIGS["C3"]
    setup(renderer, cfg)
    renderer.set_option(L.OPT_ENV_ENABLED, 0)  # the reference cannot add the sky (pathtracer.cu:233)
    spp = 8
    ref = reference(renderer, cfg)
    ref.render_pathtracer(2 * spp, 1)
    ref_ab = ref.hdr_image().cpu().numpy().copy()
    ref1 = reference(renderer, cfg)
    ref1.render_pathtracer(spp, 1)
    ref_a = ref1.hdr_image().cpu().numpy()
    ref_b = 2 * ref_ab - ref_a
    floor = rmse(ref_a, ref_b)
    imgs = []
    for leap, cache in ((1, 1), (0, 0)):
        renderer.set_option(L.OPT_LEAP, leap)
        renderer.set_option(L.OPT_PT_ENTRY_CACHE, cache)
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(spp, 1)
        torch.cuda.synchronize()
        imgs.append(renderer.hdr_image().clone())
    assert torch.equal(imgs[0], imgs[1])
    mine = imgs[0].cpu().numpy()
    assert rmse(mine, ref_a) <= 1.15 * floor
    assert abs(mine.mean() - ref_ab.mean()) < 0.02 * ref_ab.mean()
    # the product configuration (sample-parallel kernel, 32-spp launches) against the reference, 256 spp
    _statistical_parity(renderer, cfg, 1, 8, 32, lambda: None)


def test_config_c3_as_benched_with_environment_light_full_size(renderer):
    """C3 exactly as bench.py renders it -- area light + constant environment light -- at full size against the
    environment-light twin of the reference (its own sources with the line commented out at pathtracer.cu:233
    re-enabled, oracle/Makefile): path for path in the twin mode, statistically in the product mode."""
    cfg = S.CONFIGS["C3"]
    setup(renderer, cfg)
    assert cfg.env and renderer.get_option(L.OPT_ENV_ENABLED) == 1
    renderer.set_option(L.OPT_PT_MODE, 0)
    # where the reference's kernels are not built, the CPU oracle renders a band of 64 rows through the middle of the frame
    ref = oracle_reference(renderer, cfg, env=True, rows=(cfg.height // 2 - 32, cfg.height // 2 + 32))
    mine = _frames(renderer, 2, 1)
    ref.render_pathtracer(2, 1)
    theirs = ref.hdr_image().cpu().numpy()
    y0 = rows_of(ref).start or 0
    assert theirs.min() >= 0 and theirs[y0, 0, 0] == pytest.approx(0.5)   # the left edge sees the constant sky
    check_paths(mine, theirs, ref, frac=0.9999, mean_rel=1e-4)
    del ref
    renderer.set_option(L.OPT_PT_MODE, 2)
    _statistical_parity(renderer, cfg, 1, 8, 32, lambda: None, env=True)


def test_config_c1_path_trace_16spp_full_size(renderer):
    """C1 (BASELINE.json configs[0]): 128^3 u8 sphere, 512x512, the 16-spp path trace with one area light, at full
    size: the twin mode path for path against the reference's kernel, the product mode statistically."""
    cfg = S.CONFIGS["C1"]
    setup(renderer, cfg)
    renderer.set_option(L.OPT_PT_MODE, 0)
    # where the reference's kernels are not built, the CPU oracle renders a band of 128 rows through the middle of the sphere
    ref = oracle_reference(renderer, cfg, rows=(cfg.height // 2 - 64, cfg.height // 2 + 64))
    mine = _frames(renderer, cfg.spp, cfg.trace_depth)
    ref.render_pathtracer(cfg.spp, cfg.trace_depth)
    theirs = ref.hdr_image().cpu().numpy()
    assert theirs[rows_of(ref)].max() > 0
    check_paths(mine, theirs, ref, frac=0.9999, mean_rel=1e-4)
    check_u8(renderer.ldr_image().cpu().numpy(), ref)
    # one 16-sample batch == 16 frames (sample-parallel shape forced: 16 < the default minimum batch)
    renderer.set_option(L.OPT_PT_WARP_MIN_SPP, 1)
    renderer.frame_no = 0
    renderer.render_pathtracer_spp(cfg.spp, cfg.trace_depth)
    torch.cuda.synchronize()
    batched = renderer.hdr_image().cpu().numpy()
    check_paths(batched, theirs, ref, frac=0.9999)
    del ref
    renderer.set_option(L.OPT_PT_MODE, 2)
    renderer.set_option(L.OPT_PT_WARP_MIN_SPP, 32)
    _statistical_parity(renderer, cfg, cfg.trace_depth, 8, 16, lambda: None)


def test_config_c4_full_size_statistics(renderer):
    """C4: 1024^3 f16 high-albedo cloud, multiple scattering (traceDepth 32), 1920x1080 -- the regime
    where paths are long, the volume (2 GiB) misses L2 and the macrocell majorants matter most."""
    cfg = S.CONFIGS["C4"]
    setup(renderer, cfg)
    _statistical_parity(renderer, cfg, cfg.trace_depth, 8, 32, lambda: None, mean_tol=0.03)


def test_config_c5_full_size_statistics(renderer):
    """C5: 2048^3 u16 (16 GiB of voxels) at 3840x2160."""
    if torch.cuda.get_device_properties(0).total_memory < 80 * 2 ** 30:
        pytest.skip("needs ~40 GiB of device memory")
    cfg = S.CONFIGS["C5"]
    setup(renderer, cfg)
    torch.cuda.empty_cache()
    renderer.set_option(L.OPT_ENV_ENABLED, 0)  # the reference cannot add the sky (pathtracer.cu:233)
    try:
        _statistical_parity(renderer, cfg, 1, 4, 32, lambda: None, mean_tol=0.02)
    finally:
        setup(renderer, small_config())   # drop the 16 GiB array
        torch.cuda.empty_cache()


SCENE_VARIANTS = {
    "clip_planes": dict(x_clip=(-0.6, 0.35), y_clip=(-1.0, 0.5), z_clip=(-0.2, 1.0)),
    "density_and_gradient": dict(density_scale=0.6, gradient_factor=1.0),
    "thin_lens": dict(apeture=1.5, focal_length=60.0),
    "camera_inside": dict(cam_pos=(3.0, -2.0, 10.0)),
    "two_lights_exposure": dict(two_lights=True, exposure=2.5),
}


def _apply_variant(renderer, cfg, v):
    if any(k in v for k in ("x_clip", "y_clip", "z_clip", "density_scale", "gradient_factor")):
        renderer.set_volume_params(**{k: v[k] for k in ("x_clip", "y_clip", "z_clip", "density_scale", "gradient_factor") if k in v})
    cam = S.default_camera(cfg.extent, cfg.width, cfg.height, exposure=v.get("exposure", 1.0), apeture=v.get("apeture", 0.0),
                           focal_length=v.get("focal_length", 1.0))
    if "cam_pos" in v:
        cam = S.look_at_camera(v["cam_pos"], (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), image_w=cfg.width, image_h=cfg.height)
    renderer.set_camera(cam)
    if v.get("two_lights"):
        l2 = S.default_area_light(cfg.extent)
        l2.disk.center = L.Vec3(70.0, 20.0, 40.0)
        n = -np.array([70.0, 20.0, 40.0]) / np.linalg.norm([70.0, 20.0, 40.0])
        l2.disk.normal = L.Vec3(*[float(x) for x in n])
        l2.color = L.Vec3(0.4, 0.7, 1.0)
        renderer.set_area_lights([S.default_area_light(cfg.extent), l2])


@pytest.mark.parametrize("variant", sorted(SCENE_VARIANTS))
def test_scene_parameters_reach_the_path_tracer(renderer, variant):
    """Everything Canvas can change between frames -- clip planes, density scale, gradient factor, lens,
    camera pose, lights, exposure (gui/canvas.h:49-175) -- against the reference's kernel: path for path in
    the twin mode, statistically in the product mode."""
    depth = 3
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=depth)
    setup(renderer, cfg)
    _apply_variant(renderer, cfg, SCENE_VARIANTS[variant])
    renderer.set_option(L.OPT_PT_MODE, 0)
    ref = oracle_reference(renderer, cfg)
    mine = _frames(renderer, 3, depth)
    ref.render_pathtracer(3, depth)
    theirs = ref.hdr_image().cpu().numpy()
    assert theirs.max() > 0
    check_paths(mine, theirs, ref, frac=0.998, mean_rel=2e-3)
    if isinstance(ref, OracleRef):
        check_u8(renderer.ldr_image().cpu().numpy(), ref)
    else:
        assert (np.abs(renderer.ldr_image().cpu().numpy().astype(int) - ref.ldr_image().cpu().numpy().astype(int)).max(axis=2) <= 1).mean() >= 0.998
    del ref
    _statistical_parity(renderer, cfg, depth, 8, 32, lambda: renderer.set_option(L.OPT_PT_MODE, 2), mean_tol=0.02)


def test_row_bands_assemble_to_the_single_launch_frame(renderer):
    """The image split of the multi-GPU path tracer (svr_pathtracer_accumulate_bands): bands rendered by separate launches
    into one buffer are the full-frame launch bit for bit, for every kernel shape; pixels outside a launch's bands are not
    touched."""
    cfg = small_config(n=64, w=150, h=101, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    setup(renderer, cfg)
    W, H = cfg.width, cfg.height
    for shape, spp, stride in ((2, 40, 3), (1, 5, 4), (3, 40, 2), (0, 3, 5)):
        renderer.set_option(L.OPT_PT_KERNEL, shape)
        renderer.set_option(L.OPT_PT_QUEUE_MIN_DEPTH, 0)
        whole = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
        renderer.accumulate(whole, 2, 7, spp, clear=True)
        parts = torch.full((H * W * 4,), -1.0, dtype=torch.float32, device="cuda")
        rows = None
        for phase in range(stride):
            rows = renderer.accumulate_bands(parts, 2, 7, spp, phase, stride, clear=True)
            if phase == 0:   # only this launch's bands have been written
                torch.cuda.synchronize()
                v = parts.view(H, W, 4)
                band = (torch.arange(H, device="cuda") // rows) % stride
                assert bool((v[band != 0] == -1.0).all()) and bool((v[band == 0][..., 3] == spp).all())
        torch.cuda.synchronize()
        assert rows in (4, 8)
        assert torch.equal(parts, whole), shape


def test_block_split_equals_one_row_per_warp_up_to_summation_order(renderer):
    """SVR_OPT_PT_BLOCK_SPLIT: the warps of a block split the samples of one row's pixels.  Every sample is the same pure
    function of (seed, pixel, sample); four partial sums per pixel are added in a fixed order instead of one butterfly."""
    cfg = small_config(n=96, w=150, h=101, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=3)
    setup(renderer, cfg)
    W, H = cfg.width, cfg.height
    for mode, spp in ((2, 256), (2, 160), (0, 128)):
        renderer.set_option(L.OPT_PT_MODE, mode)
        imgs = {}
        for split, wp, blk in ((0, 2, 128), (1, 2, 128), (1, 1, 128), (1, 5, 64)):
            renderer.set_option(L.OPT_PT_BLOCK_SPLIT, split)
            renderer.set_option(L.OPT_PT_WARP_PIXELS, wp)
            renderer.set_option(L.OPT_PT_BLOCK, blk)
            renderer.frame_no = 0
            renderer.render_pathtracer_spp(spp, 3)
            torch.cuda.synchronize()
            imgs[(split, wp, blk)] = renderer.hdr_image().clone()
        base = imgs[(0, 2, 128)]
        assert float(base.max()) > 0
        assert torch.allclose(imgs[(1, 2, 128)], base, rtol=2e-5, atol=1e-6)
        assert torch.equal(imgs[(1, 1, 128)], imgs[(1, 2, 128)])      # the run length does not enter the result
        assert torch.allclose(imgs[(1, 5, 64)], base, rtol=2e-5, atol=1e-6)   # two warps per block: another fixed order
    # row bands (one row per band when the block is split) assemble to the single-launch frame, bit for bit
    renderer.set_option(L.OPT_PT_MODE, 2)
    renderer.set_option(L.OPT_PT_BLOCK_SPLIT, 1)
    renderer.set_option(L.OPT_PT_WARP_PIXELS, 2)
    renderer.set_option(L.OPT_PT_BLOCK, 128)
    whole = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    renderer.accumulate(whole, 3, 0, 128, clear=True)
    parts = torch.full((H * W * 4,), -1.0, dtype=torch.float32, device="cuda")
    for phase in range(3):
        rows = renderer.accumulate_bands(parts, 3, 0, 128, phase, 3, clear=True)
    torch.cuda.synchronize()
    assert rows == 1 and torch.equal(parts, whole)
    # a batch too small to give every warp a round falls back to one row per warp
    renderer.accumulate(whole, 3, 0, 64, clear=True)
    renderer.set_option(L.OPT_PT_BLOCK_SPLIT, 0)
    renderer.accumulate(parts, 3, 0, 64, clear=True)
    torch.cuda.synchronize()
    assert torch.equal(parts, whole)


def test_pixel_classification_cache_is_bit_exact_across_frames_and_scene_changes(renderer):
    """SVR_OPT_PT_PIXEL_CACHE: the 1-sample-per-call protocol keeps each pixel's classification (entry skip, light cull,
    all-sky flag) from the first frame after a change.  Only empty space is skipped: frame for frame the accumulator is the
    one the library computes when it classifies in every call -- through camera moves, transfer-function edits, new voxels,
    new lights, clip planes and option changes, in every estimator mode."""
    cfg = small_config(n=64, w=150, h=101, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    vox = setup(renderer, cfg)
    r = renderer

    def script(cache):
        r.set_option(L.OPT_PT_PIXEL_CACHE, cache)
        out = []

        def frames(n):
            for _ in range(n):
                r.render_pathtracer(2)
            torch.cuda.synchronize()
            out.append(r.hdr_image().clone())

        setup(r, cfg)
        r.set_option(L.OPT_PT_PIXEL_CACHE, cache)
        for mode in (2, 0, 1):
            r.set_option(L.OPT_PT_MODE, mode)
            r.frame_no = 0
            frames(3)
        r.set_option(L.OPT_PT_MODE, 2)
        r.set_camera(S.look_at_camera((60.0, 40.0, 110.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), image_w=cfg.width, image_h=cfg.height))
        frames(3)
        table = S.tf_table("thin")
        r.set_transfer_function(table)                 # an edit in place: same handles, new majorants
        frames(2)
        r.upload_volume(np.ascontiguousarray(vox[::-1]))   # new voxels in the same array
        frames(2)
        l2 = S.default_area_light(cfg.extent)
        l2.disk.center = L.Vec3(10.0, 5.0, 70.0)       # a light in view of the moved camera
        l2.disk.normal = L.Vec3(0.0, 0.0, 1.0)
        r.set_area_lights([S.default_area_light(cfg.extent), l2])
        frames(2)
        r.set_volume_params(x_clip=(-0.5, 0.8), density_scale=0.7)
        frames(2)
        r.set_option(L.OPT_LEAP, 0)
        frames(2)
        r.set_option(L.OPT_LEAP, 1)
        return out

    with_cache, without = script(1), script(0)
    r.set_option(L.OPT_PT_PIXEL_CACHE, 1)
    assert len(with_cache) == len(without) == 9
    for i, (a, b) in enumerate(zip(with_cache, without)):
        assert float(a.max()) > 0, i
        assert torch.equal(a, b), i
    # and the cached frames are what the batched kernel computes for the same samples (summation order aside)
    setup(r, cfg)
    r.frame_no = 0
    for _ in range(6):
        r.render_pathtracer(2)
    torch.cuda.synchronize()
    one_by_one = r.hdr_image().clone()
    r.frame_no = 0
    r.render_pathtracer_spp(6, 2)
    torch.cuda.synchronize()
    assert torch.allclose(r.hdr_image(), one_by_one, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("depth", [1, 3])
def test_sample_lookahead_is_bit_exact_frame_for_frame(renderer, depth):
    """SVR_OPT_PT_LOOKAHEAD: from frame 16 of an undisturbed progressive render, render_pathtracer computes the next 32
    samples of every pixel in one sample-parallel launch and later calls only fold their frame's sample into the running mean.
    hdrBuffer and image after EVERY call are those of one sample per call, bit for bit -- through camera moves and edits in the
    middle of a kept batch, frame counters that jump or restart, another traceDepth, every estimator mode."""
    cfg = small_config(n=64, w=150, h=101, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=depth)
    vox = setup(renderer, cfg)
    r = renderer

    def script(ahead):
        setup(r, cfg)
        r.set_option(L.OPT_PT_LOOKAHEAD, ahead)
        out = []

        def frames(n, every=1):
            for i in range(n):
                r.render_pathtracer(depth)
                if (i + 1) % every == 0 or i + 1 == n:
                    torch.cuda.synchronize()
                    out.append((r.hdr_image().clone(), r.ldr_image().clone()))

        frames(70, every=7)                              # 16 singles, a batch of 32, 22 frames into the next one
        r.set_camera(S.look_at_camera((60.0, 40.0, 110.0), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), image_w=cfg.width, image_h=cfg.height))
        r.frame_no = 0                                   # what a host does after a camera move
        frames(21, every=5)                              # 5 frames of a kept batch are used ...
        r.set_transfer_function(S.tf_table("thin"))      # ... when the transfer function changes WITHOUT a restart of the counter
        frames(30, every=6)
        r.frame_no = 100                                 # a counter that jumps
        frames(3)
        r.upload_volume(np.ascontiguousarray(vox[::-1]))
        frames(40, every=8)                              # upload_volume restarts the counter
        for mode in (0, 1):
            r.set_option(L.OPT_PT_MODE, mode)
            r.frame_no = 0
            frames(36, every=9)
        r.set_option(L.OPT_PT_MODE, 2)
        return out

    batches0 = r.lib.svr_lookahead_batch_count()
    ahead = script(-32)   # forced: what the timing-based switch would decide is not the subject here
    batches = r.lib.svr_lookahead_batch_count() - batches0
    plain = script(0)
    assert r.lib.svr_lookahead_batch_count() - batches0 == batches   # none with the option off
    assert batches == 8
    r.set_option(L.OPT_PT_LOOKAHEAD, 32)
    assert len(ahead) == len(plain)
    for i, ((ha, la), (hb, lb)) in enumerate(zip(ahead, plain)):
        assert float(ha.max()) > 0, i
        assert torch.equal(ha, hb), i
        assert torch.equal(la, lb), i


def test_sample_lookahead_launch_pattern_and_fallbacks(renderer):
    """80 undisturbed frames = 16 single launches and two batches of 32 with 32 folds each; counters on, a traceDepth that takes
    the scatter-queue kernel, or the option at 0 leave one launch per call."""
    cfg = small_config(n=48, w=96, h=64, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    setup(renderer, cfg)
    r = renderer

    def launches(n, depth=2):
        r.frame_no = 0
        r.render_pathtracer(depth)   # the frame that refreshes the grid after a change
        torch.cuda.synchronize()
        l0, b0 = r.launch_count(), r.lib.svr_lookahead_batch_count()
        for _ in range(n - 1):
            r.render_pathtracer(depth)
        torch.cuda.synchronize()
        return r.launch_count() - l0, r.lib.svr_lookahead_batch_count() - b0

    r.set_option(L.OPT_PT_LOOKAHEAD, -32)                # forced (a positive value lets the library's timing decide)
    assert launches(80) == (15 + (1 + 32) + (1 + 32), 2)
    r.set_option(L.OPT_PT_LOOKAHEAD, -8)
    assert launches(32) == (15 + (1 + 8) + (1 + 8), 2)
    r.set_option(L.OPT_PT_LOOKAHEAD, 0)
    assert launches(40) == (39, 0)
    r.set_option(L.OPT_PT_LOOKAHEAD, -32)
    r.set_option(L.OPT_COUNTERS, 1)
    assert launches(40) == (39, 0)
    r.set_option(L.OPT_COUNTERS, 0)
    assert launches(40, depth=8) == (39, 0)              # SVR_OPT_PT_QUEUE_MIN_DEPTH: the scatter-queue kernel's territory
    assert launches(40)[1] == 1
    r.set_option(L.OPT_PT_LOOKAHEAD, 32)                 # the default: batches as long as the library's own timing says they pay
    l, b = launches(200)
    # 15 single launches, then every call is a launch (a fold or, once batching is found not to pay, a single sample) plus one per batch
    assert 1 <= b <= 6 and l == 199 + b


def test_config_c3_protocol_and_streamed_upload_full_size(renderer):
    """C3 at full size through the two paths round 2 added behind unchanged entry points: (a) 80 calls of render_pathtracer with
    sample look-ahead (16 single launches, two batches of 32) against one sample per call -- hdrBuffer and image bit-equal;
    (b) svr_volume_upload from a device buffer as one pass (array fill + macrocell ranges) against copy + range kernel -- same
    image, bit for bit, from the re-uploaded voxels."""
    cfg = S.CONFIGS["C3"]
    vox = setup(renderer, cfg)
    r = renderer
    frames = {}
    for ahead in (-32, 0):
        r.set_option(L.OPT_PT_LOOKAHEAD, ahead)
        r.frame_no = 0
        for _ in range(80):
            r.render_pathtracer(cfg.trace_depth)
        torch.cuda.synchronize()
        frames[ahead] = (r.hdr_image().clone(), r.ldr_image().clone())
    r.set_option(L.OPT_PT_LOOKAHEAD, 32)
    assert float(frames[0][0].max()) > 0
    assert torch.equal(frames[-32][0], frames[0][0]) and torch.equal(frames[-32][1], frames[0][1])
    imgs = {}
    src = torch.from_numpy(np.ascontiguousarray(vox[::-1])).cuda().view(torch.uint8)   # other voxels than the bound ones
    for fused in (1, 0):
        r.set_option(L.OPT_FUSED_UPLOAD, fused)
        f0 = r.lib.svr_fused_upload_count()
        r.upload_volume(src)
        assert r.lib.svr_fused_upload_count() - f0 == fused
        r.render_pathtracer_spp(32, cfg.trace_depth)
        torch.cuda.synchronize()
        imgs[fused] = r.hdr_image().clone()
    r.set_option(L.OPT_FUSED_UPLOAD, 1)
    assert float(imgs[1].max()) > 0 and torch.equal(imgs[1], imgs[0])
    assert not torch.equal(imgs[1], frames[0][0])
