"""Adaptive sampling (svr_pathtracer_accumulate_adaptive, Renderer.accumulate_adaptive) on the GPU.

A path is a pure function of (seed, pixel, sample) and every pixel is summed by one warp in a fixed order, so an adaptive render
is held bit for bit to the uniform svr_pathtracer_accumulate sequence (first, min) + (first + min + k batch, batch) truncated per
pixel; the odd-sample half to single-sample renders; the stopping rule to a numpy restatement of it; the image to a uniform
render at 16 x maxSamples."""
import ctypes as C

import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S
from sunvolumerender_b200.render import setup_config

from _gpu_common import setup, small_config

pytestmark = pytest.mark.gpu

ESTIMATORS = {"mode0": (0, False), "mode1": (1, False), "mode2": (2, False), "env_nee": (2, True)}


def _scene(r, w=96, h=64, est="mode2", lens=False):
    cfg = small_config(n=64, w=w, h=h, gen=L.GEN_CT, fmt=L.VOXEL_U16, env=True)
    setup(r, cfg)
    mode, nee = ESTIMATORS[est]
    r.set_option(L.OPT_PT_MODE, mode)
    r.set_option(L.OPT_ENV_NEE, 1 if nee else 0)
    if lens:
        r.set_camera(S.default_camera(cfg.extent, w, h, apeture=1.5, focal_length=60.0))
    return cfg


@pytest.fixture
def scene(renderer):
    """The renderer, with the options the rest of the suite expects restored afterwards."""
    yield renderer
    renderer.set_option(L.OPT_ENV_NEE, 0)
    renderer.set_option(L.OPT_PT_MODE, 2)
    renderer.set_option(L.OPT_COUNTERS, 0)


def _hw(r):
    return r.camera.imageH, r.camera.imageW


def _adaptive(r, depth, first, mn, mx, batch, threshold):
    H, W = _hw(r)
    s = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    h = torch.zeros_like(s)
    e = torch.zeros(H * W, dtype=torch.float32, device="cuda")
    info = r.accumulate_adaptive(s, h, depth, first, mn, mx, batch, threshold, err=e)
    torch.cuda.synchronize()
    return s.view(H, W, 4).cpu().numpy(), h.view(H, W, 4).cpu().numpy(), e.view(H, W).cpu().numpy(), info


def _uniform(r, depth, first, mn, mx, batch):
    """Snapshots of the uniform sequence after each round: accumulate(first, mn, clear), then batches."""
    H, W = _hw(r)
    buf = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    r.accumulate(buf, depth, first, mn, clear=True)
    torch.cuda.synchronize()
    snaps, w = [buf.view(H, W, 4).cpu().numpy().copy()], mn
    while w < mx:
        n = min(batch, mx - w)
        r.accumulate(buf, depth, first + w, n, clear=False)
        torch.cuda.synchronize()
        snaps.append(buf.view(H, W, 4).cpu().numpy().copy())
        w += n
    return snaps


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def _tone_map(x, exposure):
    return (1.0 - np.exp(-x * 16.0 * exposure)) ** 2.2


def _err_map(s, h, exposure):
    """The convergence pass, restated: d = max_c |tm(even mean) - tm(odd mean)| / 2, err = RMS of d over the 3 x 3 window
    (coordinates clamped to the image)."""
    we, hw = s[..., 3] - h[..., 3], h[..., 3]
    ok = (hw > 0) & (we > 0)
    with np.errstate(divide="ignore", invalid="ignore"):
        even = ((s[..., :3] - h[..., :3]) / we[..., None]).astype(np.float64)
        odd = (h[..., :3] / hw[..., None]).astype(np.float64)
        d = np.abs(_tone_map(even, exposure) - _tone_map(odd, exposure)).max(axis=-1) / 2.0
    d = np.where(ok, d, 0.0)
    H, W = d.shape
    p = np.pad(d, 1, mode="edge")
    e2 = sum(p[j:j + H, i:i + W] ** 2 for j in range(3) for i in range(3)) / 9.0
    return np.sqrt(e2)


def _pick_threshold(r, depth, first, mn):
    """A threshold that stops some pixels after mn samples and keeps others going: 0.6 x the median error at mn samples."""
    _, _, e, _ = _adaptive(r, depth, first, mn, mn, 32, 0.0)
    return float(0.6 * np.median(e[e > 0]))


# ---- 1. never converging equals the uniform sequence, bit for bit
@pytest.mark.parametrize("lens", [False, True], ids=["pinhole", "thin_lens"])
@pytest.mark.parametrize("depth", [1, 6])
@pytest.mark.parametrize("est", list(ESTIMATORS))
def test_threshold_zero_equals_the_uniform_sequence(scene, est, depth, lens):
    r = scene
    _scene(r, est=est, lens=lens)
    first, mn, mx, batch = 7, 64, 160, 32
    s, h, e, info = _adaptive(r, depth, first, mn, mx, batch, 0.0)
    ref = _uniform(r, depth, first, mn, mx, batch)[-1]
    assert (s[..., 3] == mx).all() and (h[..., 3] == mx // 2).all()
    assert np.array_equal(_bits(s), _bits(ref))
    assert info["rounds"] == 4 and info["samples"] == s.shape[0] * s.shape[1] * mx
    assert info["unconverged"] == s.shape[0] * s.shape[1]  # err >= 0 everywhere


# ---- 2 and 4: truncation and the stopping rule
@pytest.fixture
def stopped(scene):
    r = scene
    _scene(r, w=128, h=96)
    depth, first, mn, mx, batch = 1, 3, 64, 256, 64
    T = _pick_threshold(r, depth, first, mn)
    s, h, e, info = _adaptive(r, depth, first, mn, mx, batch, T)
    snaps = _uniform(r, depth, first, mn, mx, batch)
    # (sum, half) of every pixel after round k: threshold 0 with maxSamples = mn + k batch
    halves = [_adaptive(r, depth, first, mn, mn + k * batch, batch, 0.0)[:2] for k in range(len(snaps))]
    return dict(r=r, T=T, s=s, h=h, e=e, info=info, snaps=snaps, halves=halves, mn=mn, mx=mx, batch=batch)


def test_truncation_equals_the_uniform_snapshots(stopped):
    c = stopped
    s, mn, mx, batch = c["s"], c["mn"], c["mx"], c["batch"]
    w = s[..., 3]
    allowed = set(range(mn, mx + 1, batch)) | {mx}
    assert set(np.unique(w).astype(int)) <= allowed
    k = ((w - mn) // batch).astype(int)
    assert 0 < (w < mx).mean() < 1, "the threshold should stop some pixels early and not others"
    for j, snap in enumerate(c["snaps"]):
        sel = k == j
        assert np.array_equal(_bits(s[sel]), _bits(snap[sel])), j
        assert np.array_equal(_bits(c["halves"][j][0][sel]), _bits(snap[sel]))  # threshold 0 reproduces the snapshot too
        assert np.array_equal(_bits(c["h"][sel]), _bits(c["halves"][j][1][sel]))
    assert c["info"]["samples"] == int(w.sum())


def test_stopping_rule_matches_numpy(stopped):
    c = stopped
    r, T, s, h, e = c["r"], c["T"], c["s"], c["h"], c["e"]
    exposure = r.camera.exposure
    # the error map of the final pass
    mine = _err_map(s, h, exposure)
    assert np.abs(mine - e).max() <= 1e-5
    assert c["info"]["unconverged"] == int((e >= T).sum())
    clear = np.abs(mine - T) > 1e-4
    assert abs(c["info"]["unconverged"] - int((mine >= T).sum())) <= int((~clear).sum())
    # every pass, given the states the library's decisions produced: a pixel still listed after pass k took the next round
    w = s[..., 3]
    kstop = ((w - c["mn"]) // c["batch"]).astype(int)
    last = len(c["snaps"]) - 1
    for k in range(last + 1):
        idx = np.minimum(kstop, k)
        S_ = np.choose(idx[..., None], [hs[0] for hs in c["halves"]])
        H_ = np.choose(idx[..., None], [hs[1] for hs in c["halves"]])
        err = _err_map(S_, H_, exposure)
        took = kstop >= k  # took round k: judged by this pass
        keep = took & (err >= T) & (k < last)
        mine_keep = took & (kstop > k)
        sure = took & (np.abs(err - T) > 1e-4)
        assert np.array_equal(keep[sure], mine_keep[sure]), k
        # a pixel that stopped before maxSamples did so with err below the threshold
        stop = took & ~mine_keep & (k < last)
        assert (err[stop & sure] < T).all()


# ---- 3. the half buffer holds the odd samples
def test_half_holds_the_odd_samples(scene):
    r = scene
    _scene(r, w=64, h=48, est="mode1")
    H, W = _hw(r)
    first, n = 5, 32
    s, h, _, _ = _adaptive(r, 1, first, n, n, 32, 0.0)
    acc = np.zeros((H, W, 3), np.float64)
    one = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    for j in range(1, n, 2):
        r.accumulate(one, 1, first + j, 1, clear=True)
        torch.cuda.synchronize()
        acc += one.view(H, W, 4).cpu().numpy()[..., :3]
    assert (h[..., 3] == s[..., 3] / 2).all()
    assert np.allclose(h[..., :3], acc, rtol=1e-5, atol=1e-6)


# ---- 5. quality and bias against the product's uniform render at 16 x maxSamples
def _tile_stats(mean, var, tile=16):
    H, W, Cc = mean.shape
    th, tw = H // tile, W // tile
    m = mean[: th * tile, : tw * tile].reshape(th, tile, tw, tile, Cc)
    v = var[: th * tile, : tw * tile].reshape(th, tile, tw, tile, Cc)
    return m.mean(axis=(1, 3)), np.sqrt(v.sum(axis=(1, 3))) / (tile * tile)


def test_quality_and_bias(scene):
    r = scene
    _scene(r, w=128, h=128)
    H, W = _hw(r)
    depth, mn, mx, batch = 1, 64, 256, 64
    T = _pick_threshold(r, depth, 0, mn)
    s, h, _, _ = _adaptive(r, depth, 0, mn, mx, batch, T)
    w, hw = s[..., 3:4].astype(np.float64), h[..., 3:4].astype(np.float64)
    mean = s[..., :3] / w
    even, odd = (s[..., :3] - h[..., :3]) / (w - hw), h[..., :3] / hw
    var = ((even - odd) / 2.0) ** 2  # of the full mean, one degree of freedom per pixel
    # reference: 16 x maxSamples in two halves (their difference gives the reference's variance the same way)
    halves = []
    for j in range(2):
        buf = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
        for b in range(8):
            r.accumulate(buf, depth, 1_000_000 + (8 * j + b) * mx, mx, clear=b == 0)
        torch.cuda.synchronize()
        v = buf.view(H, W, 4).cpu().numpy().astype(np.float64)
        halves.append(v[..., :3] / v[..., 3:4])
    ref = (halves[0] + halves[1]) / 2.0
    ref_var = ((halves[0] - halves[1]) / 2.0) ** 2
    ma, sa = _tile_stats(mean, var)
    mr, sr = _tile_stats(ref, ref_var)
    ok = np.abs(ma - mr) <= 4.5 * np.sqrt(sa ** 2 + sr ** 2) + 1e-6 * np.abs(mr)  # (all-sky tiles: rounding only)
    assert ok.all(axis=-1).mean() >= 0.995, float(ok.all(axis=-1).mean())
    converged = s[..., 3] < mx
    assert converged.any()
    disp = np.abs(_tone_map(mean, r.camera.exposure) - _tone_map(ref, r.camera.exposure)).max(axis=-1)
    assert np.sqrt((disp[converged] ** 2).mean()) <= 1.5 * T, (float(np.sqrt((disp[converged] ** 2).mean())), T)


# ---- 6. edges
def test_sky_and_depth_zero_stop_after_min(scene):
    r = scene
    _scene(r, w=64, h=48)
    mn, mx = 64, 256
    # depth 0: every sample is black, d = 0
    s, h, e, info = _adaptive(r, 0, 0, mn, mx, 64, 1e-6)
    assert (s[..., 3] == mn).all() and (s[..., :3] == 0).all() and (e == 0).all()
    assert info["rounds"] == 1 and info["unconverged"] == 0
    # a camera that looks away from the volume: every pixel is the constant sky
    c = r.camera
    r.set_area_lights([])
    r.set_camera(S.make_camera((c.pos.x, c.pos.y, c.pos.z), (-1, 0, 0), (0, 1, 0), (0, 0, -1), 45.0, 0.0, 1.0, 1.0, 64, 48))
    s, h, e, info = _adaptive(r, 1, 0, mn, mx, 64, 1e-6)
    assert (s[..., 3] == mn).all() and (e == 0).all() and (s[..., :3] > 0).all()
    assert np.array_equal(_bits(h[..., :3] * 2), _bits(s[..., :3]))
    assert info["rounds"] == 1 and info["samples"] == 64 * 48 * mn


def test_odd_canvas(scene):
    r = scene
    _scene(r, w=131, h=77, est="mode2")
    s, h, e, info = _adaptive(r, 2, 11, 32, 96, 32, 0.0)
    ref = _uniform(r, 2, 11, 32, 96, 32)[-1]
    assert np.array_equal(_bits(s), _bits(ref))
    assert np.abs(_err_map(s, h, r.camera.exposure) - e).max() <= 1e-5


@pytest.mark.parametrize("bad", [
    dict(sum=None), dict(half=None), dict(mn=0), dict(mn=48), dict(mx=100), dict(batch=0), dict(batch=16),
    dict(mn=128, mx=64), dict(T=-1.0), dict(T=float("nan")), dict(counters=1),
])
def test_rejected_arguments(scene, bad):
    r = scene
    _scene(r, w=32, h=32)
    H, W = _hw(r)
    s = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    h = torch.zeros_like(s)
    a = dict(sum=C.c_void_p(s.data_ptr()), half=C.c_void_p(h.data_ptr()), mn=64, mx=128, batch=32, T=0.01, counters=0)
    a.update(bad)
    r.set_option(L.OPT_COUNTERS, a["counters"])
    torch.cuda.synchronize()
    before = r.launch_count()
    rc = r.lib.svr_pathtracer_accumulate_adaptive(a["sum"], a["half"], None, 1, 0, a["mn"], a["mx"], a["batch"], a["T"], None, None, None)
    assert rc != 0
    assert r.lib.svr_last_error()
    assert r.launch_count() == before
    r.set_option(L.OPT_COUNTERS, 0)


# ---- 7. full size
def test_full_size_c3(scene):
    r = scene
    cfg = S.CONFIGS["C3"]
    setup(r, small_config(n=64, w=64, h=64))  # the suite's options
    setup_config(r, cfg)
    H, W = _hw(r)
    mn, mx, batch, T = 64, 1024, 64, 1.0 / 255.0
    s, h, e, info = _adaptive(r, cfg.trace_depth, 0, mn, mx, batch, T)
    w = s[..., 3]
    assert info["samples"] == int(w.astype(np.int64).sum()) < H * W * mx
    assert set(np.unique(w).astype(int)) <= set(range(mn, mx + 1, batch))
    mine = _err_map(s, h, r.camera.exposure)
    assert np.abs(mine - e).max() <= 1e-5
    assert info["unconverged"] == int((e >= T).sum())
    # the pixels the final pass stopped (every other stop was decided on an earlier state)
    wl = int(w.max())
    assert info["rounds"] == (wl - mn) // batch + 1
    if wl < mx:
        sel = (w == wl) & (np.abs(mine - T) > 1e-4)
        assert (mine[sel] < T).all()
