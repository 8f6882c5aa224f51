"""svr_set_device with every cache populated: the library drops what it holds on the device and rebuilds it.

svr_set_device(current device) in the middle of a render must leave the render's results bit for bit what they are without it:
look-ahead launches a new batch, the macrocell grid, pixel classification and environment sampler are rebuilt, and a denoised
progressive display starts again at the render's next frameNo 0 (until then render_pathtracer shows the raw image, and hdrBuffer
is unaffected throughout).  Rebinding over and over must not leak device memory."""
import torch
import pytest

from sunvolumerender_b200 import _lib as L

from _gpu_common import setup, small_config

pytestmark = pytest.mark.gpu

W, H = 96, 64


@pytest.fixture
def rr(renderer):
    """The session's renderer; the options these tests change are restored, so later tests render as before."""
    yield renderer
    for key, value in ((L.OPT_PT_LOOKAHEAD, 32), (L.OPT_PT_DENOISE, 0), (L.OPT_ENV_NEE, 0), (L.OPT_PT_MODE, 2)):
        renderer.set_option(key, value)


def _rebind(r):
    L.check(r.lib.svr_set_device(torch.cuda.current_device()), "svr_set_device")


def _snap(r, out):
    torch.cuda.synchronize()
    out.append(r.hdr.clone())
    out.append(r.img.clone())


def _lookahead(r, rebind, out):
    """A forced look-ahead render past frame 16: the rebind falls inside the first batch (frames 16 .. 47)."""
    setup(r, small_config(n=48, w=W, h=H, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2))
    r.set_option(L.OPT_PT_LOOKAHEAD, -32)
    r.frame_no = 0
    for f in range(60):
        if f == 24:
            rebind()
        r.render_pathtracer(2)
        if f in (23, 24, 30, 59):
            _snap(r, out)


def _denoised(r, rebind, out):
    """A denoised progressive render, rebound at frame 20, continued to frame 30, then restarted at frameNo 0."""
    setup(r, small_config(n=64, w=W, h=H, gen=L.GEN_CT, fmt=L.VOXEL_U16, env=True))
    r.set_option(L.OPT_PT_DENOISE, 4)
    r.frame_no = 0
    for f in range(30):
        if f == 20:
            rebind()
        r.render_pathtracer(1)
        torch.cuda.synchronize()
        out.append(r.hdr.clone())  # the display is raw between the rebind and the restart: only the running mean is compared
        if f < 20:
            out.append(r.img.clone())
    r.frame_no = 0
    for f in range(20):
        r.render_pathtracer(1)
        _snap(r, out)
    r.set_option(L.OPT_PT_DENOISE, 0)


def _adaptive(r, rebind, out):
    """Two adaptive accumulates with the rebind between them."""
    setup(r, small_config(n=64, w=W, h=H, gen=L.GEN_CT, fmt=L.VOXEL_U16, env=True))
    npix = W * H
    for first in (0, 256):
        s = torch.empty(npix * 4, dtype=torch.float32, device=r.device)
        half = torch.empty_like(s)
        err = torch.empty(npix, dtype=torch.float32, device=r.device)
        stats = r.accumulate_adaptive(s, half, 1, first, 32, 256, 32, 2.0 / 255.0, err=err)
        torch.cuda.synchronize()
        out.extend([s, half, err, torch.tensor([stats["rounds"], stats["samples"], stats["unconverged"]])])
        if first == 0:
            rebind()


def _env_nee(r, rebind, out):
    """A progressive render with environment next-event estimation, rebound at frame 10."""
    setup(r, small_config(n=64, w=W, h=H, gen=L.GEN_CT, fmt=L.VOXEL_U16, env=True))
    r.set_option(L.OPT_ENV_NEE, 1)
    r.frame_no = 0
    for f in range(20):
        if f == 10:
            rebind()
        r.render_pathtracer(1)
        if f in (9, 10, 19):
            _snap(r, out)
    r.render_pathtracer_spp(64)
    _snap(r, out)
    r.set_option(L.OPT_ENV_NEE, 0)


RENDERS = {"lookahead": _lookahead, "denoised": _denoised, "adaptive": _adaptive, "env_nee": _env_nee}


@pytest.mark.parametrize("name", list(RENDERS))
def test_set_device_mid_render_is_bit_identical(rr, name):
    plain, rebound = [], []
    RENDERS[name](rr, lambda: None, plain)
    RENDERS[name](rr, lambda: _rebind(rr), rebound)
    assert len(plain) == len(rebound) > 0
    assert float(plain[0].abs().max()) > 0
    for i, (a, b) in enumerate(zip(plain, rebound)):
        assert torch.equal(a, b), f"{name}: result {i} differs after svr_set_device"


def test_set_device_releases_every_cache(rr):
    """Five cycles of rebind + all four renders: free device memory returns to where the first cycle left it."""
    free = []
    for _ in range(5):
        _rebind(rr)
        for render in RENDERS.values():
            render(rr, lambda: None, [])
        torch.cuda.synchronize()
        free.append(torch.cuda.mem_get_info()[0])
    assert abs(free[-1] - free[0]) <= 1 << 20, [f - free[0] for f in free]
