"""Denoised progressive display (SVR_OPT_PT_DENOISE, svr_pathtracer_set_denoise_params, Renderer.set_denoise_params).

render_pathtracer with the option on must leave hdrBuffer bit-identical to the option-off run and write, per frame, exactly
what svr_pathtracer_denoise writes for sums and guides rebuilt outside the mode: the even and odd frames' samples from
svr_pathtracer_accumulate(., s, 1), sum = even + odd in float32, guides from svr_pathtracer_guides at the option's ray count
(16 from frame 16 on).  Calls that do not continue the followed render give the option-off image.  The canvas, which paints
through render_pathtracer, gets the same.  The option and parameter checks at the end run without a GPU."""
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
GOOD = dict(iterations=5, sigmaLuminance=4.0, sigmaNormal=128.0, sigmaDepth=1.0, sigmaCoverage=0.1)
CUSTOM = dict(iterations=3, sigma_luminance=2.0, sigma_normal=32.0, sigma_depth=2.0, sigma_coverage=0.3)


# ---------------------------------------------------------------------------------------------------------------------
# GPU helpers
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture
def pd(renderer):
    """The session's renderer; the options and parameters these tests change are restored, so later tests render as before."""
    yield renderer
    renderer.set_option(L.OPT_PT_DENOISE, 0)
    renderer.set_denoise_params(None)
    for key, value in ((L.OPT_PT_MODE, 2), (L.OPT_ENV_NEE, 0), (L.OPT_COUNTERS, 0), (L.OPT_PT_KERNEL, 2), (L.OPT_PT_WARP_MIN_SPP, 32)):
        renderer.set_option(key, value)


def _scene(r, n=64, w=96, h=64, env=True, apeture=0.0):
    from _gpu_common import setup, small_config

    cfg = small_config(n=n, w=w, h=h, gen=L.GEN_CT, fmt=L.VOXEL_U16, env=env)
    setup(r, cfg)
    if apeture:
        cam = r.camera
        r.set_camera(S.default_camera(cfg.extent, w, h, apeture=apeture, focal_length=0.8 * cam.pos.z))
    return cfg


def _sync():
    import torch

    torch.cuda.synchronize()


def _host(t):
    _sync()
    return t.cpu().numpy().copy()


def _frame(r, frame_no, depth=1, hdr=None):
    rp = L.RenderParams(depth, frame_no, (r.hdr if hdr is None else hdr).data_ptr())
    r.lib.render_pathtracer(C.c_void_p(r.img.data_ptr()), C.byref(rp))


def _params(kw):
    p = L.DenoiseParams()
    L.check(L.load().svr_denoise_defaults(C.byref(p)), "svr_denoise_defaults")
    names = {"iterations": "iterations", "sigma_luminance": "sigmaLuminance", "sigma_normal": "sigmaNormal", "sigma_depth": "sigmaDepth",
             "sigma_coverage": "sigmaCoverage"}
    for k, v in (kw or {}).items():
        setattr(p, names[k], v)
    return p


class Expected:
    """The denoised frames rebuilt outside the mode: even / odd sums from svr_pathtracer_accumulate, guides from
    svr_pathtracer_guides, the image from svr_pathtracer_denoise.  add(f) renders sample f of the bound scene into its half
    (frame 0 clears both); image(f) is the frame the mode must show after it."""

    def __init__(self, r, rays, params=None, depth=1):
        import torch

        self.r, self.rays, self.depth, self.p = r, rays, depth, _params(params)
        npix = r.camera.imageW * r.camera.imageH
        self.even, self.odd, self.ac, self.nd = (torch.zeros(npix * 4, dtype=torch.float32, device="cuda") for _ in range(4))
        self.img = torch.zeros(npix * 4, dtype=torch.uint8, device="cuda")

    def add(self, f):
        if f == 0:
            self.odd.zero_()
        self.r.accumulate(self.even if f % 2 == 0 else self.odd, self.depth, f, 1, clear=f == 0)

    def image(self, f):
        r = self.r
        s = self.even + self.odd
        L.check(r.lib.svr_pathtracer_guides(C.c_void_p(self.ac.data_ptr()), C.c_void_p(self.nd.data_ptr()), 16 if f >= 16 else self.rays),
                "svr_pathtracer_guides")
        L.check(r.lib.svr_pathtracer_denoise(C.c_void_p(self.img.data_ptr()), None, C.c_void_p(s.data_ptr()), C.c_void_p(self.odd.data_ptr()),
                                             C.c_void_p(self.ac.data_ptr()), C.c_void_p(self.nd.data_ptr()), C.byref(self.p)), "svr_pathtracer_denoise")
        return _host(self.img)


def _run(r, frames, value, depth=1):
    """hdr and img after each of `frames` render_pathtracer calls from frameNo 0, with SVR_OPT_PT_DENOISE = value."""
    r.set_option(L.OPT_PT_DENOISE, value)
    hdrs, imgs = [], []
    for f in range(frames):
        _frame(r, f, depth)
        hdrs.append(_host(r.hdr))
        imgs.append(_host(r.img))
    return hdrs, imgs


# ---- 1. hdrBuffer is the option-off running mean, bit for bit
HDR_CASES = {
    "mode0": ({L.OPT_PT_MODE: 0}, 1, 0.0),
    "mode1": ({L.OPT_PT_MODE: 1}, 1, 0.0),
    "mode2": ({}, 1, 0.0),
    "env_nee": ({L.OPT_ENV_NEE: 1}, 1, 0.0),
    "depth8": ({}, 8, 0.0),
    "depth8_warp": ({L.OPT_PT_WARP_MIN_SPP: 1}, 8, 0.0),
    "thin_lens": ({}, 1, 0.4),
    "kernel0": ({L.OPT_PT_KERNEL: 0}, 1, 0.0),
    "kernel1": ({L.OPT_PT_KERNEL: 1}, 1, 0.0),
    "kernel2_warp": ({L.OPT_PT_KERNEL: 2, L.OPT_PT_WARP_MIN_SPP: 1}, 1, 0.0),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(HDR_CASES))
def test_hdr_is_bit_identical(pd, case):
    """40 frames (across frame 16, where look-ahead starts batching and the guides go to 16 rays) with the option off and on."""
    r = pd
    opts, depth, apeture = HDR_CASES[case]
    _scene(r, apeture=apeture)
    for k, v in opts.items():
        r.set_option(k, v)
    off, off_img = _run(r, 40, 0, depth)
    on, on_img = _run(r, 40, 4, depth)
    for f in range(40):
        assert np.array_equal(off[f], on[f]), f
    assert off[-1].max() > 0
    # the display is the denoised one (the first frames of a 1-spp render differ everywhere the volume is)
    assert not np.array_equal(off_img[1], on_img[1])


# ---- 2. every denoised frame is svr_pathtracer_denoise of the sums and guides rebuilt outside the mode
@pytest.mark.gpu
@pytest.mark.parametrize("case", ["defaults_4", "custom_1", "mode0_16", "thin_lens_4", "iterations0_4"])
def test_frames_match_denoise(pd, case):
    r = pd
    rays = int(case.rsplit("_", 1)[1])
    params = {"custom_1": CUSTOM, "iterations0_4": dict(iterations=0)}.get(case)
    _scene(r, apeture=0.4 if case.startswith("thin_lens") else 0.0)
    if case.startswith("mode0"):
        r.set_option(L.OPT_PT_MODE, 0)
    r.set_denoise_params(params)
    _, imgs = _run(r, 40, rays)
    exp = Expected(r, rays, params)
    for f in range(40):
        exp.add(f)
        assert np.array_equal(imgs[f], exp.image(f)), f
    if case == "iterations0_4":  # the filter's identity: the running mean's tone map up to the float division
        _, off_imgs = _run(r, 4, 0)
        assert np.abs(imgs[3].astype(int) - off_imgs[3].astype(int)).max() <= 1


# ---- 3. the calls that are not denoised frames
def _sequence(r, steps, value, start=None):
    """Runs `steps` ((kind, args) tuples) with the option at `value` (`start` before the first step, if given); returns
    (hdr, img) after every frame step."""
    import torch

    other = torch.zeros_like(r.hdr)
    r.set_option(L.OPT_PT_DENOISE, value if start is None else start)
    out = []
    for kind, *args in steps:
        if kind == "frame":
            f, depth, which = args
            _frame(r, f, depth, other if which else None)
            out.append((_host(other if which else r.hdr), _host(r.img)))
        elif kind == "option":
            r.set_option(*args)
        elif kind == "spp":
            rp = L.RenderParams(1, args[0], r.hdr.data_ptr())
            L.check(r.lib.svr_render_pathtracer_spp(C.c_void_p(r.img.data_ptr()), C.byref(rp), args[1]), "svr_render_pathtracer_spp")
    return out


def _frames(fs, depth=1, which=0):
    return [("frame", f, depth, which) for f in fs]


TRACKING = {
    # name: (steps, frame-step indices shown as with the option off, option value before the first step)
    "skipped_frame": (_frames(range(6)) + _frames([7, 8, 9]) + _frames([0, 1]), range(6, 9), None),
    "other_hdr": (_frames(range(6)) + _frames([6, 7], which=1) + _frames([8, 0, 1]), range(6, 9), None),
    "trace_depth": (_frames(range(6)) + _frames([6, 7], depth=2) + _frames([8]) + _frames([0, 1]), range(6, 9), None),
    "counters": (_frames(range(6)) + [("option", L.OPT_COUNTERS, 1)] + _frames([6]) + [("option", L.OPT_COUNTERS, 0)] + _frames([7, 8, 0, 1]),
                 range(6, 9), None),
    "turned_on_mid_render": (_frames(range(6)) + [("option", L.OPT_PT_DENOISE, 4)] + _frames([6, 7, 8, 0, 1]), range(0, 9), 0),
    "interleaved_spp": (_frames(range(6)) + [("spp", 6, 2)] + _frames([8, 9, 10]) + _frames([0, 1]), range(6, 9), None),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(TRACKING))
def test_tracking_rules(pd, case):
    """After the break, every frame until the next frameNo = 0 is the option-off image; hdr is the option-off one throughout;
    frames 0 and 1 after the restart are denoised again."""
    r = pd
    _scene(r)
    steps, plain, start = TRACKING[case]
    off = _sequence(r, [s for s in steps if s[:2] != ("option", L.OPT_PT_DENOISE)], 0)
    on = _sequence(r, steps, 4, start)
    assert len(off) == len(on) == 11
    for i, ((h0, i0), (h1, i1)) in enumerate(zip(off, on)):
        assert np.array_equal(h0, h1), i
        if i in plain:
            assert np.array_equal(i0, i1), i
    for i in [i for i in range(len(on)) if i not in plain]:
        assert not np.array_equal(off[i][1], on[i][1]), i  # denoised


@pytest.mark.gpu
def test_camera_change_without_restart_remakes_the_guides(pd):
    """The canvas's quirk: a repaint with a new camera before frameNo is reset continues the sums under the new camera, with
    guides of the new one."""
    r = pd
    cfg = _scene(r)
    r.set_option(L.OPT_PT_DENOISE, 4)
    cam0 = r.camera
    cam1 = S.make_camera((4.0, -3.0, cam0.pos.z * 0.9), (1, 0, 0), (0, 1, 0), (0, 0, 1), 45.0, 0.0, 1.0, 1.0, cfg.width, cfg.height)
    shown = []
    for f in range(8):
        if f == 5:
            r.lib.setup_camera(C.byref(cam1))
        _frame(r, f)
        shown.append(_host(r.img))
    r.lib.setup_camera(C.byref(cam0))
    exp = Expected(r, 4)
    for f in range(8):
        if f == 5:
            r.lib.setup_camera(C.byref(cam1))
        exp.add(f)
        assert np.array_equal(shown[f], exp.image(f)), f
    r.lib.setup_camera(C.byref(cam0))


@pytest.mark.gpu
def test_restart_clears_both_sums(pd):
    """frameNo = 0 after 20 frames (guides at 16 rays by then) starts over: the same images as the first frames of a render,
    4-ray guides again."""
    r = pd
    _scene(r)
    r.set_option(L.OPT_PT_DENOISE, 4)
    shown = []
    for f in list(range(20)) + [0, 1, 2]:
        _frame(r, f)
        shown.append(_host(r.img))
    for f in range(3):
        assert np.array_equal(shown[f], shown[20 + f]), f


# ---- 4. the canvas
@pytest.mark.gpu
def test_canvas_interaction(pd):
    """A scripted path-traced interaction with immediate repaints (press, left and middle drags, wheel, key, setters, plain
    paints), once with the option off and once on.  After every action the canvas shows its last paint; with the option on
    that is the denoised frame rebuilt from the samples of the paints since the last restart (each action's paints share
    one scene and have consecutive frame numbers, so they are re-rendered right after it with svr_pathtracer_accumulate), or
    the option-off image where the paint did not continue the followed render.  svr_canvas_hdr is the option-off buffer,
    bit for bit, after every action."""
    from sunvolumerender_b200.canvas import Canvas

    r = pd
    cfg = _scene(r, w=128, h=96, env=False)
    W, H = cfg.width, cfg.height
    actions = [("set", dict(render_mode=L.RENDER_MODE_PATHTRACER)), ("paint", 3), ("press", 60, 40, L.BUTTON_LEFT),
               ("move", 70, 44, L.BUTTON_LEFT), ("paint", 2), ("move", 75, 40, L.BUTTON_LEFT | L.BUTTON_MID), ("paint", 18),
               ("wheel", -120), ("paint", 1), ("set", dict(density_scale=1.5)), ("paint", 4), ("key", L.KEY_LEFT), ("paint", 2),
               ("set", dict(exposure=1.3)), ("paint", 20), ("set", dict(fov=40.0)), ("paint", 1)]

    def replay(value, exp):
        import torch

        r.set_option(L.OPT_PT_DENOISE, value)
        canvas = Canvas(W, H)
        try:
            canvas.set_volume(r.volume, cfg.extent, S.raycast_step_size())
            canvas.set_transfer_function(r.tf)
            canvas.set_area_lights(r.lights)
            hdr = torch.zeros(H * W * 3, dtype=torch.float32, device="cuda")
            out, following, last = [], False, -1
            for kind, *args in actions:
                f0, p0 = canvas.frame_no, canvas.paint_count
                if kind == "set":
                    canvas.set(**args[0])
                elif kind == "paint":
                    canvas.paint(args[0])
                else:
                    getattr(canvas, {"press": "mouse_press", "move": "mouse_move", "wheel": "wheel", "key": "key"}[kind])(*args)
                n = canvas.paint_count - p0
                L.check(r.lib.svr_stage_copy(C.c_void_p(hdr.data_ptr()), C.c_void_p(canvas.hdr_ptr()), hdr.numel() * 4, None), "copy")
                entry = {"paints": n, "hdr": _host(hdr), "img": canvas.image().reshape(-1)}
                if exp is not None and n:
                    for f in range(f0, f0 + n):  # the paints of this action, under the scene still bound
                        following = f == 0 or (following and f == last + 1)
                        last = f
                        if following:
                            exp.add(f)
                    entry["expected"] = exp.image(f0 + n - 1) if following else None
                out.append(entry)
            return out
        finally:
            canvas.close()
            r.lib.setup_env_lights(C.byref(r.env))

    off = replay(0, None)
    on = replay(4, Expected(r, 4))
    denoised = 0
    for i, (a, b) in enumerate(zip(off, on)):
        assert a["paints"] == b["paints"], i
        assert np.array_equal(a["hdr"], b["hdr"]), i
        if b["paints"] == 0:
            continue
        if b["expected"] is None:
            assert np.array_equal(a["img"], b["img"]), i
        else:
            assert np.array_equal(b["img"], b["expected"]), i
            denoised += 1
    assert denoised >= 10


# ---- 5. quality against a high-spp render
@pytest.mark.gpu
def test_quality(pd):
    """Display RMSE of the shown u8 image (raw: the option-off image, the running mean's tone map; denoised: the mode's)
    against the u8 image of 8192 spp, on the denoise tests' 192 x 128 CT scene, 4-ray guides (16 from frame 16), default parameters.
    Expected: denoised below raw at 1, 2, 4, 8, 16 and 64 frames; within 1.1 x raw at 1024.  Measured on a B200 (1000 W), raw /
    denoised: 1 frame 0.0818 / 0.0502, 2: 0.0628 / 0.0425, 4: 0.0486 / 0.0317, 8: 0.0373 / 0.0238, 16: 0.0263 / 0.0162,
    64: 0.0132 / 0.0091, 1024: 0.00354 / 0.00353 (1.00 x)."""
    import torch

    r = pd
    from _gpu_common import setup, small_config

    cfg = small_config(n=128, w=192, h=128, gen=L.GEN_CT, fmt=L.VOXEL_U16, env=True)
    setup(r, cfg)
    H, W, ex = cfg.height, cfg.width, r.camera.exposure
    ref = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    for b in range(8):
        r.accumulate(ref, 1, (1 << 24) + b * 1024, 1024, clear=b == 0)
    v = _host(ref).reshape(H, W, 4).astype(np.float64)
    ref_disp = np.floor(((1.0 - np.exp(-(v[..., :3] / v[..., 3:4]) * 16.0 * ex)) ** 2.2) * 255.0) / 255.0  # truncated as pack_u8x4
    marks = (1, 2, 4, 8, 16, 64, 1024)
    rmse = {}
    for value in (0, 4):
        r.set_option(L.OPT_PT_DENOISE, value)
        for f in range(max(marks)):
            _frame(r, f)
            if f + 1 in marks:
                disp = _host(r.img).reshape(H, W, 4)[..., :3] / 255.0
                rmse.setdefault(f + 1, []).append(float(np.sqrt(((disp - ref_disp) ** 2).mean())))
    print("frames: (raw, denoised) display RMSE", {k: tuple(round(x, 6) for x in v) for k, v in rmse.items()})
    for n in (1, 2, 4, 8, 16, 64):
        assert rmse[n][1] < rmse[n][0], (n, rmse)
    assert rmse[1024][1] <= 1.1 * rmse[1024][0], rmse


# ---- 6. checks without a GPU
def test_option_values():
    lib = L.load()
    assert L.OPT_PT_DENOISE == 26
    before = lib.svr_get_option(L.OPT_PT_DENOISE)
    for bad in (2, 3, -1, 32):
        assert lib.svr_set_option(L.OPT_PT_DENOISE, bad) != 0
        assert b"SVR_OPT_PT_DENOISE" in lib.svr_last_error()
        assert lib.svr_get_option(L.OPT_PT_DENOISE) == before
    for good in (1, 4, 16, 0):
        assert lib.svr_set_option(L.OPT_PT_DENOISE, good) == 0
        assert lib.svr_get_option(L.OPT_PT_DENOISE) == good


def test_set_denoise_params_checks():
    """Each bad field is rejected with svr_pathtracer_denoise's message (prefixed with the entry point) before any CUDA call;
    NULL restores the defaults."""
    lib = L.load()
    bad_params = [dict(iterations=9)] + [{k: v} for k in ("sigmaLuminance", "sigmaDepth", "sigmaCoverage") for v in (0.0, -1.0, math.inf, math.nan)] + \
                 [dict(sigmaNormal=v) for v in (-1.0, math.inf, math.nan)]
    for bad in bad_params:
        p = L.DenoiseParams(**dict(GOOD, **bad))
        assert lib.svr_pathtracer_set_denoise_params(C.byref(p)) != 0, bad
        msg = lib.svr_last_error()
        assert msg.startswith(b"svr_pathtracer_set_denoise_params: "), msg
        assert (b"iterations" if "iterations" in bad else b"sigma") in msg
    assert lib.svr_pathtracer_set_denoise_params(C.byref(L.DenoiseParams(**dict(GOOD, iterations=0, sigmaNormal=0.0)))) == 0
    assert lib.svr_pathtracer_set_denoise_params(None) == 0
    # svr_pathtracer_denoise keeps its own messages (the pointers are never dereferenced: the parameters are bad)
    f = [C.c_void_p(256 * (i + 1)) for i in range(6)]
    assert lib.svr_pathtracer_denoise(*f, C.byref(L.DenoiseParams(**dict(GOOD, iterations=9)))) != 0
    assert lib.svr_last_error() == b"svr_pathtracer_denoise: iterations above 8"
    assert lib.svr_pathtracer_denoise(*f, C.byref(L.DenoiseParams(**dict(GOOD, sigmaNormal=-1.0)))) != 0
    assert lib.svr_last_error() == b"svr_pathtracer_denoise: sigmaNormal must be >= 0 and finite"


def test_renderer_binding_forwards_params():
    """Renderer.set_denoise_params maps its keyword names onto the struct and raises on a rejected value (no device: the
    checks come first)."""
    from sunvolumerender_b200.render import Renderer

    r = Renderer.__new__(Renderer)  # the binding only; no device set-up
    r.lib = L.load()
    r.set_denoise_params(dict(iterations=2, sigma_luminance=3.0))
    r.set_denoise_params(None)
    with pytest.raises(L.SvrError, match="sigmaLuminance"):
        r.set_denoise_params(dict(sigma_luminance=-1.0))
    with pytest.raises(L.SvrError, match="iterations"):
        r.set_denoise_params(dict(iterations=12))


def test_environment_switch():
    """SVR_PT_DENOISE is read once from the environment: 4 reads back as 4; 3 leaves the default 0 and warns."""
    code = "import sys; sys.path.insert(0, %r)\nfrom sunvolumerender_b200 import _lib as L\nprint(L.load().svr_get_option(L.OPT_PT_DENOISE))\n" % ROOT
    for value, expect, warns in (("4", 4, False), ("16", 16, False), ("3", 0, True), ("-1", 0, True)):
        env = dict(os.environ, SVR_PT_DENOISE=value)
        out = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, check=True)
        assert int(out.stdout.strip()) == expect, (value, out)
        assert ("ignoring SVR_PT_DENOISE=%s (out of range)" % value in out.stderr) == warns, out.stderr


def test_headless_denoise_command(tmp_path):
    """tools/svr_headless --interact parses the whole script before it touches the device: `denoise 4` is a command (the
    malformed line after it is the one reported), `denoise 3` and `denoise` are malformed."""
    exe = os.path.join(ROOT, "tools", "svr_headless")
    if not os.path.exists(exe):
        pytest.skip("tools/svr_headless not built (make tools)")
    cases = (("denoise 4\nfrobnicate 1\n", ":2: cannot parse 'frobnicate 1'"), ("denoise 3\n", ":1: cannot parse 'denoise 3'"),
             ("# comment\ndenoise\n", ":2: cannot parse 'denoise'"))
    for i, (text, err) in enumerate(cases):
        script = tmp_path / f"s{i}.txt"
        script.write_text(text)
        out = subprocess.run([exe, "--config", "C1", "--n", "32", "--w", "64", "--h", "64", "--interact", str(script)], capture_output=True, text=True,
                             timeout=300)
        assert out.returncode == 2 and err in out.stderr, (text, out.stderr)
