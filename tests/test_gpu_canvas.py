"""GPU tests of the windowless Canvas (include/svr_canvas.h, SURVEY.md section 8f rank 4): the frame protocol of
gui/canvas.cpp:63-117 and gui/canvas.h:43-47 on top of the seven entry points, and a scripted interaction whose frames
are compared with the reference's own kernels (the CPU oracle where they are not built) given the camera the canvas
arrived at."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import metaimage_oracle as M
from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S
from sunvolumerender_b200.canvas import Canvas

from _gpu_common import OracleRef, check_paths, check_u8, oracle_reference, setup, small_config

pytestmark = pytest.mark.gpu
W = H = 128   # a canvas size the reference is compiled for (WIDTH / HEIGHT are compile-time there)


@pytest.fixture()
def scene(renderer):
    cfg = small_config(n=64, w=W, h=H, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    setup(renderer, cfg)
    canvas = Canvas(W, H)
    yield renderer, cfg, canvas
    canvas.close()
    renderer.lib.setup_env_lights(C.byref(renderer.env))


def _hdr(canvas):
    """The canvas's accumulation buffer (RenderParams::hdrBuffer) on the host."""
    host = np.zeros((H, W, 3), np.float32)
    rt = C.CDLL("libcudart.so.12")
    assert rt.cudaMemcpy(C.c_void_p(host.ctypes.data), C.c_void_p(canvas.hdr_ptr()), host.nbytes, 2) == 0  # device to host
    return host


def _attach(renderer, cfg, canvas):
    size = cfg.extent
    canvas.set_volume(renderer.volume, size, S.raycast_step_size())
    canvas.set_transfer_function(renderer.tf)
    canvas.set_area_lights(renderer.lights)


def test_fresh_canvas_and_raycast_frame(scene):
    renderer, cfg, canvas = scene
    canvas.paint()
    assert canvas.paint_count == 0 and canvas.frame_no == 0          # not ready: paintGL returns early (canvas.cpp:67)
    e = canvas.env_light()
    assert (e.tex, e.defaultRadiance.tuple(), e.intensity) == (0, (1.0, 1.0, 1.0), 0.5)   # canvas.cpp:11-13
    _attach(renderer, cfg, canvas)
    v = canvas.volume()
    assert v.gradientFactor == 0.5 and v.densityScale == 1.0 and v.x_clip.x == -1.0 and v.z_clip.y == 1.0
    # the camera a freshly loaded volume gets (canvas.cpp:35-38)
    cam, ref_cam = canvas.camera(), S.default_camera(cfg.extent, W, H)
    assert cam.pos.tuple() == pytest.approx(ref_cam.pos.tuple(), rel=1e-6) and cam.w.tuple() == (0.0, 0.0, 1.0)
    # default mode is ray casting (canvas.h:226); one paint = one frame
    before = canvas.paint_count
    canvas.paint()
    assert canvas.paint_count == before + 1
    img = canvas.image()
    assert img[..., 3].max() > 128
    renderer.set_camera(cam)
    renderer.render_raycasting()
    torch.cuda.synchronize()
    assert np.array_equal(img, renderer.ldr_image().cpu().numpy())
    ref = oracle_reference(renderer, cfg)
    ref.render_raycasting(S.raycast_step_size())
    check_u8(img, ref)


def test_frame_protocol_and_restart(scene):
    renderer, cfg, canvas = scene
    _attach(renderer, cfg, canvas)
    canvas.set(render_mode=L.RENDER_MODE_PATHTRACER, scatter_times=2.0)
    assert canvas.frame_no == 0
    canvas.paint(5)
    assert canvas.frame_no == 5                                       # frameNo++ per paint (canvas.cpp:116)
    # the accumulator is the running mean of frames 0..4 of the same scene rendered through the Renderer
    host = _hdr(canvas)
    renderer.set_camera(canvas.camera())
    renderer.frame_no = 0
    for _ in range(5):
        renderer.render_pathtracer(2)
    torch.cuda.synchronize()
    assert np.array_equal(host, renderer.hdr_image().cpu().numpy())
    # a setter repaints once (updateGL inside ReStartRender) and resets the counter (canvas.h:43-47)
    paints = canvas.paint_count
    canvas.set(density_scale=0.7)
    assert canvas.frame_no == 0 and canvas.paint_count == paints + 1 and canvas.volume().densityScale == np.float32(0.7)
    canvas.paint(2)
    assert canvas.frame_no == 2
    # events: wheel = UpdateCamera + ReStartRender (1 repaint); key = updateGL + ReStartRender (2); a left drag = 2 per move
    for action, repaints in ((lambda: canvas.wheel(120), 1), (lambda: canvas.key(L.KEY_LEFT), 2),
                             (lambda: (canvas.mouse_press(64, 64, L.BUTTON_LEFT), canvas.mouse_move(70, 60, L.BUTTON_LEFT)), 2)):
        canvas.paint(1)
        paints = canvas.paint_count
        action()
        assert canvas.frame_no == 0 and canvas.paint_count == paints + repaints
    # batch hosts can switch the immediate repaints off; the counter is still reset
    canvas.set_immediate_repaint(False)
    canvas.paint(3)
    paints = canvas.paint_count
    canvas.set(exposure=2.0, fov=50.0, x_clip=(-0.5, 1.0))
    assert canvas.frame_no == 0 and canvas.paint_count == paints
    cam = canvas.camera()
    assert cam.exposure == 2.0 and cam.tanFovxOverTwo == pytest.approx(np.tan(np.radians(25.0)), rel=1e-6)
    assert canvas.volume().x_clip.x == -0.5
    # cudaEnvironmentLight::Set(radiance) resets the intensity (cuda_environment_light.h:25-31)
    canvas.set(env_intensity=3.0)
    assert canvas.env_light().intensity == 3.0
    canvas.set(env_background=(0.2, 0.3, 0.4))
    e = canvas.env_light()
    assert e.intensity == 1.0 and e.defaultRadiance.tuple() == pytest.approx((0.2, 0.3, 0.4))


def test_scripted_interaction_against_the_reference_kernels(scene):
    renderer, cfg, canvas = scene
    renderer.set_option(L.OPT_PT_MODE, 0)     # the reference's random streams: path for path
    renderer.set_option(L.OPT_PT_KERNEL, 1)
    _attach(renderer, cfg, canvas)
    canvas.set_immediate_repaint(False)
    canvas.set(render_mode=L.RENDER_MODE_PATHTRACER, scatter_times=2.0)
    canvas.mouse_press(40, 90, L.BUTTON_LEFT | L.BUTTON_MID)
    for px, py in ((48, 84), (60, 80), (75, 70)):
        canvas.mouse_move(px, py, L.BUTTON_LEFT | L.BUTTON_MID)
    canvas.wheel(-240)
    canvas.key(L.KEY_DOWN)
    canvas.set(fov=38.0, exposure=1.5)
    canvas.paint(4)
    assert canvas.frame_no == 4
    img = canvas.image()
    host = _hdr(canvas)
    assert host.max() > 0
    # the reference's kernels with the camera the canvas arrived at
    renderer.camera = canvas.camera()
    ref = oracle_reference(renderer, cfg)
    ref.frame_no = 0
    ref.render_pathtracer(4, 2)
    theirs = ref.hdr_image().cpu().numpy()
    check_paths(host, theirs, ref)
    if isinstance(ref, OracleRef):
        check_u8(img, ref)
    else:
        assert (np.abs(img.astype(int) - ref.ldr_image().cpu().numpy().astype(int)) <= 1).mean() > 0.999
    # and the ray caster from the same view
    canvas.set(render_mode=L.RENDER_MODE_RAYCASTING)
    canvas.paint()
    ref.render_raycasting(S.raycast_step_size())
    check_u8(canvas.image(), ref)
    renderer.set_option(L.OPT_PT_MODE, 2)
    renderer.set_option(L.OPT_PT_KERNEL, 2)


def test_load_volume_from_a_metaimage_file(scene, tmp_path):
    renderer, cfg, canvas = scene
    rng = np.random.default_rng(2)
    n = (40, 36, 30)   # z, y, x
    z, y, x = np.meshgrid(*[np.linspace(-1, 1, k) for k in n], indexing="ij")
    data = (np.clip(1.2 - np.sqrt(x * x + y * y + z * z), 0, 1) * 2000 + rng.normal(0, 5, n)).astype(np.int16)
    path = M.write_metaimage(tmp_path / "vol.mhd", data, spacing=(0.8, 1.0, 1.25), element_type="MET_SHORT")
    canvas.load_volume(path)
    canvas.set_transfer_function(renderer.tf)
    size = (n[2] * 0.8, n[1] * 1.0, n[0] * 1.25)
    cam = canvas.camera()
    assert cam.pos.z == pytest.approx(1.5 * max(size) / (2 * np.tan(np.radians(22.5))), rel=1e-5)
    v = canvas.volume()
    assert v.bbox.vmax.x == pytest.approx(0.5 * size[0]) and v.spacing.z == np.float32(1.25) and v.gradientFactor == 0.5
    canvas.paint()
    img = canvas.image()
    assert img[..., 3].max() > 100 and img[0, 0, 3] == 0
    with pytest.raises(L.SvrError):
        canvas.load_volume(tmp_path / "missing.mhd")
    canvas.paint()   # still usable


def test_headless_driver_replays_an_interaction_script(tmp_path):
    """tools/svr_headless --interact: the C++ host of the canvas (events, setters, paints, saved frames)."""
    import json
    import os
    import subprocess

    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "tools", "svr_headless")
    if not os.path.exists(exe):
        pytest.skip("tools/svr_headless not built (make tools)")
    script = tmp_path / "session.txt"
    script.write_text("\n".join([
        "# ray-cast view, then a drag, a zoom and a path-traced refinement",
        "paint 1", f"save {tmp_path}/rc0",
        "press 100 100 1", "move 130 90 1", "move 160 95 1", "wheel -120", "key left",
        "paint 1", f"save {tmp_path}/rc1",
        "mode pt", "depth 2", "exposure 1.5", "repaint 0", "clip x -0.5 1", "paint 16", f"save {tmp_path}/pt",
    ]) + "\n")
    out = subprocess.run([exe, "--config", "C1", "--n", "64", "--w", "256", "--h", "192", "--interact", str(script)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr
    info = json.loads(out.stdout.strip().splitlines()[-1])
    # paints: 2 (the driver's SetTransferFunction and SetAreaLights each repaint) + 1 + (2 per left-drag move) * 2
    # + 1 (wheel) + 2 (key) + 1 + 1 (mode) + 1 (depth) + 1 (exposure) + 16
    assert info["paints"] == 2 + 1 + 4 + 1 + 2 + 1 + 3 + 16 and info["frame_no"] == 16
    imgs = {}
    for name in ("rc0", "rc1", "pt"):
        raw = (tmp_path / f"{name}.ppm").read_bytes()
        assert raw.startswith(b"P6\n256 192\n255\n")
        imgs[name] = np.frombuffer(raw[len(b"P6\n256 192\n255\n"):], np.uint8)
        assert imgs[name].size == 256 * 192 * 3 and imgs[name].max() > 0
    assert not np.array_equal(imgs["rc0"], imgs["rc1"])
    bad = tmp_path / "bad.txt"
    bad.write_text("frobnicate 1\n")
    out = subprocess.run([exe, "--config", "C1", "--n", "32", "--w", "64", "--h", "64", "--interact", str(bad)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 2 and "cannot parse" in out.stderr
