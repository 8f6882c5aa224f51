"""GPU tests of label maps (svr_render_labels, svr_render_label_slices, svr_labels_create, svr_labels_load_metaimage): parity
with the CPU restatement (tests/label_oracle.cpp), bit-exact skipping through the label presence grid, visibility changes that
rebuild nothing, new voxels, exact overlays against numpy, the MetaImage loader, no effect on the other renderers and the
headless driver.  Every option a test changes is restored (the session's renderer is shared)."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _label_oracle as LO
from _gpu_common import setup, small_config

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STEP = S.raycast_step_size()
H_STEP = 0.5 * STEP
ALL = S.label_table(S.label_palette(3))


@pytest.fixture(autouse=True)
def restore_options(renderer):
    saved = {k: renderer.get_option(k) for k in range(L.OPT_PT_DENOISE + 1)}
    yield
    for k, v in saved.items():
        renderer.set_option(k, v)
    renderer.free_labels()


def ct_labels(r, n=64, fmt=L.VOXEL_U16):
    """Skin (1), soft tissue (2) and bone (3) of the generated CT, as the tools derive them."""
    vox = r.generate_volume(L.GEN_CT, fmt, n).cpu().numpy().view(S.VOXEL_DTYPES[fmt]).reshape(n, n, n)
    return S.labels_from_thresholds(vox, S.CT_LABEL_LEVELS)


def ball_labels(n, R, lab=1, centre=(0.0, 0.0, 0.0)):
    c = np.arange(n) + 0.5 - n / 2
    d2 = (c[:, None, None] - centre[2]) ** 2 + (c[None, :, None] - centre[1]) ** 2 + (c[None, None, :] - centre[0]) ** 2
    return (d2 <= R * R).astype(np.uint8) * lab


def render(r, table, phase=0, stride=1):
    H, W = r.camera.imageH, r.camera.imageW
    surface = torch.full((H * W * 4,), -3.0, dtype=torch.float32, device="cuda")
    lab = torch.full((H * W,), 77, dtype=torch.uint8, device="cuda")
    r.img.fill_(0x5A)
    r.render_labels(table, STEP, surface=surface, labels=lab, phase=phase, stride=stride)
    torch.cuda.synchronize()
    return surface.view(H, W, 4).clone(), r.ldr_image().clone(), lab.view(H, W).clone()


def oblique_camera(n, w, h):
    return S.look_at_camera((0.9 * n, 0.7 * n, 1.1 * n), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), fovx=45.0, image_w=w, image_h=h)


def check_vs_oracle(got, ref):
    """Hit masks agree on >= 99 % of the pixels; where both hit, the depth is within h (a rounding difference of a position can
    move the first sample that reaches 1/2), the label is equal and u8 within 2 LSB on >= 99 % of them.  Misses are
    (0, 0, 0, +inf), a zero image and label 0 on both sides."""
    s, u, lab = (x.cpu().numpy() for x in got)
    rs, ru, rlab = ref
    hit, ref_hit = np.isfinite(s[..., 3]), np.isfinite(rs[..., 3])
    assert ref_hit.mean() > 0.01
    assert (hit == ref_hit).mean() >= 0.99, float((hit == ref_hit).mean())
    both = hit & ref_hit
    assert (np.abs(s[..., 3][both] - rs[..., 3][both]) <= H_STEP).mean() >= 0.99
    assert (lab[both] == rlab[both]).mean() >= 0.99, float((lab[both] == rlab[both]).mean())
    du = np.abs(u[both].astype(int) - ru[both].astype(int)).max(axis=1)
    assert (du <= 2).mean() >= 0.99, float((du <= 2).mean())
    miss = ~hit
    assert np.all(s[miss][:, :3] == 0) and np.all(s[miss][:, 3] == np.inf) and np.all(u[miss] == 0) and np.all(lab[miss] == 0)
    assert np.all(u[hit][:, 3] == 255) and np.all(lab[hit] != 0)


@pytest.mark.parametrize("kind", ["ct", "ball"])
def test_matches_cpu_restatement(renderer, kind):
    n, W, H = 64, 112, 96
    lab = ct_labels(renderer, n) if kind == "ct" else ball_labels(n, 13.0, 5, (3.0, -2.0, 1.0))
    spacing = (1.0, 1.0, 1.0)
    vol = renderer.load_labels(lab, spacing)
    tables = (ALL, S.label_table({3: (1.0, 1.0, 1.0, 1.0), 2: (0.2, 0.9, 0.3, 0.0)})) if kind == "ct" else (
        S.label_table({5: (0.3, 0.6, 0.9, 1.0)}),)
    for cam in (S.default_camera((n, n, n), W, H), oblique_camera(n, W, H)):
        renderer.set_camera(cam)
        orc = LO.oracle(lab, vol, cam)
        for table in tables:
            check_vs_oracle(render(renderer, table), LO.labels(orc, table, STEP))


SUBSETS = [{1: (1.0, 0.8, 0.6, 1.0), 2: (0.8, 0.3, 0.3, 1.0), 3: (1.0, 1.0, 0.9, 1.0)}, {3: (1.0, 1.0, 0.9, 1.0)},
           {2: (0.8, 0.3, 0.3, 0.5)}, {1: (0.2, 0.2, 1.0, 1.0), 3: (1.0, 1.0, 1.0, 0.1)}, {}]


def test_skipping_is_bit_exact(renderer):
    """img, surface and label with skipping off and on, for cell edges 2 .. 16, several visibility subsets (including none), clip
    planes and a camera inside the volume."""
    n, W, H = 48, 80, 64
    renderer.load_labels(ct_labels(renderer, n, L.VOXEL_U8), (1.0, 1.0, 1.0))
    inside = S.make_camera((3.0, -2.0, 6.0), (1, 0, 0), (0, 1, 0), (0, 0, 1), 60.0, 0.0, 1.0, 1.0, W, H)
    views = [(S.default_camera((n, n, n), W, H), (-1.0, 1.0)), (oblique_camera(n, W, H), (-0.4, 0.3)), (inside, (-1.0, 1.0))]
    for cam, clip in views:
        renderer.set_camera(cam)
        for a in "xyz":
            setattr(renderer.labels, a + "_clip", L.Vec2(*clip))
        hits = 0
        for colors in SUBSETS:
            table = S.label_table(colors)
            renderer.set_option(L.OPT_RC_SKIP, 0)
            ref = render(renderer, table)
            hits += int(torch.isfinite(ref[0][..., 3]).sum())
            renderer.set_option(L.OPT_RC_SKIP, 1)
            for cell in (2, 4, 8, 16):
                renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
                got = render(renderer, table)
                for g, f in zip(got, ref):
                    assert torch.equal(g, f), (clip, cell, colors)
        assert hits > 0, clip


def test_skipping_skips(renderer):
    """On sparse labels (a ball of radius 6 in 64^3, and the CT's bone alone) the steps are the same with skipping on and off,
    and more than half of them are skipped."""
    n = 64
    renderer.set_camera(S.default_camera((n, n, n), 128, 128))
    renderer.set_option(L.OPT_COUNTERS, 1)
    for lab, table in ((ball_labels(n, 6.0, 2), S.label_table({2: (1.0, 0.0, 0.0, 1.0)})),
                       (ct_labels(renderer, n), S.label_table({3: (1.0, 1.0, 1.0, 1.0)}))):
        renderer.load_labels(lab)
        counts = {}
        for skip in (0, 1):
            renderer.set_option(L.OPT_RC_SKIP, skip)
            renderer.reset_counters()
            got = render(renderer, table)
            counts[skip] = renderer.counters()
            counts[skip]["hits"] = int(torch.isfinite(got[0][..., 3]).sum())
        print({k: {m: c[m] for m in ("steps", "skipped", "shade_taps", "cells", "hits")} for k, c in counts.items()})
        off, on = counts[0], counts[1]
        assert off["steps"] == on["steps"] and off["hits"] == on["hits"] > 0
        assert off["skipped"] == 0 and off["shade_taps"] == off["steps"]
        assert on["shade_taps"] + on["skipped"] == on["steps"]
        assert on["skipped"] > 0.5 * on["steps"], on


def test_visibility_changes_rebuild_nothing(renderer):
    """After the first call (which builds the presence grid), every call with a new table is one launch."""
    n = 48
    renderer.load_labels(ct_labels(renderer, n, L.VOXEL_U8))
    renderer.set_camera(S.default_camera((n, n, n), 64, 64))
    renderer.set_option(L.OPT_RC_SKIP, 1)
    renderer.set_option(L.OPT_COUNTERS, 0)
    renderer.render_labels(ALL)
    for colors in SUBSETS * 2:
        before = renderer.launch_count()
        renderer.render_labels(S.label_table(colors))
        assert renderer.launch_count() == before + 1, colors


@pytest.mark.parametrize("how", ["host", "device", "recreate"])
def test_new_voxels_are_seen(renderer, how):
    n, W, H = 48, 80, 64
    first = ct_labels(renderer, n, L.VOXEL_U8)
    renderer.load_labels(first)
    renderer.set_camera(S.default_camera((n, n, n), W, H))
    table = S.label_table({1: (1.0, 0.0, 0.0, 1.0), 3: (0.0, 1.0, 0.0, 1.0), 4: (0.0, 0.0, 1.0, 1.0)})
    render(renderer, table)  # presence grid of the CT
    second = ball_labels(n, 10.0, 4)
    if how == "host":
        renderer.upload_labels(second)
    elif how == "device":
        renderer.upload_labels(torch.from_numpy(second.copy()).cuda())
    else:
        renderer.load_labels(second)
    got = render(renderer, table)
    check_vs_oracle(got, LO.labels(LO.oracle(second, renderer.labels, renderer.camera), table, STEP))
    renderer.set_option(L.OPT_RC_SKIP, 0)
    for g, f in zip(render(renderer, table), got):
        assert torch.equal(g, f)


def _label_planes(lab, axis):
    """The label planes axis_slice's full stack shows: (count, H, W)."""
    if axis == "z":
        return lab
    if axis == "y":
        return np.ascontiguousarray(lab.transpose(1, 0, 2))  # slice y: rows z, columns x
    return np.ascontiguousarray(lab.transpose(2, 0, 1))      # slice x: rows z, columns y


def test_axis_slices_are_the_label_planes(renderer):
    rng = np.random.default_rng(5)
    nx, ny, nz = 28, 24, 20
    spacing = (0.8, 1.25, 1.5)
    lab = rng.integers(0, 6, size=(nz, ny, nx)).astype(np.uint8)
    renderer.load_labels(lab, spacing)
    for axis in "xyz":
        a = "xyz".index(axis)
        p = S.axis_slice((nx, ny, nz), spacing, axis, 0, count=(nx, ny, nz)[a])
        got, _ = renderer.render_label_slices(p, ALL)
        assert np.array_equal(got.cpu().numpy(), _label_planes(lab, axis)), axis
    # a clip plane: pixels whose centre lies outside the clipped box read 0
    renderer.labels.z_clip = L.Vec2(-1.0, 0.0)
    got, _ = renderer.render_label_slices(S.axis_slice((nx, ny, nz), spacing, "z", 0, count=nz), ALL)
    want = lab.copy()
    want[nz // 2:] = 0
    assert np.array_equal(got.cpu().numpy(), want)


def _composite(grey, lab, colors, outline):
    """numpy float32 restatement of the overlay: trunc((1 - a) in + a (255 c) + 1/2), a = 1 on outline pixels."""
    out = grey.copy()
    f = np.float32
    vis = np.zeros(256, bool)
    table = np.zeros((256, 4), np.float32)
    for l, c in colors.items():
        table[l] = np.array(c, np.float32)
        vis[l] = l != 0 and table[l, 3] > 0
    edge = np.zeros(lab.shape, bool)
    if outline:
        edge[:, :, 1:] |= lab[:, :, 1:] != lab[:, :, :-1]
        edge[:, :, :-1] |= lab[:, :, :-1] != lab[:, :, 1:]
        edge[:, 1:, :] |= lab[:, 1:, :] != lab[:, :-1, :]
        edge[:, :-1, :] |= lab[:, :-1, :] != lab[:, 1:, :]
    m = vis[lab]
    a = np.where(edge, f(1), table[lab, 3])[m]
    for ch in range(3):
        v = (f(1) - a) * grey[..., ch][m].astype(np.float32) + a * (f(255) * table[lab, ch][m])
        out[..., ch][m] = (v + f(0.5)).astype(np.uint32).astype(np.uint8)
    out[..., 3][m] = 255
    return out, m, edge & m


@pytest.mark.parametrize("outline", [False, True])
def test_overlay_equals_numpy(renderer, outline):
    rng = np.random.default_rng(11)
    nx, ny, nz = 40, 36, 12
    lab = np.zeros((nz, ny, nx), np.uint8)
    for l in range(1, 6):  # boxes of labels 1..5, so that the outline has runs and corners
        x0, y0 = rng.integers(0, nx - 8), rng.integers(0, ny - 8)
        lab[:, y0:y0 + rng.integers(4, 14), x0:x0 + rng.integers(4, 14)] = l
    renderer.load_labels(lab)
    colors = {1: (1.0, 0.0, 0.0, 0.5), 2: (0.1, 0.7, 0.3, 0.3), 3: (0.2, 0.4, 0.9, 0.0), 4: (0.9, 0.9, 0.1, 1.0), 5: (0.33, 0.66, 0.99, 0.77)}
    table = S.label_table(colors)
    p = S.axis_slice((nx, ny, nz), (1.0, 1.0, 1.0), "z", 0, count=nz)
    grey = torch.from_numpy(rng.integers(0, 256, size=(nz, ny, nx, 4)).astype(np.uint8)).cuda()
    img = grey.clone()
    got_lab, _ = renderer.render_label_slices(p, table, img=img, outline=outline)
    torch.cuda.synchronize()
    g = got_lab.cpu().numpy()
    assert np.array_equal(g, lab)
    want, drawn, edge = _composite(grey.cpu().numpy(), lab, colors, outline)
    mine = img.cpu().numpy()
    assert np.array_equal(mine, want)
    assert drawn.any() and (edge.any() if outline else True)
    assert np.array_equal(mine[~drawn], grey.cpu().numpy()[~drawn])  # background and hidden labels (3) untouched
    # the same composite again over a fresh copy of the grey image
    img2 = grey.clone()
    renderer.render_label_slices(p, table, img=img2, labels=None, outline=outline)
    assert torch.equal(img2, img)


def test_oblique_overlay_matches_cpu_restatement(renderer):
    n = 48
    lab = ct_labels(renderer, n, L.VOXEL_U8)
    vol = renderer.load_labels(lab)
    p = S.oblique_slice((1.0, -2.0, 0.5), (0.3, 0.5, 0.8), (0.0, 1.0, 0.0), 0.7, 96, 80, count=3, slice_step=2.0)
    orc = LO.oracle(lab, vol, S.default_camera((n, n, n), 8, 8))
    rng = np.random.default_rng(3)
    grey = rng.integers(0, 256, size=(3, 80, 96, 4)).astype(np.uint8)
    img = torch.from_numpy(grey).cuda()
    got, _ = renderer.render_label_slices(p, ALL, img=img, outline=True)
    ref, ref_img = LO.label_slices(orc, p, ALL, img=grey, outline=True)
    g = got.cpu().numpy()
    assert (g != 0).mean() > 0.1
    assert (g == ref).mean() >= 0.999, float((g == ref).mean())
    assert (np.all(img.cpu().numpy() == ref_img, axis=3)).mean() >= 0.99


@pytest.mark.parametrize("name,etype,dtype,compressed,msb", [("a.mha", "MET_UCHAR", np.uint8, False, False),
                                                             ("b.mha", "MET_USHORT", np.uint16, True, True),
                                                             ("c.mhd", "MET_INT", np.int32, False, False),
                                                             ("d.mhd", "MET_CHAR", np.int8, True, False)])
def test_metaimage_labels_round_trip(renderer, tmp_path, name, etype, dtype, compressed, msb):
    rng = np.random.default_rng(2)
    nx, ny, nz = 13, 9, 7
    lab = rng.integers(0, 128, size=(nz, ny, nx)).astype(dtype)
    path = LO.write_metaimage(tmp_path / name, lab, etype, compressed=compressed, msb=msb, detached=name.endswith(".mhd"))
    assert renderer.load_label_metaimage(path) == int(lab.max())
    out = np.zeros((nz, ny, nx), np.uint8)
    L.check(renderer.lib.svr_volume_download(C.byref(renderer.labels), C.c_void_p(out.ctypes.data), out.nbytes), "svr_volume_download")
    assert np.array_equal(out, lab.astype(np.uint8))
    v = renderer.labels
    assert (v.spacing.x, v.spacing.y, v.spacing.z) == (1.5, 1.0, 2.0)
    assert abs(v.bbox.vmax.x - nx * 1.5 / 2) < 1e-6 and abs(v.bbox.vmax.z - nz * 2.0 / 2) < 1e-6


def test_grey_volume_is_not_a_label_volume(renderer):
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U8, w=32, h=32)
    setup(renderer, cfg)
    before = renderer.launch_count()
    with pytest.raises(L.SvrError, match="not a label volume"):
        L.check(renderer.lib.svr_render_labels(C.c_void_p(renderer.img.data_ptr()), None, None, C.byref(renderer.volume),
                                               C.byref(renderer.camera), C.byref(ALL), STEP, 0, 1, None), "svr_render_labels")
    with pytest.raises(L.SvrError, match="not a label volume"):
        L.check(renderer.lib.svr_render_label_slices(C.c_void_p(renderer.img.data_ptr()), None, C.byref(renderer.volume),
                                                     C.byref(S.axis_slice((64, 64, 64), (1, 1, 1), "z", 3)), C.byref(ALL), 0),
                "svr_render_label_slices")
    assert renderer.launch_count() == before


def _grid_info(r):
    dims, cell = (C.c_int32 * 3)(), C.c_int32(0)
    L.check(r.lib.svr_grid_info(dims, C.byref(cell)), "svr_grid_info")
    return tuple(dims), int(cell.value)


def test_other_renderers_are_unchanged(renderer):
    """Label renders between grey renders change none of projection, isosurface, slices, ray caster and path tracer, and leave
    the grey volume's range grid (svr_grid_info) as it was."""
    cfg = small_config(gen=L.GEN_CT, fmt=L.VOXEL_U16, w=96, h=80, depth=2)
    setup(renderer, cfg)
    renderer.set_option(L.OPT_MACROCELL_SIZE, 0)
    n = cfg.n
    sl = S.axis_slice((n, n, n), (1.0, 1.0, 1.0), "y", 20, thickness_voxels=9, count=4)

    def grey():
        out = {}
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(4, 2)
        torch.cuda.synchronize()
        out["pt"] = (renderer.hdr.clone(), renderer.img.clone())
        rc = torch.zeros(cfg.width * cfg.height * 4, dtype=torch.float32, device="cuda")
        renderer.render_raycasting_f32(rc, STEP, img=renderer.img)
        torch.cuda.synchronize()
        out["rc"] = (rc, renderer.img.clone())
        val = torch.zeros(cfg.width * cfg.height, dtype=torch.float32, device="cuda")
        renderer.render_projection("max", out=val)
        torch.cuda.synchronize()
        out["mip"] = (val, renderer.img.clone())
        surf = torch.zeros(cfg.width * cfg.height * 4, dtype=torch.float32, device="cuda")
        renderer.render_isosurface(0.7, STEP, surface=surf)
        torch.cuda.synchronize()
        out["iso"] = (surf, renderer.img.clone())
        out["slice"] = tuple(x.clone() for x in renderer.render_slices(sl))
        out["grid"] = _grid_info(renderer)
        return out

    ref = grey()
    renderer.load_labels(ct_labels(renderer, n))
    for table in (ALL, S.label_table({3: (1.0, 1.0, 1.0, 1.0)})):
        render(renderer, table)
        renderer.render_label_slices(sl, table, img=renderer.render_slices(sl)[1], outline=True)
        assert _grid_info(renderer) == ref["grid"]
        now = grey()
        for k in ref:
            if k == "grid":
                assert now[k] == ref[k]
            else:
                for a, b in zip(now[k], ref[k]):
                    assert torch.equal(a, b), k


def _headless_camera(n, W, H):
    libm = C.CDLL("libm.so.6")
    libm.tanf.restype, libm.tanf.argtypes = C.c_float, [C.c_float]
    cam = L.Camera()
    cam.imageW, cam.imageH, cam.exposure, cam.apeture, cam.focalLength = W, H, 1.0, 0.0, 1.0
    cam.aspectRatio = float(np.float32(W) / np.float32(H))
    cam.tanFovxOverTwo = libm.tanf(float(np.float32(float(np.float32(45.0) * np.float32(0.5)) * math.pi / float(np.float32(180.0)))))
    cam.pos = L.Vec3(0.0, 0.0, float(np.float32(1.5 * n / (2.0 * math.tan(45.0 * 0.5 * math.pi / 180.0)))))
    cam.u, cam.v, cam.w = L.Vec3(1, 0, 0), L.Vec3(0, 1, 0), L.Vec3(0, 0, 1)
    return cam


def _ppm(path, W, H):
    with open(path, "rb") as f:
        data = f.read()
    return np.frombuffer(data[-W * H * 3:], np.uint8).reshape(H, W, 3)[::-1]


def test_headless_driver_writes_the_python_images(renderer, tmp_path):
    exe = os.path.join(ROOT, "tools", "svr_headless")
    if not os.path.exists(exe):
        pytest.skip("tools/svr_headless was not built (make tools)")
    n = 64
    sphere = S.sphere_volume(n, L.VOXEL_U8)
    lab = S.labels_from_thresholds(sphere, (0.3, 0.6, 0.85))
    path = LO.write_metaimage(tmp_path / "labels.mha", lab, "MET_UCHAR")
    with open(path, "rb") as f:  # the writer's spacing is (1.5, 1, 2); the driver's volume has spacing 1
        text = f.read().replace(b"ElementSpacing = 1.5 1 2", b"ElementSpacing = 1 1 1")
    with open(path, "wb") as f:
        f.write(text)
    W, H = 96, 80
    out = str(tmp_path / "labels")
    subprocess.check_call([exe, "--config", "C1", "--n", str(n), "--w", str(W), "--h", str(H), "--mode", "labels", "--labels", path,
                           "--reps", "1", "--out", out], cwd=str(tmp_path))
    ppm = _ppm(out + ".ppm", W, H)
    renderer.load_labels(lab)
    renderer.set_camera(_headless_camera(n, W, H))
    step = float(np.float32(0.5) * np.sqrt(np.float32(3.0)))
    renderer.img.zero_()
    renderer.render_labels(S.label_table(S.label_palette(int(lab.max()))), step)
    torch.cuda.synchronize()
    mine = renderer.ldr_image().cpu().numpy()[..., :3]
    assert mine.max() > 100
    assert np.array_equal(ppm, mine)
    # the slice overlay: the grey axial slice through voxel n / 2, the labels at half opacity, outlines opaque
    out = str(tmp_path / "overlay")
    subprocess.check_call([exe, "--config", "C1", "--n", str(n), "--w", str(n), "--h", str(n), "--mode", "slice", "--labels", path,
                           "--outline", "--reps", "1", "--out", out], cwd=str(tmp_path))
    ppm = _ppm(out + ".ppm", n, n)
    setup(renderer, small_config(n=n, w=n, h=n, gen=L.GEN_SPHERE, fmt=L.VOXEL_U8))
    renderer.load_volume(renderer.generate_volume(L.GEN_SPHERE, L.VOXEL_U8, n, 1234), L.VOXEL_U8, (n, n, n))
    p = S.axis_slice((n, n, n), (1.0, 1.0, 1.0), "z", n // 2)
    _, img = renderer.render_slices(p)
    renderer.render_label_slices(p, S.label_table(S.label_palette(int(lab.max()), 0.5)), img=img, outline=True)
    torch.cuda.synchronize()
    mine = img[0, ..., :3].cpu().numpy()
    assert np.array_equal(ppm, mine)
    assert (mine[..., 0] != mine[..., 1]).any()  # coloured pixels
