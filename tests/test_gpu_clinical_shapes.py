"""GPU tests of the projection-family renderers (projection, slices, curved reformation, isosurface, labels) on a volume shaped
like clinical data: 67 x 45 x 29 voxels with spacing (0.7, 1.0, 1.9) (tests/test_clinical_shapes_cpu.py), off-axis cameras, one of
them inside the box, and a ragged image size.
  a. the float64 closed forms of test_clinical_shapes_cpu on the kernels' own outputs, with the same bounds: the check that shares
     no code with the product (rays, boxes, slab samples and curve points in numpy);
  b. parity with the CPU restatements on a CT-like body (u16, and i16 through the MetaImage preprocessing) and on label blocks, at
     the tolerances of the renderers' own GPU files;
  c. bit-exact macrocell skipping on grids whose last cell is partial on every axis, and counters that show the skipping happened.
Every option a test changes is restored (the session's renderer is shared)."""
import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _curved_oracle as CO
import _isosurface_oracle as IO
import _label_oracle as LO
import _projection_oracle as PO
import _slice_oracle as SO
import test_clinical_shapes_cpu as CS
from test_gpu_anisotropic import _voxels
from test_gpu_isosurface import check_vs_oracle as check_iso_vs_oracle
from test_gpu_labels import check_vs_oracle as check_labels_vs_oracle
from test_gpu_projection import _tie_volume, check_vs_oracle

pytestmark = pytest.mark.gpu
DIMS, SPACING, STEP, MODES = CS.DIMS, CS.SPACING, CS.STEP, CS.MODES
WINDOW = (0.4, 0.3)
CELLS = (4, 8, 16, 32)
BODY_ISO = (0.2, 0.5)
TIE_ISO = (61 / 255,)   # one of the tie volume's levels (u16: 61 * 257 / 65535, the same value)
LABEL_TABLES = (S.label_table(S.label_palette(4)), S.label_table({2: (0.8, 0.3, 0.3, 1.0), 4: (0.2, 0.9, 0.4, 0.6)}))


@pytest.fixture(autouse=True)
def restore_options(renderer):
    saved = {k: renderer.get_option(k) for k in range(L.OPT_PT_DENOISE + 1)}
    renderer.set_option(L.OPT_RC_SKIP, 1)
    renderer.set_option(L.OPT_MACROCELL_SIZE, 8)
    renderer.set_option(L.OPT_COUNTERS, 0)
    yield
    for k, v in saved.items():
        renderer.set_option(k, v)
    renderer.free_labels()


def body():
    """The two ellipsoids of test_gpu_anisotropic at DIMS, u16; air is 0."""
    return _voxels(DIMS)


def ties(fmt=L.VOXEL_U16):
    """Blocks of 5 voxels at four integer levels (test_gpu_projection._tie_volume) cut to DIMS."""
    return np.ascontiguousarray(_tie_volume(max(DIMS), fmt)[:DIMS[2], :DIMS[1], :DIMS[0]])


def label_blocks(seed=3):
    """Blocks of 5 voxels holding label 0..4."""
    rng = np.random.default_rng(seed)
    b = [(d + 4) // 5 for d in DIMS[::-1]]
    blocks = rng.integers(0, 5, size=b).astype(np.uint8)
    lab = np.repeat(np.repeat(np.repeat(blocks, 5, 0), 5, 1), 5, 2)
    return np.ascontiguousarray(lab[:DIMS[2], :DIMS[1], :DIMS[0]])


def load(r, vox, fmt, clip=None):
    r.load_volume(vox, fmt, DIMS, spacing=SPACING)
    clip = clip or [(-1.0, 1.0)] * 3
    r.set_volume_params(x_clip=clip[0], y_clip=clip[1], z_clip=clip[2])


def project(r, mode):
    H, W = r.camera.imageH, r.camera.imageW
    out = torch.zeros(H * W, dtype=torch.float32, device="cuda")
    r.img.zero_()
    r.render_projection(mode, WINDOW, STEP, out=out)
    torch.cuda.synchronize()
    return out.view(H, W).clone(), r.ldr_image().clone()


def iso(r, value):
    H, W = r.camera.imageH, r.camera.imageW
    surface = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    r.img.zero_()
    r.render_isosurface(value, STEP, (0.9, 0.8, 0.6), surface=surface)
    torch.cuda.synchronize()
    return surface.view(H, W, 4).clone(), r.ldr_image().clone()


def labels(r, table):
    H, W = r.camera.imageH, r.camera.imageW
    surface = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    lab = torch.zeros(H * W, dtype=torch.uint8, device="cuda")
    r.img.zero_()
    r.render_labels(table, STEP, surface=surface, labels=lab)
    torch.cuda.synchronize()
    return surface.view(H, W, 4).clone(), r.ldr_image().clone(), lab.view(H, W).clone()


def slices(r, p):
    value, img = r.render_slices(p)
    torch.cuda.synchronize()
    return value, img


def curved(r, pts, p):
    value, img = r.render_curved(pts, p)
    torch.cuda.synchronize()
    return value, img


# ---- a. the closed forms on the kernels' outputs ---------------------------------------------------------------------------------

def test_projection_of_the_ramp_is_the_closed_form(renderer):
    for fmt in (L.VOXEL_F32, L.VOXEL_U16):
        load(renderer, CS.ramp(fmt), fmt, CS.CLIP)
        for cam in (CS.outside_camera(), CS.inside_camera()):
            renderer.set_camera(cam)
            worst = CS.check_projection({m: project(renderer, m)[0].cpu().numpy() for m in MODES}, cam, fmt)
            print("projection", fmt, worst, "bound", CS.ramp_bound(fmt))


def test_oblique_slices_and_slabs_of_the_ramp_are_the_closed_form(renderer):
    for fmt in (L.VOXEL_F32, L.VOXEL_U16):
        load(renderer, CS.ramp(fmt), fmt, CS.CLIP)
        worst = 0.0
        for thickness, count in CS.SLABS:
            for mode in MODES:
                p = CS.oblique(mode, thickness, count)
                o, n = CS.slice_origins(p)
                want, taken, ok = CS.slab_want(o, np.broadcast_to(n, o.shape), thickness, p.sampleSpacing)
                value, img = slices(renderer, p)
                worst = max(worst, CS.check_slab(value.cpu().numpy(), img.cpu().numpy(), want[mode], taken, ok, fmt, 3000))
        print("slices", fmt, worst, "bound", CS.ramp_bound(fmt))


def test_curved_reformation_of_the_ramp_is_the_closed_form(renderer):
    pts = CS.centerline()
    for fmt in (L.VOXEL_F32, L.VOXEL_U16):
        load(renderer, CS.ramp(fmt), fmt, CS.CLIP)
        worst = 0.0
        for make, thickness in CS.CURVES:
            for mode in MODES:
                p = make(mode, thickness)
                value, img = curved(renderer, pts, p)
                want, taken, ok = CS.curved_want(p, pts, mode)
                worst = max(worst, CS.check_slab(value.cpu().numpy(), img.cpu().numpy(), want, taken, ok, fmt, 2000))
        print("curved", fmt, worst, "bound", CS.ramp_bound(fmt))


def test_isosurface_of_the_ramp_is_the_plane(renderer):
    for fmt in (L.VOXEL_F32, L.VOXEL_U16):
        load(renderer, CS.rising_ramp(fmt), fmt, CS.CLIP)
        for cam in (CS.outside_camera(), CS.inside_camera()):
            renderer.set_camera(cam)
            for value in CS.ISO_VALUES:
                surface, u8 = iso(renderer, value)
                s = surface.cpu().numpy()
                worst = CS.check_iso_surface(s, cam, value, fmt, 300 if cam.pos.x < CS.EXT[0] / 2 else 500)
                assert np.all(u8.cpu().numpy()[np.isfinite(s[..., 3])][:, 3] == 255)
                print("isosurface", fmt, value, "depth, normal (99 %), normal (max)", worst)


def test_label_half_spaces_put_the_surface_on_the_voxel_face(renderer):
    cam = CS.outside_camera(112, 96)
    renderer.set_camera(cam)
    for axis in range(3):
        renderer.load_labels(CS.half_space(axis), SPACING)
        surface, _, lab = labels(renderer, CS.HALF_TABLE)
        worst = CS.check_half_space(surface.cpu().numpy(), lab.cpu().numpy(), cam, axis)
        print("labels", "xyz"[axis], "depth", worst)


# ---- b. parity with the CPU restatements -----------------------------------------------------------------------------------------

# (camera, clip): the ragged image size from outside over the whole box, and the camera inside a clipped box
def views():
    inner = [(-0.6, 0.7), (-0.7, 0.6), (-0.8, 0.8)]
    return [(CS.outside_camera(150, 101), None), (CS.inside_camera(), inner)]


def i16_body(r):
    """The body as MetaImage MET_SHORT values through the preprocessing (svr_volume_from_raw); returns the stored u16 voxels."""
    data = (body().astype(np.float64) / 65535.0 * 3000.0 - 1000.0).round().astype(np.int16)
    r.load_raw(data, L.MET_SHORT, DIMS, spacing=SPACING)
    return r.download_volume(DIMS, np.uint16)


@pytest.mark.parametrize("kind", ["body", "i16"])
def test_projection_and_isosurface_match_cpu_restatements(renderer, kind):
    vox = body() if kind == "body" else None
    for cam, clip in views():
        if kind == "body":
            load(renderer, vox, L.VOXEL_U16, clip)
        else:
            vox = i16_body(renderer)
            if clip:
                renderer.set_volume_params(x_clip=clip[0], y_clip=clip[1], z_clip=clip[2])
        renderer.set_camera(cam)
        for mode in MODES:
            value, u8 = project(renderer, mode)
            ref_value, ref_u8 = PO.project(PO.oracle(vox, L.VOXEL_U16, DIMS, renderer.volume, cam), mode, STEP, WINDOW)
            assert mode == "min" or ref_value.max() > 0.1
            check_vs_oracle(value, u8, ref_value, ref_u8)
        orc = IO.oracle(vox, L.VOXEL_U16, DIMS, renderer.volume, cam)
        for value in BODY_ISO:
            surface, u8 = iso(renderer, value)
            check_iso_vs_oracle(surface, u8, *IO.isosurface(orc, value, STEP, (0.9, 0.8, 0.6)))


def test_slices_and_curved_match_cpu_restatements(renderer):
    vox = body()
    load(renderer, vox, L.VOXEL_U16)
    so = SO.oracle(vox, L.VOXEL_U16, DIMS, renderer.volume)
    co = CO.oracle(vox, L.VOXEL_U16, DIMS, renderer.volume)
    pts = CS.centerline()
    for mode in MODES:
        for thickness, count in CS.SLABS:
            p = CS.oblique(mode, thickness, count, size=(75, 61))
            value, img = slices(renderer, p)
            ref_value, ref_u8 = SO.slices(so, p)
            assert ref_value.max() > 0.1
            check_vs_oracle(value, img, ref_value, ref_u8)
            assert np.array_equal(img[..., 3].cpu().numpy(), ref_u8[..., 3])
        for make, thickness in CS.CURVES:
            p = make(mode, thickness)
            value, img = curved(renderer, pts, p)
            ref_value, ref_u8 = CO.curved(co, p, pts)
            assert ref_value.max() > 0.1
            check_vs_oracle(value, img, ref_value, ref_u8)
            # inclusion can flip only for a sample on the box's surface (test_gpu_curved)
            assert (img[..., 3].cpu().numpy() != ref_u8[..., 3]).mean() <= 1e-3


def test_labels_match_cpu_restatements(renderer):
    lab = label_blocks()
    vol = renderer.load_labels(lab, SPACING)
    for cam, clip in views():
        for a, c in zip("xyz", clip or [(-1.0, 1.0)] * 3):
            setattr(renderer.labels, a + "_clip", L.Vec2(*c))
        renderer.set_camera(cam)
        orc = LO.oracle(lab, renderer.labels, cam)
        for table in LABEL_TABLES:
            check_labels_vs_oracle(labels(renderer, table), LO.labels(orc, table, STEP))
    # the oblique overlay at SPACING, over a grey stack, with outlines
    for a in "xyz":
        setattr(renderer.labels, a + "_clip", L.Vec2(-1.0, 1.0))
    p = CS.oblique("max", 0.0, 3, size=(75, 61))
    orc = LO.oracle(lab, vol, S.default_camera(DIMS, 8, 8))
    grey = np.random.default_rng(3).integers(0, 256, size=(3, 61, 75, 4)).astype(np.uint8)
    img = torch.from_numpy(grey).cuda()
    got, _ = renderer.render_label_slices(p, LABEL_TABLES[0], img=img, outline=True)
    ref, ref_img = LO.label_slices(orc, p, LABEL_TABLES[0], img=grey, outline=True)
    g = got.cpu().numpy()
    assert (g != 0).mean() > 0.1
    assert (g == ref).mean() >= 0.999, float((g == ref).mean())
    assert (np.all(img.cpu().numpy() == ref_img, axis=3)).mean() >= 0.99


# ---- c. bit-exact skipping on the ragged grid ------------------------------------------------------------------------------------

def skipping_is_exact(r, run, what):
    """run() with skipping off, then on for every cell edge of CELLS (each grid's last cell is partial on every axis): equal, tensor
    for tensor.  Then once more at cell 8 with the counters on (the counting variant): the same outputs, and shade_taps + skipped
    = steps.  Returns the skipped count."""
    r.set_option(L.OPT_RC_SKIP, 0)
    ref = run()
    r.set_option(L.OPT_RC_SKIP, 1)
    for cell in CELLS:
        r.set_option(L.OPT_MACROCELL_SIZE, cell)
        for g, f in zip(run(), ref):
            assert torch.equal(g, f), (what, cell, int((g != f).sum()))
    r.set_option(L.OPT_MACROCELL_SIZE, 8)
    r.set_option(L.OPT_COUNTERS, 1)
    r.reset_counters()
    got = run()
    c = r.counters()
    r.set_option(L.OPT_COUNTERS, 0)
    for g, f in zip(got, ref):
        assert torch.equal(g, f), (what, "counted")
    assert c["steps"] > 0 and c["shade_taps"] + c["skipped"] == c["steps"], (what, c)
    return c["skipped"]


VOLUMES = {"body": body, "ties": ties}


def test_projection_and_isosurface_skipping_is_bit_exact(renderer):
    skipped = {}
    for kind, make in VOLUMES.items():
        for cam, clip in views():
            load(renderer, make(), L.VOXEL_U16, clip)
            renderer.set_camera(cam)
            for mode in MODES:
                skipped[mode] = skipped.get(mode, 0) + skipping_is_exact(renderer, lambda: project(renderer, mode), (kind, mode))
            for value in BODY_ISO if kind == "body" else TIE_ISO:
                skipped["iso"] = skipped.get("iso", 0) + skipping_is_exact(renderer, lambda: iso(renderer, value), (kind, value))
    print("skipped", skipped)
    assert all(v > 0 for v in skipped.values()), skipped


def test_slice_and_curved_skipping_is_bit_exact(renderer):
    pts = CS.centerline()
    skipped = {}
    for kind, make in VOLUMES.items():
        load(renderer, make(), L.VOXEL_U16)
        for mode in MODES:
            # slabs of 36 and 40 samples: the curved walk needs at least CURVED_WALK_MIN_K = 32
            runs = [("slice", lambda: slices(renderer, CS.oblique(mode, 20.0, 2))),
                    ("straightened", lambda: curved(renderer, pts, CS.straightened(mode, 22.0))),
                    ("cross", lambda: curved(renderer, pts, CS.cross_sections(mode, 22.0)))]
            for name, run in runs:
                skipped[name, mode] = skipped.get((name, mode), 0) + skipping_is_exact(renderer, run, (kind, name, mode))
    print("skipped", skipped)
    assert all(v > 0 for v in skipped.values()), skipped


def test_label_skipping_is_bit_exact(renderer):
    skipped = 0
    for lab in (label_blocks(), S.labels_from_thresholds(body(), (0.1, 0.3, 0.6))):
        renderer.load_labels(lab, SPACING)
        for cam, clip in views():
            for a, c in zip("xyz", clip or [(-1.0, 1.0)] * 3):
                setattr(renderer.labels, a + "_clip", L.Vec2(*c))
            renderer.set_camera(cam)
            for table in LABEL_TABLES:
                skipped += skipping_is_exact(renderer, lambda: labels(renderer, table), "labels")
    assert skipped > 0
