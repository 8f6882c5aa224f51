"""The projection-family renderers on a volume shaped like clinical data, held to float64 closed forms (no GPU): 67 x 45 x 29
voxels (no axis a multiple of 2, so every macrocell grid has a partial last cell on every axis) with spacing (0.7, 1.0, 1.9), as a
MetaImage from a scanner hands over.  On a cube with spacing 1 an axis mix-up or a missing spacing factor gives the same image;
here it moves a world-linear ramp's value by many times the bounds below.

The checkers are the CPU restatements (tests/*_oracle.cpp); tests/test_gpu_clinical_shapes.py applies the same closed forms to
the kernels' own outputs.  The closed forms share no code with either: rays, boxes, slab samples and curve points are float64
numpy from the camera and parameter structs.

Bounds.  The texture unit rounds each texel coordinate to 1/256 voxel (at most 1/512 off) and each trilinear weight to 1/256 in
two stages; for a linear function the summed weight of the upper texels of an axis equals the rounded fraction, or one unit more
where two roundings tie (test_isosurface_cpu.test_linear_ramp_gives_a_plane).  So a fetch of the ramp c0 + a . x is within
3/512 voxel per axis of the ramp at its position: |error| <= 3/512 sum_i |a_i s_i| (RAMP_BOUND), plus the storage: fp32
rounding of values near 1/2, or for u16 half an LSB when stored and half an LSB when the filter rounds its 16-bit sum."""
import math

import numpy as np

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _curved_oracle as CO
import _isosurface_oracle as IO
import _label_oracle as LO
import _projection_oracle as PO
import _slice_oracle as SO
from test_isosurface_cpu import _hit_points, _rays

DIMS = (67, 45, 29)            # x, y, z
SPACING = (0.7, 1.0, 1.9)
SP = np.array(SPACING)
EXT = np.array(DIMS) * SP      # the box spans +-EXT / 2
STEP = S.raycast_step_size(SPACING)
H_STEP = 0.5 * STEP
MODES = ("max", "min", "mean")

# the world-linear ramp c0 + a . x at the voxel centres, per world unit
RAMP_A = np.array([0.004, -0.006, 0.005])
RAMP_C0 = 0.5
RAMP_BOUND = 3.0 / 512 * float(np.sum(np.abs(RAMP_A * SP)))
STORAGE = {L.VOXEL_F32: 1e-6, L.VOXEL_U16: 1.0 / 65535}
INSET = 2                      # clip planes this many voxels in on every face: no tap reads the zero border
CLIP = [(-1.0 + 2.0 * INSET / d, 1.0 - 2.0 * INSET / d) for d in DIMS]
BOX_HI = 0.5 * EXT * (1.0 - 2.0 * INSET / np.array(DIMS))   # the clipped box [-BOX_HI, BOX_HI]
FACE_MARGIN = 1e-4             # samples this close to a clip face (world units) are left out: fp32 positions (|x| < 30) may fall
                               # on either side


def voxel_centres():
    """World coordinates of the voxel centres per axis: (i + 1/2) s - dim s / 2."""
    return [(np.arange(d) + 0.5) * s - 0.5 * d * s for d, s in zip(DIMS, SPACING)]


def ramp(fmt, a=RAMP_A, c0=RAMP_C0):
    """c0 + a . x at the voxel centres, (z, y, x), stored as fmt."""
    xs, ys, zs = voxel_centres()
    f = c0 + a[0] * xs[None, None, :] + a[1] * ys[None, :, None] + a[2] * zs[:, None, None]
    return S.encode_voxels(f.astype(np.float32), fmt)


def ramp_bound(fmt):
    return RAMP_BOUND + STORAGE[fmt]


def clip_volume(vol):
    vol.x_clip, vol.y_clip, vol.z_clip = (L.Vec2(*c) for c in CLIP)
    return vol


def ramp_volume():
    return clip_volume(S.host_volume_struct(DIMS, SPACING))


def outside_camera(w=96, h=80):
    """Off-axis: no ray is parallel to a grid axis."""
    return S.look_at_camera((0.9 * EXT[0], 0.55 * EXT[1], 1.6 * EXT[2]), (0.0, 0.0, 0.0), (0.0, 1.0, 0.0), fovx=45.0, image_w=w, image_h=h)


def inside_camera(w=96, h=80):
    """Inside the box, looking off-axis across it."""
    return S.look_at_camera((0.2 * EXT[0], -0.15 * EXT[1], 0.1 * EXT[2]), (-0.3 * EXT[0], 0.1 * EXT[1], -0.25 * EXT[2]), (0.0, 1.0, 0.0),
                            fovx=60.0, image_w=w, image_h=h)


def ray_samples(cam, lo, hi):
    """float64 (d, o, t0, K, sure) of camera_ray_center's rays against the box [lo, hi]: K samples at t0 + (k + 1/2) h; sure leaves
    out the pixels where (tFar - t0) / h + 1/2 lies within 1e-3 of an integer, where K is decided by rounding."""
    d = _rays(cam)
    o = np.array(cam.pos.tuple())
    with np.errstate(divide="ignore", invalid="ignore"):
        t1, t2 = (lo - o) / d, (hi - o) / d
    tn, tf = np.minimum(t1, t2).max(axis=2), np.maximum(t1, t2).min(axis=2)
    t0 = np.maximum(tn, 0.0)
    q = (tf - t0) / H_STEP + 0.5
    K = np.where(tf > t0, np.floor(q), 0.0)
    sure = ~(np.abs(q - np.round(q)) < 1e-3)
    return d, o, t0, K, sure


def projection_want(cam):
    """The ramp's projections in float64: MEAN = c0 + a . (the mean sample position), MAX and MIN the values at the first and
    last sample (the ramp is linear along a ray).  Returns ({mode: want}, compared mask, the rays sure to take no sample)."""
    d, o, t0, K, sure = ray_samples(cam, -BOX_HI, BOX_HI)
    first = RAMP_C0 + (o + d * (t0 + 0.5 * H_STEP)[..., None]) @ RAMP_A
    last = RAMP_C0 + (o + d * (t0 + (K - 0.5) * H_STEP)[..., None]) @ RAMP_A
    mean = RAMP_C0 + (o + d * (t0 + 0.5 * K * H_STEP)[..., None]) @ RAMP_A
    return {"max": np.maximum(first, last), "min": np.minimum(first, last), "mean": mean}, sure & (K > 0), sure & (K == 0)


def check_projection(got, cam, fmt, min_pixels=1500):
    """got: {mode: value (H, W)}; 0 where no sample is taken.  Returns the largest error per mode."""
    want, ok, miss = projection_want(cam)
    assert ok.sum() >= min_pixels, int(ok.sum())
    bound = ramp_bound(fmt)
    worst = {}
    for mode in MODES:
        err = np.abs(np.asarray(got[mode], np.float64) - want[mode])[ok]
        worst[mode] = float(err.max())
        assert worst[mode] <= bound, (mode, worst[mode], bound)
        assert np.all(np.asarray(got[mode])[miss] == 0), mode
    return worst


def test_projection_of_the_ramp_is_the_closed_form():
    for fmt in (L.VOXEL_F32, L.VOXEL_U16):
        vox = ramp(fmt)
        for cam in (outside_camera(), inside_camera()):
            orc = PO.oracle(vox, fmt, DIMS, ramp_volume(), cam)
            check_projection({m: PO.project(orc, m, STEP)[0] for m in MODES}, cam, fmt)


# ---- slices and slabs: the slab rule in float64 -------------------------------------------------------------------------------

def oblique(mode="max", thickness=0.0, count=2, size=(80, 64)):
    """An oblique stack through the ragged volume: its normal has no zero component, its pixels run off the clipped box."""
    return S.oblique_slice((1.3, -0.8, 0.6), (0.5, 0.35, 1.0), (0.1, 1.0, 0.2), 0.6, size[0], size[1], count=count, slice_step=3.0,
                           thickness=thickness, sample_spacing=0.55, mode=mode, window=(0.4, 0.3))


def _inside(x):
    """(inside the clipped box, within FACE_MARGIN of one of its faces)"""
    gap = np.min(BOX_HI - np.abs(x), axis=-1)
    return gap >= 0.0, np.abs(gap) < FACE_MARGIN


def slab_want(o, d, thickness, sample_spacing):
    """The slab rule (include/svr_render.h) in float64 on the rays o + t d, o and d (..., 3): K = max(1, floor(thickness / h + 1/2))
    samples h = sampleSpacing apart centred on t = 0 (a thin image: one sample at 0); the included ones are those inside the
    clipped box.  MEAN is the ramp at their centroid, MAX and MIN its values at the end samples.  Returns ({mode: want}, taken,
    compared mask: no sample within FACE_MARGIN of a clip face)."""
    if thickness > 0.0:
        h = float(sample_spacing)
        K = max(1, int(math.floor(thickness / h + 0.5)))
    else:
        h, K = 0.0, 1
    t = -0.5 * K * h + (np.arange(K) + 0.5) * h
    x = o[..., None, :] + t[:, None] * d[..., None, :]
    inside, near = _inside(x)
    taken = inside.sum(axis=-1)
    v = RAMP_C0 + x @ RAMP_A
    k = np.arange(K)
    first = np.where(inside, k, K).min(axis=-1)
    last = np.where(inside, k, -1).max(axis=-1)
    vf = np.take_along_axis(v, np.minimum(first, K - 1)[..., None], -1)[..., 0]
    vl = np.take_along_axis(v, np.maximum(last, 0)[..., None], -1)[..., 0]
    centroid = (x * inside[..., None]).sum(axis=-2) / np.maximum(taken, 1)[..., None]
    want = {"max": np.maximum(vf, vl), "min": np.minimum(vf, vl), "mean": RAMP_C0 + centroid @ RAMP_A}
    return {m: np.where(taken > 0, w, 0.0) for m, w in want.items()}, taken, ~near.any(axis=-1)


def slice_origins(p):
    """float64 pixel centres (count, H, W, 3) of svr_render_slices, c + fx U + fy V + j W, and the slab direction U x V / |U x V|."""
    c, u, v, w = (np.array(list(a), np.float64) for a in (p.center, p.axisU, p.axisV, p.axisW))
    fx = np.arange(p.imageW) + 0.5 - 0.5 * p.imageW
    fy = np.arange(p.imageH) + 0.5 - 0.5 * p.imageH
    j = np.arange(p.count)
    o = c + fx[None, None, :, None] * u + fy[None, :, None, None] * v + j[:, None, None, None] * (w if p.count > 1 else 0.0)
    n = np.cross(u, v)
    return o, n / np.linalg.norm(n)


def check_slab(value, u8, want, taken, ok, fmt, min_pixels):
    """value (count, H, W), u8 (count, H, W, 4) against slab_want: a pixel with a sample is within the ramp bound and opaque, one
    without is 0 and transparent.  Returns the largest error."""
    value, u8 = np.asarray(value, np.float64), np.asarray(u8)
    some = ok & (taken > 0)
    assert some.sum() >= min_pixels, int(some.sum())
    assert np.all(u8[..., 3][ok] == np.where(taken > 0, 255, 0)[ok])
    assert np.all(value[ok & (taken == 0)] == 0)
    err = float(np.abs(value - want)[some].max())
    assert err <= ramp_bound(fmt), (err, ramp_bound(fmt))
    return err


SLABS = ((0.0, 2), (12.0, 2))   # (thickness, count): thin slices, and 22-sample slabs


def test_oblique_slices_and_slabs_of_the_ramp_are_the_closed_form():
    for fmt in (L.VOXEL_F32, L.VOXEL_U16):
        orc = SO.oracle(ramp(fmt), fmt, DIMS, ramp_volume())
        for thickness, count in SLABS:
            for mode in MODES:
                p = oblique(mode, thickness, count)
                o, n = slice_origins(p)
                want, taken, ok = slab_want(o, np.broadcast_to(n, o.shape), thickness, p.sampleSpacing)
                value, u8 = SO.slices(orc, p)
                check_slab(value, u8, want[mode], taken, ok, fmt, 3000)


# ---- curved planar reformation: the pixels' points from the frame table --------------------------------------------------------

def centerline(m=300):
    """A non-planar curve through the ragged box."""
    u = np.linspace(0.0, 1.0, m)
    return np.stack([12.0 * np.sin(2 * np.pi * u), (u - 0.5) * 30.0, 9.0 * np.cos(np.pi * u)], 1).astype(np.float32)


def straightened(mode="max", thickness=0.0, count=2):
    return S.straightened_curve(64, 40, 0.7, station_spacing=0.9, up=(0, 0, 1), count=count, angle0=0.3, angle_step=1.1,
                                thickness=thickness, sample_spacing=0.55, mode=mode, window=(0.4, 0.3))


def cross_sections(mode="max", thickness=0.0, count=5):
    return S.curve_cross_sections(40, 36, count, 0.6, 7.0, up=(0, 0, 1), angle=0.4, thickness=thickness, sample_spacing=0.55, mode=mode,
                                  window=(0.4, 0.3))


def curve_origins(p, points):
    """float64 ray origins (count, H, W, 3), directions (count, H, W, 3) and the valid-station mask of svr_render_curved, from the
    frame table of S.curve_frames: straightened row y at angle theta_j is c_y + fx ps a (a = cos r + sin b), its slab along
    e = cos b - sin r; cross-section j is c_j + fx ps a + fy ps e, its slab along t."""
    cross = p.layout == L.CURVED_CROSS
    F = S.curve_frames(points, list(p.up), p.stationSpacing, CO.stations(p)).astype(np.float64)
    c, t, r, b, valid = F[:, 0, :3], F[:, 1, :3], F[:, 2, :3], F[:, 3, :3], F[:, 0, 3] != 0
    theta = p.angle0 + (np.zeros(1) if cross else np.arange(p.count) * p.angleStep)
    cs, sn = np.cos(theta), np.sin(theta)
    fx = (np.arange(p.imageW) + 0.5 - 0.5 * p.imageW) * p.pixelSpacing
    if cross:
        fy = (np.arange(p.imageH) + 0.5 - 0.5 * p.imageH) * p.pixelSpacing
        a = cs[0] * r + sn[0] * b                                   # (count, 3): one station per image
        e = cs[0] * b - sn[0] * r
        o = c[:, None, None] + fx[None, None, :, None] * a[:, None, None] + fy[None, :, None, None] * e[:, None, None]
        d = np.broadcast_to(t[:, None, None], o.shape)
        ok = np.broadcast_to(valid[:, None, None], o.shape[:3])
    else:
        a = cs[:, None, None] * r[None] + sn[:, None, None] * b[None]  # (count, H, 3)
        e = cs[:, None, None] * b[None] - sn[:, None, None] * r[None]
        o = c[None, :, None] + fx[None, None, :, None] * a[:, :, None]
        d = np.broadcast_to(e[:, :, None], o.shape)
        ok = np.broadcast_to(valid[None, :, None], o.shape[:3])
    return o, d, ok


def curved_want(p, points, mode):
    o, d, valid = curve_origins(p, points)
    want, taken, ok = slab_want(o, d, p.thickness, p.sampleSpacing)
    taken = np.where(valid, taken, 0)
    return np.where(valid, want[mode], 0.0), taken, ok


CURVES = ((straightened, 0.0), (straightened, 12.0), (cross_sections, 0.0), (cross_sections, 12.0))


def test_curved_reformation_of_the_ramp_is_the_closed_form():
    pts = centerline()
    for fmt in (L.VOXEL_F32, L.VOXEL_U16):
        orc = CO.oracle(ramp(fmt), fmt, DIMS, ramp_volume())
        for make, thickness in CURVES:
            for mode in MODES:
                p = make(mode, thickness)
                value, u8 = CO.curved(orc, p, pts)
                want, taken, ok = curved_want(p, pts, mode)
                check_slab(value, u8, want, taken, ok, fmt, 2000)


# ---- isosurface of the rising ramp --------------------------------------------------------------------------------------------

ISO_VALUES = (0.45, 0.5, 0.55)


def check_iso_surface(surface, cam, iso, fmt, min_pixels=500):
    """surface (H, W, 4) of the isosurface of 1 - ramp (b = -a, c1 = 1 - c0: the value rises where b . d > 0) at iso.  Compared
    where b . d > 0.3 |b| and the crossing lies clearly between the first and the last sample:
      depth   the float64 ray-plane crossing c1 + b . x = iso, within e / (b . d) along the ray (a fetch within e of the plane's
              function crosses iso within e / slope of it, and the linear interpolation ending the refinement keeps that) plus
              2e-4 for fp32 positions at depths about 90;
      normal  b / |b| turned to the camera (= a / |a|), the world-space direction: gradient_at's taps are +-spacing, scaled by
              1 / (2 spacing).  The two taps of an axis have the same fixed-point fractions, so their difference is exact up to
              the storage error q of each tap (STORAGE): a component is off by at most q / s_i, the unit normal by
              2 |(q / s_i)_i| / |a|.  Where a tap lies within fp32 rounding of a 1/512 boundary, the two taps round apart (the
              one pixel of 1386 seen at iso 0.5 on the CPU): each tap is then off by up to e, the component by e / s_i and the
              normal by 2 |(e / s_i)_i| / |a|.  At most 1 % of the pixels may take that second bound.
    Returns (largest depth error, largest normal error on the 99 %, largest normal error)."""
    b, c1 = -RAMP_A, 1.0 - RAMP_C0
    d, o, t0, K, sure = ray_samples(cam, -BOX_HI, BOX_HI)
    ok = sure & (K > 0)
    slope = d @ b
    e = ramp_bound(fmt)
    first = c1 + (o + d * (t0 + 0.5 * H_STEP)[..., None]) @ b
    last = c1 + (o + d * (t0 + (K - 0.5) * H_STEP)[..., None]) @ b
    cmp = ok & (slope > 0.3 * np.linalg.norm(b)) & (first < iso - 2 * e) & (last >= iso + 2 * e)
    assert cmp.sum() >= min_pixels, int(cmp.sum())
    hit = np.isfinite(surface[..., 3])
    assert hit[cmp].all()
    back = -np.array(cam.w.tuple())
    t_hit = (iso - c1 - o @ b) / slope
    db = d @ back
    dz = np.abs(surface[..., 3] - t_hit * db)[cmp]
    bound = (e / slope * db + 2e-4)[cmp]
    assert np.all(dz <= bound), float((dz / bound).max())
    want_n = RAMP_A / np.linalg.norm(RAMP_A)
    dn = np.abs(surface[..., :3][cmp] - want_n).max(axis=1)
    same = 2.0 * np.linalg.norm(STORAGE[fmt] / SP) / np.linalg.norm(RAMP_A)
    tie = 2.0 * np.linalg.norm(e / SP) / np.linalg.norm(RAMP_A)
    assert (dn <= same).mean() >= 0.99, (float((dn <= same).mean()), same)
    assert dn.max() <= tie, (float(dn.max()), tie)
    return float(dz.max()), float(np.quantile(dn, 0.99)), float(dn.max())


def rising_ramp(fmt):
    return ramp(fmt, -RAMP_A, 1.0 - RAMP_C0)


def test_isosurface_of_the_ramp_is_the_plane():
    for fmt in (L.VOXEL_F32, L.VOXEL_U16):
        vox = rising_ramp(fmt)
        for cam in (outside_camera(), inside_camera()):
            orc = IO.oracle(vox, fmt, DIMS, ramp_volume(), cam)
            for iso in ISO_VALUES:
                surface, u8 = IO.isosurface(orc, iso, STEP)
                check_iso_surface(surface, cam, iso, fmt, 300 if cam.pos.x < EXT[0] / 2 else 500)
                assert np.all(u8[np.isfinite(surface[..., 3])][:, 3] == 255)


# ---- label half-spaces: the surface on the voxel face --------------------------------------------------------------------------

HALF = {0: 40, 1: 27, 2: 18}   # label 1 on voxels i < HALF[axis] of that axis: the face lies at HALF s - dim s / 2
HALF_LABEL = 3


def half_space(axis):
    lab = np.zeros(DIMS[::-1], np.uint8)
    sl = [slice(None)] * 3
    sl[2 - axis] = slice(0, HALF[axis])
    lab[tuple(sl)] = HALF_LABEL
    return lab


def check_half_space(surface, label, cam, axis, min_pixels=500):
    """Along the axis the indicator of label HALF_LABEL falls linearly from 1 at the centre of voxel HALF - 1 to 0 at that of voxel
    HALF: 1/2 on the face between them.  The camera lies on the + side, so the rays meet the face from outside the labels;
    compared where the float64 crossing lies at least one voxel inside the box on the other two axes (no side face is met first)
    and d_axis < -0.15.  The indicator is plain fp32 (no 8-bit weights) and linear across the face, so the depth is the
    plane's within 1e-3 (fp32 positions), the normal is +axis (the gradient is -axis / s, turned to the camera) and the label is
    HALF_LABEL.  Returns the largest depth error."""
    d = _rays(cam)
    o = np.array(cam.pos.tuple())
    plane = HALF[axis] * SPACING[axis] - 0.5 * EXT[axis]
    t = (plane - o[axis]) / d[..., axis]
    x = o + d * t[..., None]
    others = [i for i in range(3) if i != axis]
    cmp = (d[..., axis] < -0.15) & (t > 0)
    for i in others:
        cmp &= np.abs(x[..., i]) <= 0.5 * EXT[i] - SPACING[i]
    assert cmp.sum() >= min_pixels, int(cmp.sum())
    assert np.isfinite(surface[..., 3][cmp]).all()
    back = -np.array(cam.w.tuple())
    dz = np.abs(surface[..., 3] - t * (d @ back))[cmp]
    assert dz.max() <= 1e-3, float(dz.max())
    want_n = np.eye(3)[axis]
    assert np.abs(surface[..., :3][cmp] - want_n).max() <= 1e-6
    assert np.all(label[cmp] == HALF_LABEL)
    xh = _hit_points(cam, surface)[cmp]
    assert np.abs(xh[:, axis] - plane).max() <= 1e-3
    return float(dz.max())


HALF_TABLE = S.label_table({HALF_LABEL: (0.9, 0.5, 0.2, 1.0)})


def test_label_half_spaces_put_the_surface_on_the_voxel_face():
    vol = S.host_volume_struct(DIMS, SPACING)
    cam = outside_camera(112, 96)
    for axis in range(3):
        surface, u8, label = LO.labels(LO.oracle(half_space(axis), vol, cam), HALF_TABLE, STEP)
        check_half_space(surface, label, cam, axis)
