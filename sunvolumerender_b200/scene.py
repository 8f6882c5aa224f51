"""Host-side scene construction -- the part of gui/canvas.cpp, gui/mainwindow.cpp and
core/VolumeReader.cpp that decides WHAT the render entry points are called with.  Pure numpy /
ctypes: no GPU needed, so the `-m "not gpu"` tests cover it.

Synthetic configurations C1..C5 are the ones SURVEY.md section 8(d) and BASELINE.json name.
"""
import math
from dataclasses import dataclass, field

import numpy as np

from . import _lib as L

TF_TABLE_SIZE = 1024  # gui/transferfunction.h:29

# colour nodes of the default transfer function, gui/mainwindow.cpp:57-62
_COLOR_NODES = [
    (0.0, (69.0 / 255, 199.0 / 255, 186.0 / 255)),
    (0.2, (172.0 / 255, 3.0 / 255, 57.0 / 255)),
    (0.4, (169.0 / 255, 83.0 / 255, 58.0 / 255)),
    (0.6, (43.0 / 255, 32.0 / 255, 161.0 / 255)),
    (0.8, (247.0 / 255, 158.0 / 255, 97.0 / 255)),
    (1.0, (183.0 / 255, 7.0 / 255, 140.0 / 255)),
]


def make_camera(pos, u, v, w, fovx=45.0, apeture=0.0, focal_length=1.0, exposure=1.0, image_w=640, image_h=480):
    """cudaCamera::Setup(pos, u, v, w, ...) -- core/cuda_camera.h:34-47 (field `apeture` as spelled there)."""
    cam = L.Camera()
    cam.pos = L.Vec3(*pos)
    cam.u = L.Vec3(*u)
    cam.v = L.Vec3(*v)
    cam.w = L.Vec3(*w)
    cam.imageW = int(image_w)
    cam.imageH = int(image_h)
    cam.aspectRatio = np.float32(image_w) / np.float32(image_h)
    # tanf(fovx * 0.5f * M_PI / 180.f): the product is evaluated in double, then tanf of its float value
    cam.tanFovxOverTwo = float(np.tan(np.float32(np.float32(fovx) * np.float32(0.5) * math.pi / 180.0), dtype=np.float32))
    cam.exposure = exposure
    cam.focalLength = focal_length
    cam.apeture = apeture
    return cam


def look_at_camera(pos, target, up, **kw):
    """cudaCamera::Setup(pos, target, up, ...) -- core/cuda_camera.h:49-62."""
    pos = np.asarray(pos, np.float32)
    target = np.asarray(target, np.float32)
    up = np.asarray(up, np.float32)
    w = pos - target
    w = w / np.sqrt(np.dot(w, w))
    u = np.cross(up, w)
    v = np.cross(w, u)
    return make_camera(pos, u, v, w, **kw)


def eye_distance(extent, fov=45.0):
    """Canvas::ZoomToExtent, gui/canvas.cpp:191-197."""
    return 1.5 * max(extent) / (2.0 * math.tan(math.radians(fov * 0.5)))


def default_camera(extent, image_w, image_h, fov=45.0, exposure=1.0, apeture=0.0, focal_length=1.0):
    """Camera as Canvas frames a freshly loaded volume: on +z looking at the origin (gui/canvas.cpp:31-38, 179-188)."""
    d = eye_distance(extent, fov)
    return make_camera((0.0, 0.0, d), (1, 0, 0), (0, 1, 0), (0, 0, 1), fov, apeture, focal_length, exposure, image_w, image_h)


def default_area_light(extent, n_ref=128.0, intensity=500.0):
    """MainWindow::onAddLight, gui/mainwindow.cpp:229-240: disk of radius 10 facing -y, placed
    1.5 * boundingSphereRadius + 1 above the volume.  The radius scales with the volume so that the
    light subtends the same solid angle at every config size (SURVEY.md section 8d)."""
    R = 0.5 * math.sqrt(sum(e * e for e in extent))
    light = L.AreaLight()
    light.disk.radius = 10.0 * (max(extent) / n_ref)
    light.disk.center = L.Vec3(0.0, 1.5 * R + 1.0, 0.0)
    light.disk.normal = L.Vec3(0.0, -1.0, 0.0)
    light.color = L.Vec3(1.0, 1.0, 1.0)
    light.intensity = intensity
    return light


def constant_env_light(radiance=(0.5, 0.5, 0.5), intensity=1.0):
    """Lights::SetEnvionmentLight(radiance), core/lights/lights.cpp:77-80; default radiance gui/canvas.cpp:11-12."""
    env = L.EnvLight()
    env.tex = 0
    env.defaultRadiance = L.Vec3(*radiance)
    env.intensity = intensity
    env.offset = L.Vec2(0.0, 0.0)
    return env


def _color_table(n=TF_TABLE_SIZE):
    x = np.linspace(0.0, 1.0, n)  # vtkColorTransferFunction::GetTable(0, 1, n, ...) samples both ends
    xs = np.array([c[0] for c in _COLOR_NODES])
    out = np.empty((n, 3), np.float32)
    for ch in range(3):
        out[:, ch] = np.interp(x, xs, np.array([c[1][ch] for c in _COLOR_NODES]))
    return out


def tf_table(kind="default", n=TF_TABLE_SIZE):
    """n x (r, g, b, opacity) float32 table in the layout TransferFunction uploads
    (gui/transferfunction.cpp:17-29).  Opacity ramps (SURVEY.md section 8d):
      default: 0 at 0 rising linearly to 0.5 at 0.1, then flat (stand-in for mainwindow.cpp:51-55)
      thin   : 0.02 * clamp((i - 0.1) / 0.9, 0, 1)
      cloud  : 0.5 * i, white
    """
    x = np.linspace(0.0, 1.0, n)
    t = np.empty((n, 4), np.float32)
    t[:, :3] = _color_table(n)
    if kind == "default":
        t[:, 3] = np.clip(x / 0.1, 0.0, 1.0) * 0.5
    elif kind == "thin":
        t[:, 3] = 0.02 * np.clip((x - 0.1) / 0.9, 0.0, 1.0)
    elif kind == "cloud":
        t[:, :3] = 1.0
        t[:, 3] = 0.5 * x
    else:
        raise ValueError(kind)
    return np.ascontiguousarray(t)


def build_tf_table(opacity_nodes, color_nodes, n=TF_TABLE_SIZE):
    """TransferFunction's composite table from node lists (gui/transferfunction.cpp:17-29) through the C
    ABI (svr_tf_build_table): opacity nodes (x, y[, midpoint, sharpness]), colour nodes (x, r, g, b[,
    midpoint, sharpness]).  Returns (table n x 4 float32, maxOpacity)."""
    import ctypes as C

    lib = L.load()
    on = (L.TfOpacityNode * max(1, len(opacity_nodes)))(*[L.TfOpacityNode(*(tuple(p) + (0.5, 0.0))[:4]) for p in opacity_nodes])
    cn = (L.TfColorNode * max(1, len(color_nodes)))(*[L.TfColorNode(*(tuple(p) + (0.5, 0.0))[:6]) for p in color_nodes])
    table = np.zeros((n, 4), np.float32)
    mx = C.c_float()
    L.check(lib.svr_tf_build_table(on, len(opacity_nodes), cn, len(color_nodes), C.c_void_p(table.ctypes.data), n, C.byref(mx)), "svr_tf_build_table")
    return table, float(mx.value)


def default_tf_nodes():
    """The start-up transfer function of the application (gui/mainwindow.cpp:46-62) as node lists."""
    import ctypes as C

    lib = L.load()
    on, cn = (L.TfOpacityNode * 16)(), (L.TfColorNode * 16)()
    no, nc = C.c_uint32(16), C.c_uint32(16)
    L.check(lib.svr_tf_default_nodes(on, C.byref(no), cn, C.byref(nc)), "svr_tf_default_nodes")
    return ([(o.x, o.y, o.midpoint, o.sharpness) for o in on[: no.value]],
            [(c.x, c.r, c.g, c.b, c.midpoint, c.sharpness) for c in cn[: nc.value]])


def raycast_step_size(spacing=(1.0, 1.0, 1.0)):
    """VolumeReader::GetElementBoundingSphereRadius, core/VolumeReader.cpp:198-201 (passed at gui/canvas.cpp:92)."""
    return 0.5 * math.sqrt(sum(s * s for s in spacing))


def sphere_volume(n, fmt=L.VOXEL_U8):
    """C1 generator on the host (numpy) for CPU-only tests: rho = clamp(1 - r/(0.45 n), 0, 1)."""
    c = 0.5 * n
    ax = (np.arange(n, dtype=np.float32) + 0.5 - c).astype(np.float32)
    z, y, x = np.meshgrid(ax, ax, ax, indexing="ij")
    r = np.sqrt(x * x + y * y + z * z, dtype=np.float32)
    d = np.clip(1.0 - r / np.float32(0.45 * n), 0.0, 1.0).astype(np.float32)
    return encode_voxels(d, fmt)


def encode_voxels(d, fmt):
    if fmt == L.VOXEL_U8:
        return (d * 255.0 + 0.5).astype(np.uint8)
    if fmt == L.VOXEL_U16:
        return (d * 65535.0 + 0.5).astype(np.uint16)
    if fmt == L.VOXEL_F16:
        return d.astype(np.float16)
    return d.astype(np.float32)


VOXEL_DTYPES = {L.VOXEL_U8: np.uint8, L.VOXEL_U16: np.uint16, L.VOXEL_F16: np.float16, L.VOXEL_F32: np.float32}


def host_volume_struct(n_xyz, spacing=(1.0, 1.0, 1.0), max_grad_mag=1.0):
    """cudaVolume as VolumeReader::CreateDeviceVolume + Canvas::LoadVolume leave it, without a
    texture (core/VolumeReader.cpp:174-185; gui/canvas.cpp:31-32).  Used by the CPU oracle."""
    v = L.Volume()
    size = [np.float32(n) * np.float32(s) for n, s in zip(n_xyz, spacing)]
    vmax = [s - s * np.float32(0.5) for s in size]
    v.bbox.vmin = L.Vec3(*[-x for x in vmax])
    v.bbox.vmax = L.Vec3(*vmax)
    v.bbox.invSize = L.Vec3(*[np.float32(1.0) / (x + x) for x in vmax])
    v.densityScale = 1.0
    v.invMaxMagnitude = 1.0 / max_grad_mag
    v.gradientFactor = 0.5
    v.spacing = L.Vec3(*spacing)
    v.invSpacing = L.Vec3(*[1.0 / s for s in spacing])
    v.x_clip = L.Vec2(-1.0, 1.0)
    v.y_clip = L.Vec2(-1.0, 1.0)
    v.z_clip = L.Vec2(-1.0, 1.0)
    return v


# slice orientations (svr_render_slices): the world axes of a pixel row (U) and of a row step (V) per slice normal axis
_SLICE_AXES = {"z": (0, 1), "y": (0, 2), "x": (1, 2)}  # axial, coronal, sagittal


def axis_slice(dims, spacing, axis, index, thickness_voxels=0, count=1, mode="max", window=(0.5, 1.0)):
    """svr_slice_params of an axial (axis "z": U = +x, V = +y), coronal ("y": U = +x, V = +z) or sagittal ("x": U = +y,
    V = +z) slice through voxel `index` of a dims (x, y, z) volume with the given spacing (the box of host_volume_struct,
    centred on the origin).  Pixel centres lie on voxel centres; a stack of `count` slices advances one voxel per slice.  A
    slab of thickness_voxels > 0 voxels is projected with `mode` and a sample spacing of one voxel, centred on the slice."""
    a = "xyz".index(axis)
    iu, iv = _SLICE_AXES[axis]
    sp = [np.float32(x) for x in spacing]
    p = L.SliceParams()
    center = [0.0, 0.0, 0.0]
    center[a] = float((np.float32(index) + np.float32(0.5) - np.float32(0.5) * np.float32(dims[a])) * sp[a])
    p.center[:] = center
    p.axisU[:] = [float(sp[iu]) if i == iu else 0.0 for i in range(3)]
    p.axisV[:] = [float(sp[iv]) if i == iv else 0.0 for i in range(3)]
    p.axisW[:] = [float(sp[a]) if i == a else 0.0 for i in range(3)]
    p.imageW, p.imageH, p.count = int(dims[iu]), int(dims[iv]), int(count)
    p.mode = L.PROJECT_MODES[mode]
    p.thickness = float(np.float32(thickness_voxels) * sp[a])
    p.sampleSpacing = float(sp[a])
    p.windowCenter, p.windowWidth = window
    return p


def oblique_slice(center, normal, up, pixel_size, image_w, image_h, count=1, slice_step=None, thickness=0.0, sample_spacing=None,
                  mode="max", window=(0.5, 1.0)):
    """svr_slice_params of a slice centred on `center` with the given normal: U = pixel_size * normalize(cross(up, normal)),
    V = pixel_size * cross(normalize(normal), normalize(U)), so cross(U, V) points along the normal and V along the part of
    `up` across it.  A stack steps slice_step (default pixel_size) along the normal; a slab of `thickness` world units is
    sampled every sample_spacing (default pixel_size)."""
    n = np.asarray(normal, np.float64)
    n = n / np.linalg.norm(n)
    u = np.cross(np.asarray(up, np.float64), n)
    u = u / np.linalg.norm(u)
    v = np.cross(n, u)
    p = L.SliceParams()
    p.center[:] = [float(x) for x in center]
    p.axisU[:] = [float(x) for x in pixel_size * u]
    p.axisV[:] = [float(x) for x in pixel_size * v]
    p.axisW[:] = [float(x) for x in (pixel_size if slice_step is None else slice_step) * n]
    p.imageW, p.imageH, p.count = int(image_w), int(image_h), int(count)
    p.mode = L.PROJECT_MODES[mode]
    p.thickness = float(thickness)
    p.sampleSpacing = float(pixel_size if sample_spacing is None else sample_spacing)
    p.windowCenter, p.windowWidth = window
    return p


def _curved(layout, image_w, image_h, count, pixel_spacing, station_spacing, up, angle0, angle_step, thickness, sample_spacing, mode,
            window):
    p = L.CurvedParams()
    p.up[:] = [float(x) for x in up]
    p.layout = L.CURVED_LAYOUTS[layout]
    p.imageW, p.imageH, p.count = int(image_w), int(image_h), int(count)
    p.mode = L.PROJECT_MODES[mode]
    p.pixelSpacing, p.stationSpacing = float(pixel_spacing), float(station_spacing)
    p.angle0, p.angleStep = float(angle0), float(angle_step)
    p.thickness = float(thickness)
    p.sampleSpacing = float(pixel_spacing if sample_spacing is None else sample_spacing)
    p.windowCenter, p.windowWidth = window
    return p


def straightened_curve(image_w, n_stations, pixel_spacing, station_spacing=None, up=(0.0, 0.0, 1.0), count=1, angle0=0.0,
                       angle_step=None, thickness=0.0, sample_spacing=None, mode="max", window=(0.5, 1.0)):
    """svr_curved_params of a straightened CPR (svr_render_curved): one row per station (n_stations rows, station_spacing apart
    along the curve, default pixel_spacing), image_w columns pixel_spacing apart across it.  count > 1 is the rotational stack,
    image j at angle0 + j angle_step about the tangent (default a full turn over the count).  A slab of `thickness` world units
    across the image plane is sampled every sample_spacing (default pixel_spacing)."""
    step = 2.0 * math.pi / count if angle_step is None else angle_step
    return _curved("straightened", image_w, n_stations, count, pixel_spacing, pixel_spacing if station_spacing is None else station_spacing,
                   up, angle0, step, thickness, sample_spacing, mode, window)


def curve_cross_sections(image_w, image_h, count, pixel_spacing, station_spacing, up=(0.0, 0.0, 1.0), angle=0.0, thickness=0.0,
                         sample_spacing=None, mode="max", window=(0.5, 1.0)):
    """svr_curved_params of `count` cross-sections (svr_render_curved): image j is the image_w x image_h plane perpendicular to
    the curve at station j (station_spacing apart), pixel_spacing between pixels, its columns along the frame's
    cos(angle) r + sin(angle) b.  A slab of `thickness` world units along the tangent is sampled every sample_spacing."""
    return _curved("cross", image_w, image_h, count, pixel_spacing, station_spacing, up, angle, 0.0, thickness, sample_spacing, mode, window)


def polyline_length(points):
    """Arc length of the polyline `points` ((n, 3)), in float64."""
    p = np.asarray(points, np.float64).reshape(-1, 3)
    return float(np.linalg.norm(np.diff(p, axis=0), axis=1).sum())


def curve_frames(points, up, station_spacing, n):
    """The library's frames of n stations of the polyline `points` (svr_curve_frames; no GPU): (n, 4, 4) float32, rows
    (c, valid), (t, 0), (r, 0), (b, 0).  The world position of CPR pixel column x of a straightened row y at angle theta is
    c_y + (x + 1/2 - W/2) pixelSpacing (cos(theta) r_y + sin(theta) b_y)."""
    import ctypes as C

    pts = np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1, 3))
    upv = np.ascontiguousarray(np.asarray(up, np.float32).reshape(3))
    out = np.zeros((int(n), 4, 4), np.float32)
    lib = L.load()
    L.check(lib.svr_curve_frames(pts.ctypes.data, len(pts), upv.ctypes.data, C.c_float(station_spacing), int(n), out.ctypes.data),
            "svr_curve_frames")
    return out


# label maps (svr_render_labels, svr_render_label_slices): the levels of the generated CT's skin, soft tissue and bone, on its
# normalised values (svr_generate_volume writes shells at 0.25, 0.45 and 0.85)
CT_LABEL_LEVELS = (0.15, 0.35, 0.7)


def label_table(colors):
    """svr_label_params from {label id: (r, g, b, a)}; every other id is hidden (all zero).  a = 0 hides a label; in 2D
    overlays a is the fill opacity."""
    p = L.LabelParams()
    for lab, rgba in colors.items():
        if not 0 <= int(lab) <= 255:
            raise ValueError(f"label_table: label id {lab} is outside 0..255")
        p.color[int(lab)][:] = [float(np.float32(c)) for c in rgba]
    return p


def label_palette(n, alpha=1.0):
    """A deterministic colour per label id 1..n, {id: (r, g, b, alpha)}, distinct for every id (the red byte (73 id + 91) mod 256
    alone differs between any two ids).  Each channel is byte / 255 in float32, as tools/svr_headless.cpp computes it."""
    out = {}
    for lab in range(1, int(n) + 1):
        rgb = ((73 * lab + 91) & 255, (151 * lab + 17) & 255, (29 * lab + 193) & 255)
        out[lab] = tuple(float(np.float32(c) / np.float32(255)) for c in rgb) + (float(alpha),)
    return out


def labels_from_thresholds(volume, levels):
    """u8 labels of a grey volume: the number of `levels` (increasing) at or below each voxel's value, so that
    levels = CT_LABEL_LEVELS gives 1 skin, 2 soft tissue and 3 bone on the generated CT.  Values are compared as the volume
    texture returns them: unsigned integer voxels over their type's maximum (normalised reads), floats as stored."""
    v = np.asarray(volume)
    if np.issubdtype(v.dtype, np.unsignedinteger):
        v = v.astype(np.float32) / np.float32(np.iinfo(v.dtype).max)
    out = np.zeros(v.shape, np.uint8)
    for level in levels:
        out += (v >= np.float32(level)).astype(np.uint8)
    return out


@dataclass
class Config:
    """One BASELINE.json configuration."""
    name: str
    n: int                 # volume edge
    fmt: int               # voxel format
    gen: int               # svr_volume_kind
    width: int
    height: int
    tf: str
    trace_depth: int = 1
    spp: int = 16
    env: bool = False
    gen_seed: int = 1234
    notes: str = ""
    extent: tuple = field(init=False)

    def __post_init__(self):
        self.extent = (float(self.n),) * 3

    @property
    def voxel_bytes(self):
        return L.VOXEL_BYTES[self.fmt]


CONFIGS = {
    "C1": Config("C1", 128, L.VOXEL_U8, L.GEN_SPHERE, 512, 512, "default", 1, 16),
    "C2": Config("C2", 256, L.VOXEL_U8, L.GEN_CT, 1024, 1024, "thin", 1, 1),
    "C3": Config("C3", 512, L.VOXEL_U16, L.GEN_CT, 1920, 1080, "default", 1, 256, env=True),
    "C4": Config("C4", 1024, L.VOXEL_F16, L.GEN_CLOUD, 1920, 1080, "cloud", 32, 512, gen_seed=42),
    "C5": Config("C5", 2048, L.VOXEL_U16, L.GEN_CT, 3840, 2160, "default", 1, 1024, env=True),
}


def split_samples(total, world_size):
    """Sample-index ranges per rank: rank r renders [first, first+count) (SURVEY.md section 8e)."""
    base, rem = divmod(total, world_size)
    out, first = [], 0
    for r in range(world_size):
        cnt = base + (1 if r < rem else 0)
        out.append((first, cnt))
        first += cnt
    return out


def split_rows(height, world_size, align=4):
    """Row ranges per rank for the ray caster's image-tile split, aligned to the warp tile height."""
    rows = (height + align - 1) // align
    base, rem = divmod(rows, world_size)
    out, y = [], 0
    for r in range(world_size):
        cnt = (base + (1 if r < rem else 0)) * align
        y1 = min(height, y + cnt)
        out.append((y, y1))
        y = y1
    return out
