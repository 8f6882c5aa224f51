"""ctypes binding of libsvr_b200.so (include/svr_render.h, include/svr_types.h).

The structures below are the plain-C mirrors of the reference's scene PODs (core/cuda_volume.h:111-121,
core/cuda_camera.h:98-106, ...); sizes and offsets are asserted at import so a drift from the C
headers fails loudly.  There is NO fallback: if the CUDA library is missing, importing this module
raises.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SVR_B200_LIB selects an alternative build of the same library (A/B experiments with compiler flags)
LIB_PATH = os.environ.get("SVR_B200_LIB") or os.path.join(_HERE, "libsvr_b200.so")


class Vec2(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float)]


class Vec3(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]

    def __init__(self, x=0.0, y=0.0, z=0.0):
        super().__init__(float(x), float(y), float(z))

    def tuple(self):
        return (self.x, self.y, self.z)


class Vec4(C.Structure):
    _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float), ("w", C.c_float)]


class BBox(C.Structure):
    _fields_ = [("vmin", Vec3), ("vmax", Vec3), ("invSize", Vec3)]


class Volume(C.Structure):  # cudaVolume
    _fields_ = [
        ("bbox", BBox),
        ("_pad0", C.c_uint32),
        ("tex", C.c_ulonglong),
        ("densityScale", C.c_float),
        ("invMaxMagnitude", C.c_float),
        ("gradientFactor", C.c_float),
        ("spacing", Vec3),
        ("invSpacing", Vec3),
        ("x_clip", Vec2),
        ("y_clip", Vec2),
        ("z_clip", Vec2),
        ("_pad1", C.c_uint32),
    ]


class TransferFunction(C.Structure):  # cudaTransferFunction
    _fields_ = [("tex", C.c_ulonglong), ("maxOpacity", C.c_float), ("_pad0", C.c_uint32)]


class Camera(C.Structure):  # cudaCamera
    _fields_ = [
        ("imageW", C.c_uint32),
        ("imageH", C.c_uint32),
        ("exposure", C.c_float),
        ("apeture", C.c_float),
        ("focalLength", C.c_float),
        ("aspectRatio", C.c_float),
        ("tanFovxOverTwo", C.c_float),
        ("pos", Vec3),
        ("u", Vec3),
        ("v", Vec3),
        ("w", Vec3),
    ]


class Disk(C.Structure):  # cudaDisk
    _fields_ = [("radius", C.c_float), ("center", Vec3), ("normal", Vec3)]


class AreaLight(C.Structure):  # cudaAreaLight
    _fields_ = [("disk", Disk), ("color", Vec3), ("intensity", C.c_float)]


class EnvLight(C.Structure):  # cudaEnvironmentLight
    _fields_ = [("tex", C.c_ulonglong), ("defaultRadiance", Vec3), ("intensity", C.c_float), ("offset", Vec2)]


class RenderParams(C.Structure):  # RenderParams
    _fields_ = [("traceDepth", C.c_uint32), ("frameNo", C.c_uint32), ("hdrBuffer", C.c_void_p)]


assert C.sizeof(Vec3) == 12 and C.sizeof(BBox) == 36
assert C.sizeof(Volume) == 112 and Volume.tex.offset == 40 and Volume.spacing.offset == 60 and Volume.z_clip.offset == 100
assert C.sizeof(TransferFunction) == 16 and TransferFunction.maxOpacity.offset == 8
assert C.sizeof(Camera) == 76 and Camera.pos.offset == 28 and Camera.w.offset == 64
assert C.sizeof(Disk) == 28 and C.sizeof(AreaLight) == 44
assert C.sizeof(EnvLight) == 32 and EnvLight.intensity.offset == 20
assert C.sizeof(RenderParams) == 16 and RenderParams.hdrBuffer.offset == 8


class DenoiseParams(C.Structure):  # svr_denoise_params
    _fields_ = [("iterations", C.c_uint32), ("sigmaLuminance", C.c_float), ("sigmaNormal", C.c_float), ("sigmaDepth", C.c_float),
                ("sigmaCoverage", C.c_float)]


assert C.sizeof(DenoiseParams) == 20


class ProjectionParams(C.Structure):  # svr_projection_params
    _fields_ = [("mode", C.c_int32), ("stepSize", C.c_float), ("windowCenter", C.c_float), ("windowWidth", C.c_float)]


assert C.sizeof(ProjectionParams) == 16
# enum svr_projection_mode
PROJECT_MAX, PROJECT_MIN, PROJECT_MEAN = range(3)
PROJECT_MODES = {"max": PROJECT_MAX, "min": PROJECT_MIN, "mean": PROJECT_MEAN}


class IsosurfaceParams(C.Structure):  # svr_isosurface_params
    _fields_ = [("isoValue", C.c_float), ("stepSize", C.c_float), ("color", C.c_float * 3)]


assert C.sizeof(IsosurfaceParams) == 20


class SliceParams(C.Structure):  # svr_slice_params
    _fields_ = [("center", C.c_float * 3), ("axisU", C.c_float * 3), ("axisV", C.c_float * 3), ("axisW", C.c_float * 3),
                ("imageW", C.c_uint32), ("imageH", C.c_uint32), ("count", C.c_uint32), ("mode", C.c_int32), ("thickness", C.c_float),
                ("sampleSpacing", C.c_float), ("windowCenter", C.c_float), ("windowWidth", C.c_float)]


assert C.sizeof(SliceParams) == 80


class CurvedParams(C.Structure):  # svr_curved_params
    _fields_ = [("up", C.c_float * 3), ("layout", C.c_int32), ("imageW", C.c_uint32), ("imageH", C.c_uint32), ("count", C.c_uint32),
                ("mode", C.c_int32), ("pixelSpacing", C.c_float), ("stationSpacing", C.c_float), ("angle0", C.c_float),
                ("angleStep", C.c_float), ("thickness", C.c_float), ("sampleSpacing", C.c_float), ("windowCenter", C.c_float),
                ("windowWidth", C.c_float)]


assert C.sizeof(CurvedParams) == 64

class LabelParams(C.Structure):  # svr_label_params
    _fields_ = [("color", (C.c_float * 4) * 256)]


assert C.sizeof(LabelParams) == 4096

# enum svr_curved_layout
CURVED_STRAIGHTENED, CURVED_CROSS = 0, 1
CURVED_LAYOUTS = {"straightened": CURVED_STRAIGHTENED, "cross": CURVED_CROSS}

# enum svr_option
(OPT_PT_MODE, OPT_SHADOW_ESTIMATOR, OPT_ENV_ENABLED, OPT_MACROCELL_SIZE, OPT_RC_SKIP, OPT_SEED, OPT_COUNTERS,
 OPT_PT_BLOCK, OPT_RC_BLOCK, OPT_PT_KERNEL, OPT_PT_ROUNDS, OPT_LEAP, OPT_PT_ENTRY_CACHE, OPT_PT_WARP_PIXELS,
 OPT_PT_WARP_MIN_SPP, OPT_PT_QUEUE_MIN_DEPTH, OPT_SETUP_SYNC, OPT_PT_LIGHT_CULL, OPT_PT_PROFILE, OPT_PT_REFILL, OPT_PT_POOL_PIXELS, OPT_ENV_NEE, OPT_PT_BLOCK_SPLIT, OPT_PT_PIXEL_CACHE,
 OPT_FUSED_UPLOAD, OPT_PT_LOOKAHEAD, OPT_PT_DENOISE) = range(27)
# enum svr_voxel_format
VOXEL_U8, VOXEL_U16, VOXEL_F16, VOXEL_F32 = range(4)
VOXEL_BYTES = {VOXEL_U8: 1, VOXEL_U16: 2, VOXEL_F16: 2, VOXEL_F32: 4}
# enum svr_volume_kind
GEN_SPHERE, GEN_CT, GEN_CLOUD = range(3)
# enum svr_counter
CNT_TRACK_TAPS, CNT_SHADOW_TAPS, CNT_SHADE_TAPS, CNT_TF_LOOKUPS, CNT_SCATTERS, CNT_PATHS, CNT_CELLS, CNT_STEPS, CNT_SKIPPED = range(9)
CNT_NAMES = ["track_taps", "shadow_taps", "shade_taps", "tf_lookups", "scatters", "paths", "cells", "steps", "skipped"]

# every symbol include/svr_render.h declares: (name, restype, argtypes)
_P = C.c_void_p
SIGNATURES = [
    # Part 1 -- the reference boundary (pathtracer.h:17-24, raycasting.h:8)
    ("render_pathtracer", None, [_P, C.POINTER(RenderParams)]),
    ("setup_volume", None, [C.POINTER(Volume)]),
    ("setup_transferfunction", None, [C.POINTER(TransferFunction)]),
    ("setup_camera", None, [C.POINTER(Camera)]),
    ("setup_env_lights", None, [C.POINTER(EnvLight)]),
    ("setup_area_lights", None, [C.POINTER(AreaLight), C.c_uint32]),
    ("render_raycasting", None, [_P, C.POINTER(Volume), C.POINTER(TransferFunction), C.POINTER(Camera), C.c_float]),
    # Part 2 -- headless extension
    ("svr_version", C.c_int, []),
    ("svr_last_error", C.c_char_p, []),
    ("svr_set_stream", C.c_int, [_P]),
    ("svr_set_device", C.c_int, [C.c_int]),
    ("svr_set_option", C.c_int, [C.c_int, C.c_int]),
    ("svr_get_option", C.c_int, [C.c_int]),
    ("svr_render_pathtracer_spp", C.c_int, [_P, C.POINTER(RenderParams), C.c_uint32]),
    ("svr_pathtracer_accumulate", C.c_int, [_P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int]),
    ("svr_pathtracer_accumulate_bands", C.c_int, [_P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32)]),
    ("svr_pathtracer_resolve", C.c_int, [_P, _P, _P]),
    ("svr_pathtracer_accumulate_adaptive", C.c_int, [_P, _P, _P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float,
                                                     C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    ("svr_pathtracer_guides", C.c_int, [_P, _P, C.c_uint32]),
    ("svr_denoise_defaults", C.c_int, [C.POINTER(DenoiseParams)]),
    ("svr_pathtracer_denoise", C.c_int, [_P, _P, _P, _P, _P, _P, C.POINTER(DenoiseParams)]),
    ("svr_pathtracer_set_denoise_params", C.c_int, [C.POINTER(DenoiseParams)]),
    ("svr_render_raycasting_f32", C.c_int, [_P, C.POINTER(Volume), C.POINTER(TransferFunction), C.POINTER(Camera), C.c_float]),
    ("svr_render_raycasting_rows", C.c_int, [_P, _P, C.POINTER(Volume), C.POINTER(TransferFunction), C.POINTER(Camera), C.c_float, C.c_uint32, C.c_uint32]),
    ("svr_volume_create", C.c_int, [C.POINTER(Volume), _P, C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.c_float]),
    ("svr_volume_destroy", C.c_int, [C.POINTER(Volume)]),
    ("svr_render_raycasting_bands", C.c_int, [_P, _P, C.POINTER(Volume), C.POINTER(TransferFunction), C.POINTER(Camera), C.c_float, C.c_uint32, C.c_uint32,
                                            C.POINTER(C.c_uint32)]),
    ("svr_volume_upload", C.c_int, [C.POINTER(Volume), _P, C.c_int]),
    ("svr_stage_alloc", C.c_int, [C.POINTER(C.c_void_p), C.c_uint64]),
    ("svr_stage_free", C.c_int, [_P]),
    ("svr_stage_export", C.c_int, [_P, C.POINTER(C.c_ubyte * 64)]),
    ("svr_stage_import", C.c_int, [C.POINTER(C.c_ubyte * 64), C.POINTER(C.c_void_p)]),
    ("svr_stage_release", C.c_int, [_P]),
    ("svr_stage_copy", C.c_int, [_P, _P, C.c_uint64, _P]),
    ("svr_peer_signal", C.c_int, [_P]),
    ("svr_peer_wait", C.c_int, [_P, C.c_uint32, C.c_uint32]),
    ("svr_volume_invalidate_cache", C.c_int, []),
    ("svr_tf_create", C.c_int, [C.POINTER(TransferFunction), _P, C.c_uint32]),
    ("svr_tf_destroy", C.c_int, [C.POINTER(TransferFunction)]),
    ("svr_tf_upload", C.c_int, [C.POINTER(TransferFunction), _P, C.c_uint32]),
    ("svr_env_create", C.c_int, [C.POINTER(EnvLight), _P, C.c_uint32, C.c_uint32]),
    ("svr_env_destroy", C.c_int, [C.POINTER(EnvLight)]),
    ("svr_generate_volume", C.c_int, [_P, C.c_int, C.c_int, C.c_uint32, C.c_uint32]),
    ("svr_max_gradient_magnitude", C.c_int, [_P, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float)]),
    ("svr_counters_reset", C.c_int, []),
    ("svr_counters_read", C.c_int, [C.POINTER(C.c_uint64), C.c_uint32]),
    ("svr_launch_count", C.c_uint64, []),
    ("svr_fused_upload_count", C.c_uint64, []),
    ("svr_lookahead_batch_count", C.c_uint64, []),
    ("svr_microbench_taps", C.c_int, [C.POINTER(Volume), C.c_int, C.c_uint32, C.c_uint32, _P, C.POINTER(C.c_uint64)]),
    ("svr_layout_brick", C.c_int, [_P, _P, C.c_uint32]),
    ("svr_microbench_soft_taps", C.c_int, [_P, C.c_uint32, C.c_int, C.c_int, C.c_uint32, C.c_uint32, _P, C.POINTER(C.c_uint64)]),
    ("svr_debug_sample_volume", C.c_int, [C.POINTER(Volume), _P, C.c_uint32, _P]),
    ("svr_debug_sample_tf", C.c_int, [C.POINTER(TransferFunction), _P, C.c_uint32, _P]),
    ("svr_grid_info", C.c_int, [C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    ("svr_grid_copy", C.c_int, [_P, _P]),
    ("svr_render_projection", C.c_int, [_P, _P, C.POINTER(Volume), C.POINTER(Camera), C.POINTER(ProjectionParams), C.c_uint32, C.c_uint32,
                                        C.POINTER(C.c_uint32)]),
    ("svr_render_isosurface", C.c_int, [_P, _P, C.POINTER(Volume), C.POINTER(Camera), C.POINTER(IsosurfaceParams), C.c_uint32, C.c_uint32,
                                        C.POINTER(C.c_uint32)]),
    ("svr_render_slices", C.c_int, [_P, _P, C.POINTER(Volume), C.POINTER(SliceParams)]),
    ("svr_curve_frames", C.c_int, [_P, C.c_uint32, _P, C.c_float, C.c_uint32, _P]),
    ("svr_render_curved", C.c_int, [_P, _P, C.POINTER(Volume), C.POINTER(CurvedParams), _P, C.c_uint32]),
    ("svr_render_labels", C.c_int, [_P, _P, _P, C.POINTER(Volume), C.POINTER(Camera), C.POINTER(LabelParams), C.c_float, C.c_uint32, C.c_uint32,
                                    C.POINTER(C.c_uint32)]),
    ("svr_render_label_slices", C.c_int, [_P, _P, C.POINTER(Volume), C.POINTER(SliceParams), C.POINTER(LabelParams), C.c_int]),
    ("svr_labels_create", C.c_int, [C.POINTER(Volume), _P, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float]),
]


# ---- include/svr_volume_io.h
MET_UCHAR, MET_CHAR, MET_USHORT, MET_SHORT, MET_UINT, MET_INT, MET_FLOAT, MET_DOUBLE = range(8)


class MetaImageHeader(C.Structure):  # svr_metaimage_header
    _fields_ = [
        ("ndims", C.c_uint32),
        ("dim", C.c_uint32 * 3),
        ("spacing", C.c_float * 3),
        ("element_type", C.c_int32),
        ("channels", C.c_uint32),
        ("msb", C.c_int32),
        ("compressed", C.c_int32),
        ("header_size", C.c_int64),
        ("compressed_size", C.c_uint64),
        ("data_offset", C.c_uint64),
        ("data_file", C.c_char * 1024),
    ]


class VolumeStats(C.Structure):  # svr_volume_stats
    _fields_ = [
        ("dim", C.c_uint32 * 3),
        ("spacing", C.c_float * 3),
        ("data_min", C.c_float),
        ("data_max", C.c_float),
        ("max_gradient_magnitude", C.c_float),
        ("histogram_bins", C.c_uint32),
        ("histogram_total", C.c_uint64),
    ]


SIGNATURES_IO = [
    ("svr_metaimage_read_header", C.c_int, [C.c_char_p, C.POINTER(MetaImageHeader)]),
    ("svr_volume_from_raw", C.c_int, [_P, C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_float,
                                      C.POINTER(Volume), C.POINTER(VolumeStats), _P, C.c_uint32]),
    ("svr_volume_load_metaimage", C.c_int, [C.c_char_p, C.POINTER(Volume), C.POINTER(VolumeStats), _P, C.c_uint32]),
    ("svr_labels_load_metaimage", C.c_int, [C.c_char_p, C.POINTER(Volume), C.POINTER(C.c_uint32)]),
    ("svr_volume_download", C.c_int, [C.POINTER(Volume), _P, C.c_uint64]),
]


# ---- include/svr_tf_io.h
class TfOpacityNode(C.Structure):  # svr_tf_opacity_node: vtkPiecewiseFunction node, 4 doubles
    _fields_ = [("x", C.c_double), ("y", C.c_double), ("midpoint", C.c_double), ("sharpness", C.c_double)]


class TfColorNode(C.Structure):  # svr_tf_color_node: vtkColorTransferFunction node, 6 doubles
    _fields_ = [("x", C.c_double), ("r", C.c_double), ("g", C.c_double), ("b", C.c_double), ("midpoint", C.c_double), ("sharpness", C.c_double)]


SIGNATURES_TF = [
    ("svr_tf_build_table", C.c_int, [C.POINTER(TfOpacityNode), C.c_uint32, C.POINTER(TfColorNode), C.c_uint32, _P, C.c_uint32, C.POINTER(C.c_float)]),
    ("svr_tf_default_nodes", C.c_int, [C.POINTER(TfOpacityNode), C.POINTER(C.c_uint32), C.POINTER(TfColorNode), C.POINTER(C.c_uint32)]),
    ("svr_tf_file_write", C.c_int, [C.c_char_p, C.POINTER(TfOpacityNode), C.c_uint32, C.POINTER(TfColorNode), C.c_uint32]),
    ("svr_tf_file_read", C.c_int, [C.c_char_p, C.POINTER(TfOpacityNode), C.POINTER(C.c_uint32), C.POINTER(TfColorNode), C.POINTER(C.c_uint32)]),
]


# ---- include/svr_env_io.h
SIGNATURES_ENV = [
    ("svr_hdr_read", C.c_int, [C.c_char_p, _P, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    ("svr_env_load_hdr", C.c_int, [C.c_char_p, C.POINTER(EnvLight)]),
    ("svr_env_sampler_copy", C.c_int, [_P, _P, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
]


# ---- include/svr_canvas.h
class View(C.Structure):  # svr_view: the camera-related members of Canvas (gui/canvas.h:210-217)
    _fields_ = [("viewMat", C.c_float * 16), ("eyeDist", C.c_float), ("translate", C.c_float * 2), ("fov", C.c_float),
                ("apeture", C.c_float), ("focalLength", C.c_float), ("exposure", C.c_float), ("mouseStart", C.c_float * 2)]


BUTTON_LEFT, BUTTON_MID = 1, 4
KEY_LEFT, KEY_RIGHT, KEY_DOWN = 0, 1, 2
RENDER_MODE_PATHTRACER, RENDER_MODE_RAYCASTING, RENDER_MODE_PROJECTION = 0, 1, 2
_F3 = C.POINTER(C.c_float * 3)
_V = C.POINTER(View)

SIGNATURES_CANVAS = [
    ("svr_view_init", None, [_V]),
    ("svr_view_zoom_to_extent", None, [_V, _F3]),
    ("svr_view_reset", None, [_V, _F3]),
    ("svr_view_rotate", None, [_V, C.c_float, C.c_float, C.c_float, C.c_float]),
    ("svr_view_pixel_to_view", None, [C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.POINTER(C.c_float * 2)]),
    ("svr_view_mouse_press", C.c_int, [_V, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_int]),
    ("svr_view_mouse_move", C.c_int, [_V, C.c_uint32, C.c_uint32, C.c_float, C.c_float, C.c_int, _F3]),
    ("svr_view_wheel", C.c_int, [_V, C.c_int, _F3]),
    ("svr_view_key", C.c_int, [_V, C.c_int]),
    ("svr_view_camera", None, [_V, C.c_uint32, C.c_uint32, C.POINTER(Camera)]),
    ("svr_canvas_create", _P, [C.c_uint32, C.c_uint32]),
    ("svr_canvas_destroy", None, [_P]),
    ("svr_canvas_load_volume", C.c_int, [_P, C.c_char_p]),
    ("svr_canvas_set_volume", C.c_int, [_P, C.POINTER(Volume), _F3, C.c_float]),
    ("svr_canvas_set_transfer_function", C.c_int, [_P, C.POINTER(TransferFunction)]),
    ("svr_canvas_set_density_scale", C.c_int, [_P, C.c_double]),
    ("svr_canvas_set_gradient_factor", C.c_int, [_P, C.c_double]),
    ("svr_canvas_set_scatter_times", C.c_int, [_P, C.c_double]),
    ("svr_canvas_set_render_mode", C.c_int, [_P, C.c_int]),
    ("svr_canvas_set_env_background", C.c_int, [_P, C.c_float, C.c_float, C.c_float]),
    ("svr_canvas_set_env_map", C.c_int, [_P, C.c_char_p]),
    ("svr_canvas_set_env_offset", C.c_int, [_P, C.c_float, C.c_float]),
    ("svr_canvas_set_env_intensity", C.c_int, [_P, C.c_float]),
    ("svr_canvas_set_area_lights", C.c_int, [_P, C.POINTER(AreaLight), C.c_uint32]),
    ("svr_canvas_set_fov", C.c_int, [_P, C.c_float]),
    ("svr_canvas_set_apeture", C.c_int, [_P, C.c_float]),
    ("svr_canvas_set_focal_length", C.c_int, [_P, C.c_float]),
    ("svr_canvas_set_exposure", C.c_int, [_P, C.c_float]),
    ("svr_canvas_set_clip_plane", C.c_int, [_P, C.c_int, C.c_double, C.c_double]),
    ("svr_canvas_set_projection", C.c_int, [_P, C.c_int, C.c_float, C.c_float]),
    ("svr_canvas_mouse_press", C.c_int, [_P, C.c_float, C.c_float, C.c_int]),
    ("svr_canvas_mouse_move", C.c_int, [_P, C.c_float, C.c_float, C.c_int]),
    ("svr_canvas_wheel", C.c_int, [_P, C.c_int]),
    ("svr_canvas_key", C.c_int, [_P, C.c_int]),
    ("svr_canvas_paint", C.c_int, [_P]),
    ("svr_canvas_paint_into", C.c_int, [_P, _P]),
    ("svr_canvas_set_immediate_repaint", None, [_P, C.c_int]),
    ("svr_canvas_image", _P, [_P]),
    ("svr_canvas_hdr", _P, [_P]),
    ("svr_canvas_read_image", C.c_int, [_P, _P]),
    ("svr_canvas_frame_no", C.c_uint32, [_P]),
    ("svr_canvas_paint_count", C.c_uint64, [_P]),
    ("svr_canvas_get_view", None, [_P, _V]),
    ("svr_canvas_get_camera", None, [_P, C.POINTER(Camera)]),
    ("svr_canvas_get_volume", None, [_P, C.POINTER(Volume)]),
    ("svr_canvas_get_env_light", None, [_P, C.POINTER(EnvLight)]),
]


class SvrError(RuntimeError):
    pass


_lib = None


def load():
    """Load libsvr_b200.so and bind every declared symbol.  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `make lib` (or __graft_entry__.build()). "
            "sunvolumerender_b200 has no CPU or PyTorch fallback."
        )
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_LOCAL)
    for name, res, args in SIGNATURES + SIGNATURES_IO + SIGNATURES_TF + SIGNATURES_ENV + SIGNATURES_CANVAS:
        fn = getattr(lib, name)  # AttributeError if a declared symbol is not exported
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().svr_last_error()
        raise SvrError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
