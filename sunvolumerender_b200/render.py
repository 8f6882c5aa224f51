"""Python host side of the render path: a thin mirror of what gui/canvas.cpp does with the seven
entry points (SetUp* -> setup_*, paintGL -> render_*), on top of the C ABI.  torch is used only for
device buffers, streams and torch.distributed; every pixel is produced by libsvr_b200.so.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L
from . import scene as S


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


class Renderer:
    """One scene on one GPU (the library, like the reference, holds one scene per process)."""

    def __init__(self, device=0):
        if not torch.cuda.is_available():
            raise RuntimeError("sunvolumerender_b200 needs a CUDA device; there is no CPU path")
        self.lib = L.load()
        self.device = torch.device("cuda", device)
        torch.cuda.set_device(self.device)
        L.check(self.lib.svr_set_device(device), "svr_set_device")
        self.sync_stream()
        self.volume = None
        self.labels = None
        self.tf = None
        self._tf_size = 0
        self.camera = None
        self.env = None
        self.lights = []
        self.hdr = None
        self.img = None
        self.frame_no = 0

    # ---- plumbing
    def sync_stream(self):
        L.check(self.lib.svr_set_stream(C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)), "svr_set_stream")

    def set_option(self, key, value):
        L.check(self.lib.svr_set_option(key, int(value)), "svr_set_option")

    def get_option(self, key):
        return self.lib.svr_get_option(key)

    def counters(self, reset=False):
        buf = (C.c_uint64 * 16)()
        L.check(self.lib.svr_counters_read(buf, 16), "svr_counters_read")
        out = {name: int(buf[i]) for i, name in enumerate(L.CNT_NAMES)}
        if reset:
            L.check(self.lib.svr_counters_reset(), "svr_counters_reset")
        return out

    def reset_counters(self):
        L.check(self.lib.svr_counters_reset(), "svr_counters_reset")

    def launch_count(self):
        return int(self.lib.svr_launch_count())

    # ---- resources (VolumeReader / TransferFunction / Lights stand-ins)
    def generate_volume(self, kind, fmt, n, seed=1234):
        """Synthetic volume in device memory (x fastest), as a torch uint8 byte tensor."""
        nbytes = n * n * n * L.VOXEL_BYTES[fmt]
        buf = torch.empty(nbytes, dtype=torch.uint8, device=self.device)
        L.check(self.lib.svr_generate_volume(_ptr(buf), kind, fmt, n, seed), "svr_generate_volume")
        return buf

    def load_volume(self, data, fmt, dims, spacing=(1.0, 1.0, 1.0), max_grad_mag=0.0):
        """Canvas::LoadVolume: upload voxels (host numpy array or device byte tensor), bind the
        texture, publish with setup_volume (gui/canvas.cpp:27-41)."""
        self.free_volume()
        vol = L.Volume()
        nx, ny, nz = dims
        if isinstance(data, torch.Tensor):
            on_device = 1 if data.is_cuda else 0
            ptr = _ptr(data)
        else:
            data = np.ascontiguousarray(data)
            on_device = 0
            ptr = C.c_void_p(data.ctypes.data)
        L.check(
            self.lib.svr_volume_create(C.byref(vol), ptr, on_device, fmt, nx, ny, nz, spacing[0], spacing[1], spacing[2], max_grad_mag),
            "svr_volume_create",
        )
        self.volume = vol
        self._vol_nbytes = nx * ny * nz * L.VOXEL_BYTES[fmt]
        self.lib.setup_volume(C.byref(vol))
        return vol

    def load_metaimage(self, path, histogram_capacity=65536):
        """Canvas::LoadVolume on a MetaImage file (gui/canvas.cpp:27-41 -> core/VolumeReader.cpp:13-94):
        returns (stats, histogram)."""
        self.free_volume()
        vol, stats = L.Volume(), L.VolumeStats()
        hist = np.zeros(histogram_capacity, np.uint32)
        L.check(self.lib.svr_volume_load_metaimage(str(path).encode(), C.byref(vol), C.byref(stats), C.c_void_p(hist.ctypes.data), histogram_capacity),
                "svr_volume_load_metaimage")
        self.volume = vol
        self.lib.setup_volume(C.byref(vol))
        self.frame_no = 0
        return stats, hist[: min(stats.histogram_bins, histogram_capacity)]

    def load_raw(self, data, met_type, dims, spacing=(1.0, 1.0, 1.0), msb=False, histogram_capacity=65536):
        """The preprocessing half of VolumeReader::Read for voxels already in host memory (any MetaImage element type)."""
        self.free_volume()
        data = np.ascontiguousarray(data)
        vol, stats = L.Volume(), L.VolumeStats()
        hist = np.zeros(histogram_capacity, np.uint32)
        L.check(self.lib.svr_volume_from_raw(C.c_void_p(data.ctypes.data), met_type, 1 if msb else 0, dims[0], dims[1], dims[2],
                                             spacing[0], spacing[1], spacing[2], C.byref(vol), C.byref(stats), C.c_void_p(hist.ctypes.data), histogram_capacity),
                "svr_volume_from_raw")
        self.volume = vol
        self.lib.setup_volume(C.byref(vol))
        self.frame_no = 0
        return stats, hist[: min(stats.histogram_bins, histogram_capacity)]

    def download_volume(self, dims, dtype=np.uint16):
        out = np.zeros((dims[2], dims[1], dims[0]), dtype)
        L.check(self.lib.svr_volume_download(C.byref(self.volume), C.c_void_p(out.ctypes.data), out.nbytes), "svr_volume_download")
        return out

    def upload_volume(self, data):
        """Replace the voxels of the bound volume (same dims/format) from a host numpy array, a pinned
        host tensor or a device tensor."""
        if isinstance(data, torch.Tensor):
            on_device, ptr = (1 if data.is_cuda else 0), _ptr(data)
        else:
            data = np.ascontiguousarray(data)
            on_device, ptr = 0, C.c_void_p(data.ctypes.data)
        L.check(self.lib.svr_volume_upload(C.byref(self.volume), ptr, on_device), "svr_volume_upload")
        self.lib.setup_volume(C.byref(self.volume))
        self.frame_no = 0

    def volume_nbytes(self):
        """Size in bytes of the bound volume's voxels (volumes made by load_volume)."""
        if getattr(self, "_vol_nbytes", None) is None:
            raise RuntimeError("volume_nbytes: no volume loaded with load_volume")
        return self._vol_nbytes

    def free_volume(self):
        if self.volume is not None:
            L.check(self.lib.svr_volume_destroy(C.byref(self.volume)), "svr_volume_destroy")
            self.volume = None

    def set_volume_params(self, density_scale=None, gradient_factor=None, x_clip=None, y_clip=None, z_clip=None):
        """Canvas::SetDensityScale / SetGradientFactor / Set?ClipPlane (gui/canvas.h:49-175)."""
        v = self.volume
        if density_scale is not None:
            v.densityScale = density_scale
        if gradient_factor is not None:
            v.gradientFactor = gradient_factor
        if x_clip is not None:
            v.x_clip = L.Vec2(*x_clip)
        if y_clip is not None:
            v.y_clip = L.Vec2(*y_clip)
        if z_clip is not None:
            v.z_clip = L.Vec2(*z_clip)
        self.lib.setup_volume(C.byref(v))
        self.frame_no = 0

    def set_transfer_function(self, table):
        table = np.ascontiguousarray(table, dtype=np.float32)
        if self.tf is not None and self._tf_size == table.shape[0]:
            # an edit of the bound table: new contents into the same array
            L.check(self.lib.svr_tf_upload(C.byref(self.tf), C.c_void_p(table.ctypes.data), table.shape[0]), "svr_tf_upload")
            self.lib.setup_transferfunction(C.byref(self.tf))
            self.frame_no = 0
            return self.tf
        if self.tf is not None:
            L.check(self.lib.svr_tf_destroy(C.byref(self.tf)), "svr_tf_destroy")
        tf = L.TransferFunction()
        L.check(self.lib.svr_tf_create(C.byref(tf), C.c_void_p(table.ctypes.data), table.shape[0]), "svr_tf_create")
        self.tf = tf
        self._tf_size = table.shape[0]
        self.lib.setup_transferfunction(C.byref(tf))
        self.frame_no = 0
        return tf

    def set_camera(self, cam):
        if self.camera is None or (cam.imageW, cam.imageH) != (self.camera.imageW, self.camera.imageH):
            # RenderParams::SetupHDRBuffer (core/render_parameters.h:17-23) + the PBO of gui/canvas.cpp:50-55
            self.hdr = torch.zeros(cam.imageH * cam.imageW * 3, dtype=torch.float32, device=self.device)
            self.img = torch.zeros(cam.imageH * cam.imageW * 4, dtype=torch.uint8, device=self.device)
        self.camera = cam
        self.lib.setup_camera(C.byref(cam))
        self.frame_no = 0

    def set_area_lights(self, lights):
        self.lights = list(lights)
        arr = (L.AreaLight * max(1, len(self.lights)))(*self.lights)
        self.lib.setup_area_lights(arr, len(self.lights))
        self.frame_no = 0

    def set_env_light(self, env, enabled=True):
        self.env = env
        self.lib.setup_env_lights(C.byref(env))
        self.set_option(L.OPT_ENV_ENABLED, 1 if enabled else 0)
        self.frame_no = 0

    def load_env_map(self, path, intensity=1.0, offset=(0.0, 0.0), enabled=True):
        """Lights::SetEnvironmentLight(filename) + SetEnvironmentLightIntensity / Offset (core/lights/lights.cpp:31-90)."""
        env = L.EnvLight()
        L.check(self.lib.svr_env_load_hdr(str(path).encode(), C.byref(env)), "svr_env_load_hdr")
        if getattr(self, "_env_owned", None) is not None:
            self.lib.svr_env_destroy(C.byref(self._env_owned))
        self._env_owned = env
        env.intensity = intensity
        env.offset = L.Vec2(*offset)
        self.set_env_light(env, enabled)
        return env

    # ---- rendering
    def render_pathtracer(self, trace_depth=1):
        """One reference-style frame: one sample per pixel, frame counter advanced by the caller
        (gui/canvas.cpp:96,116)."""
        rp = L.RenderParams(trace_depth, self.frame_no, self.hdr.data_ptr())
        self.lib.render_pathtracer(_ptr(self.img), C.byref(rp))
        self.frame_no += 1

    def render_pathtracer_spp(self, spp, trace_depth=1, tonemap=True):
        rp = L.RenderParams(trace_depth, self.frame_no, self.hdr.data_ptr())
        L.check(self.lib.svr_render_pathtracer_spp(_ptr(self.img if tonemap else None), C.byref(rp), spp), "svr_render_pathtracer_spp")
        self.frame_no += spp

    def accumulate(self, sum_buf, trace_depth, first_sample, n_samples, clear=True):
        L.check(self.lib.svr_pathtracer_accumulate(_ptr(sum_buf), trace_depth, first_sample, n_samples, 1 if clear else 0), "svr_pathtracer_accumulate")

    def accumulate_bands(self, sum_buf, trace_depth, first_sample, n_samples, phase, stride, clear=True):
        """The image split: this rank's row bands (phase, phase + stride, ...) of the float4 sum buffer -- a tensor or a raw
        device pointer (e.g. distributed.PeerFrame.img_ptr, a peer mapping of rank 0's buffer).  Returns the band height."""
        rows = C.c_uint32(0)
        ptr = sum_buf if isinstance(sum_buf, C.c_void_p) else _ptr(sum_buf)
        L.check(self.lib.svr_pathtracer_accumulate_bands(ptr, trace_depth, first_sample, n_samples, 1 if clear else 0, phase, stride, C.byref(rows)),
                "svr_pathtracer_accumulate_bands")
        return int(rows.value)

    def accumulate_adaptive(self, sum_buf, half_buf, trace_depth, first_sample, min_samples, max_samples, batch, threshold, err=None):
        """Adaptive sampling (svr_pathtracer_accumulate_adaptive): every pixel takes min_samples, then batches of `batch` until its
        display-space error estimate falls below `threshold` or it has max_samples.  sum_buf / half_buf: float4 per pixel (all
        samples / the odd ones); err: optional float per pixel, the final error estimate.  Returns {"rounds", "samples",
        "unconverged"}."""
        rounds, samples, unconverged = C.c_uint32(0), C.c_uint64(0), C.c_uint32(0)
        L.check(self.lib.svr_pathtracer_accumulate_adaptive(_ptr(sum_buf), _ptr(half_buf), _ptr(err), trace_depth, first_sample, min_samples, max_samples,
                                                            batch, threshold, C.byref(rounds), C.byref(samples), C.byref(unconverged)),
                "svr_pathtracer_accumulate_adaptive")
        return {"rounds": int(rounds.value), "samples": int(samples.value), "unconverged": int(unconverged.value)}

    def guides(self, albedo_cov=None, normal_depth=None, rays_per_pixel=4):
        """Guide images of the bound scene for denoise() (svr_pathtracer_guides): float4 (albedo rgb, coverage) and float4
        (normal xyz, view-space depth) per pixel, allocated here when not given.  Returns (albedo_cov, normal_depth)."""
        n = self.camera.imageW * self.camera.imageH * 4
        if albedo_cov is None:
            albedo_cov = torch.empty(n, dtype=torch.float32, device=self.device)
        if normal_depth is None:
            normal_depth = torch.empty(n, dtype=torch.float32, device=self.device)
        L.check(self.lib.svr_pathtracer_guides(_ptr(albedo_cov), _ptr(normal_depth), rays_per_pixel), "svr_pathtracer_guides")
        return albedo_cov, normal_depth

    def denoise(self, sum_buf, half_buf, guides, iterations=None, sigma_luminance=None, sigma_normal=None, sigma_depth=None,
                sigma_coverage=None, want_hdr=True):
        """Filtered resolve of an adaptive render (svr_pathtracer_denoise) into self.img and, with want_hdr, self.hdr, as
        resolve() writes them.  sum_buf / half_buf: float4 per pixel as accumulate_adaptive leaves them; guides: the pair
        guides() returns.  Parameters not given take the library's defaults."""
        p = L.DenoiseParams()
        L.check(self.lib.svr_denoise_defaults(C.byref(p)), "svr_denoise_defaults")
        for field, value in (("iterations", iterations), ("sigmaLuminance", sigma_luminance), ("sigmaNormal", sigma_normal),
                             ("sigmaDepth", sigma_depth), ("sigmaCoverage", sigma_coverage)):
            if value is not None:
                setattr(p, field, value)
        albedo_cov, normal_depth = guides
        L.check(self.lib.svr_pathtracer_denoise(_ptr(self.img), _ptr(self.hdr if want_hdr else None), _ptr(sum_buf), _ptr(half_buf),
                                                _ptr(albedo_cov), _ptr(normal_depth), C.byref(p)), "svr_pathtracer_denoise")

    def set_denoise_params(self, params=None):
        """Filter parameters of the denoised progressive display (OPT_PT_DENOISE, svr_pathtracer_set_denoise_params): a dict
        with any of iterations, sigma_luminance, sigma_normal, sigma_depth, sigma_coverage (the others take the library's
        defaults), or None for the defaults."""
        if params is None:
            L.check(self.lib.svr_pathtracer_set_denoise_params(None), "svr_pathtracer_set_denoise_params")
            return
        p = L.DenoiseParams()
        L.check(self.lib.svr_denoise_defaults(C.byref(p)), "svr_denoise_defaults")
        names = {"iterations": "iterations", "sigma_luminance": "sigmaLuminance", "sigma_normal": "sigmaNormal", "sigma_depth": "sigmaDepth",
                 "sigma_coverage": "sigmaCoverage"}
        for key, value in params.items():
            setattr(p, names[key], value)
        L.check(self.lib.svr_pathtracer_set_denoise_params(C.byref(p)), "svr_pathtracer_set_denoise_params")

    def resolve(self, sum_buf, want_hdr=True):
        ptr = sum_buf if isinstance(sum_buf, C.c_void_p) else _ptr(sum_buf)
        L.check(self.lib.svr_pathtracer_resolve(_ptr(self.img), _ptr(self.hdr if want_hdr else None), ptr), "svr_pathtracer_resolve")

    def render_raycasting(self, step_size=None):
        if step_size is None:
            step_size = S.raycast_step_size(self.volume.spacing.tuple())
        self.lib.render_raycasting(_ptr(self.img), C.byref(self.volume), C.byref(self.tf), C.byref(self.camera), step_size)

    def render_raycasting_f32(self, out, step_size=None, rows=None, img=None):
        if step_size is None:
            step_size = S.raycast_step_size(self.volume.spacing.tuple())
        y0, y1 = rows if rows is not None else (0, self.camera.imageH)
        L.check(
            self.lib.svr_render_raycasting_rows(_ptr(img), _ptr(out), C.byref(self.volume), C.byref(self.tf), C.byref(self.camera), step_size, y0, y1),
            "svr_render_raycasting_rows",
        )

    def render_raycasting_bands(self, phase, stride, step_size=None, out=None, img_ptr=None):
        """Row bands phase, phase + stride, ... of the u8 image (the balanced multi-GPU split); returns the band height.
        img_ptr: a raw device pointer to render into instead of self.img (e.g. a peer mapping of another rank's image)."""
        if step_size is None:
            step_size = S.raycast_step_size(self.volume.spacing.tuple())
        rows = C.c_uint32(0)
        L.check(self.lib.svr_render_raycasting_bands(img_ptr if img_ptr is not None else _ptr(self.img), _ptr(out), C.byref(self.volume), C.byref(self.tf), C.byref(self.camera), step_size,
                                                     phase, stride, C.byref(rows)), "svr_render_raycasting_bands")
        return int(rows.value)

    def render_projection(self, mode="max", window=(0.5, 1.0), step_size=None, out=None, img_ptr=None, phase=0, stride=1):
        """Maximum, minimum or average intensity projection (svr_render_projection) of the bound volume from the bound camera:
        mode "max", "min" or "mean"; window (center, width) maps the projected value to the grey u8 image; out: optional
        float tensor, one value per pixel.  The u8 image goes to self.img, or to img_ptr, a raw device pointer (e.g.
        distributed.PeerFrame.img_ptr).  phase / stride: the row bands of render_raycasting_bands.  Returns the band height."""
        if step_size is None:
            step_size = S.raycast_step_size(self.volume.spacing.tuple())
        p = L.ProjectionParams(L.PROJECT_MODES[mode], step_size, window[0], window[1])
        rows = C.c_uint32(0)
        L.check(self.lib.svr_render_projection(img_ptr if img_ptr is not None else _ptr(self.img), _ptr(out), C.byref(self.volume), C.byref(self.camera),
                                               C.byref(p), phase, stride, C.byref(rows)), "svr_render_projection")
        return int(rows.value)

    def render_isosurface(self, iso, step_size=None, color=(1.0, 1.0, 1.0), surface=None, img_ptr=None, phase=0, stride=1):
        """Isosurface (svr_render_isosurface) of the bound volume from the bound camera: the first point along each pixel-centre
        ray where tex3D * densityScale reaches iso, shaded in color with the ray caster's headlight.  surface: optional float
        tensor, four values per pixel (normal facing the camera, view-space depth; (0, 0, 0, +inf) where the ray misses).  The
        u8 image goes to self.img, or to img_ptr, a raw device pointer.  phase / stride: the row bands of
        render_raycasting_bands.  Returns the band height."""
        if step_size is None:
            step_size = S.raycast_step_size(self.volume.spacing.tuple())
        p = L.IsosurfaceParams(iso, step_size, (C.c_float * 3)(*color))
        rows = C.c_uint32(0)
        L.check(self.lib.svr_render_isosurface(img_ptr if img_ptr is not None else _ptr(self.img), _ptr(surface), C.byref(self.volume),
                                               C.byref(self.camera), C.byref(p), phase, stride, C.byref(rows)), "svr_render_isosurface")
        return int(rows.value)

    def render_slices(self, params, value=None, img=None):
        """Slices or slabs (svr_render_slices) of the bound volume; params: an L.SliceParams (scene.axis_slice,
        scene.oblique_slice).  value: float32 (count, H, W) and img: uint8 (count, H, W, 4) device tensors, allocated when not
        given.  Returns (value, img)."""
        shape = (params.count, params.imageH, params.imageW)
        if value is None:
            value = torch.empty(shape, dtype=torch.float32, device=self.device)
        if img is None:
            img = torch.empty(shape + (4,), dtype=torch.uint8, device=self.device)
        L.check(self.lib.svr_render_slices(_ptr(img), _ptr(value), C.byref(self.volume), C.byref(params)), "svr_render_slices")
        return value, img

    def render_curved(self, points, params, value=None, img=None):
        """Curved planar reformation (svr_render_curved) of the bound volume along the polyline `points` ((n, 3) world xyz on
        the host); params: an L.CurvedParams (scene.straightened_curve, scene.curve_cross_sections).  value: float32
        (count, H, W) and img: uint8 (count, H, W, 4) device tensors, allocated when not given.  Returns (value, img)."""
        pts = np.ascontiguousarray(np.asarray(points, np.float32).reshape(-1, 3))
        shape = (params.count, params.imageH, params.imageW)
        if value is None:
            value = torch.empty(shape, dtype=torch.float32, device=self.device)
        if img is None:
            img = torch.empty(shape + (4,), dtype=torch.uint8, device=self.device)
        L.check(self.lib.svr_render_curved(_ptr(img), _ptr(value), C.byref(self.volume), C.byref(params), pts.ctypes.data, len(pts)),
                "svr_render_curved")
        return value, img

    # ---- label maps (one label volume per renderer, on the grid of the bound volume when dims and spacing match)
    def load_labels(self, data, spacing=(1.0, 1.0, 1.0)):
        """A label volume (svr_labels_create) from u8 label ids shaped (nz, ny, nx): a host numpy array or a device tensor.
        Replaces the renderer's label volume."""
        self.free_labels()
        if isinstance(data, torch.Tensor):
            if data.dtype != torch.uint8 or data.dim() != 3:
                raise ValueError("load_labels: a uint8 tensor shaped (nz, ny, nx)")
            data = data.contiguous()
            on_device, ptr = (1 if data.is_cuda else 0), _ptr(data)
        else:
            data = np.ascontiguousarray(data)
            if data.dtype != np.uint8 or data.ndim != 3:
                raise ValueError("load_labels: a uint8 array shaped (nz, ny, nx)")
            on_device, ptr = 0, C.c_void_p(data.ctypes.data)
        nz, ny, nx = data.shape
        vol = L.Volume()
        L.check(self.lib.svr_labels_create(C.byref(vol), ptr, on_device, nx, ny, nz, spacing[0], spacing[1], spacing[2]), "svr_labels_create")
        self.labels = vol
        return vol

    def load_label_metaimage(self, path):
        """A label volume from a MetaImage file (svr_labels_load_metaimage); returns the largest label id."""
        self.free_labels()
        vol, max_label = L.Volume(), C.c_uint32(0)
        L.check(self.lib.svr_labels_load_metaimage(str(path).encode(), C.byref(vol), C.byref(max_label)), "svr_labels_load_metaimage")
        self.labels = vol
        return int(max_label.value)

    def upload_labels(self, data):
        """New label ids (same dims) into the label volume: a host numpy array or a host or device uint8 tensor."""
        if isinstance(data, torch.Tensor):
            data = data.contiguous()
            on_device, ptr = (1 if data.is_cuda else 0), _ptr(data)
        else:
            data = np.ascontiguousarray(data, dtype=np.uint8)
            on_device, ptr = 0, C.c_void_p(data.ctypes.data)
        L.check(self.lib.svr_volume_upload(C.byref(self.labels), ptr, on_device), "svr_volume_upload")

    def free_labels(self):
        if self.labels is not None:
            L.check(self.lib.svr_volume_destroy(C.byref(self.labels)), "svr_volume_destroy")
            self.labels = None

    def render_labels(self, table, step_size=None, surface=None, labels=None, img_ptr=None, phase=0, stride=1):
        """3D label surfaces (svr_render_labels) of the label volume from the bound camera; table: an L.LabelParams
        (scene.label_table).  surface: optional float tensor, four values per pixel (normal, view-space depth); labels: optional
        uint8 tensor, the label hit per pixel (0 = none).  The u8 image goes to self.img, or to img_ptr, a raw device pointer.
        phase / stride: the row bands of render_raycasting_bands.  Returns the band height."""
        if step_size is None:
            step_size = S.raycast_step_size(self.labels.spacing.tuple())
        rows = C.c_uint32(0)
        L.check(self.lib.svr_render_labels(img_ptr if img_ptr is not None else _ptr(self.img), _ptr(surface), _ptr(labels), C.byref(self.labels),
                                           C.byref(self.camera), C.byref(table), step_size, phase, stride, C.byref(rows)), "svr_render_labels")
        return int(rows.value)

    def render_label_slices(self, params, table, img=None, labels=None, outline=False):
        """Label overlays (svr_render_label_slices) on the slices of params (an L.SliceParams, as given to render_slices):
        img, a uint8 (count, H, W, 4) device tensor holding the grey slices, is composited in place where given; labels, uint8
        (count, H, W), receives the label per pixel and is allocated when not given.  Returns (labels, img)."""
        if labels is None:
            labels = torch.empty((params.count, params.imageH, params.imageW), dtype=torch.uint8, device=self.device)
        L.check(self.lib.svr_render_label_slices(_ptr(img), _ptr(labels), C.byref(self.labels), C.byref(params), C.byref(table),
                                                 1 if outline else 0), "svr_render_label_slices")
        return labels, img

    # ---- results
    def hdr_image(self):
        return self.hdr.view(self.camera.imageH, self.camera.imageW, 3)

    def ldr_image(self):
        return self.img.view(self.camera.imageH, self.camera.imageW, 4)

    def close(self):
        self.free_volume()
        self.free_labels()
        if self.tf is not None:
            self.lib.svr_tf_destroy(C.byref(self.tf))
            self.tf = None
        if getattr(self, "_env_owned", None) is not None:
            self.lib.svr_env_destroy(C.byref(self._env_owned))
            self._env_owned = None


class VolumeStream:
    """A sequence of host-resident volumes (a time series: same dimensions and voxel format) rendered one after the
    other, with the NEXT volume's host-to-device transfer overlapped with the CURRENT volume's rendering.

        vs = VolumeStream(renderer)
        vs.prefetch(host_volume[0])
        for i in range(n):
            vs.bind()                                  # volume i becomes the renderer's volume (device-to-device + setup_volume)
            ...setup_* calls of the frame...
            if i + 1 < n: vs.prefetch(host_volume[i + 1])  # PCIe transfer runs beside the launches below
            renderer.accumulate(...) / render_pathtracer_spp(...)

    The voxels cross PCIe on a copy stream into one of two linear staging buffers in HBM; bind() copies the
    staged voxels into the bound volume's cudaArray on the render stream (svr_volume_upload, data_on_device = 1: one
    kernel that fills the array and reduces the macrocell ranges, 256 MiB in 0.24 ms), so the caller's cudaArray / texture
    object never change.
    prefetch() must come AFTER the frame's setup_* calls: like the reference's (pathtracer.cu:34-68) they
    cudaDeviceSynchronize, which would wait for the transfer.

    One process per GPU, world_size > 1 (every rank constructs the stream and calls prefetch / bind in the same
    order; the volume is replicated, SURVEY.md section 8e) -- `fanout` says how the voxels reach every GPU:
      "p2p"    rank `src` uploads once over PCIe and pushes the staged voxels into the other ranks' staging buffers
               with copy engines over NVLink (CUDA IPC peer mappings, svr_stage_*; no SMs, so the pushes run beside a
               render kernel that fills every SM).  Cross-process ordering: interprocess CUDA events plus one
               host-side (gloo) barrier per prefetch, which guarantees an event's record has been CALLED before a
               peer waits on it.  Falls back to "nvlink" when CUDA IPC is unavailable.
      "nvlink" rank `src` uploads, then an NCCL broadcast (an SM kernel: beside a full-machine render kernel it only
               gets scheduled in that kernel's tail).
      "pcie"   every rank uploads its own host copy over its own PCIe link (no collective).
    """

    def __init__(self, renderer, nbytes=None, group=None, src=0, fanout="p2p", host_group=None):
        import torch.distributed as dist

        if fanout not in ("p2p", "nvlink", "pcie"):
            raise ValueError("VolumeStream: fanout must be 'p2p', 'nvlink' or 'pcie'")
        self.r = renderer
        self.lib = renderer.lib
        self.group, self.src = group, src
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1
        self.fanout = fanout if multi else "local"
        self.dist = dist if multi else None
        self.world = dist.get_world_size(group) if multi else 1
        self.rank = dist.get_rank(group) if multi else src
        dev = renderer.device
        self.nbytes = int(nbytes if nbytes is not None else renderer.volume_nbytes())
        self.copy_stream = torch.cuda.Stream(device=dev)
        self.head = 0      # next slot to fill
        self.tail = 0      # next slot to bind
        self.inflight = 0
        self.stage = None
        self.stage_ptr = [None, None]
        self.peer_ptr = {}
        if self.fanout == "p2p":
            try:
                # host-side barrier and handle exchange; gloo needs a resolvable local address on every rank
                self.host_group = host_group if host_group is not None else dist.new_group(backend="gloo")
            except Exception:
                self.host_group = None
            if self.host_group is None or not self._setup_p2p():
                self.fanout = "nvlink"
        if self.fanout != "p2p":
            self.stage = [torch.empty(self.nbytes, dtype=torch.uint8, device=dev) for _ in range(2)]
            for t in self.stage:
                t.record_stream(self.copy_stream)
            self.stage_ptr = [C.c_void_p(t.data_ptr()) for t in self.stage]
            self.ready = [torch.cuda.Event(), torch.cuda.Event()]      # staging buffer filled (copy stream)
            self.consumed = [torch.cuda.Event(), torch.cuda.Event()]   # staging buffer copied into the array (render stream)

    # ---- "p2p": exportable staging buffers, peer mappings on the uploading rank, interprocess events
    def _setup_p2p(self):
        dist, lib, dev = self.dist, self.lib, self.r.device
        ok, handles, consumed_h = True, [], []
        try:
            for i in range(2):
                p = C.c_void_p(0)
                L.check(lib.svr_stage_alloc(C.byref(p), self.nbytes), "svr_stage_alloc")
                self.stage_ptr[i] = p
                h = (C.c_ubyte * 64)()
                L.check(lib.svr_stage_export(p, C.byref(h)), "svr_stage_export")
                handles.append(bytes(h))
            self.consumed = [torch.cuda.Event(interprocess=True), torch.cuda.Event(interprocess=True)]
            consumed_h = [e.ipc_handle() for e in self.consumed]
        except Exception:
            ok = False
        everyone = [None] * self.world
        dist.all_gather_object(everyone, (ok, handles, consumed_h), group=self.host_group)
        ok = all(e[0] for e in everyone)
        landed_h = [None, None]
        if ok and self.rank == self.src:
            try:
                for r in range(self.world):
                    if r == self.src:
                        continue
                    ptrs = []
                    for hb in everyone[r][1]:
                        q = C.c_void_p(0)
                        h = (C.c_ubyte * 64).from_buffer_copy(hb)
                        L.check(lib.svr_stage_import(C.byref(h), C.byref(q)), "svr_stage_import")
                        ptrs.append(q)
                    self.peer_ptr[r] = ptrs
                self.peer_consumed = {r: [torch.cuda.Event.from_ipc_handle(dev, h) for h in everyone[r][2]]
                                      for r in range(self.world) if r != self.src}
                self.ready = [torch.cuda.Event(interprocess=True), torch.cuda.Event(interprocess=True)]
                landed_h = [e.ipc_handle() for e in self.ready]
            except Exception:
                ok = False
        box = [(ok, landed_h)]
        dist.broadcast_object_list(box, src=self.src, group=self.host_group)
        ok, landed_h = box[0]
        if ok and self.rank != self.src:
            try:
                self.ready = [torch.cuda.Event.from_ipc_handle(dev, h) for h in landed_h]
            except Exception:
                ok = False
        flags = [None] * self.world
        dist.all_gather_object(flags, ok, group=self.host_group)
        if not all(flags):
            self._release_p2p()
            return False
        return True

    def _release_p2p(self):
        for ptrs in self.peer_ptr.values():
            for q in ptrs:
                self.lib.svr_stage_release(q)
        self.peer_ptr = {}
        for i, p in enumerate(self.stage_ptr):
            if p is not None and self.stage is None:
                self.lib.svr_stage_free(p)
            self.stage_ptr[i] = None

    def close(self):
        """Collective for fanout "p2p": peer mappings are released before their owners free the buffers."""
        torch.cuda.synchronize(self.r.device)
        if self.fanout == "p2p":
            for ptrs in self.peer_ptr.values():
                for q in ptrs:
                    self.lib.svr_stage_release(q)
            self.peer_ptr = {}
            self.dist.barrier(group=self.host_group)
            self._release_p2p()
        self.stage = None

    def prefetch(self, host_volume):
        """Start the transfer of the next volume (a pinned host uint8 tensor; read on rank `src` only, unless
        fanout is "pcie").  Collective when world_size > 1."""
        if self.inflight >= 2:
            raise RuntimeError("VolumeStream.prefetch: both staging buffers are in flight; bind() first")
        slot = self.head
        cs = self.copy_stream
        uploads = self.fanout in ("local", "pcie") or self.rank == self.src
        with torch.cuda.stream(cs):
            cs.wait_event(self.consumed[slot])  # the slot's previous contents have left for the array
            if self.fanout == "p2p":
                if uploads:
                    for evs in self.peer_consumed.values():
                        cs.wait_event(evs[slot])
                    src_ptr = C.c_void_p(host_volume.data_ptr())
                    L.check(self.lib.svr_stage_copy(self.stage_ptr[slot], src_ptr, self.nbytes, C.c_void_p(cs.cuda_stream)), "svr_stage_copy")
                    for ptrs in self.peer_ptr.values():   # NVLink, copy engines
                        L.check(self.lib.svr_stage_copy(ptrs[slot], self.stage_ptr[slot], self.nbytes, C.c_void_p(cs.cuda_stream)), "svr_stage_copy")
                    self.ready[slot].record(cs)
            else:
                if uploads:
                    self.stage[slot].copy_(host_volume.view(torch.uint8).reshape(-1), non_blocking=True)
                if self.fanout == "nvlink":
                    self.dist.broadcast(self.stage[slot], src=self.src, group=self.group)
                self.ready[slot].record(cs)
        if self.fanout == "p2p":
            self.dist.barrier(group=self.host_group)  # rank src has CALLED record: the others may wait on the event
        self.head ^= 1
        self.inflight += 1

    def bind(self):
        """Make the oldest prefetched volume the renderer's volume."""
        if self.inflight == 0:
            raise RuntimeError("VolumeStream.bind: nothing prefetched")
        slot = self.tail
        main = torch.cuda.current_stream(self.r.device)
        main.wait_event(self.ready[slot])
        L.check(self.lib.svr_volume_upload(C.byref(self.r.volume), self.stage_ptr[slot], 1), "svr_volume_upload")
        self.consumed[slot].record(main)
        # no setup_volume: the svr_volume struct is unchanged, and the upload itself has invalidated what depends on the voxels
        # (a setup_volume here would make the next render re-check the array behind the handle: one more host round trip per frame)
        self.r.frame_no = 0
        self.tail ^= 1
        self.inflight -= 1


def setup_config(r, cfg, volume_bytes=None):
    """Populate a Renderer with one of the BASELINE.json configurations (scene.CONFIGS)."""
    if volume_bytes is None:
        volume_bytes = r.generate_volume(cfg.gen, cfg.fmt, cfg.n, cfg.gen_seed)
    r.load_volume(volume_bytes, cfg.fmt, (cfg.n,) * 3)
    r.set_transfer_function(S.tf_table(cfg.tf))
    r.set_camera(S.default_camera(cfg.extent, cfg.width, cfg.height))
    r.set_area_lights([S.default_area_light(cfg.extent)])
    r.set_env_light(S.constant_env_light(), enabled=cfg.env)
    return volume_bytes
