"""TEST INFRASTRUCTURE -- not product code.  ctypes bindings of the two checkers:

  * oracle/libsvr_oracle.so  -- CPU restatement of the reference's render path (svr_oracle.cpp)
  * oracle/_ref/libsvr_ref_<W>x<H>[_r32].so -- the reference's own unmodified pathtracer.cu +
    raycasting.cu compiled headless (oracle/Makefile); needs a GPU to run.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import this.
"""
import ctypes as C
import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(_HERE))
from sunvolumerender_b200 import _lib as L  # noqa: E402  (struct layouts only; does not load the product .so)

CPU_LIB = os.path.join(_HERE, "libsvr_oracle.so")
REF_DIR = os.path.join(_HERE, "_ref")


class OracleScene(C.Structure):  # svr_oracle_scene
    _fields_ = [
        ("voxels", C.c_void_p),
        ("format", C.c_int32),
        ("nx", C.c_uint32),
        ("ny", C.c_uint32),
        ("nz", C.c_uint32),
        ("volume", L.Volume),
        ("tfTable", C.c_void_p),
        ("tfSize", C.c_uint32),
        ("tf", L.TransferFunction),
        ("camera", L.Camera),
        ("lights", L.AreaLight * 8),
        ("numLights", C.c_uint32),
        ("env", L.EnvLight),
        ("envEnabled", C.c_int32),
        ("filterMode", C.c_int32),
    ]


CNT = {"track_taps": 0, "shadow_taps": 1, "shade_taps": 2, "tf_lookups": 3, "scatters": 4, "paths": 5, "steps": 7}

_cpu = None


def cpu():
    global _cpu
    if _cpu is None:
        lib = C.CDLL(CPU_LIB)
        P = C.POINTER(OracleScene)
        lib.svr_oracle_threads.restype = C.c_int
        lib.svr_oracle_set_threads.argtypes = [C.c_int]
        lib.svr_oracle_raycast.argtypes = [P, C.c_float, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.svr_oracle_pathtrace.argtypes = [P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
        lib.svr_oracle_pathtrace_strided.argtypes = [P, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p]
        lib.svr_oracle_tonemap.argtypes = [C.c_void_p, C.c_float, C.c_uint64, C.c_void_p]
        lib.svr_oracle_tex3d.restype = C.c_float
        lib.svr_oracle_tex3d.argtypes = [P, C.c_float, C.c_float, C.c_float]
        lib.svr_oracle_tf.argtypes = [P, C.c_float, C.c_void_p]
        lib.svr_oracle_wang_hash.restype = C.c_uint32
        lib.svr_oracle_wang_hash.argtypes = [C.c_uint32]
        lib.svr_oracle_xorwow_uniforms.argtypes = [C.c_uint64, C.c_uint32, C.c_void_p]
        _cpu = lib
    return _cpu


class CpuOracle:
    """Host scene + the CPU restatement.  Keeps the numpy arrays alive."""

    def __init__(self, voxels, fmt, dims, volume, tf_table, camera, lights=(), env=None, env_enabled=False, filter_mode=0):
        self.voxels = np.ascontiguousarray(voxels)
        self.tf_table = np.ascontiguousarray(tf_table, dtype=np.float32)
        s = OracleScene()
        s.voxels = self.voxels.ctypes.data
        s.format = fmt
        s.nx, s.ny, s.nz = dims
        s.volume = volume
        s.tfTable = self.tf_table.ctypes.data
        s.tfSize = self.tf_table.shape[0]
        s.tf.maxOpacity = float(self.tf_table[:, 3].max())
        s.camera = camera
        for i, l in enumerate(lights):
            s.lights[i] = l
        s.numLights = len(lights)
        if env is not None:
            s.env = env
        s.envEnabled = 1 if env_enabled else 0
        s.filterMode = filter_mode
        self.scene = s

    def raycast(self, step_size, rows=None):
        W, H = self.scene.camera.imageW, self.scene.camera.imageH
        y0, y1 = rows if rows else (0, H)
        rgba = np.zeros((H, W, 4), np.float32)
        u8 = np.zeros((H, W, 4), np.uint8)
        cnt = np.zeros(16, np.uint64)
        cpu().svr_oracle_raycast(C.byref(self.scene), step_size, W, y0, y1, rgba.ctypes.data, u8.ctypes.data, cnt.ctypes.data)
        return rgba, u8, cnt

    def pathtrace(self, trace_depth, frame0, nframes, rows=None, hdr=None, row_step=1):
        W, H = self.scene.camera.imageW, self.scene.camera.imageH
        y0, y1 = rows if rows else (0, H)
        if hdr is None:
            hdr = np.zeros((H, W, 3), np.float32)
        cnt = np.zeros(16, np.uint64)
        cpu().svr_oracle_pathtrace_strided(C.byref(self.scene), trace_depth, frame0, nframes, W, y0, y1, row_step, hdr.ctypes.data, cnt.ctypes.data)
        return hdr, cnt

    def tonemap(self, hdr):
        hdr = np.ascontiguousarray(hdr, np.float32)
        out = np.zeros(hdr.shape[:-1] + (4,), np.uint8)
        cpu().svr_oracle_tonemap(hdr.ctypes.data, self.scene.camera.exposure, hdr.size // 3, out.ctypes.data)
        return out


def ref_lib_path(width, height, r32=False, f32=False, env=False):
    h16 = (height + 15) // 16 * 16
    suffix = "_r32" if r32 else ("_f32" if f32 else ("_env" if env else ""))
    return os.path.join(REF_DIR, f"libsvr_ref_{width}x{h16}{suffix}.so")


_ref_cache = {}


def ref(width, height, r32=False, f32=False, env=False):
    """The reference's own kernels for a WIDTH x HEIGHT canvas (HEIGHT rounded up to 16: the launch
    has no bounds guard, pathtracer.cu:294-295).  r32 = built with the shipped -maxrregcount=32;
    f32 = float twin (img holds 4 floats per pixel, see glm_shim); env = environment-light twin (the line
    commented out at pathtracer.cu:233 re-enabled, see oracle/Makefile).  None when not prebuilt."""
    path = ref_lib_path(width, height, r32, f32, env)
    if path in _ref_cache:
        return _ref_cache[path]
    if not os.path.exists(path):
        return None
    lib = C.CDLL(path, mode=C.RTLD_LOCAL)
    for name, res, args in L.SIGNATURES[:7]:
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    lib.buffer_height = (height + 15) // 16 * 16
    _ref_cache[path] = lib
    return lib


GOLDEN_KERNELS = os.path.join(os.path.dirname(_HERE), "tests", "golden", "reference_kernels.npz")


def load_golden_scene(r, g, name):
    """Loads scene `name` of tests/golden/reference_kernels.npz (what the reference's own kernels rendered, stored by
    tests/golden/make_golden.py) into the product renderer r; returns (step size, trace depth, frames)."""
    from sunvolumerender_b200 import scene as S

    n, fmt, W, H, depth, frames, nl = [int(v) for v in g[f"{name}_meta"]]
    r.load_volume(g[f"{name}_vox"], fmt, (n, n, n))
    stored = L.Volume.from_buffer_copy(bytes(g[f"{name}_volume"]))
    for f in ("densityScale", "invMaxMagnitude", "gradientFactor"):
        assert getattr(r.volume, f) == getattr(stored, f), f
    assert r.volume.bbox.vmin.tuple() == stored.bbox.vmin.tuple() and r.volume.bbox.invSize.tuple() == stored.bbox.invSize.tuple()
    r.set_transfer_function(g[f"{name}_tf"])
    r.set_camera(L.Camera.from_buffer_copy(bytes(g[f"{name}_camera"])))
    lb = bytes(g[f"{name}_lights"])
    r.set_area_lights([L.AreaLight.from_buffer_copy(lb[i * 44:(i + 1) * 44]) for i in range(nl)])
    r.set_env_light(S.constant_env_light(), enabled=False)
    return float(g[f"{name}_step"]), depth, frames


REFSCENE_LIB = os.path.join(REF_DIR, "libsvr_refscene.so")


class RefScene:
    """Scene resources of bench.py's reference arm, built by oracle/ref_scene.cu with plain CUDA runtime calls (same
    descriptors as the reference's loaders, same synthetic voxels as the product's generator): the arm's process never
    maps the product library."""

    def __init__(self, cfg, tf_table):
        if not os.path.exists(REFSCENE_LIB):
            raise FileNotFoundError(REFSCENE_LIB)
        self.lib = C.CDLL(REFSCENE_LIB, mode=C.RTLD_LOCAL)
        self.lib.ref_scene_create.argtypes = [C.c_int, C.c_int, C.c_uint32, C.c_uint32, C.c_void_p, C.c_uint32, C.POINTER(L.Volume), C.POINTER(L.TransferFunction)]
        self.lib.ref_scene_destroy.argtypes = [C.POINTER(L.Volume), C.POINTER(L.TransferFunction)]
        self.lib.ref_scene_download.argtypes = [C.POINTER(L.Volume), C.c_void_p, C.c_uint64]
        table = np.ascontiguousarray(tf_table, dtype=np.float32)
        self.volume, self.tf = L.Volume(), L.TransferFunction()
        rc = self.lib.ref_scene_create(cfg.gen, cfg.fmt, cfg.n, cfg.gen_seed, table.ctypes.data, table.shape[0], C.byref(self.volume), C.byref(self.tf))
        if rc != 0:
            raise RuntimeError(f"ref_scene_create failed: CUDA error {rc}")

    def download(self, dtype, n):
        out = np.zeros((n, n, n), dtype)
        rc = self.lib.ref_scene_download(C.byref(self.volume), out.ctypes.data, out.nbytes)
        if rc != 0:
            raise RuntimeError(f"ref_scene_download failed: {rc}")
        return out

    def close(self):
        self.lib.ref_scene_destroy(C.byref(self.volume), C.byref(self.tf))


class RefCuda:
    """Drives the reference's own kernels the way gui/canvas.cpp does: setup_* once, then
    render_pathtracer per frame with frameNo = 0, 1, ... (canvas.cpp:96,116), or render_raycasting.
    Texture objects come from the caller (same descriptors as the reference's loaders)."""

    def __init__(self, width, height, r32=False, f32=False, device=None, env=False):
        import torch

        self.torch = torch
        self.f32 = f32
        self.lib = ref(width, height, r32, f32, env)
        if self.lib is None:
            raise FileNotFoundError(ref_lib_path(width, height, r32, f32, env))
        self.W, self.H = width, height
        self.HB = self.lib.buffer_height
        dev = device if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.hdr = torch.zeros(self.HB * self.W * 3, dtype=torch.float32, device=dev)
        self.img = torch.zeros(self.HB * self.W * 4, dtype=torch.float32 if f32 else torch.uint8, device=dev)
        self.frame_no = 0

    def setup(self, volume, tf, camera, lights, env):
        lib = self.lib
        assert camera.imageW == self.W and camera.imageH == self.H
        lib.setup_volume(C.byref(volume))
        lib.setup_transferfunction(C.byref(tf))
        lib.setup_camera(C.byref(camera))
        lib.setup_env_lights(C.byref(env))
        arr = (L.AreaLight * max(1, len(lights)))(*lights)
        lib.setup_area_lights(arr, len(lights))
        self.volume, self.tf, self.camera = volume, tf, camera
        self.frame_no = 0

    def render_pathtracer(self, frames, trace_depth=1):
        # the reference launches on the legacy default stream; order it after torch's stream
        self.torch.cuda.current_stream().synchronize()
        for _ in range(frames):
            rp = L.RenderParams(trace_depth, self.frame_no, self.hdr.data_ptr())
            self.lib.render_pathtracer(C.c_void_p(self.img.data_ptr()), C.byref(rp))
            self.frame_no += 1

    def render_raycasting(self, step_size):
        self.torch.cuda.current_stream().synchronize()
        self.lib.render_raycasting(C.c_void_p(self.img.data_ptr()), C.byref(self.volume), C.byref(self.tf), C.byref(self.camera), step_size)

    def hdr_image(self):
        self.torch.cuda.synchronize()
        return self.hdr.view(self.HB, self.W, 3)[: self.H]

    def ldr_image(self):
        """u8 RGBA; for the float twin: the four products the kernel hands to u8vec4 (L*255), as floats."""
        self.torch.cuda.synchronize()
        return self.img.view(self.HB, self.W, 4)[: self.H]
