"""Shared helpers of the GPU parity tests: scene setup through the C ABI, the reference's own
kernels (oracle/_ref, test infrastructure) on the same texture objects, the CPU oracle on the same
voxels."""
import ctypes as C

import numpy as np
import torch

from oracle import binding as B
from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S
from sunvolumerender_b200.render import setup_config


def small_config(name="S", n=64, w=128, h=128, fmt=L.VOXEL_U8, gen=L.GEN_SPHERE, tf="default", depth=1, env=False):
    return S.Config(name, n, fmt, gen, w, h, tf, trace_depth=depth, spp=1, env=env)


def setup(r, cfg):
    """Loads cfg into the renderer; returns the voxels as a host numpy array (z, y, x)."""
    r.set_option(L.OPT_PT_MODE, 2)
    r.set_option(L.OPT_PT_KERNEL, 2)
    r.set_option(L.OPT_PT_WARP_PIXELS, 0)
    r.set_option(L.OPT_PT_WARP_MIN_SPP, 32)
    r.set_option(L.OPT_PT_QUEUE_MIN_DEPTH, 8)
    r.set_option(L.OPT_SHADOW_ESTIMATOR, 0)
    r.set_option(L.OPT_RC_SKIP, 1)
    r.set_option(L.OPT_LEAP, 1)
    r.set_option(L.OPT_PT_ENTRY_CACHE, 1)
    r.set_option(L.OPT_PT_LIGHT_CULL, 1)
    r.set_option(L.OPT_PT_PROFILE, 0)
    r.set_option(L.OPT_PT_REFILL, 0)
    r.set_option(L.OPT_PT_POOL_PIXELS, 0)
    r.set_option(L.OPT_ENV_NEE, 0)
    r.set_option(L.OPT_PT_BLOCK_SPLIT, 0)
    r.set_option(L.OPT_PT_PIXEL_CACHE, 1)
    r.set_option(L.OPT_FUSED_UPLOAD, 1)
    r.set_option(L.OPT_PT_LOOKAHEAD, 32)
    r.set_option(L.OPT_MACROCELL_SIZE, 8)
    r.set_option(L.OPT_COUNTERS, 0)
    r.set_option(L.OPT_SEED, 0x5EED)
    vb = setup_config(r, cfg)
    vox = vb.cpu().numpy().view(S.VOXEL_DTYPES[cfg.fmt]).reshape(cfg.n, cfg.n, cfg.n)
    return vox


def reference(r, cfg, f32=False, r32=False, env=False):
    """env=True: the environment-light twin (pathtracer.cu:233 re-enabled at build time, oracle/Makefile)."""
    ref = ref_cuda(r, cfg.width, cfg.height, r32=r32, f32=f32, env=env)
    ref.setup(r.volume, r.tf, r.camera, r.lights, r.env)
    return ref


def ref_cuda(r, width, height, r32=False, f32=False, env=False):
    """The reference's own kernels (oracle/_ref) where they are built from the reference's sources; elsewhere the
    product's reference-twin path (TwinRef), which tests/test_gpu_reference_golden.py holds to the reference's stored
    outputs.  Only the statistical-parity tests take this arm (thousands of frames: too many for the CPU oracle); every
    deterministic comparison uses oracle_reference."""
    if B.ref(width, height, r32, f32, env) is not None:
        return B.RefCuda(width, height, r32=r32, f32=f32, env=env)
    assert not f32, "the float twin of the ray caster: use oracle_reference"
    return TwinRef(r, width, height, env=env)


def oracle_reference(r, cfg, f32=False, env=False, lights=None, rows=None):
    """The reference's own kernels where they are built; elsewhere the CPU oracle (oracle/svr_oracle.cpp, held to the
    reference's stored outputs by tests/test_oracle_golden.py), independent of the product.  Compare with check_rgba /
    check_u8 / check_paths: the oracle computes in IEEE arithmetic, the reference and the product with fast math.
    cfg.dims (x, y, z) where the volume is not cfg.n^3; lights: instead of r.lights; rows: (y0, y1), the only rows the
    oracle renders (full-size images at the oracle's speed; compare them through rows_of)."""
    lights = r.lights if lights is None else lights
    if B.ref(cfg.width, cfg.height, f32=f32, env=env) is not None:
        ref = ref_cuda(r, cfg.width, cfg.height, f32=f32, env=env)
    else:
        ref = OracleRef(r, cfg.fmt, getattr(cfg, "dims", None) or (cfg.n,) * 3, env=env, rows=rows)
    ref.setup(r.volume, r.tf, r.camera, lights, r.env)
    return ref


def rows_of(ref):
    """The rows of the image a reference arm rendered."""
    rows = getattr(ref, "rows", None)
    return slice(*rows) if rows else slice(None)


TWIN_OPTIONS = {L.OPT_PT_MODE: 0, L.OPT_SHADOW_ESTIMATOR: 0, L.OPT_ENV_NEE: 0, L.OPT_PT_KERNEL: 1, L.OPT_PT_LOOKAHEAD: 0}


class TwinRef:
    """B.RefCuda's path-tracer interface on the product library: the reference-twin mode (global majorant, XORWOW streams
    in the reference's draw order, delta-tracked shadow rays, megakernel), rendering into buffers of its own.  The library's scene and options are shared with the renderer `r`: each call sets the twin's
    scene and options and restores r's afterwards."""

    def __init__(self, r, width, height, env=False):
        self.r, self.lib = r, r.lib
        self.W, self.H = width, height
        self.env = env
        self.hdr = torch.zeros(height * width * 3, dtype=torch.float32, device="cuda")
        self.img = torch.zeros(height * width * 4, dtype=torch.uint8, device="cuda")
        self.frame_no = 0

    def setup(self, volume, tf, camera, lights, env):
        assert camera.imageW == self.W and camera.imageH == self.H
        self.volume, self.tf, self.camera = L.Volume.from_buffer_copy(volume), L.TransferFunction.from_buffer_copy(tf), L.Camera.from_buffer_copy(camera)
        self.lights, self.env_light = list(lights), L.EnvLight.from_buffer_copy(env)
        self.frame_no = 0

    def _scene(self, volume, tf, camera, lights, env):
        self.lib.setup_volume(C.byref(volume))
        self.lib.setup_transferfunction(C.byref(tf))
        self.lib.setup_camera(C.byref(camera))
        self.lib.setup_env_lights(C.byref(env))
        self.lib.setup_area_lights((L.AreaLight * max(1, len(lights)))(*lights), len(lights))

    def render_pathtracer(self, frames, trace_depth=1):
        r = self.r
        options = {**TWIN_OPTIONS, L.OPT_ENV_ENABLED: 1 if self.env else 0}
        saved = {k: r.get_option(k) for k in options}
        self._scene(self.volume, self.tf, self.camera, self.lights, self.env_light)
        for k, v in options.items():
            r.set_option(k, v)
        try:
            for _ in range(frames):
                rp = L.RenderParams(trace_depth, self.frame_no, self.hdr.data_ptr())
                self.lib.render_pathtracer(C.c_void_p(self.img.data_ptr()), C.byref(rp))
                self.frame_no += 1
            torch.cuda.synchronize()
        finally:
            for k, v in saved.items():
                r.set_option(k, v)
            self._scene(r.volume, r.tf, r.camera, r.lights, r.env)

    def hdr_image(self):
        torch.cuda.synchronize()
        return self.hdr.view(self.H, self.W, 3)

    def ldr_image(self):
        torch.cuda.synchronize()
        return self.img.view(self.H, self.W, 4)


class OracleRef:
    """B.RefCuda's interface on the CPU oracle.  setup() reads the voxels and the transfer function table back from the
    renderer's resources; the oracle samples them with its own software filter (bit-exact to the texture hardware,
    tests/test_oracle_golden.py).  Images come back as CPU tensors."""

    def __init__(self, r, fmt, dims, env=False, rows=None):
        self.r, self.fmt, self.dims, self.env, self.rows = r, fmt, tuple(dims), env, rows
        self.frame_no = 0

    def _tf_table(self, tf):
        n = self.r._tf_size
        x = torch.from_numpy((np.arange(n, dtype=np.float32) + np.float32(0.5)) / np.float32(n)).cuda()
        out = torch.zeros(n * 4, dtype=torch.float32, device="cuda")
        L.check(self.r.lib.svr_debug_sample_tf(C.byref(tf), C.c_void_p(x.data_ptr()), n, C.c_void_p(out.data_ptr())), "svr_debug_sample_tf")
        return out.view(n, 4).cpu().numpy()

    def setup(self, volume, tf, camera, lights, env):
        assert not (self.env and env.tex), "the CPU oracle's environment light is the constant sky"
        nx, ny, nz = self.dims
        vox = np.zeros((nz, ny, nx), S.VOXEL_DTYPES[self.fmt])
        L.check(self.r.lib.svr_volume_download(C.byref(volume), C.c_void_p(vox.ctypes.data), vox.nbytes), "svr_volume_download")
        self.oracle = B.CpuOracle(vox, self.fmt, self.dims, volume, self._tf_table(tf), camera, list(lights)[:8], env=env, env_enabled=self.env)
        self.W, self.H = camera.imageW, camera.imageH
        self.hdr, self.img, self.rgba = None, None, None
        self.frame_no = 0

    def render_raycasting(self, step_size):
        self.rgba, self.img, _ = self.oracle.raycast(step_size, rows=self.rows)

    def render_pathtracer(self, frames, trace_depth=1):
        self.hdr, _ = self.oracle.pathtrace(trace_depth, self.frame_no, frames, rows=self.rows, hdr=None if self.frame_no == 0 else self.hdr)
        self.frame_no += frames
        self.img = self.oracle.tonemap(self.hdr)

    def hdr_image(self):
        return torch.from_numpy(self.hdr)

    def ldr_image(self):
        """u8 RGBA; after render_raycasting also rgba_image() (the float RGBA)."""
        return torch.from_numpy(self.img)

    def rgba_image(self):
        return torch.from_numpy(self.rgba)


def rgba_of(ref):
    """Float RGBA of the last ray-cast frame of a reference arm (B.RefCuda float twin: the products handed to u8vec4)."""
    if isinstance(ref, OracleRef):
        return ref.rgba_image().numpy()
    return ref.ldr_image().cpu().numpy() / 255.0


def check_rgba(mine, ref):
    """Ray-cast float RGBA: within 1e-4 per channel of the reference's float twin; against the CPU oracle the bounds of
    tests/test_gpu_raycast.py::test_against_cpu_oracle (a 1-ulp coordinate difference can flip an 8-bit filter weight)."""
    rows = rows_of(ref)
    d = np.abs(np.asarray(mine)[rows] - rgba_of(ref)[rows])
    if isinstance(ref, OracleRef):
        assert d.mean() < 5e-5 and (d.max(axis=2) < 1e-4).mean() > 0.99, (float(d.mean()), float((d.max(axis=2) < 1e-4).mean()))
    else:
        assert d.max() <= 1e-4, float(d.max())


def check_u8(mine_u8, ref):
    """u8 image: 1 LSB of the reference's; against the CPU oracle 1 LSB on >= 99 % of the pixels (the float bound of
    check_rgba, quantised: a pixel whose filter weight flipped can differ by several LSB)."""
    rows = rows_of(ref)
    d = np.abs(np.asarray(mine_u8)[rows].astype(int) - ref.ldr_image().cpu().numpy()[rows].astype(int)).max(axis=2)
    if isinstance(ref, OracleRef):
        assert (d <= 1).mean() > 0.99, float((d <= 1).mean())
    else:
        assert d.max() <= 1, int(d.max())


def check_paths(mine, theirs, ref, frac=0.999, mean_rel=None, scaled=False):
    """Twin-mode HDR, path for path: within 1e-4 on `frac` of the pixels of the reference's; against the CPU oracle (IEEE
    libm flips a few accept/reject decisions) the bounds of tests/test_gpu_pathtrace.py::test_twin_mode_matches_cpu_oracle.
    scaled: the bound is relative above 1 (a light in view or a bright sky: radiance where 1e-4 is below one float ulp)."""
    rows = rows_of(ref)
    mine, theirs = np.asarray(mine)[rows], np.asarray(theirs)[rows]
    d = np.abs(mine - theirs).max(axis=2)
    if scaled:
        d = d / np.maximum(1.0, np.abs(theirs).max(axis=2))
    if isinstance(ref, OracleRef):
        assert (d < 1e-3).mean() > 0.95 and abs(mine.mean() - theirs.mean()) < 0.03 * theirs.mean(), (float((d < 1e-3).mean()), mine.mean(), theirs.mean())
    else:
        assert (d <= 1e-4).mean() >= frac, (float(d.max()), float((d <= 1e-4).mean()))
        assert mean_rel is None or abs(mine.mean() - theirs.mean()) <= mean_rel * theirs.mean()


def cpu_oracle(r, cfg, vox, env_enabled=False):
    return B.CpuOracle(vox, cfg.fmt, (cfg.n,) * 3, r.volume, S.tf_table(cfg.tf), r.camera, r.lights, env=r.env, env_enabled=env_enabled)


def raycast_f32(r, rows=None):
    H, W = r.camera.imageH, r.camera.imageW
    out = torch.zeros(H * W * 4, dtype=torch.float32, device="cuda")
    r.render_raycasting_f32(out, rows=rows, img=r.img)
    torch.cuda.synchronize()
    return out.view(H, W, 4)


def rmse(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.sqrt(((a - b) ** 2).mean()))
