"""Slices and slabs (svr_render_slices) without a GPU: the parameter struct's layout, the argument checks (all made before
any CUDA call), and closed forms on the CPU restatement (tests/slice_oracle.cpp) that the GPU tests hold the kernel to."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

import _slice_oracle as SO

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("center", "axisU", "axisV", "axisW", "imageW", "imageH", "count", "mode", "thickness", "sampleSpacing", "windowCenter",
          "windowWidth")


def test_slice_params_layout_matches_header(tmp_path):
    probe = tmp_path / "probe.c"
    offs = ", ".join(f"offsetof(svr_slice_params, {f})" for f in FIELDS)
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "svr_render.h"\n'
                     f'int main(void){{printf("{"%zu " * (len(FIELDS) + 1)}\\n", sizeof(svr_slice_params), {offs});return 0;}}\n')
    exe = tmp_path / "probe"
    subprocess.check_call(["/usr/bin/gcc", "-std=c11", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)])
    got = [int(x) for x in subprocess.check_output([str(exe)], text=True).split()]
    P = L.SliceParams
    assert got == [C.sizeof(P)] + [getattr(P, f).offset for f in FIELDS]


def test_argument_errors_are_reported_before_any_cuda_call():
    lib = L.load()
    vol = S.host_volume_struct((8, 8, 8))
    out = C.c_void_p(16)  # never dereferenced: every call below fails its checks first
    inf, nan = float("inf"), float("nan")

    def call(img=out, value=out, volume=vol, params=True, **kw):
        p = S.axis_slice((8, 8, 8), (1, 1, 1), "z", 3, thickness_voxels=4)
        for k, v in kw.items():
            if k in ("axisU", "axisV", "axisW"):
                getattr(p, k)[:] = v
            else:
                setattr(p, k, v)
        rc = lib.svr_render_slices(img, value, C.byref(volume) if volume is not None else None, C.byref(p) if params else None)
        return rc, lib.svr_last_error().decode()

    bad = [dict(volume=None), dict(params=False), dict(img=None, value=None),
           dict(axisU=(inf, 0, 0)), dict(axisU=(nan, 0, 0)), dict(axisV=(0, nan, 0)), dict(axisV=(2, 0, 0)), dict(axisU=(0, 0, 0)),
           dict(axisU=(1e30, 0, 0), axisV=(0, 1e30, 0)), dict(count=2, axisW=(0, 0, nan)), dict(count=2, axisW=(inf, 0, 0)),
           dict(imageW=0), dict(imageH=0), dict(imageW=16385), dict(imageH=16385), dict(count=0), dict(count=65536),
           dict(mode=-1), dict(mode=3), dict(thickness=-1.0), dict(thickness=inf), dict(thickness=nan),
           dict(sampleSpacing=0.0), dict(sampleSpacing=-1.0), dict(sampleSpacing=inf), dict(sampleSpacing=nan),
           dict(thickness=65537.0, sampleSpacing=1.0), dict(windowWidth=0.0), dict(windowWidth=-1.0), dict(windowWidth=inf),
           dict(windowWidth=nan), dict(windowCenter=nan)]
    for kw in bad:
        rc, msg = call(**kw)
        assert rc != 0, kw
        assert "svr_render_slices" in msg, (kw, msg)


def _volume(dims, spacing=(1.0, 1.0, 1.0), fmt=L.VOXEL_U16, seed=3):
    """Random voxels (z, y, x) and their normalised values."""
    rng = np.random.default_rng(seed)
    nx, ny, nz = dims
    d = rng.random((nz, ny, nx), dtype=np.float32)
    vox = S.encode_voxels(d, fmt)
    norm = {L.VOXEL_U8: 255.0, L.VOXEL_U16: 65535.0}.get(fmt, 1.0)
    return vox, (vox.astype(np.float32) / np.float32(norm)).astype(np.float32)


def _orc(vox, fmt, dims, spacing=(1.0, 1.0, 1.0), vol=None):
    vol = vol or S.host_volume_struct(dims, spacing)
    return SO.oracle(vox, fmt, dims, vol), vol


DIMS, SPACING = (20, 14, 10), (0.8, 1.0, 1.3)  # non-cubic, anisotropic


def plane(ref, axis, index):
    """The voxels (z, y, x) of an axis slice in its image layout (V rows, U columns)."""
    return {"z": lambda: ref[index], "y": lambda: ref[:, index, :], "x": lambda: ref[:, :, index]}[axis]()


@pytest.mark.parametrize("fmt", [L.VOXEL_U8, L.VOXEL_F32])
def test_axis_slices_are_the_voxels_of_their_plane(fmt):
    vox, ref = _volume(DIMS, SPACING, fmt)
    orc, _ = _orc(vox, fmt, DIMS, SPACING)
    for axis, index in (("z", 4), ("y", 9), ("x", 13)):
        value, u8 = SO.slices(orc, S.axis_slice(DIMS, SPACING, axis, index))
        want = plane(ref, axis, index)
        assert value.shape == (1,) + want.shape
        assert np.abs(value[0] - want).max() <= np.spacing(np.float32(1)), axis  # a fetch at a texel centre has weights 0 and 1
        assert np.all(u8[..., 3] == 255)


def test_a_stack_of_every_axial_slice_is_the_volume():
    vox, ref = _volume(DIMS, SPACING, L.VOXEL_F32)
    orc, _ = _orc(vox, L.VOXEL_F32, DIMS, SPACING)
    value, _ = SO.slices(orc, S.axis_slice(DIMS, SPACING, "z", 0, count=DIMS[2]))
    assert np.array_equal(value, ref)


def test_whole_depth_slab_gives_column_max_min_and_mean():
    vox, ref = _volume(DIMS, SPACING, L.VOXEL_F32)
    orc, _ = _orc(vox, L.VOXEL_F32, DIMS, SPACING)
    nz = DIMS[2]
    for mode in ("max", "min", "mean"):
        p = S.axis_slice(DIMS, SPACING, "z", 0, thickness_voxels=nz, mode=mode)
        p.center[2] = 0.0  # the volume's middle: the nz samples lie on the nz voxel centres of each column
        value = SO.slices(orc, p)[0][0]
        if mode == "max":
            want = ref.max(axis=0)
        elif mode == "min":
            want = ref.min(axis=0)
        else:
            acc = np.zeros(ref.shape[1:], np.float32)
            for k in range(nz):
                acc = (acc + ref[k]).astype(np.float32)
            want = (acc / np.float32(nz)).astype(np.float32)
        assert np.array_equal(value, want), mode


def test_constant_volume_slab_mean_is_the_constant_under_clip_planes():
    n, c = 24, np.float32(0.37)
    vox = np.full((n, n, n), c, np.float32)
    vol = S.host_volume_struct((n, n, n))
    vol.z_clip = L.Vec2(-0.25, 0.5)
    vol.x_clip = L.Vec2(-1.0, 0.75)
    orc, _ = _orc(vox, L.VOXEL_F32, (n, n, n), vol=vol)
    # an oblique slab far thicker than the clipped box: the clip planes exclude many of its samples
    p = S.oblique_slice((0.0, 0.0, 0.0), (0.3, 0.2, 1.0), (0.0, 1.0, 0.0), 0.5, 32, 32, thickness=3.0 * n, sample_spacing=0.5, mode="mean")
    value, u8 = SO.slices(orc, p)
    hit = u8[..., 3] == 255
    assert hit.mean() > 0.5
    assert np.abs(value[hit] - c).max() <= 1e-6
    assert np.all(value[~hit] == 0)


def test_pixels_outside_the_clipped_box_give_zero_and_alpha_zero():
    n = 16
    vox = np.full((n, n, n), 200, np.uint8)
    vol = S.host_volume_struct((n, n, n))
    vol.x_clip = L.Vec2(-1.0, 0.0)  # x <= 0 only
    orc, _ = _orc(vox, L.VOXEL_U8, (n, n, n), vol=vol)
    for thick in (0, 4):
        p = S.axis_slice((n, n, n), (1, 1, 1), "z", 8, thickness_voxels=thick)
        p.imageW, p.imageH = 2 * n, 2 * n  # twice the box: the outer ring misses it
        value, u8 = SO.slices(orc, p)
        x = (np.arange(2 * n) + 0.5 - n)[None, :]
        y = (np.arange(2 * n) + 0.5 - n)[:, None]
        inside = (x <= 0) & (x >= -n / 2) & (np.abs(y) <= n / 2)
        inside = np.broadcast_to(inside, value[0].shape)
        assert np.all(value[0][~inside] == 0) and np.all(u8[0][~inside] == 0)
        assert np.all(u8[0][inside][:, 3] == 255) and value[0][inside].min() > 0.3


def test_density_scale_two_doubles_the_value_exactly():
    vox, _ = _volume(DIMS, SPACING, L.VOXEL_U8)
    orc1, vol = _orc(vox, L.VOXEL_U8, DIMS, SPACING)
    vol2 = L.Volume.from_buffer_copy(vol)
    vol2.densityScale = 2.0
    orc2, _ = _orc(vox, L.VOXEL_U8, DIMS, SPACING, vol=vol2)
    for mode in ("max", "min", "mean"):
        p = S.oblique_slice((0.5, -0.3, 0.2), (1.0, 0.5, 0.7), (0.0, 0.0, 1.0), 0.7, 24, 20, thickness=5.0, sample_spacing=0.6, mode=mode)
        a, b = SO.slices(orc1, p)[0], SO.slices(orc2, p)[0]
        assert np.array_equal(b, np.float32(2) * a), mode


def test_window_mapping_follows_the_formula():
    vox, _ = _volume(DIMS, SPACING, L.VOXEL_U16)
    orc, _ = _orc(vox, L.VOXEL_U16, DIMS, SPACING)
    for center, width in ((0.5, 1.0), (0.3, 0.2), (0.9, 0.05), (-1.0, 3.5)):
        p = S.oblique_slice((0.0, 0.0, 0.0), (1.0, 1.0, 1.0), (0.0, 1.0, 0.0), 0.6, 40, 30, thickness=3.0, sample_spacing=0.5,
                            window=(center, width))
        value, u8 = SO.slices(orc, p)
        c, w = np.float32(center), np.float32(width)
        g = np.clip((value - (c - np.float32(0.5) * w)) / w, np.float32(0), np.float32(1)).astype(np.float32)
        q = (np.float32(255) * g).astype(np.int32).astype(np.uint8)
        hit = u8[..., 3] == 255
        assert 0.2 < hit.mean() < 1.0
        for ch in range(3):
            assert np.array_equal(u8[..., ch][hit], q[hit]) and np.all(u8[..., ch][~hit] == 0)
    assert len(np.unique(u8[..., 0])) > 2
