"""The product against what the reference's own kernels rendered (tests/golden/reference_kernels.npz, stored by
tests/golden/make_golden.py from oracle/_ref on a B200): the same voxels, transfer function, camera and lights.

This holds the ray caster and the reference-twin path tracer to the reference itself wherever the reference's kernels
are not built; parity tests that have no independent arm use that twin path as their reference (tests/_gpu_common.py::TwinRef).
Tolerances as for the reference's kernels themselves (tests/test_gpu_raycast.py, tests/test_gpu_pathtrace.py): ray
casting within 1e-4 per channel of the float twin and 1 LSB of the u8 image; the twin-mode path trace within 1e-4 on
>= 99.9 % of the pixels of every frame, the image mean within 1e-3, the tone-mapped image within 1 LSB."""
import os

import numpy as np
import pytest
import torch

from oracle import binding as B

from _gpu_common import TWIN_OPTIONS

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def kern():
    return np.load(B.GOLDEN_KERNELS)


@pytest.mark.parametrize("name", ["ct_u16", "sphere_u8", "ct_u8_thin"])
def test_product_renders_what_the_reference_kernels_rendered(renderer, kern, name):
    assert os.path.exists(B.GOLDEN_KERNELS)
    step, depth, frames = B.load_golden_scene(renderer, kern, name)
    out = torch.zeros(renderer.camera.imageH * renderer.camera.imageW * 4, dtype=torch.float32, device="cuda")
    renderer.render_raycasting_f32(out, step, img=renderer.img)
    mine = out.view(renderer.camera.imageH, renderer.camera.imageW, 4).cpu().numpy()
    assert np.abs(mine - kern[f"{name}_rc_f32x255"] / np.float32(255.0)).max() <= 1e-4
    assert np.abs(renderer.ldr_image().cpu().numpy().astype(int) - kern[f"{name}_rc_u8"].astype(int)).max() <= 1

    saved = {k: renderer.get_option(k) for k in TWIN_OPTIONS}
    try:
        for k, v in TWIN_OPTIONS.items():
            renderer.set_option(k, v)
        renderer.frame_no = 0
        for f in range(frames):
            renderer.render_pathtracer(depth)
            torch.cuda.synchronize()
            hdr, ref = renderer.hdr_image().cpu().numpy(), kern[f"{name}_pt_hdr"][f]
            assert (ref.max(axis=2) > 0).mean() > 0.01
            d = np.abs(hdr - ref).max(axis=2)
            assert (d <= 1e-4).mean() >= 0.999, (f, d.max(), (d <= 1e-4).mean())
            assert abs(float(hdr.mean()) - float(ref.mean())) <= 1e-3 * float(ref.mean())
        assert np.abs(renderer.ldr_image().cpu().numpy().astype(int) - kern[f"{name}_pt_u8"].astype(int)).max() <= 1
    finally:
        for k, v in saved.items():
            renderer.set_option(k, v)
