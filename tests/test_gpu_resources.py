"""GPU tests of the resource builders and synthetic generators behind the render path."""
import ctypes as C

import numpy as np
import pytest
import torch

from sunvolumerender_b200 import _lib as L
from sunvolumerender_b200 import scene as S

from _gpu_common import OracleRef, raycast_f32, ref_cuda, setup, small_config

pytestmark = pytest.mark.gpu


def test_generators_are_deterministic_and_match_host_formula(renderer):
    n = 32
    a = renderer.generate_volume(L.GEN_SPHERE, L.VOXEL_U8, n).cpu().numpy().reshape(n, n, n)
    b = renderer.generate_volume(L.GEN_SPHERE, L.VOXEL_U8, n).cpu().numpy().reshape(n, n, n)
    assert np.array_equal(a, b)
    host = S.sphere_volume(n, L.VOXEL_U8)
    assert np.abs(a.astype(int) - host.astype(int)).max() <= 1  # fast-math sqrt/div vs numpy
    ct = renderer.generate_volume(L.GEN_CT, L.VOXEL_U16, n, 1234).cpu().numpy().view(np.uint16)
    ct2 = renderer.generate_volume(L.GEN_CT, L.VOXEL_U16, n, 99).cpu().numpy().view(np.uint16)
    assert ct.max() > 40000 and (ct == 0).mean() > 0.2  # bone present, air exactly zero
    assert not np.array_equal(ct, ct2)
    cloud = renderer.generate_volume(L.GEN_CLOUD, L.VOXEL_F16, n, 42).cpu().numpy().view(np.float16)
    assert 0 < cloud.max() <= 1.0 and cloud.min() == 0.0


@pytest.mark.parametrize("fmt", [L.VOXEL_U8, L.VOXEL_U16, L.VOXEL_F32])
def test_max_gradient_magnitude(renderer, fmt):
    """VolumeReader.cpp:70-76 semantics: max central-difference gradient magnitude of the raw data."""
    n = 24
    rng = np.random.default_rng(3)
    d = rng.uniform(0, 1, (n, n, n)).astype(np.float32)
    vox = S.encode_voxels(d, fmt)
    raw = vox.astype(np.float64) * {L.VOXEL_U8: 257.0, L.VOXEL_U16: 1.0, L.VOXEL_F32: 65535.0}[fmt]
    sx, sy, sz = 1.0, 2.0, 0.5
    p = np.pad(raw, 1, mode="edge")
    gx = (p[1:-1, 1:-1, 2:] - p[1:-1, 1:-1, :-2]) * 0.5 / sx
    gy = (p[1:-1, 2:, 1:-1] - p[1:-1, :-2, 1:-1]) * 0.5 / sy
    gz = (p[2:, 1:-1, 1:-1] - p[:-2, 1:-1, 1:-1]) * 0.5 / sz
    expect = np.sqrt(gx * gx + gy * gy + gz * gz).max()
    dev = torch.from_numpy(vox.view(np.uint8).reshape(-1)).cuda()
    out = C.c_float()
    L.check(renderer.lib.svr_max_gradient_magnitude(C.c_void_p(dev.data_ptr()), fmt, n, n, n, sx, sy, sz, C.byref(out)))
    assert out.value == pytest.approx(expect, rel=1e-4)


def test_volume_from_host_equals_volume_from_device(renderer):
    cfg = small_config(n=48, w=64, h=64, gen=L.GEN_CT, fmt=L.VOXEL_U16)
    vox = setup(renderer, cfg)
    a = raycast_f32(renderer).clone()
    inv_a = renderer.volume.invMaxMagnitude
    renderer.load_volume(vox, cfg.fmt, (cfg.n,) * 3)  # host numpy path (H2D inside the C ABI)
    b = raycast_f32(renderer)
    assert torch.equal(a, b)
    assert renderer.volume.invMaxMagnitude == inv_a
    v = renderer.volume
    assert (v.bbox.vmin.x, v.bbox.vmax.x) == (-24.0, 24.0)
    assert v.densityScale == 1.0 and v.gradientFactor == 0.5 and v.x_clip.x == -1.0


def test_texture_fetch_matches_oracle_sampler(renderer, oracle_cpu):
    """The hardware linear filter, with its 8-bit weights, against the oracle's software sampler --
    this is what pins oracle/svr_oracle.cpp's filterMode 0."""
    n = 16
    rng = np.random.default_rng(5)
    vox = rng.integers(0, 65536, (n, n, n), dtype=np.uint16)
    renderer.load_volume(vox, L.VOXEL_U16, (n, n, n), max_grad_mag=1.0)
    tf = S.tf_table("default")
    renderer.set_transfer_function(tf)
    m = 20000
    uvw = rng.uniform(-0.1, 1.1, (m, 3)).astype(np.float32)
    d_uvw = torch.from_numpy(uvw).cuda()
    d_o = torch.zeros(m, dtype=torch.float32, device="cuda")
    L.check(renderer.lib.svr_debug_sample_volume(C.byref(renderer.volume), C.c_void_p(d_uvw.data_ptr()), m, C.c_void_p(d_o.data_ptr())))
    got = d_o.cpu().numpy()
    o = oracle_cpu.CpuOracle(vox, L.VOXEL_U16, (n, n, n), renderer.volume, tf, S.default_camera((n,) * 3, 16, 16))
    lib = oracle_cpu.cpu()
    expect = np.array([lib.svr_oracle_tex3d(C.byref(o.scene), float(a), float(b), float(c)) for a, b, c in uvw], np.float32)
    d = np.abs(got - expect)
    assert (d < 2e-6).mean() > 0.995  # a weight lands on a rounding tie for a handful of samples
    assert d.max() < 1.0 / 256 + 1e-6
    xs = rng.uniform(-0.05, 1.05, 5000).astype(np.float32)
    d_x = torch.from_numpy(xs).cuda()
    d_t = torch.zeros(5000 * 4, dtype=torch.float32, device="cuda")
    L.check(renderer.lib.svr_debug_sample_tf(C.byref(renderer.tf), C.c_void_p(d_x.data_ptr()), 5000, C.c_void_p(d_t.data_ptr())))
    got_tf = d_t.view(5000, 4).cpu().numpy()
    out = np.zeros(4, np.float32)
    exp_tf = np.zeros((5000, 4), np.float32)
    for i, x in enumerate(xs):
        lib.svr_oracle_tf(C.byref(o.scene), float(x), out.ctypes.data)
        exp_tf[i] = out
    assert np.abs(got_tf - exp_tf).max() < 2e-6 + np.abs(np.diff(tf, axis=0)).max() / 256


def test_error_paths_return_codes_not_exit(renderer):
    lib = renderer.lib
    vol = L.Volume()
    assert lib.svr_volume_create(C.byref(vol), None, 0, L.VOXEL_U8, 4, 4, 4, 1.0, 1.0, 1.0, 1.0) != 0
    assert b"svr_volume_create" in lib.svr_last_error()
    assert lib.svr_pathtracer_accumulate(None, 1, 0, 1, 1) != 0
    assert lib.svr_counters_reset() == 0


def test_upload_into_bound_resources_equals_fresh_load(renderer):
    """svr_volume_upload / svr_tf_upload replace contents behind the same handles (what bench.py's e2e
    step does every step); derived data (macrocell ranges, majorants) must follow."""
    cfg = small_config(n=48, w=96, h=64, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    vox = setup(renderer, cfg)

    def render():
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(4, 2)
        rc = raycast_f32(renderer).clone()
        torch.cuda.synchronize()
        return renderer.hdr_image().clone(), rc

    pt_a, rc_a = render()
    # different voxels and table through the same handles
    other = (vox[::-1, :, ::-1] // 2).copy()
    renderer.upload_volume(other)
    renderer.set_transfer_function(S.tf_table("thin"))
    pt_b, rc_b = render()
    assert not torch.equal(pt_a, pt_b) and not torch.equal(rc_a, rc_b)
    # fresh load of the same data gives the same images bit for bit
    renderer.load_volume(other, cfg.fmt, (cfg.n,) * 3, max_grad_mag=1.0 / renderer.volume.invMaxMagnitude)
    L.check(renderer.lib.svr_tf_destroy(C.byref(renderer.tf)))
    renderer.tf = None  # force a new array + texture
    renderer.set_transfer_function(S.tf_table("thin"))
    pt_c, rc_c = render()
    assert torch.equal(pt_b, pt_c) and torch.equal(rc_b, rc_c)
    # and back again
    renderer.upload_volume(torch.from_numpy(vox.copy()).cuda().view(torch.uint8))
    renderer.set_transfer_function(S.tf_table(cfg.tf))
    pt_d, rc_d = render()
    assert torch.equal(pt_a, pt_d) and torch.equal(rc_a, rc_d)


@pytest.mark.parametrize("fmt", [L.VOXEL_U8, L.VOXEL_U16, L.VOXEL_F16, L.VOXEL_F32])
@pytest.mark.parametrize("cell", [2, 4, 8, 16])
@pytest.mark.parametrize("dims", [(45, 38, 29), (64, 21, 19)])  # x, y, z; rows of a multiple of 32 voxels take the 16-byte kernel
def test_range_grid_follows_uploads_from_host_and_device(renderer, fmt, cell, dims):
    """The macrocell ranges after svr_volume_upload (host or device source) are those of a fresh load of
    the same voxels, float for float -- every u8 / u16 value, a volume whose dimensions are not multiples
    of the cell (zero border), every brick-kernel cell size.  A device source takes the one-pass kernel that fills
    the array and reduces the ranges together (SVR_OPT_FUSED_UPLOAD): same array contents, same ranges as the copy +
    read-back path."""
    rng = np.random.default_rng(11)
    nvox = dims[0] * dims[1] * dims[2]
    dt = S.VOXEL_DTYPES[fmt]

    def volume(seed):
        r_ = np.random.default_rng(seed)
        if fmt == L.VOXEL_U8:
            v = r_.integers(0, 256, nvox).astype(dt)
            v[:256] = np.arange(256)
        elif fmt == L.VOXEL_U16:
            v = r_.integers(0, 65536, nvox).astype(dt)
            v[:16384] = np.arange(0, 65536, 4) + seed % 4
        else:
            v = r_.random(nvox).astype(dt)
        v = v.reshape(dims[2], dims[1], dims[0])
        v[:, :, : dims[0] // 3] = 0  # an empty region
        return v

    def ranges():
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(1, 1)  # brings the grid up to date
        torch.cuda.synchronize()
        g, c = (C.c_int32 * 3)(), C.c_int32()
        L.check(renderer.lib.svr_grid_info(g, C.byref(c)))
        assert c.value == cell
        out = np.zeros((g[2], g[1], g[0], 2), np.float32)
        L.check(renderer.lib.svr_grid_copy(None, C.c_void_p(out.ctypes.data)))
        return out

    a, b = volume(1), volume(2)
    setup(renderer, small_config(n=16, w=32, h=32))
    renderer.set_option(L.OPT_MACROCELL_SIZE, cell)
    renderer.load_volume(a, fmt, dims, max_grad_mag=1000.0)
    renderer.set_camera(S.default_camera(dims, 32, 32))
    ra_tex = ranges()                                    # fresh load
    renderer.upload_volume(b)                            # host source
    rb_tex = ranges()
    assert not np.array_equal(ra_tex, rb_tex)
    fused0 = renderer.lib.svr_fused_upload_count()
    renderer.upload_volume(torch.from_numpy(a.copy()).cuda().view(torch.uint8))   # device source: one pass
    ra_lin = ranges()
    assert np.array_equal(renderer.download_volume(dims, dt).view(np.uint8), a.view(np.uint8))
    renderer.upload_volume(torch.from_numpy(b.copy()).cuda().view(torch.uint8))
    rb_lin = ranges()
    assert np.array_equal(renderer.download_volume(dims, dt).view(np.uint8), b.view(np.uint8))
    assert renderer.lib.svr_fused_upload_count() == fused0 + 2
    assert np.array_equal(ra_tex.view(np.uint32), ra_lin.view(np.uint32))
    assert np.array_equal(rb_tex.view(np.uint32), rb_lin.view(np.uint32))
    renderer.set_option(L.OPT_FUSED_UPLOAD, 0)                                    # device source: copy, ranges from the array
    renderer.upload_volume(torch.from_numpy(a.copy()).cuda().view(torch.uint8))
    assert np.array_equal(ranges().view(np.uint32), ra_lin.view(np.uint32))
    assert renderer.lib.svr_fused_upload_count() == fused0 + 2
    renderer.set_option(L.OPT_FUSED_UPLOAD, 1)
    assert ra_lin[..., 0].min() == 0.0 and ra_lin[..., 1].max() > 0.9
    # against numpy on the same voxels, every cell (the last one of each axis partial): min / max over texels cC-1 .. (c+1)C with
    # a zero border
    norm = {L.VOXEL_U8: 255.0, L.VOXEL_U16: 65535.0}.get(fmt, 1.0)
    for vox, got in ((a, ra_lin), (b, rb_lin)):
        assert got.shape[:3] == tuple(-(-d // cell) for d in dims[::-1])
        pad = np.zeros((dims[2] + 2 * cell + 2, dims[1] + 2 * cell + 2, dims[0] + 2 * cell + 2), np.float64)
        pad[1:1 + dims[2], 1:1 + dims[1], 1:1 + dims[0]] = vox.astype(np.float64) / norm
        win = np.lib.stride_tricks.sliding_window_view(pad, (cell + 2,) * 3)[::cell, ::cell, ::cell]
        win = win[:got.shape[0], :got.shape[1], :got.shape[2]]
        assert np.array_equal(got[..., 0], win.min(axis=(3, 4, 5)).astype(np.float32))
        assert np.array_equal(got[..., 1], win.max(axis=(3, 4, 5)).astype(np.float32))


def test_volume_stream_equals_direct_uploads(renderer):
    """render.VolumeStream (the transfer of frame i+1 overlapped with the rendering of frame i, what bench.py's
    e2e loop does) renders a sequence of volumes to the same images, bit for bit, as uploading each one directly."""
    from sunvolumerender_b200.render import VolumeStream

    cfg = small_config(n=48, w=96, h=64, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    vox = setup(renderer, cfg)
    frames = [vox.copy(), (vox[::-1, :, ::-1] // 2).copy(), (vox[:, ::-1, :] // 3 * 2).copy(), vox.copy()]

    def render():
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(64, 2)  # the sample-parallel kernel
        return renderer.hdr_image().clone()

    direct = []
    for f in frames:
        renderer.upload_volume(f)
        direct.append(render())
    torch.cuda.synchronize()
    assert not torch.equal(direct[0], direct[1]) and not torch.equal(direct[1], direct[2])

    pinned = [torch.from_numpy(f).view(torch.uint8).reshape(-1).pin_memory() for f in frames]
    vs = VolumeStream(renderer)
    with pytest.raises(RuntimeError):
        vs.bind()
    vs.prefetch(pinned[0])
    streamed = []
    for i in range(len(frames)):
        vs.bind()
        renderer.set_transfer_function(S.tf_table(cfg.tf))  # a frame's setup_* calls come before the prefetch
        if i + 1 < len(frames):
            vs.prefetch(pinned[i + 1])
        streamed.append(render())
    torch.cuda.synchronize()
    for a, b in zip(direct, streamed):
        assert torch.equal(a, b)
    vs.prefetch(pinned[0])
    vs.prefetch(pinned[1])
    with pytest.raises(RuntimeError):
        vs.prefetch(pinned[2])
    torch.cuda.synchronize()


def test_automatic_macrocell_size_follows_the_mean_free_path(renderer):
    """SVR_OPT_MACROCELL_SIZE = 0: an opaque medium (mean free path ~2 voxels) gets 4-voxel cells, a thin
    one large cells; the choice follows transfer-function edits and never changes a ray-cast image."""
    cfg = small_config(n=64, w=96, h=96, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=1)
    setup(renderer, cfg)

    def cell_after_render():
        renderer.frame_no = 0
        renderer.render_pathtracer_spp(2, 1)
        torch.cuda.synchronize()
        dims, cell = (C.c_int32 * 3)(), C.c_int32()
        L.check(renderer.lib.svr_grid_info(dims, C.byref(cell)))
        return cell.value

    renderer.set_option(L.OPT_MACROCELL_SIZE, 8)
    fixed = raycast_f32(renderer).clone()
    assert cell_after_render() == 8
    renderer.set_option(L.OPT_MACROCELL_SIZE, 0)
    assert cell_after_render() == 4                      # TF-default: opacity 0.5 per voxel inside the body
    assert torch.equal(raycast_f32(renderer), fixed)     # skipping only removes exact zeros, whatever the cell size
    renderer.set_transfer_function(S.tf_table("thin"))   # opacity <= 0.02: mean free path > 50 voxels
    assert cell_after_render() == 32
    renderer.set_transfer_function(S.tf_table("cloud"))
    assert cell_after_render() in (8, 16)
    renderer.set_volume_params(density_scale=0.05)       # thinner again through the density scale
    assert cell_after_render() == 32
    renderer.set_option(L.OPT_MACROCELL_SIZE, 8)


def test_application_default_transfer_function_renders_like_the_reference(renderer):
    """The start-up transfer function of the application (gui/mainwindow.cpp:46-62: a sharpness-0.5 opacity
    ramp, not the linear stand-in of the synthetic configurations), built by svr_tf_build_table, edited in
    place, against the reference's kernels on the same table."""
    from _gpu_common import check_paths, check_rgba, oracle_reference

    cfg = small_config(n=64, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    setup(renderer, cfg)
    op, col = S.default_tf_nodes()
    table, mx = S.build_tf_table(op, col)
    renderer.set_transfer_function(table)                      # in-place upload into the bound texture
    assert renderer.tf.maxOpacity == pytest.approx(mx)
    ref = oracle_reference(renderer, cfg, f32=True)
    ref.render_raycasting(S.raycast_step_size())
    mine = raycast_f32(renderer).cpu().numpy()
    check_rgba(mine, ref)
    # an edit of one opacity node (what dragging a point in the CTK widget does) is picked up by both renderers
    op[2], op[3] = (0.2, 0.02, 0.5, 0.0), (0.3, 0.02, 0.5, 0.9)   # the skin (intensity 0.25) turns nearly transparent
    table2, _ = S.build_tf_table(op, col)
    renderer.set_transfer_function(table2)
    ref = oracle_reference(renderer, cfg, f32=True)
    ref.render_raycasting(S.raycast_step_size())
    mine2 = raycast_f32(renderer).cpu().numpy()
    check_rgba(mine2, ref)
    assert np.abs(mine2 - mine).max() > 1e-2
    renderer.set_option(L.OPT_PT_MODE, 0)
    renderer.frame_no = 0
    renderer.render_pathtracer(2)
    ref2 = oracle_reference(renderer, cfg)
    ref2.render_pathtracer(1, 2)
    torch.cuda.synchronize()
    check_paths(renderer.hdr_image().cpu().numpy(), ref2.hdr_image().cpu().numpy(), ref2)


def _cudart():
    import glob
    import os

    cands = glob.glob(os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "lib64", "libcudart.so*"))
    rt = C.CDLL(sorted(cands)[-1])
    rt.cudaGetTextureObjectResourceDesc.argtypes = [C.c_void_p, C.c_uint64]
    rt.cudaDestroyTextureObject.argtypes = [C.c_uint64]
    rt.cudaFreeArray.argtypes = [C.c_void_p]
    return rt


def test_host_that_frees_and_reallocates_the_array_itself_gets_fresh_macrocells(renderer):
    """A host following the reference's own flow (VolumeReader::ClearDevice: cudaDestroyTextureObject + cudaFreeArray,
    then cudaMalloc3DArray for the next volume; core/VolumeReader.cpp:108-122, 138-172) never calls svr_volume_destroy,
    and the new array may get the freed one's handle.  The macrocell cache must not survive that: same dims, same box,
    same gradient normalisation, other voxels -> the image is the one a cold library renders."""
    rt = _cudart()
    cfg = small_config(n=64, w=96, h=96, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=2)
    setup(renderer, cfg)
    r = renderer
    n = cfg.n

    def render():
        r.set_option(L.OPT_PT_MODE, 2)
        r.frame_no = 0
        r.render_pathtracer_spp(33, 2)
        torch.cuda.synchronize()
        return r.hdr_image().clone(), raycast_f32(r).clone()

    vox_a = r.generate_volume(L.GEN_CT, L.VOXEL_U16, n, 1234)
    # volume B: the body moved and thinned, air where A had tissue and the other way round
    host_b = np.roll(vox_a.cpu().numpy().view(np.uint16).reshape(n, n, n), (9, -7, 5), axis=(0, 1, 2)).copy()
    host_b[:, : n // 3] = 0
    reused = 0
    for attempt in range(3):
        r.load_volume(vox_a, cfg.fmt, (n,) * 3, max_grad_mag=1000.0)
        img_a, rc_a = render()   # builds ranges / majorants for A
        old = (int(r.volume.tex), None)
        # the host tears the resources down behind the library's back, as VolumeReader::ClearDevice does
        desc = (C.c_uint64 * 8)()
        assert rt.cudaGetTextureObjectResourceDesc(desc, r.volume.tex) == 0
        arr = desc[1]
        torch.cuda.synchronize()
        assert rt.cudaDestroyTextureObject(r.volume.tex) == 0
        assert rt.cudaFreeArray(C.c_void_p(arr)) == 0
        r.volume = None  # nothing for Renderer.free_volume to destroy
        r.load_volume(host_b, cfg.fmt, (n,) * 3, max_grad_mag=1000.0)   # cudaMalloc3DArray + setup_volume
        assert rt.cudaGetTextureObjectResourceDesc(desc, r.volume.tex) == 0
        reused += int(desc[1] == arr and int(r.volume.tex) == old[0])
        img_b, rc_b = render()
        # ground truth: the same volume with the cache dropped explicitly
        L.check(r.lib.svr_volume_invalidate_cache())
        img_b_cold, rc_b_cold = render()
        assert torch.equal(img_b, img_b_cold) and torch.equal(rc_b, rc_b_cold), f"stale macrocells (attempt {attempt}, handles reused: {reused})"
        assert not torch.equal(img_b, img_a)
    print("array + texture handles reused in", reused, "of 3 attempts")


def test_reference_arm_scene_builder_makes_the_same_scene_without_the_product_library(renderer):
    """bench.py --impl reference builds its volume / transfer function with oracle/ref_scene.cu (plain CUDA runtime, the
    generator's device code shared through svr_generate.cuh): the voxels, the cudaVolume fields and the images the
    reference's kernels render from them are those of the product's resource builders, bit for bit."""
    from oracle import binding as B

    cfg = small_config(n=64, gen=L.GEN_CT, fmt=L.VOXEL_U16, depth=1)
    vox = setup(renderer, cfg)
    rs = B.RefScene(cfg, S.tf_table(cfg.tf))
    try:
        assert np.array_equal(rs.download(np.uint16, cfg.n), vox)
        a, b = rs.volume, renderer.volume
        for f in ("densityScale", "invMaxMagnitude", "gradientFactor"):
            assert getattr(a, f) == getattr(b, f), f
        assert a.bbox.vmin.tuple() == b.bbox.vmin.tuple() and a.bbox.invSize.tuple() == b.bbox.invSize.tuple()
        assert rs.tf.maxOpacity == renderer.tf.maxOpacity
        imgs = []
        for vol, tf in ((rs.volume, rs.tf), (renderer.volume, renderer.tf)):
            ref = ref_cuda(renderer, cfg.width, cfg.height) if B.ref(cfg.width, cfg.height) else OracleRef(renderer, cfg.fmt, (cfg.n,) * 3)
            ref.setup(vol, tf, renderer.camera, renderer.lights, renderer.env)
            ref.render_pathtracer(3, 1)
            imgs.append(ref.hdr_image().clone())
        assert float(imgs[0].max()) > 0 and torch.equal(imgs[0].cpu(), imgs[1].cpu())
    finally:
        rs.close()


def test_raycaster_notices_a_table_edited_behind_an_unchanged_handle(renderer):
    """The reference's host re-creates the transfer-function texture on every edit (gui/transferfunction.cpp:128-151) and
    hands render_raycasting the struct by reference: new contents can sit behind the handle the majorants were built for.
    The drop-in entry point compares the table's hash on every call (one small launch, no host synchronisation: a frame whose
    table differs renders without empty-space skipping, the next call rebuilds)."""
    rt = _cudart()
    rt.cudaMemcpy2DToArray.argtypes = [C.c_void_p, C.c_size_t, C.c_size_t, C.c_void_p, C.c_size_t, C.c_size_t, C.c_size_t, C.c_int]
    cfg = small_config(n=64, w=96, h=96, gen=L.GEN_CT, fmt=L.VOXEL_U16, tf="default")
    setup(renderer, cfg)
    r = renderer
    r.render_raycasting()
    torch.cuda.synchronize()
    before = r.ldr_image().clone()
    launches0 = r.launch_count()
    r.render_raycasting()
    torch.cuda.synchronize()
    assert r.launch_count() - launches0 == 2          # unchanged table: the hash check + the ray-cast kernel, no rebuild
    assert torch.equal(r.ldr_image(), before)
    # new contents behind the same array and texture object, without telling the library: air becomes fog
    table = S.tf_table("thin").copy()
    table[:, 3] = np.maximum(table[:, 3], 0.01)
    desc = (C.c_uint64 * 8)()
    assert rt.cudaGetTextureObjectResourceDesc(desc, r.tf.tex) == 0
    assert rt.cudaMemcpy2DToArray(C.c_void_p(desc[1]), 0, 0, C.c_void_p(table.ctypes.data), table.shape[0] * 16, table.shape[0] * 16, 1, 1) == 0
    r.tf.maxOpacity = float(table[:, 3].max())
    r.render_raycasting()
    torch.cuda.synchronize()
    edited = r.ldr_image().clone()
    assert not torch.equal(edited, before)
    # that call found out on the device (its kernel did not skip); the next one rebuilds the majorants, the one after is back to
    # hash + ray cast -- and all three render the same image
    launches0 = r.launch_count()
    r.render_raycasting()
    torch.cuda.synchronize()
    assert r.launch_count() - launches0 > 2 and torch.equal(r.ldr_image(), edited)
    launches0 = r.launch_count()
    r.render_raycasting()
    torch.cuda.synchronize()
    assert r.launch_count() - launches0 == 2 and torch.equal(r.ldr_image(), edited)
    # ground truth: the same table through the announced path, and without empty-space skipping at all
    r.set_transfer_function(table)
    r.render_raycasting()
    torch.cuda.synchronize()
    assert torch.equal(r.ldr_image(), edited)
    r.set_option(L.OPT_RC_SKIP, 0)
    r.render_raycasting()
    torch.cuda.synchronize()
    assert torch.equal(r.ldr_image(), edited)
    r.set_option(L.OPT_RC_SKIP, 1)


def test_peer_frame_on_one_gpu_is_the_plain_image(renderer):
    """distributed.PeerFrame with a single rank: bands rendered into the stage buffer, frame_done a no-op."""
    from sunvolumerender_b200 import distributed as D

    cfg = small_config(n=48, w=80, h=64, gen=L.GEN_CT, fmt=L.VOXEL_U16, tf="thin")
    setup(renderer, cfg)
    renderer.render_raycasting()
    torch.cuda.synchronize()
    whole = renderer.ldr_image().clone()
    pf = D.PeerFrame(renderer, cfg.width * cfg.height * 4)
    for phase in range(3):   # three "ranks" one after the other on this GPU
        renderer.render_raycasting_bands(phase, 3, img_ptr=pf.img_ptr)
    pf.frame_done()
    assert torch.equal(pf.image().view(cfg.height, cfg.width, 4), whole)
    pf.close()


def test_layout_study_software_taps_read_the_same_voxels(renderer):
    """The layout microbenchmarks (bench.py: layout_study) fetch from a linear and from a Morton-bricked copy of the voxels:
    the bricked copy is a permutation of the linear one, brick by brick (8^3 voxels contiguous)."""
    n = 32
    vox = renderer.generate_volume(L.GEN_CT, L.VOXEL_U16, n, 7)
    bricked = torch.empty_like(vox)
    L.check(renderer.lib.svr_layout_brick(C.c_void_p(vox.data_ptr()), C.c_void_p(bricked.data_ptr()), n))
    torch.cuda.synchronize()
    lin = vox.cpu().numpy().view(np.uint16).reshape(n, n, n)
    br = bricked.cpu().numpy().view(np.uint16)
    assert np.array_equal(np.sort(br), np.sort(lin.reshape(-1)))

    def morton(bx, by, bz):
        m = 0
        for b in range(10):
            m |= ((bx >> b) & 1) << (3 * b) | ((by >> b) & 1) << (3 * b + 1) | ((bz >> b) & 1) << (3 * b + 2)
        return m

    for (bx, by, bz) in ((0, 0, 0), (1, 0, 0), (0, 1, 0), (3, 2, 1), (3, 3, 3)):
        brick = br[morton(bx, by, bz) * 512: morton(bx, by, bz) * 512 + 512].reshape(8, 8, 8)
        assert np.array_equal(brick, lin[bz * 8: bz * 8 + 8, by * 8: by * 8 + 8, bx * 8: bx * 8 + 8])
    sink = torch.zeros(4, dtype=torch.float32, device="cuda")
    taps = C.c_uint64(0)
    for layout, buf in ((1, vox), (2, bricked)):
        for rnd in (0, 1):
            L.check(renderer.lib.svr_microbench_soft_taps(C.c_void_p(buf.data_ptr()), n, layout, rnd, 4096, 16, C.c_void_p(sink.data_ptr()), C.byref(taps)))
    torch.cuda.synchronize()
    assert taps.value == 4096 * 16
    assert renderer.lib.svr_layout_brick(C.c_void_p(vox.data_ptr()), C.c_void_p(bricked.data_ptr()), 30) != 0   # not a multiple of 8
