// svr_api.cu -- library state, options, the setup_* half of the reference boundary
// (pathtracer.cu:34-68), resource builders that mirror the reference's loaders, synthetic volume
// generators (SURVEY.md section 8d), gradient-magnitude reduction, counters, tap microbenchmarks.
#include <cuda_fp16.h>

#include <cstring>
#include <vector>

#include "svr_generate.cuh"
#include "svr_state.h"

namespace svr {

// SVR_OPT_PT_DENOISE: off, or the guide rays per pixel svr_pathtracer_guides takes
static bool denoise_value_ok(long v) { return v == 0 || v == 1 || v == 4 || v == 16; }

HostState& state()
{
    static HostState* s = [] {
        HostState* p = new HostState();
        memset(&p->scene, 0, sizeof(p->scene));
        memset(p->options, 0, sizeof(p->options));
        p->options[SVR_OPT_PT_MODE] = 2;
        p->options[SVR_OPT_SHADOW_ESTIMATOR] = 0;
        p->options[SVR_OPT_ENV_ENABLED] = 0;
        p->options[SVR_OPT_MACROCELL_SIZE] = 0;  // chosen from the scene (svr_macrocell.cu: auto_cell)
        p->options[SVR_OPT_RC_SKIP] = 1;
        p->options[SVR_OPT_SEED] = 0x5EED;
        p->options[SVR_OPT_COUNTERS] = 0;
        p->options[SVR_OPT_PT_BLOCK] = 128;
        p->options[SVR_OPT_RC_BLOCK] = 64;  // 16 x 4 pixel tiles: shorter blocks, fuller last wave (1.35 vs 1.40 ms on C2 TF-thin)
        // sample-parallel warp for batches of >= 32 spp (1.37x the megakernel on C3, profiles/r01), megakernel below;
        // the phase-scheduled shape measured 2.5x slower than the megakernel
        p->options[SVR_OPT_PT_KERNEL] = 2;
        p->options[SVR_OPT_LEAP] = 1;
        p->options[SVR_OPT_PT_ENTRY_CACHE] = 1;
        // 0 = chosen per launch (launch_pathtrace): one pixel per warp for launches of 128 samples or more, two below.  While a
        // warp classified its run's pixels itself, runs of 2 were best at every length (8.22 ms on C3 against 8.81 with 1, 8.47
        // with 4); with the classification made once per scene by a kernel of its own the shortest run balances long launches
        // best -- C3 at 256 spp: 7.48 / 7.60 / 7.98 ms for runs of 1 / 2 / 4 pixels, at 128 spp 3.89 / 3.92 / 4.11 -- while short
        // launches still want fewer, longer blocks: 64 spp 2.12 / 2.08 / 2.14, 32 spp 1.24 / 1.15 / 1.17 (tools/gpu_run_length.py)
        p->options[SVR_OPT_PT_WARP_PIXELS] = 0;
        p->options[SVR_OPT_PT_WARP_MIN_SPP] = 32;
        p->options[SVR_OPT_PT_QUEUE_MIN_DEPTH] = 8;
        p->options[SVR_OPT_SETUP_SYNC] = 1;
        p->options[SVR_OPT_PT_LIGHT_CULL] = 1;
        p->options[SVR_OPT_PT_PROFILE] = 0;  // measured slower than shape 2 on every BASELINE configuration (DESIGN.md section 3.1)
        p->options[SVR_OPT_PT_REFILL] = 0;
        p->options[SVR_OPT_PT_PIXEL_CACHE] = 1;
        p->options[SVR_OPT_FUSED_UPLOAD] = 1;
        p->options[SVR_OPT_PT_LOOKAHEAD] = 32;
        p->options[SVR_OPT_PT_DENOISE] = 0;
        svr_denoise_defaults(&p->progParams);
        // A host that only knows the reference's seven entry points (gui/canvas.cpp) cannot call
        // svr_set_option: the same switches are read once from the environment.  `ok`, where given, replaces the range.
        static const struct { const char* name; int key, lo, hi; bool (*ok)(long); } kEnv[] = {
            {"SVR_PT_MODE", SVR_OPT_PT_MODE, 0, 2},           {"SVR_SHADOW_ESTIMATOR", SVR_OPT_SHADOW_ESTIMATOR, 0, 1},
            {"SVR_ENV_ENABLED", SVR_OPT_ENV_ENABLED, 0, 1},   {"SVR_RC_SKIP", SVR_OPT_RC_SKIP, 0, 1},
            {"SVR_SEED", SVR_OPT_SEED, INT32_MIN, INT32_MAX}, {"SVR_PT_KERNEL", SVR_OPT_PT_KERNEL, 0, 5},
            {"SVR_PT_DENOISE", SVR_OPT_PT_DENOISE, 0, 16, denoise_value_ok},
        };
        for (const auto& e : kEnv) {
            const char* v = getenv(e.name);
            if (!v || !*v) continue;
            long x = strtol(v, nullptr, 0);
            if (e.ok ? e.ok(x) : (x >= e.lo && x <= e.hi)) p->options[e.key] = (int)x;
            else fprintf(stderr, "libsvr_b200: ignoring %s=%s (out of range)\n", e.name, v);
        }
        return p;
    }();
    return *s;
}

void DeviceState::reset()
{
    if (volPointTex) cudaDestroyTextureObject(volPointTex);
    if (uploadSurf) cudaDestroySurfaceObject(uploadSurf);
    if (aheadEvReady)
        for (cudaEvent_t e : aheadEv) cudaEventDestroy(e);  // events belong to the device they were created on
    if (tfCheckEvent) cudaEventDestroy(tfCheckEvent);
    if (hMailbox) cudaFreeHost(hMailbox);
    *this = DeviceState();  // the DevBufs swapped out here free themselves
}

int fail(const char* where, cudaError_t e)
{
    char buf[512];
    snprintf(buf, sizeof(buf), "%s: %s (%s)", where, cudaGetErrorString(e), cudaGetErrorName(e));
    state().lastError = buf;
    cudaGetLastError();  // clear the sticky-free error so later calls can proceed
    return (int)e == 0 ? -1 : (int)e;
}

int fail_msg(const char* msg)
{
    state().lastError = msg;
    return -1;
}

}  // namespace svr

using namespace svr;

// ------------------------------------------------------------------------------------------------
// Part 1: setup_* (pathtracer.cu:34-68).  The PODs are copied into the host snapshot that every
// later launch passes as its kernel parameter block; like the reference they return only after
// the device is idle (cudaDeviceSynchronize), except setup_area_lights (pathtracer.cu:57-61).
// ------------------------------------------------------------------------------------------------
// Does `b` describe the same device resources and geometry as `a`?  Everything a slider tick of the canvas leaves
// alone (densityScale, gradientFactor and the clip planes are what gui/canvas.h:49-175 edits between frames).
static bool same_volume_resource(const svr_volume& a, const svr_volume& b)
{
    return a.tex == b.tex && memcmp(&a.bbox, &b.bbox, sizeof(a.bbox)) == 0 && memcmp(&a.spacing, &b.spacing, sizeof(a.spacing)) == 0 &&
           a.invMaxMagnitude == b.invMaxMagnitude;
}

extern "C" void setup_volume(const svr_volume* vol)
{
    HostState& st = state();
    // The macrocell cache is keyed on the cudaArray handle.  A host that follows the reference's flow
    // (VolumeReader::ClearDevice: cudaFreeArray + cudaDestroyTextureObject, then cudaMalloc3DArray for the next
    // volume, core/VolumeReader.cpp:108-122, 138-172) never passes through svr_volume_destroy, and the driver is free
    // to hand the new array and texture object the handle values of the freed ones.  So the handle alone proves
    // nothing: any change of texture handle, box, spacing or gradient normalisation drops the cache (ranges,
    // dims and the point-sampled view bound to the old array); and when the struct is unchanged in all of those a
    // sampled fingerprint of the voxels is compared against the one taken when the ranges were built.
    if (st.dev.gridArray && !same_volume_resource(st.scene.vol, *vol)) release_grid(st);
    st.scene.vol = *vol;
    st.sceneEpoch++;
    st.dev.majorantValid = false;  // densityScale / array may have changed
    st.dev.fingerprintDue = true;  // checked at the next grid use (needs the stream; setup_* must stay cheap)
    if (st.options[SVR_OPT_SETUP_SYNC]) SVR_FATAL(cudaDeviceSynchronize());
}

extern "C" void setup_transferfunction(const svr_transfer_function* tf)
{
    HostState& st = state();
    st.scene.tf = *tf;
    st.sceneEpoch++;
    st.dev.majorantValid = false;  // every TF edit invalidates the local majorants
    if (st.options[SVR_OPT_SETUP_SYNC]) SVR_FATAL(cudaDeviceSynchronize());
}

extern "C" void setup_camera(const svr_camera* cam)
{
    HostState& st = state();
    st.scene.cam = *cam;
    st.sceneEpoch++;
    if (st.options[SVR_OPT_SETUP_SYNC]) SVR_FATAL(cudaDeviceSynchronize());
}

extern "C" void setup_env_lights(const svr_env_light* light)
{
    HostState& st = state();
    st.scene.env = *light;
    st.sceneEpoch++;
    if (st.options[SVR_OPT_SETUP_SYNC]) SVR_FATAL(cudaDeviceSynchronize());
}

extern "C" void setup_area_lights(svr_area_light* lights, uint32_t n)
{
    // the reference overruns its 8-entry constant array for n > 8 (lights.cpp:94 lets a 9th through)
    if (n > SVR_MAX_LIGHT_SOURCES) n = SVR_MAX_LIGHT_SOURCES;
    HostState& st = state();
    st.scene.numLights = n;
    st.sceneEpoch++;
    for (uint32_t i = 0; i < n; ++i) st.scene.lights[i] = lights[i];
}

// ------------------------------------------------------------------------------------------------
// Part 2: library management
// ------------------------------------------------------------------------------------------------
extern "C" int svr_version(void) { return SVR_VERSION; }
extern "C" const char* svr_last_error(void) { return state().lastError.c_str(); }

extern "C" int svr_set_stream(void* cuda_stream)
{
    state().stream = (cudaStream_t)cuda_stream;
    return 0;
}

extern "C" int svr_set_device(int device)
{
    HostState& st = state();
    SVR_TRY(cudaSetDevice(device));
    st.dev.reset();  // derived data lives on the previous device: drop it
    cudaGetLastError();
    st.sceneEpoch++;
    return 0;
}

extern "C" int svr_set_option(int key, int value)
{
    if (key < 0 || key >= SVR_OPT_COUNT_) return fail_msg("svr_set_option: unknown key");
    HostState& st = state();
    switch (key) {
        case SVR_OPT_PT_MODE:
            if (value < 0 || value > 2) return fail_msg("SVR_OPT_PT_MODE must be 0, 1 or 2");
            break;
        case SVR_OPT_MACROCELL_SIZE:
            if (value != 0 && (value < 2 || value > 64 || (value & (value - 1))))
                return fail_msg("SVR_OPT_MACROCELL_SIZE must be 0 (automatic) or a power of two in 2..64");
            if (value != st.options[key]) {
                release_grid(st);
                st.dev.autoCell = 0;
            }
            break;
        case SVR_OPT_PT_BLOCK:
            // the path-tracing kernels are compiled for at most 128 threads per block (register budget)
            if (value != 64 && value != 128) return fail_msg("path-tracer block size must be 64 or 128");
            break;
        case SVR_OPT_RC_BLOCK:
            if (value != 64 && value != 128 && value != 256) return fail_msg("block size must be 64, 128 or 256");
            break;
        case SVR_OPT_PT_KERNEL:
            if (value < 0 || value > 5) return fail_msg("SVR_OPT_PT_KERNEL must be 0 .. 5");
            break;
        case SVR_OPT_PT_WARP_PIXELS:
            if (value < 0 || value > 64) return fail_msg("SVR_OPT_PT_WARP_PIXELS must be in 0..64");
            break;
        case SVR_OPT_PT_WARP_MIN_SPP:
            if (value < 1) return fail_msg("SVR_OPT_PT_WARP_MIN_SPP must be >= 1");
            break;
        case SVR_OPT_PT_QUEUE_MIN_DEPTH:
            if (value < 0) return fail_msg("SVR_OPT_PT_QUEUE_MIN_DEPTH must be >= 0");
            break;
        case SVR_OPT_PT_POOL_PIXELS:
            if (value < 0 || value > 16) return fail_msg("SVR_OPT_PT_POOL_PIXELS must be in 0..16");
            break;
        case SVR_OPT_PT_REFILL:
            if (value < 0 || value > 32) return fail_msg("SVR_OPT_PT_REFILL must be in 0..32");
            break;
        case SVR_OPT_PT_ROUNDS:
            if (value < 0) return fail_msg("SVR_OPT_PT_ROUNDS must be >= 0");
            break;
        case SVR_OPT_PT_DENOISE:
            if (!denoise_value_ok(value)) return fail_msg("SVR_OPT_PT_DENOISE must be 0 (off), 1, 4 or 16");
            break;
        default: break;
    }
    st.options[key] = value;
    st.sceneEpoch++;
    return 0;
}

extern "C" int svr_get_option(int key)
{
    if (key < 0 || key >= SVR_OPT_COUNT_) return -1;
    return state().options[key];
}

extern "C" uint64_t svr_launch_count(void) { return state().launches; }
extern "C" uint64_t svr_fused_upload_count(void) { return state().fusedUploads; }
extern "C" uint64_t svr_lookahead_batch_count(void) { return state().aheadBatches; }

extern "C" int svr_volume_invalidate_cache(void)
{
    release_grid(state());
    return 0;
}

// ------------------------------------------------------------------------------------------------
// counters
// ------------------------------------------------------------------------------------------------
namespace svr {
Counters* device_counters()
{
    HostState& st = state();
    if (!st.dev.counters.p) {
        if (st.dev.counters.reserve(1) != cudaSuccess) return nullptr;
        cudaMemset(st.dev.counters.p, 0, sizeof(Counters));
    }
    return st.dev.counters.p;
}
}  // namespace svr

extern "C" int svr_counters_reset(void)
{
    Counters* c = device_counters();
    if (!c) return fail_msg("svr_counters_reset: allocation failed");
    SVR_TRY(cudaMemsetAsync(c, 0, sizeof(Counters), state().stream));
    return 0;
}

extern "C" int svr_counters_read(uint64_t* host_out, uint32_t n)
{
    Counters* c = device_counters();
    if (!c) return fail_msg("svr_counters_read: allocation failed");
    Counters h;
    SVR_TRY(cudaStreamSynchronize(state().stream));
    SVR_TRY(cudaMemcpy(&h, c, sizeof(h), cudaMemcpyDeviceToHost));
    for (uint32_t i = 0; i < n && i < 16; ++i) host_out[i] = h.v[i];
    return 0;
}

// ------------------------------------------------------------------------------------------------
// resource builders
// ------------------------------------------------------------------------------------------------
static size_t voxel_bytes(int format)
{
    switch (format) {
        case SVR_VOXEL_U8: return 1;
        case SVR_VOXEL_U16: return 2;
        case SVR_VOXEL_F16: return 2;
        case SVR_VOXEL_F32: return 4;
        default: return 0;
    }
}

static cudaChannelFormatDesc voxel_channel(int format)
{
    switch (format) {
        case SVR_VOXEL_U8: return cudaCreateChannelDesc(8, 0, 0, 0, cudaChannelFormatKindUnsigned);
        case SVR_VOXEL_U16: return cudaCreateChannelDesc(16, 0, 0, 0, cudaChannelFormatKindUnsigned);
        case SVR_VOXEL_F16: return cudaCreateChannelDesc(16, 0, 0, 0, cudaChannelFormatKindFloat);
        default: return cudaCreateChannelDesc(32, 0, 0, 0, cudaChannelFormatKindFloat);
    }
}

extern "C" int svr_max_gradient_magnitude(const void* dev_data, int format, uint32_t nx, uint32_t ny, uint32_t nz,
                                          float sx, float sy, float sz, float* host_out);

// core/VolumeReader.cpp:138-185
extern "C" int svr_volume_create(svr_volume* out, const void* data, int data_on_device, int format, uint32_t nx,
                                 uint32_t ny, uint32_t nz, float sx, float sy, float sz, float maxGradMag)
{
    size_t bpe = voxel_bytes(format);
    if (!bpe || !out || !data || !nx || !ny || !nz) return fail_msg("svr_volume_create: bad argument");
    HostState& st = state();
    cudaChannelFormatDesc ch = voxel_channel(format);
    cudaExtent extent = make_cudaExtent(nx, ny, nz);
    cudaArray_t arr = nullptr;
    // surface stores allowed: svr_volume_upload fills the array and reduces the macrocell ranges in one pass (svr_macrocell.cu)
    SVR_TRY(cudaMalloc3DArray(&arr, &ch, extent, cudaArraySurfaceLoadStore));

    cudaMemcpy3DParms cp;
    memset(&cp, 0, sizeof(cp));
    cp.dstArray = arr;
    cp.extent = extent;
    cp.kind = data_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
    cp.srcPtr = make_cudaPitchedPtr(const_cast<void*>(data), nx * bpe, nx, ny);
    cudaError_t e = cudaMemcpy3DAsync(&cp, st.stream);
    if (e != cudaSuccess) {
        cudaFreeArray(arr);
        return fail("cudaMemcpy3DAsync(volume)", e);
    }

    cudaResourceDesc rd;
    memset(&rd, 0, sizeof(rd));
    rd.resType = cudaResourceTypeArray;
    rd.res.array.array = arr;
    cudaTextureDesc td;
    memset(&td, 0, sizeof(td));
    td.addressMode[0] = td.addressMode[1] = td.addressMode[2] = cudaAddressModeBorder;
    td.filterMode = cudaFilterModeLinear;
    // integer formats read as normalised float (VolumeReader.cpp:168); float formats as stored
    td.readMode = (format == SVR_VOXEL_U8 || format == SVR_VOXEL_U16) ? cudaReadModeNormalizedFloat : cudaReadModeElementType;
    td.normalizedCoords = 1;
    cudaTextureObject_t tex = 0;
    e = cudaCreateTextureObject(&tex, &rd, &td, nullptr);
    if (e != cudaSuccess) {
        cudaFreeArray(arr);
        return fail("cudaCreateTextureObject(volume)", e);
    }

    // from here on every error path releases the array and the texture object
    auto drop = [&](int rc) {
        cudaDestroyTextureObject(tex);
        cudaFreeArray(arr);
        return rc;
    };
    if (!(maxGradMag > 0.f)) {
        if (!data_on_device) {
            // stage once on the device for the reduction
            void* tmp = nullptr;
            size_t bytes = (size_t)nx * ny * nz * bpe;
            e = cudaMalloc(&tmp, bytes);
            if (e != cudaSuccess) return drop(fail("cudaMalloc(gradient staging)", e));
            e = cudaMemcpyAsync(tmp, data, bytes, cudaMemcpyHostToDevice, st.stream);
            int rc = e != cudaSuccess ? fail("cudaMemcpyAsync(gradient staging)", e)
                                      : svr_max_gradient_magnitude(tmp, format, nx, ny, nz, sx, sy, sz, &maxGradMag);
            cudaFree(tmp);
            if (rc) return drop(rc);
        } else {
            int rc = svr_max_gradient_magnitude(data, format, nx, ny, nz, sx, sy, sz, &maxGradMag);
            if (rc) return drop(rc);
        }
        if (!(maxGradMag > 0.f)) maxGradMag = 1.f;
    }
    e = cudaStreamSynchronize(st.stream);
    if (e != cudaSuccess) return drop(fail("cudaStreamSynchronize(svr_volume_create)", e));

    memset(out, 0, sizeof(*out));
    float3 size = f3(nx * sx, ny * sy, nz * sz);
    float3 vmax = size - size * 0.5f;  // VolumeReader.cpp:178-180
    out->bbox.vmin = {-vmax.x, -vmax.y, -vmax.z};
    out->bbox.vmax = {vmax.x, vmax.y, vmax.z};
    out->bbox.invSize = {1.f / (vmax.x + vmax.x), 1.f / (vmax.y + vmax.y), 1.f / (vmax.z + vmax.z)};
    out->tex = tex;
    out->densityScale = 1.f;          // gui/canvas.cpp:32
    out->invMaxMagnitude = 1.f / maxGradMag;
    out->gradientFactor = 0.5f;       // gui/canvas.cpp:19
    out->spacing = {sx, sy, sz};
    out->invSpacing = {1.f / sx, 1.f / sy, 1.f / sz};
    out->x_clip = out->y_clip = out->z_clip = {-1.f, 1.f};  // gui/canvas.cpp:31
    return 0;
}

extern "C" int svr_volume_upload(const svr_volume* vol, const void* data, int data_on_device)
{
    if (!vol || !vol->tex || !data) return fail_msg("svr_volume_upload: bad argument");
    HostState& st = state();
    cudaResourceDesc rd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&rd, vol->tex));
    if (rd.resType != cudaResourceTypeArray) return fail_msg("svr_volume_upload: texture is not bound to a cudaArray");
    cudaChannelFormatDesc ch;
    cudaExtent ext;
    unsigned int flags = 0;
    SVR_TRY(cudaArrayGetInfo(&ch, &ext, &flags, rd.res.array.array));
    const size_t bpe = (size_t)(ch.x + ch.y + ch.z + ch.w) / 8;
    bool fused = false;
    if (data_on_device) {
        // one pass: voxels into the array and the macrocell ranges out of the same tile, when the grid exists for this array
        int rc = upload_with_ranges(rd.res.array.array, ch, ext, flags, data, &fused);
        if (rc) return rc;
    }
    if (!fused) {
        cudaMemcpy3DParms cp;
        memset(&cp, 0, sizeof(cp));
        cp.dstArray = rd.res.array.array;
        cp.extent = ext;
        cp.kind = data_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice;
        cp.srcPtr = make_cudaPitchedPtr(const_cast<void*>(data), ext.width * bpe, ext.width, ext.height);
        SVR_TRY(cudaMemcpy3DAsync(&cp, st.stream));
        // same dims, new contents: the grid's allocations stay, its range stage reruns at the next render
        if (rd.res.array.array == st.dev.gridArray) st.dev.rangeValid = false;
    }
    st.dev.uploadEpoch++;
    st.sceneEpoch++;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Staging buffers for streamed, replicated volumes (include/svr_render.h)
// ------------------------------------------------------------------------------------------------
extern "C" int svr_stage_alloc(void** dev_ptr, uint64_t bytes)
{
    if (!dev_ptr || !bytes) return fail_msg("svr_stage_alloc: bad argument");
    SVR_TRY(cudaMalloc(dev_ptr, (size_t)bytes));
    return 0;
}

extern "C" int svr_stage_free(void* dev_ptr)
{
    if (dev_ptr) SVR_TRY(cudaFree(dev_ptr));
    return 0;
}

extern "C" int svr_stage_export(const void* dev_ptr, unsigned char handle_out[64])
{
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    if (!dev_ptr || !handle_out) return fail_msg("svr_stage_export: bad argument");
    cudaIpcMemHandle_t h;
    SVR_TRY(cudaIpcGetMemHandle(&h, const_cast<void*>(dev_ptr)));
    memcpy(handle_out, &h, sizeof(h));
    return 0;
}

extern "C" int svr_stage_import(const unsigned char handle[64], void** peer_ptr)
{
    if (!handle || !peer_ptr) return fail_msg("svr_stage_import: bad argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, sizeof(h));
    // opened from the CURRENT device: the mapping is a peer mapping (NVLink) when the buffer lives on another GPU
    SVR_TRY(cudaIpcOpenMemHandle(peer_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return 0;
}

extern "C" int svr_stage_release(void* peer_ptr)
{
    if (peer_ptr) SVR_TRY(cudaIpcCloseMemHandle(peer_ptr));
    return 0;
}

extern "C" int svr_stage_copy(void* dst, const void* src, uint64_t bytes, void* stream)
{
    if (!dst || !src) return fail_msg("svr_stage_copy: bad argument");
    SVR_TRY(cudaMemcpyAsync(dst, src, (size_t)bytes, cudaMemcpyDefault, (cudaStream_t)stream));
    return 0;
}

// The table half of TransferFunction::TransferFunction (gui/transferfunction.cpp:17-44) for a texture
// that already exists: the reference destroys and recreates array + texture object on every edit
// (transferfunction.cpp:128-151); the contents are all that changes.
extern "C" int svr_tf_upload(svr_transfer_function* tf, const float* host_rgba, uint32_t n)
{
    if (!tf || !tf->tex || !host_rgba) return fail_msg("svr_tf_upload: bad argument");
    HostState& st = state();
    cudaResourceDesc rd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&rd, tf->tex));
    if (rd.resType != cudaResourceTypeArray) return fail_msg("svr_tf_upload: texture is not bound to a cudaArray");
    cudaChannelFormatDesc ch;
    cudaExtent ext;
    unsigned int flags = 0;
    SVR_TRY(cudaArrayGetInfo(&ch, &ext, &flags, rd.res.array.array));
    if (ext.width != n) return fail_msg("svr_tf_upload: table size differs from the bound array");
    SVR_TRY(cudaMemcpy2DToArrayAsync(rd.res.array.array, 0, 0, host_rgba, sizeof(float) * 4 * n, sizeof(float) * 4 * n, 1,
                                     cudaMemcpyHostToDevice, st.stream));
    float maxOpacity = 0.f;
    for (uint32_t i = 0; i < n; ++i) maxOpacity = fmaxf(maxOpacity, host_rgba[4 * i + 3]);
    tf->maxOpacity = maxOpacity;
    st.dev.majorantValid = false;
    st.dev.uploadEpoch++;
    st.sceneEpoch++;
    return 0;
}

extern "C" int svr_volume_destroy(svr_volume* vol)
{
    if (!vol || !vol->tex) return 0;
    HostState& st = state();
    cudaResourceDesc rd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&rd, vol->tex));
    SVR_TRY(cudaDeviceSynchronize());
    if (rd.resType == cudaResourceTypeArray && rd.res.array.array == st.dev.gridArray) release_grid(st);
    SVR_TRY(cudaDestroyTextureObject(vol->tex));
    if (rd.resType == cudaResourceTypeArray) SVR_TRY(cudaFreeArray(rd.res.array.array));
    vol->tex = 0;
    return 0;
}

// gui/transferfunction.cpp:17-44
extern "C" int svr_tf_create(svr_transfer_function* out, const float* host_rgba, uint32_t n)
{
    if (!out || !host_rgba || n < 2) return fail_msg("svr_tf_create: bad argument");
    HostState& st = state();
    cudaChannelFormatDesc ch = cudaCreateChannelDesc(32, 32, 32, 32, cudaChannelFormatKindFloat);
    cudaArray_t arr = nullptr;
    SVR_TRY(cudaMallocArray(&arr, &ch, n));
    cudaError_t e = cudaMemcpy2DToArrayAsync(arr, 0, 0, host_rgba, sizeof(float) * 4 * n, sizeof(float) * 4 * n, 1,
                                             cudaMemcpyHostToDevice, st.stream);
    if (e != cudaSuccess) {
        cudaFreeArray(arr);
        return fail("cudaMemcpy2DToArrayAsync(tf)", e);
    }
    cudaResourceDesc rd;
    memset(&rd, 0, sizeof(rd));
    rd.resType = cudaResourceTypeArray;
    rd.res.array.array = arr;
    cudaTextureDesc td;
    memset(&td, 0, sizeof(td));
    td.addressMode[0] = cudaAddressModeClamp;
    td.filterMode = cudaFilterModeLinear;
    td.normalizedCoords = 1;
    td.readMode = cudaReadModeElementType;
    cudaTextureObject_t tex = 0;
    e = cudaCreateTextureObject(&tex, &rd, &td, nullptr);
    if (e != cudaSuccess) {
        cudaFreeArray(arr);
        return fail("cudaCreateTextureObject(tf)", e);
    }
    float maxOpacity = 0.f;  // transferfunction.cpp:26 (member starts at 0 in the constructor path)
    for (uint32_t i = 0; i < n; ++i) maxOpacity = fmaxf(maxOpacity, host_rgba[4 * i + 3]);
    memset(out, 0, sizeof(*out));
    out->tex = tex;
    out->maxOpacity = maxOpacity;
    SVR_TRY(cudaStreamSynchronize(st.stream));
    return 0;
}

extern "C" int svr_tf_destroy(svr_transfer_function* tf)
{
    if (!tf || !tf->tex) return 0;
    cudaResourceDesc rd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&rd, tf->tex));
    SVR_TRY(cudaDeviceSynchronize());
    if (rd.resType == cudaResourceTypeArray && rd.res.array.array == state().dev.majorantTfArray) {
        state().dev.majorantTfArray = nullptr;
        state().dev.majorantValid = false;
    }
    SVR_TRY(cudaDestroyTextureObject(tf->tex));
    if (rd.resType == cudaResourceTypeArray) SVR_TRY(cudaFreeArray(rd.res.array.array));
    tf->tex = 0;
    return 0;
}

// core/lights/lights.cpp:31-75
extern "C" int svr_env_create(svr_env_light* out, const float* host_rgba, uint32_t w, uint32_t h)
{
    if (!out || !host_rgba || !w || !h) return fail_msg("svr_env_create: bad argument");
    HostState& st = state();
    cudaChannelFormatDesc ch = cudaCreateChannelDesc<float4>();
    cudaArray_t arr = nullptr;
    SVR_TRY(cudaMallocArray(&arr, &ch, w, h));
    cudaError_t e = cudaMemcpy2DToArrayAsync(arr, 0, 0, host_rgba, sizeof(float4) * w, sizeof(float4) * w, h,
                                             cudaMemcpyHostToDevice, st.stream);
    if (e != cudaSuccess) {
        cudaFreeArray(arr);
        return fail("cudaMemcpy2DToArrayAsync(env)", e);
    }
    cudaResourceDesc rd;
    memset(&rd, 0, sizeof(rd));
    rd.resType = cudaResourceTypeArray;
    rd.res.array.array = arr;
    cudaTextureDesc td;
    memset(&td, 0, sizeof(td));
    td.addressMode[0] = td.addressMode[1] = cudaAddressModeWrap;
    td.filterMode = cudaFilterModeLinear;
    td.readMode = cudaReadModeElementType;
    td.normalizedCoords = 1;
    cudaTextureObject_t tex = 0;
    e = cudaCreateTextureObject(&tex, &rd, &td, nullptr);
    if (e != cudaSuccess) {
        cudaFreeArray(arr);
        return fail("cudaCreateTextureObject(env)", e);
    }
    memset(out, 0, sizeof(*out));
    out->tex = tex;          // cudaEnvironmentLight::Set(tex), cuda_environment_light.h:20-25
    out->intensity = 1.f;
    out->offset = {0.f, 0.f};
    SVR_TRY(cudaStreamSynchronize(st.stream));
    return 0;
}

extern "C" int svr_env_destroy(svr_env_light* env)
{
    if (!env || !env->tex) return 0;
    cudaResourceDesc rd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&rd, env->tex));
    SVR_TRY(cudaDeviceSynchronize());
    SVR_TRY(cudaDestroyTextureObject(env->tex));
    if (rd.resType == cudaResourceTypeArray) SVR_TRY(cudaFreeArray(rd.res.array.array));
    env->tex = 0;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// synthetic volumes (SURVEY.md section 8d): device code in svr_generate.cuh
// ------------------------------------------------------------------------------------------------
using namespace svr_gen;

extern "C" int svr_generate_volume(void* dev_out, int kind, int format, uint32_t n, uint32_t seed)
{
    if (!dev_out || !n || kind < 0 || kind > 2) return fail_msg("svr_generate_volume: bad argument");
    HostState& st = state();
    int blocks = 148 * 8, threads = 256;
    switch (format) {
        case SVR_VOXEL_U8: gen_kernel<uint8_t><<<blocks, threads, 0, st.stream>>>((uint8_t*)dev_out, kind, (int)n, seed); break;
        case SVR_VOXEL_U16: gen_kernel<uint16_t><<<blocks, threads, 0, st.stream>>>((uint16_t*)dev_out, kind, (int)n, seed); break;
        case SVR_VOXEL_F16: gen_kernel<__half><<<blocks, threads, 0, st.stream>>>((__half*)dev_out, kind, (int)n, seed); break;
        case SVR_VOXEL_F32: gen_kernel<float><<<blocks, threads, 0, st.stream>>>((float*)dev_out, kind, (int)n, seed); break;
        default: return fail_msg("svr_generate_volume: bad format");
    }
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

extern "C" int svr_max_gradient_magnitude(const void* dev_data, int format, uint32_t nx, uint32_t ny, uint32_t nz,
                                          float sx, float sy, float sz, float* host_out)
{
    if (!dev_data || !host_out) return fail_msg("svr_max_gradient_magnitude: bad argument");
    HostState& st = state();
    unsigned int* dBits = nullptr;
    SVR_TRY(cudaMalloc(&dBits, sizeof(unsigned int)));
    cudaMemsetAsync(dBits, 0, sizeof(unsigned int), st.stream);
    int blocks = 148 * 8, threads = 256;
    float hx = 0.5f / sx, hy = 0.5f / sy, hz = 0.5f / sz;
    switch (format) {
        case SVR_VOXEL_U8: gradmax_kernel<uint8_t><<<blocks, threads, 0, st.stream>>>((const uint8_t*)dev_data, nx, ny, nz, hx, hy, hz, dBits); break;
        case SVR_VOXEL_U16: gradmax_kernel<uint16_t><<<blocks, threads, 0, st.stream>>>((const uint16_t*)dev_data, nx, ny, nz, hx, hy, hz, dBits); break;
        case SVR_VOXEL_F16: gradmax_kernel<__half><<<blocks, threads, 0, st.stream>>>((const __half*)dev_data, nx, ny, nz, hx, hy, hz, dBits); break;
        case SVR_VOXEL_F32: gradmax_kernel<float><<<blocks, threads, 0, st.stream>>>((const float*)dev_data, nx, ny, nz, hx, hy, hz, dBits); break;
        default: cudaFree(dBits); return fail_msg("svr_max_gradient_magnitude: bad format");
    }
    count_launch();
    unsigned int bits = 0;
    cudaError_t e = cudaMemcpyAsync(&bits, dBits, sizeof(bits), cudaMemcpyDeviceToHost, st.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st.stream);
    cudaFree(dBits);
    if (e != cudaSuccess) return fail("svr_max_gradient_magnitude", e);
    memcpy(host_out, &bits, sizeof(float));
    return 0;
}

// ------------------------------------------------------------------------------------------------
// gather-roofline microbenchmarks: independent tex3D taps, coherent (neighbouring threads walk
// neighbouring rays) or random (hashed coordinates), no dependent arithmetic between taps.
// ------------------------------------------------------------------------------------------------
namespace {
__global__ void taps_kernel(svr_volume vol, int random, uint32_t tapsPerThread, float* sink)
{
    uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    float acc = 0.f;
    if (random) {
        uint32_t h = tid * 0x9E3779B1u + 12345u;
#pragma unroll 8
        for (uint32_t i = 0; i < tapsPerThread; ++i) {
            h = h * 1664525u + 1013904223u;
            uint32_t a = h ^ (h >> 15);
            a *= 0x2C1B3C6Du;
            a ^= a >> 13;
            float u = (float)(a & 0x3ffu) * (1.f / 1024.f);
            float v = (float)((a >> 10) & 0x3ffu) * (1.f / 1024.f);
            float w = (float)((a >> 20) & 0x3ffu) * (1.f / 1024.f);
            acc += tex3D<float>(vol.tex, u, v, w);
        }
    } else {
        // warp = 8x4 pixel tile of a 1024-wide virtual image, marching along +z
        uint32_t warp = tid >> 5, lane = tid & 31;
        uint32_t px = (warp % 128u) * 8u + (lane & 7u), py = ((warp / 128u) % 256u) * 4u + (lane >> 3);
        float u = ((float)px + 0.5f) * (1.f / 1024.f), v = ((float)py + 0.5f) * (1.f / 1024.f);
        float dw = 1.f / (float)tapsPerThread;
#pragma unroll 8
        for (uint32_t i = 0; i < tapsPerThread; ++i) acc += tex3D<float>(vol.tex, u, v, ((float)i + 0.5f) * dw);
    }
    if (acc == 123456.789f) sink[0] = acc;  // keep the taps alive
}
}  // namespace

extern "C" int svr_microbench_taps(const svr_volume* vol, int random, uint32_t threads, uint32_t taps_per_thread,
                                   float* dev_sink, uint64_t* host_taps)
{
    if (!vol || !vol->tex || !dev_sink) return fail_msg("svr_microbench_taps: bad argument");
    uint32_t block = 256, grid = (threads + block - 1) / block;
    taps_kernel<<<grid, block, 0, state().stream>>>(*vol, random, taps_per_thread, dev_sink);
    count_launch();
    SVR_TRY(cudaGetLastError());
    if (host_taps) *host_taps = (uint64_t)grid * block * taps_per_thread;
    return 0;
}

// ------------------------------------------------------------------------------------------------
// Layout study (north_star: "a bricked, Morton-ordered 8/16-bit density layout bound as a 3D texture object or staged
// through shared memory").  The same trilinear taps three ways, so that the choice of storage rests on a measurement:
//   0  the product's path: one TEX on the caller's cudaArray (hardware block-linear tiling, filter in the texture unit);
//   1  software trilinear from a LINEAR copy of the voxels (x fastest): eight loads, weights and the filter in the SM;
//   2  software trilinear from a BRICKED copy: 8 x 8 x 8-voxel bricks, each contiguous, bricks in Morton order.
// Coherent taps (neighbouring lanes walk neighbouring rays) or random ones (hashed positions), no dependent arithmetic
// between taps.  16-bit voxels (u16 or f16 bit patterns: the study is about addresses and sectors, not values).
// ------------------------------------------------------------------------------------------------
namespace {
__device__ __forceinline__ uint32_t part1by2(uint32_t x)  // spreads the low 10 bits: Morton interleave
{
    x &= 0x000003ffu;
    x = (x ^ (x << 16)) & 0xff0000ffu;
    x = (x ^ (x << 8)) & 0x0300f00fu;
    x = (x ^ (x << 4)) & 0x030c30c3u;
    x = (x ^ (x << 2)) & 0x09249249u;
    return x;
}

__device__ __forceinline__ size_t brick_index(int x, int y, int z)
{
    const uint32_t m = part1by2((uint32_t)x >> 3) | (part1by2((uint32_t)y >> 3) << 1) | (part1by2((uint32_t)z >> 3) << 2);
    return (size_t)m * 512u + (size_t)(((z & 7) << 6) | ((y & 7) << 3) | (x & 7));
}

__global__ void brick_reorder_kernel(const uint16_t* __restrict__ lin, uint16_t* __restrict__ bricked, int n)
{
    const size_t total = (size_t)n * n * n;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int x = (int)(i % n), y = (int)((i / n) % n), z = (int)(i / ((size_t)n * n));
        bricked[brick_index(x, y, z)] = lin[i];
    }
}

template <int LAYOUT>
__device__ __forceinline__ float voxel_at(const uint16_t* __restrict__ v, int n, int x, int y, int z)
{
    if ((unsigned)x >= (unsigned)n || (unsigned)y >= (unsigned)n || (unsigned)z >= (unsigned)n) return 0.f;  // border addressing
    const size_t i = LAYOUT == 1 ? ((size_t)z * n + y) * n + x : brick_index(x, y, z);
    return (float)__ldg(v + i) * (1.f / 65535.f);
}

template <int LAYOUT>
__device__ __forceinline__ float soft_tap(const uint16_t* __restrict__ v, int n, float u, float w1, float w2)
{
    const float xb = u * (float)n - 0.5f, yb = w1 * (float)n - 0.5f, zb = w2 * (float)n - 0.5f;
    const float fx = floorf(xb), fy = floorf(yb), fz = floorf(zb);
    const int x = (int)fx, y = (int)fy, z = (int)fz;
    const float a = xb - fx, b = yb - fy, c = zb - fz;
    const float v000 = voxel_at<LAYOUT>(v, n, x, y, z), v100 = voxel_at<LAYOUT>(v, n, x + 1, y, z);
    const float v010 = voxel_at<LAYOUT>(v, n, x, y + 1, z), v110 = voxel_at<LAYOUT>(v, n, x + 1, y + 1, z);
    const float v001 = voxel_at<LAYOUT>(v, n, x, y, z + 1), v101 = voxel_at<LAYOUT>(v, n, x + 1, y, z + 1);
    const float v011 = voxel_at<LAYOUT>(v, n, x, y + 1, z + 1), v111 = voxel_at<LAYOUT>(v, n, x + 1, y + 1, z + 1);
    const float x00 = v000 + a * (v100 - v000), x10 = v010 + a * (v110 - v010), x01 = v001 + a * (v101 - v001), x11 = v011 + a * (v111 - v011);
    const float y0 = x00 + b * (x10 - x00), y1 = x01 + b * (x11 - x01);
    return y0 + c * (y1 - y0);
}

template <int LAYOUT>
__global__ void soft_taps_kernel(const uint16_t* __restrict__ v, int n, int random, uint32_t tapsPerThread, float* sink)
{
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    float acc = 0.f;
    if (random) {
        uint32_t h = tid * 0x9E3779B1u + 12345u;
#pragma unroll 4
        for (uint32_t i = 0; i < tapsPerThread; ++i) {
            h = h * 1664525u + 1013904223u;
            uint32_t a = h ^ (h >> 15);
            a *= 0x2C1B3C6Du;
            a ^= a >> 13;
            acc += soft_tap<LAYOUT>(v, n, (float)(a & 0x3ffu) * (1.f / 1024.f), (float)((a >> 10) & 0x3ffu) * (1.f / 1024.f),
                                    (float)((a >> 20) & 0x3ffu) * (1.f / 1024.f));
        }
    } else {
        const uint32_t warp = tid >> 5, lane = tid & 31;
        const uint32_t px = (warp % 128u) * 8u + (lane & 7u), py = ((warp / 128u) % 256u) * 4u + (lane >> 3);
        const float u = ((float)px + 0.5f) * (1.f / 1024.f), w1 = ((float)py + 0.5f) * (1.f / 1024.f), dw = 1.f / (float)tapsPerThread;
#pragma unroll 4
        for (uint32_t i = 0; i < tapsPerThread; ++i) acc += soft_tap<LAYOUT>(v, n, u, w1, ((float)i + 0.5f) * dw);
    }
    if (acc == 123456.789f) sink[0] = acc;
}
}  // namespace

extern "C" int svr_layout_brick(const void* dev_linear, void* dev_bricked, uint32_t n)
{
    if (!dev_linear || !dev_bricked || !n || (n & 7u) || n > 8192u) return fail_msg("svr_layout_brick: n must be a multiple of 8 (at most 8192)");
    brick_reorder_kernel<<<148 * 8, 256, 0, state().stream>>>((const uint16_t*)dev_linear, (uint16_t*)dev_bricked, (int)n);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

extern "C" int svr_microbench_soft_taps(const void* dev_voxels16, uint32_t n, int layout, int random, uint32_t threads, uint32_t taps_per_thread,
                                        float* dev_sink, uint64_t* host_taps)
{
    if (!dev_voxels16 || !dev_sink || !n || (layout != 1 && layout != 2)) return fail_msg("svr_microbench_soft_taps: bad argument");
    const uint32_t block = 256, grid = (threads + block - 1) / block;
    if (layout == 1) soft_taps_kernel<1><<<grid, block, 0, state().stream>>>((const uint16_t*)dev_voxels16, (int)n, random, taps_per_thread, dev_sink);
    else soft_taps_kernel<2><<<grid, block, 0, state().stream>>>((const uint16_t*)dev_voxels16, (int)n, random, taps_per_thread, dev_sink);
    count_launch();
    SVR_TRY(cudaGetLastError());
    if (host_taps) *host_taps = (uint64_t)grid * block * taps_per_thread;
    return 0;
}
