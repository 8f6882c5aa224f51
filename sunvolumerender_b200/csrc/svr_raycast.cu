// svr_raycast.cu -- front-to-back emission/absorption ray caster behind render_raycasting
// (raycasting.h:8; kernel_raycasting raycasting.cu:15-67).
//
// Same image as the reference, fewer fetches.  Every sample position t_k of the reference's march
// (t_0 = tNear, t_{k+1} = t_k + stepSize*0.5 accumulated in fp32, raycasting.cu:29,58) is still
// enumerated with the same fp32 additions, so the samples that DO contribute sit at bit-identical
// positions; what is skipped is work whose contribution is exactly zero:
//   * a sample whose TF opacity is exactly 0 adds (1-L.w)*0 to L (raycasting.cu:49-53): its six
//     gradient fetches and the shading are skipped;
//   * a whole macrocell whose majorant is 0 cannot contain a sample with non-zero opacity
//     (svr_macrocell.cu): the march advances t through it with additions only.
// Dims and row stride come from cudaCamera::imageW/H with a bounds guard (the reference uses the
// compile-time WIDTH/HEIGHT, raycasting.cu:19,72).
#include "svr_state.h"

namespace svr {
Counters* device_counters();

namespace {

template <bool SKIP, bool COUNT>
__global__ void __launch_bounds__(256) raycast_kernel(const __grid_constant__ DevScene s, float stepSize, uint32_t* __restrict__ img,
                                                      float4* __restrict__ outf, uint32_t y0, uint32_t y1, uint32_t bandPhase,
                                                      uint32_t bandStride, Counters* cnt, const unsigned int* __restrict__ staleGrid)
{
    const uint2 pix = band_pixel(y0, y1, bandPhase, bandStride);
    const uint32_t idx = pix.x, idy = pix.y;
    const bool inside = idx < s.cam.imageW && idy < y1;
    LocalCounters<COUNT> lc;

    // the majorants may describe an older table than the one bound now (render_raycasting's per-call check): then no skipping
    const bool useGrid = SKIP && (staleGrid == nullptr || *staleGrid == 0u);
    float4 L = make_float4(0.f, 0.f, 0.f, 0.f);
    if (inside) {
        Ray ray = camera_ray_center(s.cam, idx, idy);
        lc.add(SVR_CNT_PATHS, 1);
        float tNear, tFar;
        if (intersect_volume(s.vol, ray, &tNear, &tFar)) {
            const float h = stepSize * 0.5f;
            const float3 camPos = f3(s.cam.pos);
            // ray in macrocell coordinates: g(t) = g0 + t * dg
            const float3 toCell = f3(s.vol.bbox.invSize) * s.grid.scale;
            const float3 dg = ray.dir * toCell;
            const float3 invDg = 1.f / dg;
            float t = tNear;
            while (t <= tFar) {
                float3 p = ray.orig + t * ray.dir;
                float3 tc = tex_coord(s.vol, p);
                if (SKIP && useGrid) {
                    float3 g = tc * s.grid.scale;
                    int cx = min(max((int)floorf(g.x), 0), s.grid.gx - 1);
                    int cy = min(max((int)floorf(g.y), 0), s.grid.gy - 1);
                    int cz = min(max((int)floorf(g.z), 0), s.grid.gz - 1);
                    float sig = s.grid.at(cx, cy, cz);
                    lc.add(SVR_CNT_CELLS, 1);
                    if (sig <= 0.f) {
                        // empty cell, and so is the cube of radius d-1 around it (svr_macrocell.cu stage 3):
                        // distance to the far faces of that cube along the ray
                        const int d = (int)(-sig) > 1 ? (int)(-sig) : 1;
                        float ex = ((dg.x > 0.f ? (float)(cx + d) : (float)(cx - d + 1)) - g.x) * invDg.x;
                        float ey = ((dg.y > 0.f ? (float)(cy + d) : (float)(cy - d + 1)) - g.y) * invDg.y;
                        float ez = ((dg.z > 0.f ? (float)(cz + d) : (float)(cz - d + 1)) - g.z) * invDg.z;
                        float tExit = t + fminf(fminf(dg.x != 0.f ? ex : FLT_MAX, dg.y != 0.f ? ey : FLT_MAX),
                                                dg.z != 0.f ? ez : FLT_MAX);
                        uint32_t skipped = 0;
                        do {
                            t += h;
                            ++skipped;
                        } while (t < tExit && t <= tFar);
                        lc.add(SVR_CNT_SKIPPED, skipped);
                        lc.add(SVR_CNT_STEPS, skipped);
                        continue;
                    }
                }
                float intensity = tex3D<float>(s.vol.tex, tc.x, tc.y, tc.z) * s.vol.densityScale;
                float4 co = tf_at(s.tf, intensity);
                lc.add(SVR_CNT_STEPS, 1);
                lc.add(SVR_CNT_SHADE_TAPS, 1);
                lc.add(SVR_CNT_TF_LOOKUPS, 1);
                if (co.w != 0.f) {
                    float3 gradient = gradient_at(s.vol, p);
                    lc.add(SVR_CNT_SHADE_TAPS, 6);
                    float gm = sqrtf(dot(gradient, gradient));
                    float cosTerm = 1.f, specularTerm = 0.f;
                    if ((double)gm > 1e-3) {  // the reference compares against a double literal (raycasting.cu:41)
                        float3 normal = normalize(gradient);
                        float3 lightDir = normalize(camPos - p);
                        cosTerm = fabsf(dot(normal, lightDir));
                        specularTerm = powf(cosTerm, 30.f);
                    }
                    co.x = co.x * co.w * cosTerm * 0.8f + co.w * specularTerm * 0.2f;
                    co.y = co.y * co.w * cosTerm * 0.8f + co.w * specularTerm * 0.2f;
                    co.z = co.z * co.w * cosTerm * 0.8f + co.w * specularTerm * 0.2f;
                    float k = 1.f - L.w;
                    L.x += k * co.x;
                    L.y += k * co.y;
                    L.z += k * co.z;
                    L.w += k * co.w;
                    if (L.w > 0.95f) break;
                }
                t += h;
            }
        }
        L.x = fminf(L.x, 1.f);
        L.y = fminf(L.y, 1.f);
        L.z = fminf(L.z, 1.f);
        size_t offset = (size_t)idy * s.cam.imageW + idx;
        if (img) img[offset] = pack_u8x4(L.x * 255.f, L.y * 255.f, L.z * 255.f, 255.f * L.w);
        if (outf) outf[offset] = L;
    }
    lc.flush(cnt);
}

int launch_raycast(uint32_t* img, float4* outf, const svr_volume* volume, const svr_transfer_function* tf,
                   const svr_camera* camera, float stepSize, uint32_t y0, uint32_t y1, uint32_t bandPhase = 0, uint32_t bandStride = 1,
                   bool checkTfContent = false)
{
    HostState& st = state();
    if (!volume || !tf || !camera) return fail_msg("render_raycasting: null scene argument");
    DevScene sc = st.scene;  // lights/env unused by the ray caster
    sc.vol = *volume;
    sc.tf = *tf;
    sc.cam = *camera;
    const bool skip = st.options[SVR_OPT_RC_SKIP] != 0;
    const bool count = st.options[SVR_OPT_COUNTERS] != 0;
    const unsigned int* staleGrid = nullptr;
    if (skip) {
        // Empty-space skipping needs majorants of the CURRENT table.  Edits that go through setup_transferfunction /
        // svr_tf_upload, and any change of handle, invalidate them (svr_macrocell.cu).  The reference's own host can also
        // put new contents behind an unchanged handle without telling anybody (gui/transferfunction.cpp:128-151 destroys and
        // re-creates the texture; render_raycasting gets the struct by reference): the drop-in entry point therefore
        // compares a hash of the live table with the hash of the table the majorants came from -- one small launch instead
        // of the six-launch rebuild it used to force on every frame, and no host synchronisation: the verdict reaches this
        // frame's kernel through device memory (stale majorants: it renders without skipping) and the host at the next
        // call, which then rebuilds.
        bool changed = false;
        if (checkTfContent) {
            int rc = tf_check_collect(&changed);  // what the previous call's hash found
            if (rc) return rc;
        }
        int rc = ensure_grid(&sc, /*force=*/changed, /*maxAutoCell=*/8);
        if (rc) return rc;
        if (checkTfContent) {
            rc = tf_check_launch(sc.tf, &staleGrid);  // this frame's table against the one the majorants came from
            if (rc) return rc;
        }
    } else {
        memset(&sc.grid, 0, sizeof(sc.grid));
    }
    if (y1 > camera->imageH) y1 = camera->imageH;
    if (y0 >= y1 || camera->imageW == 0) return 0;
    Counters* cnt = count ? device_counters() : nullptr;
    if (count && !cnt) return fail_msg("render_raycasting: counter allocation failed");
    const int block = st.options[SVR_OPT_RC_BLOCK];
    const uint32_t tileH = (uint32_t)block / 16u;  // block tile = 16 pixels x block/16 rows
    const uint32_t bands = ((y1 - y0) + tileH - 1u) / tileH;
    if (bandStride == 0 || bandPhase >= bandStride) return fail_msg("render_raycasting: band phase must be below the band stride");
    if (bandPhase >= bands) return 0;
    dim3 grid((camera->imageW + 15u) / 16u, (bands - bandPhase + bandStride - 1u) / bandStride);
    if (skip) {
        if (count) raycast_kernel<true, true><<<grid, block, 0, st.stream>>>(sc, stepSize, img, outf, y0, y1, bandPhase, bandStride, cnt, staleGrid);
        else raycast_kernel<true, false><<<grid, block, 0, st.stream>>>(sc, stepSize, img, outf, y0, y1, bandPhase, bandStride, cnt, staleGrid);
    } else {
        if (count) raycast_kernel<false, true><<<grid, block, 0, st.stream>>>(sc, stepSize, img, outf, y0, y1, bandPhase, bandStride, cnt, staleGrid);
        else raycast_kernel<false, false><<<grid, block, 0, st.stream>>>(sc, stepSize, img, outf, y0, y1, bandPhase, bandStride, cnt, staleGrid);
    }
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

}  // namespace
}  // namespace svr

using namespace svr;

// raycasting.h:8 / raycasting.cu:69-75.  Asynchronous, like the reference.
extern "C" void render_raycasting(svr_u8vec4* img, svr_volume* volume, svr_transfer_function* transferFunction,
                                  svr_camera* camera, float stepSize)
{
    int rc = launch_raycast((uint32_t*)img, nullptr, volume, transferFunction, camera, stepSize, 0, camera ? camera->imageH : 0, 0, 1,
                            /*checkTfContent=*/true);
    if (rc) {
        fprintf(stderr, "CUDA error at %s:%d code=%d \"%s\" \n", __FILE__, __LINE__, rc, svr_last_error());
        cudaDeviceReset();
        exit(EXIT_FAILURE);
    }
}

extern "C" int svr_render_raycasting_f32(svr_vec4* out, const svr_volume* volume, const svr_transfer_function* tf,
                                         const svr_camera* camera, float stepSize)
{
    return launch_raycast(nullptr, (float4*)out, volume, tf, camera, stepSize, 0, camera ? camera->imageH : 0);
}

extern "C" int svr_render_raycasting_rows(svr_u8vec4* img, svr_vec4* outOrNull, const svr_volume* volume,
                                          const svr_transfer_function* tf, const svr_camera* camera, float stepSize,
                                          uint32_t y0, uint32_t y1)
{
    return launch_raycast((uint32_t*)img, (float4*)outOrNull, volume, tf, camera, stepSize, y0, y1);
}

extern "C" int svr_render_raycasting_bands(svr_u8vec4* img, svr_vec4* outOrNull, const svr_volume* volume,
                                           const svr_transfer_function* tf, const svr_camera* camera, float stepSize,
                                           uint32_t phase, uint32_t stride, uint32_t* bandRows)
{
    if (bandRows) *bandRows = (uint32_t)state().options[SVR_OPT_RC_BLOCK] / 16u;
    return launch_raycast((uint32_t*)img, (float4*)outOrNull, volume, tf, camera, stepSize, 0, camera ? camera->imageH : 0, phase, stride);
}

// ------------------------------------------------------------------------------------------------
// Completion flags between the GPUs of a box: a rank that has rendered its bands straight into another rank's image
// (a peer mapping of that rank's buffer, svr_stage_export / svr_stage_import) raises the owner's flag, the owner's stream
// waits for all of them -- no collective, no host in the loop.
// ------------------------------------------------------------------------------------------------
namespace svr_peer {
__global__ void peer_signal_kernel(unsigned int* flag)
{
    __threadfence_system();  // this stream's earlier writes into the peer's memory are visible before the flag moves
    atomicAdd_system(flag, 1u);
}

__global__ void peer_wait_kernel(volatile unsigned int* flag, unsigned int expected, unsigned long long timeoutNs)
{
    unsigned long long t0;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
    while ((int)(flag[0] - expected) < 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        if (t - t0 > timeoutNs) {
            flag[1] = 1u;  // gave up: a peer never signalled (the caller reads this word)
            break;
        }
        __nanosleep(200);
    }
    __threadfence_system();
}
}  // namespace svr_peer

extern "C" int svr_peer_signal(void* peer_flag)
{
    if (!peer_flag) return fail_msg("svr_peer_signal: null flag");
    svr_peer::peer_signal_kernel<<<1, 1, 0, state().stream>>>((unsigned int*)peer_flag);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

extern "C" int svr_peer_wait(void* flag, uint32_t expected, uint32_t timeout_ms)
{
    if (!flag) return fail_msg("svr_peer_wait: null flag");
    svr_peer::peer_wait_kernel<<<1, 1, 0, state().stream>>>((volatile unsigned int*)flag, expected, (unsigned long long)timeout_ms * 1000000ull);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}
