// svr_project.cu -- maximum, minimum and average intensity projection (svr_render_projection).
//
// The reference has no projection mode; the sampling rule is this library's own (include/svr_render.h).  Per pixel-centre
// ray, clipped to the volume box and its clip planes and to t >= 0: K = floor((tFar - t0) / h + 1/2) samples at
// t0 + (k + 1/2) h, h = stepSize / 2, each tex3D * densityScale; P = max, min or (fp32 sum in k order) / K; 0 when K = 0.
//
// Skipping (SVR_OPT_RC_SKIP) walks the macrocell range grid along the ray and drops every sample index whose cell cannot
// change the result: MAX a cell whose maximum is at or below the running maximum, MIN a cell whose minimum is at or above
// the running minimum, MEAN a cell whose voxels are all 0 (adding +0 leaves an fp32 sum unchanged).  Max and min are
// order-free and the mean still adds every taken sample in k order, so the result is bit-identical.  Two things make that
// hold:
//   * a cell's range covers every texel a trilinear fetch positioned up to half a voxel outside the cell reads
//     (svr_macrocell.cu stage 1).  The walk assigns sample k..kEnd-1 to the cell of sample k, where kEnd is the first index
//     at or past the ray's exit from that cell: the samples lie inside the cell up to the rounding of t (1e-4 voxel),
//   * the texture unit filters with 8-bit weights and its own arithmetic, the range grid normalises integers with a
//     correctly rounded division: a filtered value may exceed a cell's max (or undercut its min) by an ulp or so, so the
//     bounds are widened by RANGE_MARGIN.
// Positions come from k by a multiplication, never by accumulation, so a sample is where it is whatever was skipped.
#include <cmath>
#include <cstring>

#include "svr_state.h"

namespace svr {
Counters* device_counters();

namespace {

// relative widening of a cell's bound (2^-20, 8 ulps)
constexpr float RANGE_MARGIN = 9.5367431640625e-7f;

struct ProjScene {
    svr_volume vol;
    svr_camera cam;
    const float2* range;  // per cell (min, max) before densityScale
    int gx, gy, gz;
    float3 scale;         // normalised texture coordinate -> cell coordinate
};

template <int OP>
SVR_DEV float fold(float acc, float v)
{
    if (OP == SVR_PROJECT_MAX) return fmaxf(acc, v);
    if (OP == SVR_PROJECT_MIN) return fminf(acc, v);
    return acc + v;
}

template <int OP, bool SKIP, bool COUNT>
__global__ void __launch_bounds__(256) project_kernel(const __grid_constant__ ProjScene s, float stepSize, float windowCenter, float windowWidth,
                                                      uint32_t* __restrict__ img, float* __restrict__ value, uint32_t y0, uint32_t y1,
                                                      uint32_t bandPhase, uint32_t bandStride, Counters* cnt)
{
    const uint2 pix = band_pixel(y0, y1, bandPhase, bandStride);
    const uint32_t idx = pix.x, idy = pix.y;
    LocalCounters<COUNT> lc;
    if (idx < s.cam.imageW && idy < y1) {
        const Ray ray = camera_ray_center(s.cam, idx, idy);
        lc.add(SVR_CNT_PATHS, 1);
        float P = 0.f;
        float tNear, tFar;
        if (intersect_volume(s.vol, ray, &tNear, &tFar)) {
            const float h = stepSize * 0.5f;
            const float t0 = fmaxf(tNear, 0.f);
            // K and the window use the fast-math division (2 ulp): the correctly rounded one is a subroutine call, around which
            // the counting variants spill.  K can then differ by one from the exact formula where (tFar - t0) / h + 1/2 is
            // within 2 ulp of an integer; it is the same with skipping on and off.
            const float span = tFar > t0 ? floorf(__fadd_rn(__fsub_rn(tFar, t0) / h, 0.5f)) : 0.f;
            const uint32_t K = (uint32_t)span;
            const float ds = s.vol.densityScale;
            auto sample = [&](uint32_t k) {
                const float t = __fadd_rn(t0, __fmul_rn((float)k + 0.5f, h));
                const float3 tc = tex_coord(s.vol, ray.orig + t * ray.dir);
                return tex3D<float>(s.vol.tex, tc.x, tc.y, tc.z) * ds;
            };
            float acc = OP == SVR_PROJECT_MAX ? -INFINITY : (OP == SVR_PROJECT_MIN ? INFINITY : 0.f);
            // samples [k, kEnd) into acc: four fetches in flight per lane, folded in k order
            auto take = [&](uint32_t k, uint32_t kEnd) {
                for (; k + 4u <= kEnd; k += 4u) {
                    float v[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) v[u] = sample(k + u);
#pragma unroll
                    for (int u = 0; u < 4; ++u) acc = fold<OP>(acc, v[u]);
                }
                for (; k < kEnd; ++k) acc = fold<OP>(acc, sample(k));
            };
            lc.add(SVR_CNT_STEPS, K);
            if constexpr (!SKIP) {
                take(0u, K);
                lc.add(SVR_CNT_SHADE_TAPS, K);
            } else {
                // the ray in cell coordinates: g(t) = g(t_k) + (t - t_k) dg
                const float3 dg = ray.dir * (f3(s.vol.bbox.invSize) * s.scale);
                const float3 invDg = 1.f / dg;
                uint32_t k = 0;
                while (k < K) {
                    const float t = __fadd_rn(t0, __fmul_rn((float)k + 0.5f, h));
                    const float3 g = tex_coord(s.vol, ray.orig + t * ray.dir) * s.scale;
                    const int cx = min(max((int)floorf(g.x), 0), s.gx - 1);
                    const int cy = min(max((int)floorf(g.y), 0), s.gy - 1);
                    const int cz = min(max((int)floorf(g.z), 0), s.gz - 1);
                    const float ex = ((dg.x > 0.f ? (float)(cx + 1) : (float)cx) - g.x) * invDg.x;
                    const float ey = ((dg.y > 0.f ? (float)(cy + 1) : (float)cy) - g.y) * invDg.y;
                    const float ez = ((dg.z > 0.f ? (float)(cz + 1) : (float)cz) - g.z) * invDg.z;
                    const float tExit = t + fminf(fminf(dg.x != 0.f ? ex : FLT_MAX, dg.y != 0.f ? ey : FLT_MAX), dg.z != 0.f ? ez : FLT_MAX);
                    // first index whose sample lies at or beyond tExit; at least one sample per visit
                    const float kf = ceilf((tExit - t0) / h - 0.5f);
                    const uint32_t kEnd = kf > (float)k ? (kf < (float)K ? (uint32_t)kf : K) : k + 1u;
                    const float2 r = __ldg(s.range + (((size_t)cz * s.gy + cy) * s.gx + cx));
                    lc.add(SVR_CNT_CELLS, 1);
                    bool skip;
                    if (OP == SVR_PROJECT_MEAN) {
                        skip = r.x == 0.f && r.y == 0.f;
                    } else {
                        const float a = r.x * ds, b = r.y * ds;
                        if (OP == SVR_PROJECT_MAX) {
                            const float hi = fmaxf(a, b);
                            skip = hi + fabsf(hi) * RANGE_MARGIN <= acc;
                        } else {
                            const float lo = fminf(a, b);
                            skip = lo - fabsf(lo) * RANGE_MARGIN >= acc;
                        }
                    }
                    if (skip) {
                        lc.add(SVR_CNT_SKIPPED, kEnd - k);
                    } else {
                        take(k, kEnd);
                        lc.add(SVR_CNT_SHADE_TAPS, kEnd - k);
                    }
                    k = kEnd;
                }
            }
            if (K > 0u) P = OP == SVR_PROJECT_MEAN ? __fdiv_rn(acc, (float)K) : acc;
        }
        const size_t offset = (size_t)idy * s.cam.imageW + idx;
        if (value) value[offset] = P;
        if (img) {
            const float g = fminf(fmaxf((P - (windowCenter - 0.5f * windowWidth)) / windowWidth, 0.f), 1.f);
            const float q = 255.f * g;
            img[offset] = pack_u8x4(q, q, q, 255.f);
        }
    }
    lc.flush(cnt);
}

template <int OP, bool SKIP>
void launch_op(bool count, dim3 grid, int block, cudaStream_t stream, const ProjScene& sc, const svr_projection_params& p, uint32_t* img,
               float* value, uint32_t y1, uint32_t phase, uint32_t stride, Counters* cnt)
{
    if (count)
        project_kernel<OP, SKIP, true><<<grid, block, 0, stream>>>(sc, p.stepSize, p.windowCenter, p.windowWidth, img, value, 0u, y1, phase, stride, cnt);
    else
        project_kernel<OP, SKIP, false><<<grid, block, 0, stream>>>(sc, p.stepSize, p.windowCenter, p.windowWidth, img, value, 0u, y1, phase, stride, cnt);
}

template <int OP>
void launch_mode(bool skip, bool count, dim3 grid, int block, cudaStream_t stream, const ProjScene& sc, const svr_projection_params& p,
                 uint32_t* img, float* value, uint32_t y1, uint32_t phase, uint32_t stride, Counters* cnt)
{
    if (skip) launch_op<OP, true>(count, grid, block, stream, sc, p, img, value, y1, phase, stride, cnt);
    else launch_op<OP, false>(count, grid, block, stream, sc, p, img, value, y1, phase, stride, cnt);
}

}  // namespace
}  // namespace svr

using namespace svr;

extern "C" int svr_render_projection(svr_u8vec4* imgOrNull, float* valueOrNull, const svr_volume* volume, const svr_camera* camera,
                                     const svr_projection_params* params, uint32_t phase, uint32_t stride, uint32_t* bandRows)
{
    HostState& st = state();
    if (!volume || !camera || !params) return fail_msg("svr_render_projection: null volume, camera or params");
    if (!imgOrNull && !valueOrNull) return fail_msg("svr_render_projection: both outputs are null");
    const svr_projection_params p = *params;
    if (p.mode < SVR_PROJECT_MAX || p.mode > SVR_PROJECT_MEAN) return fail_msg("svr_render_projection: mode must be 0 (max), 1 (min) or 2 (mean)");
    if (!(p.stepSize > 0.f) || !std::isfinite(p.stepSize)) return fail_msg("svr_render_projection: stepSize must be positive and finite");
    if (!(p.windowWidth > 0.f) || !std::isfinite(p.windowWidth) || !std::isfinite(p.windowCenter))
        return fail_msg("svr_render_projection: windowWidth must be positive and finite, windowCenter finite");
    if (phase >= stride) return fail_msg("svr_render_projection: band phase must be below the band stride");
    const int block = st.options[SVR_OPT_RC_BLOCK];
    const uint32_t tileH = (uint32_t)block / 16u;
    if (bandRows) *bandRows = tileH;

    ProjScene sc;
    memset(&sc, 0, sizeof(sc));
    sc.vol = *volume;
    sc.cam = *camera;
    const bool skip = st.options[SVR_OPT_RC_SKIP] != 0;
    const bool count = st.options[SVR_OPT_COUNTERS] != 0;
    if (skip) {
        int rc = ensure_ranges(*volume, st.options[SVR_OPT_MACROCELL_SIZE]);
        if (rc) return rc;
        sc.range = st.dev.range.p;
        sc.gx = st.dev.gridDims.x;
        sc.gy = st.dev.gridDims.y;
        sc.gz = st.dev.gridDims.z;
        sc.scale = f3((float)st.dev.volDims.x / (float)st.dev.gridCell, (float)st.dev.volDims.y / (float)st.dev.gridCell,
                      (float)st.dev.volDims.z / (float)st.dev.gridCell);
    }
    const uint32_t H = camera->imageH;
    if (H == 0 || camera->imageW == 0) return 0;
    Counters* cnt = count ? device_counters() : nullptr;
    if (count && !cnt) return fail_msg("svr_render_projection: counter allocation failed");
    const uint32_t bands = (H + tileH - 1u) / tileH;
    if (phase >= bands) return 0;
    dim3 grid((camera->imageW + 15u) / 16u, (bands - phase + stride - 1u) / stride);
    uint32_t* img = (uint32_t*)imgOrNull;
    if (p.mode == SVR_PROJECT_MAX) launch_mode<SVR_PROJECT_MAX>(skip, count, grid, block, st.stream, sc, p, img, valueOrNull, H, phase, stride, cnt);
    else if (p.mode == SVR_PROJECT_MIN) launch_mode<SVR_PROJECT_MIN>(skip, count, grid, block, st.stream, sc, p, img, valueOrNull, H, phase, stride, cnt);
    else launch_mode<SVR_PROJECT_MEAN>(skip, count, grid, block, st.stream, sc, p, img, valueOrNull, H, phase, stride, cnt);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}
