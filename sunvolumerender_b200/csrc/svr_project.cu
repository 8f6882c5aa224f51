// svr_project.cu -- maximum, minimum and average intensity projection (svr_render_projection), the isosurface
// (svr_render_isosurface), which samples the volume the same way (iso_kernel), and slices and slabs (svr_render_slices), which
// fold samples along a plane's normal as the projection folds them along a camera ray (slice_kernel).
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
#include <algorithm>
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

// The walk over the range grid shared by project_kernel, slice_kernel and iso_kernel.  visit(k) is the cell of sample k and
// kEnd, the first index whose sample lies at or beyond the ray's exit from that cell (at least k + 1, at most K); the caller
// drops or takes samples [k, kEnd) and continues at kEnd.
struct CellVisit {
    float2 range;   // the cell's (min, max) before densityScale
    uint32_t kEnd;
};

struct CellWalk {
    float3 dg, invDg;  // the ray in cell coordinates: g(t) = g(t_k) + (t - t_k) dg

    SVR_DEV CellWalk(const ProjScene& s, const Ray& ray)
    {
        dg = ray.dir * (f3(s.vol.bbox.invSize) * s.scale);
        invDg = 1.f / dg;
    }

    SVR_DEV CellVisit visit(const ProjScene& s, const Ray& ray, float t0, float h, uint32_t k, uint32_t K) const
    {
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
        CellVisit c;
        c.kEnd = kf > (float)k ? (kf < (float)K ? (uint32_t)kf : K) : k + 1u;
        c.range = __ldg(s.range + (((size_t)cz * s.gy + cy) * s.gx + cx));
        return c;
    }
};

template <int OP>
SVR_DEV float fold(float acc, float v)
{
    if (OP == SVR_PROJECT_MAX) return fmaxf(acc, v);
    if (OP == SVR_PROJECT_MIN) return fminf(acc, v);
    return acc + v;
}

// The fold of project_kernel and slice_kernel: samples [kBegin, kEnd) of the ray, sample k at t0 + (k + 1/2) h, each
// tex3D * densityScale, folded by OP in k order; with SKIP through the range grid, dropping the samples of every cell that
// cannot change the result.  Counts shade_taps, skipped and cells; the caller counts the steps.
template <int OP, bool SKIP, bool COUNT>
SVR_DEV float fold_samples(const ProjScene& s, const Ray& ray, float t0, float h, uint32_t kBegin, uint32_t kEnd, LocalCounters<COUNT>& lc)
{
    const float ds = s.vol.densityScale;
    auto sample = [&](uint32_t k) {
        const float t = __fadd_rn(t0, __fmul_rn((float)k + 0.5f, h));
        const float3 tc = tex_coord(s.vol, ray.orig + t * ray.dir);
        return tex3D<float>(s.vol.tex, tc.x, tc.y, tc.z) * ds;
    };
    float acc = OP == SVR_PROJECT_MAX ? -INFINITY : (OP == SVR_PROJECT_MIN ? INFINITY : 0.f);
    // samples [k, kStop) into acc: four fetches in flight per lane, folded in k order
    auto take = [&](uint32_t k, uint32_t kStop) {
        for (; k + 4u <= kStop; k += 4u) {
            float v[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) v[u] = sample(k + u);
#pragma unroll
            for (int u = 0; u < 4; ++u) acc = fold<OP>(acc, v[u]);
        }
        for (; k < kStop; ++k) acc = fold<OP>(acc, sample(k));
    };
    if constexpr (!SKIP) {
        take(kBegin, kEnd);
        lc.add(SVR_CNT_SHADE_TAPS, kEnd - kBegin);
    } else {
        const CellWalk walk(s, ray);
        uint32_t k = kBegin;
        while (k < kEnd) {
            const CellVisit c = walk.visit(s, ray, t0, h, k, kEnd);
            const uint32_t kNext = c.kEnd;
            const float2 r = c.range;
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
                lc.add(SVR_CNT_SKIPPED, kNext - k);
            } else {
                take(k, kNext);
                lc.add(SVR_CNT_SHADE_TAPS, kNext - k);
            }
            k = kNext;
        }
    }
    return acc;
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
            lc.add(SVR_CNT_STEPS, K);
            const float acc = fold_samples<OP, SKIP>(s, ray, t0, h, 0u, K, lc);
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

// Isosurface (include/svr_render.h): the first sample at or above iso along the projection's samples, refined by 4 bisection
// steps and a linear interpolation, shaded with the ray caster's headlight.  Skipping drops the samples of cells whose maximum is
// below iso: none of them can be the first hit, and the refinement recomputes the sample before the hit from its index.
template <bool SKIP, bool COUNT>
__global__ void __launch_bounds__(256) iso_kernel(const __grid_constant__ ProjScene s, float stepSize, float iso, float3 color,
                                                  uint32_t* __restrict__ img, float4* __restrict__ surface, uint32_t y1,
                                                  uint32_t bandPhase, uint32_t bandStride, Counters* cnt)
{
    const uint2 pix = band_pixel(0u, y1, bandPhase, bandStride);
    const uint32_t idx = pix.x, idy = pix.y;
    const bool inside = idx < s.cam.imageW && idy < y1;
    LocalCounters<COUNT> lc;
    Ray ray;
    bool found = false;
    float tHit = 0.f;
    if (inside) {
        ray = camera_ray_center(s.cam, idx, idy);
        lc.add(SVR_CNT_PATHS, 1);
        float tNear, tFar;
        if (intersect_volume(s.vol, ray, &tNear, &tFar)) {
            const float h = stepSize * 0.5f;
            const float t0 = fmaxf(tNear, 0.f);
            const float span = tFar > t0 ? floorf(__fadd_rn(__fsub_rn(tFar, t0) / h, 0.5f)) : 0.f;
            const uint32_t K = (uint32_t)span;
            const float ds = s.vol.densityScale;
            auto t_of = [&](uint32_t k) { return __fadd_rn(t0, __fmul_rn((float)k + 0.5f, h)); };
            auto value = [&](float t) {
                const float3 tc = tex_coord(s.vol, ray.orig + t * ray.dir);
                return tex3D<float>(s.vol.tex, tc.x, tc.y, tc.z) * ds;
            };
            // the first index in [k, kEnd) whose value reaches iso (its value in vHit), else kEnd: four fetches in flight per lane
            float vHit = 0.f;
            auto find = [&](uint32_t k, uint32_t kEnd) {
                for (; k + 4u <= kEnd; k += 4u) {
                    float v[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u) v[u] = value(t_of(k + u));
                    int first = 4;
#pragma unroll
                    for (int u = 3; u >= 0; --u)
                        if (v[u] >= iso) first = u, vHit = v[u];
                    if (first < 4) return k + (uint32_t)first;
                }
                for (; k < kEnd; ++k) {
                    const float v = value(t_of(k));
                    if (v >= iso) {
                        vHit = v;
                        return k;
                    }
                }
                return kEnd;
            };
            uint32_t hit = K;
            if constexpr (!SKIP) {
                hit = find(0u, K);
                lc.add(SVR_CNT_SHADE_TAPS, hit < K ? hit + 1u : K);
            } else {
                const CellWalk walk(s, ray);
                for (uint32_t k = 0; k < K;) {
                    const CellVisit c = walk.visit(s, ray, t0, h, k, K);
                    lc.add(SVR_CNT_CELLS, 1);
                    const float top = fmaxf(c.range.x * ds, c.range.y * ds);
                    if (top + fabsf(top) * RANGE_MARGIN < iso) {
                        lc.add(SVR_CNT_SKIPPED, c.kEnd - k);
                    } else {
                        const uint32_t f = find(k, c.kEnd);
                        lc.add(SVR_CNT_SHADE_TAPS, (f < c.kEnd ? f + 1u : c.kEnd) - k);
                        if (f < c.kEnd) {
                            hit = f;
                            break;
                        }
                    }
                    k = c.kEnd;
                }
            }
            lc.add(SVR_CNT_STEPS, hit < K ? hit + 1u : K);
            if (hit < K) {
                found = true;
                tHit = t_of(hit);
                if (hit > 0u) {
                    float lo = t_of(hit - 1u), hi = tHit, vLo = value(lo), vHi = vHit;
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float m = (lo + hi) * 0.5f;
                        const float vm = value(m);
                        if (vm >= iso) {
                            hi = m;
                            vHi = vm;
                        } else {
                            lo = m;
                            vLo = vm;
                        }
                    }
                    tHit = lo + (hi - lo) * (iso - vLo) / (vHi - vLo);
                }
            }
        }
    }
    // the counts are complete (the refinement and gradient taps are not counted): flushed before the shading, which then needs
    // no registers for them
    lc.flush(cnt);
    if (!inside) return;
    uint32_t rgba = 0u;
    float4 surf = make_float4(0.f, 0.f, 0.f, INFINITY);
    if (found) {
        const float3 x = ray.orig + tHit * ray.dir;
        const float3 camPos = f3(s.cam.pos);
        const float3 g = gradient_at(s.vol, x);
        const float gm = sqrtf(dot(g, g));
        float3 n = f3(0.f);
        float cosTerm = 1.f, specularTerm = 0.f;
        if ((double)gm > 1e-3) {  // as the ray caster compares
            n = normalize(g);
            if (dot(n, ray.dir) > 0.f) n = -n;
            cosTerm = fabsf(dot(n, normalize(camPos - x)));
            specularTerm = powf(cosTerm, 30.f);
        }
        const float r = fminf(color.x * cosTerm * 0.8f + specularTerm * 0.2f, 1.f);
        const float gr = fminf(color.y * cosTerm * 0.8f + specularTerm * 0.2f, 1.f);
        const float b = fminf(color.z * cosTerm * 0.8f + specularTerm * 0.2f, 1.f);
        rgba = pack_u8x4(r * 255.f, gr * 255.f, b * 255.f, 255.f);
        surf = make_float4(n.x, n.y, n.z, dot(x - camPos, -f3(s.cam.w)));
    }
    const size_t offset = (size_t)idy * s.cam.imageW + idx;
    if (img) img[offset] = rgba;
    if (surface) surface[offset] = surf;
}

// The plane geometry of svr_render_slices (include/svr_render.h), from the host: n, K, t0 and h of the slab rule, and the
// clipped box [cmin, cmax] turned so that the samples move up it: per component sg = -1 where n < 0, else +1, and
// sg x in [lo, hi] (lo = sg cmin, hi = sg cmax, swapped where sg = -1) iff x in [cmin, cmax].
struct SliceGeom {
    float3 center, u, v, w, n;
    float3 sg, lo, hi;
    uint32_t W, H, K;
    float t0, h;
};

// Slices and slabs (include/svr_render.h): pixel (x, y) of slice blockIdx.z folds the included samples [kLo, kHi) of the ray
// (c, n) with fold_samples.  Each component of x_k = c + s_k n is monotone in k (s_k and the rounded products and sums are), so
// the lower bounds of the turned box hold from kLo on and its upper bounds below kHi; two binary searches find both.  A
// component with n = 0 is constant: its two conditions hold for every k or for none.
template <int OP, bool SKIP, bool COUNT>
__global__ void __launch_bounds__(256) slice_kernel(const __grid_constant__ ProjScene s, const __grid_constant__ SliceGeom g, float windowCenter,
                                                    float windowWidth, uint32_t* __restrict__ img, float* __restrict__ value, Counters* cnt)
{
    const uint2 pix = band_pixel(0u, g.H, 0u, 1u);
    const uint32_t idx = pix.x, idy = pix.y, j = blockIdx.z;
    LocalCounters<COUNT> lc;
    if (idx < g.W && idy < g.H) {
        lc.add(SVR_CNT_PATHS, 1);
        const float fx = __fsub_rn((float)idx + 0.5f, 0.5f * (float)g.W), fy = __fsub_rn((float)idy + 0.5f, 0.5f * (float)g.H);
        Ray ray;
        ray.orig = g.center + fx * g.u + fy * g.v + (float)j * g.w;
        ray.dir = g.n;
        // sg * x_k is non-decreasing in k on every component: "sg x_k >= lo" holds from some k on, "sg x_k <= hi" up to some k
        auto at = [&](uint32_t k) { return g.sg * (ray.orig + __fadd_rn(g.t0, __fmul_rn((float)k + 0.5f, g.h)) * ray.dir); };
        auto rises = [&](uint32_t k) {
            const float3 x = at(k);
            return x.x >= g.lo.x && x.y >= g.lo.y && x.z >= g.lo.z;
        };
        auto falls = [&](uint32_t k) {
            const float3 x = at(k);
            return x.x <= g.hi.x && x.y <= g.hi.y && x.z <= g.hi.z;
        };
        // kLo = the first k in [0, K] with rises(k) (K: none), kHi = the first k in [0, K] without falls(k)
        uint32_t lo = 0u, hi = g.K;
        while (lo < hi) {
            const uint32_t m = (lo + hi) >> 1;
            if (rises(m)) hi = m;
            else lo = m + 1u;
        }
        const uint32_t kLo = lo;
        hi = g.K;
        while (lo < hi) {
            const uint32_t m = (lo + hi) >> 1;
            if (falls(m)) lo = m + 1u;
            else hi = m;
        }
        const uint32_t kHi = lo;
        const uint32_t taken = kHi > kLo ? kHi - kLo : 0u;
        float P = 0.f;
        if (taken > 0u) {
            lc.add(SVR_CNT_STEPS, taken);
            const float acc = fold_samples<OP, SKIP>(s, ray, g.t0, g.h, kLo, kHi, lc);
            P = OP == SVR_PROJECT_MEAN ? __fdiv_rn(acc, (float)taken) : acc;
        }
        // the pixel's place from the launch geometry again: nothing but P and the count stays live across the division, which
        // is a subroutine call (else the MEAN variant spills the pixel around it)
        const uint2 q = band_pixel(0u, g.H, 0u, 1u);
        const size_t offset = ((size_t)blockIdx.z * g.H + q.y) * g.W + q.x;
        if (value) value[offset] = P;
        if (img) {
            uint32_t rgba = 0u;
            if (taken > 0u) {
                const float gr = fminf(fmaxf((P - (windowCenter - 0.5f * windowWidth)) / windowWidth, 0.f), 1.f);
                const float grey = 255.f * gr;
                rgba = pack_u8x4(grey, grey, grey, 255.f);
            }
            img[offset] = rgba;
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

// The scene of a projection, isosurface or slice call (a slice has no camera: cameraOrNull null leaves cam zero); with
// skipping, the range grid (SVR_OPT_MACROCELL_SIZE, else the edge the cache holds for the volume's array, else 8) in its cell
// coordinates.
int make_scene(ProjScene* sc, const svr_volume& volume, const svr_camera* cameraOrNull, bool skip)
{
    HostState& st = state();
    memset(sc, 0, sizeof(*sc));
    sc->vol = volume;
    if (cameraOrNull) sc->cam = *cameraOrNull;
    if (skip) {
        int rc = ensure_ranges(volume, st.options[SVR_OPT_MACROCELL_SIZE]);
        if (rc) return rc;
        sc->range = st.dev.range.p;
        sc->gx = st.dev.gridDims.x;
        sc->gy = st.dev.gridDims.y;
        sc->gz = st.dev.gridDims.z;
        sc->scale = f3((float)st.dev.volDims.x / (float)st.dev.gridCell, (float)st.dev.volDims.y / (float)st.dev.gridCell,
                       (float)st.dev.volDims.z / (float)st.dev.gridCell);
    }
    return 0;
}

// The launch grid of band_pixel for bands phase, phase + stride, ... of tileH rows; false when the call has no pixels.
bool band_grid(const svr_camera& camera, uint32_t tileH, uint32_t phase, uint32_t stride, dim3* grid)
{
    const uint32_t H = camera.imageH;
    if (H == 0 || camera.imageW == 0) return false;
    const uint32_t bands = (H + tileH - 1u) / tileH;
    if (phase >= bands) return false;
    *grid = dim3((camera.imageW + 15u) / 16u, (bands - phase + stride - 1u) / stride);
    return true;
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
    const bool skip = st.options[SVR_OPT_RC_SKIP] != 0;
    const bool count = st.options[SVR_OPT_COUNTERS] != 0;
    if (int rc = make_scene(&sc, *volume, camera, skip)) return rc;
    dim3 grid;
    if (!band_grid(*camera, tileH, phase, stride, &grid)) return 0;
    Counters* cnt = count ? device_counters() : nullptr;
    if (count && !cnt) return fail_msg("svr_render_projection: counter allocation failed");
    const uint32_t H = camera->imageH;
    uint32_t* img = (uint32_t*)imgOrNull;
    if (p.mode == SVR_PROJECT_MAX) launch_mode<SVR_PROJECT_MAX>(skip, count, grid, block, st.stream, sc, p, img, valueOrNull, H, phase, stride, cnt);
    else if (p.mode == SVR_PROJECT_MIN) launch_mode<SVR_PROJECT_MIN>(skip, count, grid, block, st.stream, sc, p, img, valueOrNull, H, phase, stride, cnt);
    else launch_mode<SVR_PROJECT_MEAN>(skip, count, grid, block, st.stream, sc, p, img, valueOrNull, H, phase, stride, cnt);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

extern "C" int svr_render_isosurface(svr_u8vec4* imgOrNull, svr_vec4* surfaceOrNull, const svr_volume* volume, const svr_camera* camera,
                                     const svr_isosurface_params* params, uint32_t phase, uint32_t stride, uint32_t* bandRows)
{
    HostState& st = state();
    if (!volume || !camera || !params) return fail_msg("svr_render_isosurface: null volume, camera or params");
    if (!imgOrNull && !surfaceOrNull) return fail_msg("svr_render_isosurface: both outputs are null");
    const svr_isosurface_params p = *params;
    if (!(p.stepSize > 0.f) || !std::isfinite(p.stepSize)) return fail_msg("svr_render_isosurface: stepSize must be positive and finite");
    if (!std::isfinite(p.isoValue)) return fail_msg("svr_render_isosurface: isoValue must be finite");
    for (float c : p.color)
        if (!(c >= 0.f && c <= 1.f)) return fail_msg("svr_render_isosurface: each colour component must be in [0, 1]");
    if (phase >= stride) return fail_msg("svr_render_isosurface: band phase must be below the band stride");
    const int block = st.options[SVR_OPT_RC_BLOCK];
    const uint32_t tileH = (uint32_t)block / 16u;
    if (bandRows) *bandRows = tileH;

    ProjScene sc;
    const bool skip = st.options[SVR_OPT_RC_SKIP] != 0;
    const bool count = st.options[SVR_OPT_COUNTERS] != 0;
    if (int rc = make_scene(&sc, *volume, camera, skip)) return rc;
    dim3 grid;
    if (!band_grid(*camera, tileH, phase, stride, &grid)) return 0;
    Counters* cnt = count ? device_counters() : nullptr;
    if (count && !cnt) return fail_msg("svr_render_isosurface: counter allocation failed");
    const uint32_t H = camera->imageH;
    const float3 color = f3(p.color[0], p.color[1], p.color[2]);
    uint32_t* img = (uint32_t*)imgOrNull;
    float4* surface = (float4*)surfaceOrNull;
    if (skip) {
        if (count) iso_kernel<true, true><<<grid, block, 0, st.stream>>>(sc, p.stepSize, p.isoValue, color, img, surface, H, phase, stride, cnt);
        else iso_kernel<true, false><<<grid, block, 0, st.stream>>>(sc, p.stepSize, p.isoValue, color, img, surface, H, phase, stride, cnt);
    } else {
        if (count) iso_kernel<false, true><<<grid, block, 0, st.stream>>>(sc, p.stepSize, p.isoValue, color, img, surface, H, phase, stride, cnt);
        else iso_kernel<false, false><<<grid, block, 0, st.stream>>>(sc, p.stepSize, p.isoValue, color, img, surface, H, phase, stride, cnt);
    }
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

namespace {

template <int OP, bool SKIP>
void launch_slices(bool count, dim3 grid, int block, cudaStream_t stream, const ProjScene& sc, const SliceGeom& g, const svr_slice_params& p,
                   uint32_t* img, float* value, Counters* cnt)
{
    if (count) slice_kernel<OP, SKIP, true><<<grid, block, 0, stream>>>(sc, g, p.windowCenter, p.windowWidth, img, value, cnt);
    else slice_kernel<OP, SKIP, false><<<grid, block, 0, stream>>>(sc, g, p.windowCenter, p.windowWidth, img, value, cnt);
}

template <int OP>
void launch_slice_mode(bool skip, bool count, dim3 grid, int block, cudaStream_t stream, const ProjScene& sc, const SliceGeom& g,
                       const svr_slice_params& p, uint32_t* img, float* value, Counters* cnt)
{
    if (skip) launch_slices<OP, true>(count, grid, block, stream, sc, g, p, img, value, cnt);
    else launch_slices<OP, false>(count, grid, block, stream, sc, g, p, img, value, cnt);
}

bool finite3(const float* a) { return std::isfinite(a[0]) && std::isfinite(a[1]) && std::isfinite(a[2]); }

}  // namespace

extern "C" int svr_render_slices(svr_u8vec4* imgOrNull, float* valueOrNull, const svr_volume* volume, const svr_slice_params* params)
{
    HostState& st = state();
    if (!volume || !params) return fail_msg("svr_render_slices: null volume or params");
    if (!imgOrNull && !valueOrNull) return fail_msg("svr_render_slices: both outputs are null");
    const svr_slice_params p = *params;
    if (!finite3(p.axisU) || !finite3(p.axisV)) return fail_msg("svr_render_slices: axisU and axisV must be finite");
    const float3 u = f3(p.axisU[0], p.axisU[1], p.axisU[2]), v = f3(p.axisV[0], p.axisV[1], p.axisV[2]);
    const float3 nc = cross(u, v);
    const float nn = dot(nc, nc);
    if (!(nn > 0.f) || !std::isfinite(nn)) return fail_msg("svr_render_slices: cross(axisU, axisV) must be nonzero and finite");
    if (p.count > 1u && !finite3(p.axisW)) return fail_msg("svr_render_slices: axisW must be finite when count > 1");
    if (p.imageW == 0u || p.imageW > 16384u || p.imageH == 0u || p.imageH > 16384u)
        return fail_msg("svr_render_slices: imageW and imageH must be in 1..16384");
    if (p.count == 0u || p.count > 65535u) return fail_msg("svr_render_slices: count must be in 1..65535");
    if (p.mode < SVR_PROJECT_MAX || p.mode > SVR_PROJECT_MEAN) return fail_msg("svr_render_slices: mode must be 0 (max), 1 (min) or 2 (mean)");
    if (!(p.thickness >= 0.f) || !std::isfinite(p.thickness)) return fail_msg("svr_render_slices: thickness must be finite and not negative");
    if (p.thickness > 0.f) {
        if (!(p.sampleSpacing > 0.f) || !std::isfinite(p.sampleSpacing))
            return fail_msg("svr_render_slices: sampleSpacing must be positive and finite for a slab");
        if (!(p.thickness / p.sampleSpacing <= 65536.f)) return fail_msg("svr_render_slices: thickness / sampleSpacing must be at most 65536");
    }
    if (!(p.windowWidth > 0.f) || !std::isfinite(p.windowWidth) || !std::isfinite(p.windowCenter))
        return fail_msg("svr_render_slices: windowWidth must be positive and finite, windowCenter finite");

    SliceGeom g;
    g.center = f3(p.center[0], p.center[1], p.center[2]);
    g.u = u;
    g.v = v;
    g.w = p.count > 1u ? f3(p.axisW[0], p.axisW[1], p.axisW[2]) : f3(0.f);
    g.n = nc / std::sqrt(nn);
    g.W = p.imageW;
    g.H = p.imageH;
    g.h = p.thickness > 0.f ? p.sampleSpacing : 0.f;
    g.K = p.thickness > 0.f ? (uint32_t)std::max(1.f, std::floor(p.thickness / g.h + 0.5f)) : 1u;
    g.t0 = -((float)g.K * g.h) * 0.5f;
    const svr_volume& vo = *volume;
    const float cmin[3] = {vo.bbox.vmin.x * -vo.x_clip.x, vo.bbox.vmin.y * -vo.y_clip.x, vo.bbox.vmin.z * -vo.z_clip.x};
    const float cmax[3] = {vo.bbox.vmax.x * vo.x_clip.y, vo.bbox.vmax.y * vo.y_clip.y, vo.bbox.vmax.z * vo.z_clip.y};
    const float n3[3] = {g.n.x, g.n.y, g.n.z};
    float sg[3], lo[3], hi[3];
    for (int c = 0; c < 3; ++c) {
        sg[c] = n3[c] < 0.f ? -1.f : 1.f;
        lo[c] = n3[c] < 0.f ? -cmax[c] : cmin[c];
        hi[c] = n3[c] < 0.f ? -cmin[c] : cmax[c];
    }
    g.sg = f3(sg[0], sg[1], sg[2]);
    g.lo = f3(lo[0], lo[1], lo[2]);
    g.hi = f3(hi[0], hi[1], hi[2]);

    const int block = st.options[SVR_OPT_RC_BLOCK];
    const uint32_t tileH = (uint32_t)block / 16u;
    ProjScene sc;
    const bool skip = st.options[SVR_OPT_RC_SKIP] != 0 && g.K > 1u;  // a thin slice takes its one fetch and never walks
    const bool count = st.options[SVR_OPT_COUNTERS] != 0;
    if (int rc = make_scene(&sc, *volume, nullptr, skip)) return rc;
    Counters* cnt = count ? device_counters() : nullptr;
    if (count && !cnt) return fail_msg("svr_render_slices: counter allocation failed");
    const dim3 grid((p.imageW + 15u) / 16u, (p.imageH + tileH - 1u) / tileH, p.count);
    uint32_t* img = (uint32_t*)imgOrNull;
    if (p.mode == SVR_PROJECT_MAX) launch_slice_mode<SVR_PROJECT_MAX>(skip, count, grid, block, st.stream, sc, g, p, img, valueOrNull, cnt);
    else if (p.mode == SVR_PROJECT_MIN) launch_slice_mode<SVR_PROJECT_MIN>(skip, count, grid, block, st.stream, sc, g, p, img, valueOrNull, cnt);
    else launch_slice_mode<SVR_PROJECT_MEAN>(skip, count, grid, block, st.stream, sc, g, p, img, valueOrNull, cnt);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}
