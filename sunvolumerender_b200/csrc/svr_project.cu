// svr_project.cu -- maximum, minimum and average intensity projection (svr_render_projection), the isosurface
// (svr_render_isosurface), which samples the volume the same way (iso_kernel), slices and slabs (svr_render_slices), which
// fold samples along a plane's normal as the projection folds them along a camera ray (slice_kernel), the curved planar
// reformation (svr_render_curved), which folds them along rays set by a frame per station of a centerline (curved_kernel),
// and label maps: 3D label surfaces found like the isosurface (label_kernel) and label overlays on slices (label_slice_kernel).
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
#include <type_traits>
#include <vector>

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

// The walk over a macrocell grid shared by project_kernel, slice_kernel, curved_kernel, iso_kernel (the range grid) and
// label_kernel (the label presence grid).  visit(k) is the cell of sample k (its index, x fastest) and kEnd, the first index
// whose sample lies at or beyond the ray's exit from that cell (at least k + 1, at most K); the caller loads what its grid holds
// for the cell, drops or takes samples [k, kEnd) and continues at kEnd.  S: a scene with vol, scale and gx, gy, gz.
struct CellVisit {
    size_t cell;
    uint32_t kEnd;
};

struct CellWalk {
    float3 dg, invDg;  // the ray in cell coordinates: g(t) = g(t_k) + (t - t_k) dg

    template <class S>
    SVR_DEV CellWalk(const S& s, const Ray& ray)
    {
        dg = ray.dir * (f3(s.vol.bbox.invSize) * s.scale);
        invDg = 1.f / dg;
    }

    template <class S>
    SVR_DEV CellVisit visit(const S& s, const Ray& ray, float t0, float h, uint32_t k, uint32_t K) const
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
        c.cell = ((size_t)cz * s.gy + cy) * s.gx + cx;
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
            const float2 r = __ldg(s.range + c.cell);
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

// The samples of a camera ray through the volume on [tNear, tFar] (include/svr_render.h): K, with *t0 = max(tNear, 0) and
// *h = stepSize / 2.  K uses the fast-math division (2 ulp), as grey_rgba does: the correctly rounded one is a subroutine
// call, around which the counting variants spill.  K can then differ by one from the exact formula where
// (tFar - t0) / h + 1/2 is within 2 ulp of an integer; it is the same with skipping on and off.
SVR_DEV uint32_t sample_count(float stepSize, float tNear, float tFar, float* t0, float* h)
{
    *h = stepSize * 0.5f;
    *t0 = fmaxf(tNear, 0.f);
    const float span = tFar > *t0 ? floorf(__fadd_rn(__fsub_rn(tFar, *t0) / *h, 0.5f)) : 0.f;
    return (uint32_t)span;
}

// The grey image of a projected value P in the display window: (trunc(255 g), trunc(255 g), trunc(255 g), 255),
// g = clamp((P - (windowCenter - windowWidth / 2)) / windowWidth, 0, 1)
SVR_DEV uint32_t grey_rgba(float P, float windowCenter, float windowWidth)
{
    const float g = fminf(fmaxf((P - (windowCenter - 0.5f * windowWidth)) / windowWidth, 0.f), 1.f);
    const float q = 255.f * g;
    return pack_u8x4(q, q, q, 255.f);
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
            float t0, h;
            const uint32_t K = sample_count(stepSize, tNear, tFar, &t0, &h);
            lc.add(SVR_CNT_STEPS, K);
            const float acc = fold_samples<OP, SKIP>(s, ray, t0, h, 0u, K, lc);
            if (K > 0u) P = OP == SVR_PROJECT_MEAN ? __fdiv_rn(acc, (float)K) : acc;
        }
        const size_t offset = (size_t)idy * s.cam.imageW + idx;
        if (value) value[offset] = P;
        if (img) img[offset] = grey_rgba(P, windowCenter, windowWidth);
    }
    lc.flush(cnt);
}

// The refinement of a first hit (include/svr_render.h, svr_render_isosurface) between lo and hi, value(lo) = vLo < iso <= vHi =
// value(hi): 4 bisection steps, then the linear interpolation.  Returns (t_hit, the final bisection upper bound).
template <class V>
SVR_DEV float2 refine_crossing(const V& value, float iso, float lo, float hi, float vLo, float vHi)
{
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
    return make_float2(lo + (hi - lo) * (iso - vLo) / (vHi - vLo), hi);
}

// The first hit of iso_kernel and label_kernel (include/svr_render.h, svr_render_isosurface): the first of the K samples of the
// ray, sample k at t0 + (k + 1/2) h, whose value(t) reaches iso, with UNROLL fetches in flight per lane; with SKIP through the
// grid of S, dropping the samples of every cell for which mayHit(cell) is false.  A hit is refined by refine_crossing from the
// sample before it, recomputed from its index: *hit = (t_hit, the final bisection upper bound), both t_0 for a hit at k = 0.
// Counts steps, shade_taps, skipped and cells (the refinement's taps are not counted).
template <bool SKIP, int UNROLL, bool COUNT, class S, class V, class M>
SVR_DEV bool first_hit(const S& s, const Ray& ray, float t0, float h, uint32_t K, const V& value, float iso, const M& mayHit,
                       LocalCounters<COUNT>& lc, float2* hit)
{
    auto t_of = [&](uint32_t k) { return __fadd_rn(t0, __fmul_rn((float)k + 0.5f, h)); };
    // the first index in [k, kEnd) whose value reaches iso (its value in vHit), else kEnd
    float vHit = 0.f;
    auto find = [&](uint32_t k, uint32_t kEnd) {
        if constexpr (UNROLL > 1) {
            for (; k + (uint32_t)UNROLL <= kEnd; k += (uint32_t)UNROLL) {
                float v[UNROLL];
#pragma unroll
                for (int u = 0; u < UNROLL; ++u) v[u] = value(t_of(k + u));
                int first = UNROLL;
#pragma unroll
                for (int u = UNROLL - 1; u >= 0; --u)
                    if (v[u] >= iso) first = u, vHit = v[u];
                if (first < UNROLL) return k + (uint32_t)first;
            }
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
    uint32_t kHit = K;
    if constexpr (!SKIP) {
        kHit = find(0u, K);
        lc.add(SVR_CNT_SHADE_TAPS, kHit < K ? kHit + 1u : K);
    } else {
        const CellWalk walk(s, ray);
        for (uint32_t k = 0; k < K;) {
            const CellVisit c = walk.visit(s, ray, t0, h, k, K);
            lc.add(SVR_CNT_CELLS, 1);
            if (!mayHit(c.cell)) {
                lc.add(SVR_CNT_SKIPPED, c.kEnd - k);
            } else {
                const uint32_t f = find(k, c.kEnd);
                lc.add(SVR_CNT_SHADE_TAPS, (f < c.kEnd ? f + 1u : c.kEnd) - k);
                if (f < c.kEnd) {
                    kHit = f;
                    break;
                }
            }
            k = c.kEnd;
        }
    }
    lc.add(SVR_CNT_STEPS, kHit < K ? kHit + 1u : K);
    if (kHit >= K) return false;
    hit->x = hit->y = t_of(kHit);
    if (kHit > 0u) {
        const float lo = t_of(kHit - 1u);
        *hit = refine_crossing(value, iso, lo, hit->x, value(lo), vHit);
    }
    return true;
}

// Isosurface (include/svr_render.h): the first sample at or above iso along the projection's samples, refined by 4 bisection
// steps and a linear interpolation, shaded with the ray caster's headlight.  Skipping drops the samples of cells whose maximum is
// below iso: none of them can be the first hit.
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
    float2 hit = make_float2(0.f, 0.f);
    if (inside) {
        ray = camera_ray_center(s.cam, idx, idy);
        lc.add(SVR_CNT_PATHS, 1);
        float tNear, tFar;
        if (intersect_volume(s.vol, ray, &tNear, &tFar)) {
            float t0, h;
            const uint32_t K = sample_count(stepSize, tNear, tFar, &t0, &h);
            const float ds = s.vol.densityScale;
            auto value = [&](float t) {
                const float3 tc = tex_coord(s.vol, ray.orig + t * ray.dir);
                return tex3D<float>(s.vol.tex, tc.x, tc.y, tc.z) * ds;
            };
            // a cell may hold a hit unless its widened maximum is below iso
            auto mayHit = [&](size_t cell) {
                const float2 range = __ldg(s.range + cell);
                const float top = fmaxf(range.x * ds, range.y * ds);
                return !(top + fabsf(top) * RANGE_MARGIN < iso);
            };
            found = first_hit<SKIP, 4>(s, ray, t0, h, K, value, iso, mayHit, lc, &hit);
        }
    }
    // the counts are complete (the refinement and gradient taps are not counted): flushed before the shading, which then needs
    // no registers for them
    lc.flush(cnt);
    if (!inside) return;
    uint32_t rgba = 0u;
    float4 surf = make_float4(0.f, 0.f, 0.f, INFINITY);
    if (found) {
        const float3 x = ray.orig + hit.x * ray.dir;
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

// The clipped box [cmin, cmax] turned so that the samples of a ray along dir move up it: per component sg = -1 where
// dir < 0, else +1, and sg x in [lo, hi] (lo = sg cmin, hi = sg cmax, swapped where sg = -1) iff x in [cmin, cmax].
struct TurnedBox {
    float3 sg, lo, hi;
};

SVR_HD float turned_sign(float d) { return d < 0.f ? -1.f : 1.f; }

SVR_HD TurnedBox turn_box(float3 dir, float3 cmin, float3 cmax)
{
    TurnedBox b;
    b.sg = f3(turned_sign(dir.x), turned_sign(dir.y), turned_sign(dir.z));
    b.lo = f3(dir.x < 0.f ? -cmax.x : cmin.x, dir.y < 0.f ? -cmax.y : cmin.y, dir.z < 0.f ? -cmax.z : cmin.z);
    b.hi = f3(dir.x < 0.f ? -cmin.x : cmax.x, dir.y < 0.f ? -cmin.y : cmax.y, dir.z < 0.f ? -cmin.z : cmax.z);
    return b;
}

// The included samples [kLo, kHi) of the slab rule (include/svr_render.h, svr_render_slices) on the ray (orig, dir), sample k
// at orig + (t0 + (k + 1/2) h) dir, against the box turned for dir.  Each component of x_k is monotone in k (s_k and the
// rounded products and sums are), so the lower bounds of the turned box hold from kLo on and its upper bounds below kHi; two
// binary searches find both.  A component with dir = 0 is constant: its two conditions hold for every k or for none.
SVR_DEV uint2 included_range(const Ray& ray, float t0, float h, uint32_t K, const TurnedBox& box)
{
    const float3 &sg = box.sg, &bLo = box.lo, &bHi = box.hi;
    // sg * x_k is non-decreasing in k on every component: "sg x_k >= lo" holds from some k on, "sg x_k <= hi" up to some k
    auto at = [&](uint32_t k) { return sg * (ray.orig + __fadd_rn(t0, __fmul_rn((float)k + 0.5f, h)) * ray.dir); };
    auto rises = [&](uint32_t k) {
        const float3 x = at(k);
        return x.x >= bLo.x && x.y >= bLo.y && x.z >= bLo.z;
    };
    auto falls = [&](uint32_t k) {
        const float3 x = at(k);
        return x.x <= bHi.x && x.y <= bHi.y && x.z <= bHi.z;
    };
    // kLo = the first k in [0, K] with rises(k) (K: none), kHi = the first k in [0, K] without falls(k)
    uint32_t lo = 0u, hi = K;
    while (lo < hi) {
        const uint32_t m = (lo + hi) >> 1;
        if (rises(m)) hi = m;
        else lo = m + 1u;
    }
    const uint32_t kLo = lo;
    hi = K;
    while (lo < hi) {
        const uint32_t m = (lo + hi) >> 1;
        if (falls(m)) lo = m + 1u;
        else hi = m;
    }
    return make_uint2(kLo, lo);
}

// P and its grey image at pixel (x, y) of image blockIdx.z of a W x H stack, (0, 0, 0, 0) where no sample was taken.  The
// pixel's place comes from the launch geometry again: nothing but P and the count stays live across the MEAN division, which is
// a subroutine call (else the MEAN variants spill the pixel around it).
SVR_DEV void write_slab(float P, uint32_t taken, uint32_t W, uint32_t H, float windowCenter, float windowWidth, uint32_t* img, float* value)
{
    const uint2 q = band_pixel(0u, H, 0u, 1u);
    const size_t offset = ((size_t)blockIdx.z * H + q.y) * W + q.x;
    if (value) value[offset] = P;
    if (img) img[offset] = taken > 0u ? grey_rgba(P, windowCenter, windowWidth) : 0u;
}

// The plane geometry of svr_render_slices (include/svr_render.h), from the host: n, K, t0 and h of the slab rule, and the
// clipped box turned for n (TurnedBox).
struct SliceGeom {
    float3 center, u, v, w, n;
    TurnedBox box;
    uint32_t W, H, K;
    float t0, h;
};

// Slices and slabs (include/svr_render.h): pixel (x, y) of slice blockIdx.z folds the included samples [kLo, kHi) of the ray
// (c, n) with fold_samples.
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
        const uint2 kr = included_range(ray, g.t0, g.h, g.K, g.box);
        const uint32_t taken = kr.y > kr.x ? kr.y - kr.x : 0u;
        float P = 0.f;
        if (taken > 0u) {
            lc.add(SVR_CNT_STEPS, taken);
            const float acc = fold_samples<OP, SKIP>(s, ray, g.t0, g.h, kr.x, kr.y, lc);
            P = OP == SVR_PROJECT_MEAN ? __fdiv_rn(acc, (float)taken) : acc;
        }
        write_slab(P, taken, g.W, g.H, windowCenter, windowWidth, img, value);
    }
    lc.flush(cnt);
}

// The geometry of svr_render_curved (include/svr_render.h) that all pixels share, from the host: the slab rule's K, t0 and h,
// the clipped box, and where the per-image (cos, sin) table starts in the frame table (after the 4 float4 of every station).
// the fewest slab samples for which svr_render_curved walks the range grid (SVR_OPT_RC_SKIP)
constexpr uint32_t CURVED_WALK_MIN_K = 32u;

struct CurveGeom {
    float3 cmin, cmax;
    uint32_t W, H, K, trig;
    float t0, h, ps;
    int cross;  // SVR_CURVED_CROSS: image j is station j; else row y is station y and image j the angle j
};

// Curved planar reformation (include/svr_render.h): pixel (x, y) of image blockIdx.z reads its station's frame (c, t, r, b),
// forms its ray (p, n) or (p, t), turns the clipped box for that direction and folds the included samples with fold_samples.
template <int OP, bool SKIP, bool COUNT>
__global__ void __launch_bounds__(256) curved_kernel(const __grid_constant__ ProjScene s, const __grid_constant__ CurveGeom g,
                                                     const float4* __restrict__ frames, float windowCenter, float windowWidth,
                                                     uint32_t* __restrict__ img, float* __restrict__ value, Counters* cnt)
{
    const uint2 pix = band_pixel(0u, g.H, 0u, 1u);
    const uint32_t idx = pix.x, idy = pix.y, j = blockIdx.z;
    LocalCounters<COUNT> lc;
    if (idx < g.W && idy < g.H) {
        lc.add(SVR_CNT_PATHS, 1);
        const float4* f = frames + 4u * (g.cross ? j : idy);
        const float4 c = __ldg(f);
        uint32_t taken = 0u;
        float P = 0.f;
        if (c.w != 0.f) {  // a valid station
            const float4 t = __ldg(f + 1), r = __ldg(f + 2), b = __ldg(f + 3);
            const float4 cs = __ldg(frames + g.trig + (g.cross ? 0u : j));
            const float3 a = cs.x * f3(r.x, r.y, r.z) + cs.y * f3(b.x, b.y, b.z);
            const float3 e = cs.x * f3(b.x, b.y, b.z) - cs.y * f3(r.x, r.y, r.z);  // t x a
            const float fx = __fsub_rn((float)idx + 0.5f, 0.5f * (float)g.W);
            Ray ray;
            if (g.cross) {
                const float fy = __fsub_rn((float)idy + 0.5f, 0.5f * (float)g.H);
                ray.orig = f3(c.x, c.y, c.z) + (fx * g.ps) * a + (fy * g.ps) * e;
                ray.dir = f3(t.x, t.y, t.z);
            } else {
                ray.orig = f3(c.x, c.y, c.z) + (fx * g.ps) * a;
                ray.dir = e;
            }
            const TurnedBox box = turn_box(ray.dir, g.cmin, g.cmax);
            const uint2 kr = included_range(ray, g.t0, g.h, g.K, box);
            taken = kr.y > kr.x ? kr.y - kr.x : 0u;
            if (taken > 0u) {
                lc.add(SVR_CNT_STEPS, taken);
                const float acc = fold_samples<OP, SKIP>(s, ray, g.t0, g.h, kr.x, kr.y, lc);
                P = OP == SVR_PROJECT_MEAN ? __fdiv_rn(acc, (float)taken) : acc;
            }
        }
        write_slab(P, taken, g.W, g.H, windowCenter, windowWidth, img, value);
    }
    lc.flush(cnt);
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

// f(op, skip, count) with the kernel variant of a call as compile-time constants: op std::integral_constant<int, mode>, skip
// and count std::bool_constant.  The isosurface and label kernels take no mode: f(skip, count).
template <class F>
void with_variant(bool skip, bool count, F&& f)
{
    if (skip) {
        if (count) f(std::true_type(), std::true_type());
        else f(std::true_type(), std::false_type());
    } else {
        if (count) f(std::false_type(), std::true_type());
        else f(std::false_type(), std::false_type());
    }
}

template <class F>
void with_variant(int mode, bool skip, bool count, F&& f)
{
    auto with_op = [&](auto op) { with_variant(skip, count, [&](auto sk, auto ct) { f(op, sk, ct); }); };
    if (mode == SVR_PROJECT_MAX) with_op(std::integral_constant<int, SVR_PROJECT_MAX>());
    else if (mode == SVR_PROJECT_MIN) with_op(std::integral_constant<int, SVR_PROJECT_MIN>());
    else with_op(std::integral_constant<int, SVR_PROJECT_MEAN>());
}

// What every launch of this file takes from the options: the threads per block (SVR_OPT_RC_BLOCK) in band_pixel's blocks of
// 16 columns and tileH rows, skipping (SVR_OPT_RC_SKIP) and counting (SVR_OPT_COUNTERS)
struct LaunchOptions {
    int block;
    uint32_t tileH;
    bool skip, count;
};

LaunchOptions launch_options()
{
    const int* o = state().options;
    return {o[SVR_OPT_RC_BLOCK], (uint32_t)o[SVR_OPT_RC_BLOCK] / 16u, o[SVR_OPT_RC_SKIP] != 0, o[SVR_OPT_COUNTERS] != 0};
}

// "<who>: <what>" as the call's error
int fail_in(const char* who, const char* what) { return fail_msg((std::string(who) + ": " + what).c_str()); }

// The device counters into *cnt when counting, else null; the error of `who` when they cannot be allocated
int launch_counters(const char* who, bool count, Counters** cnt)
{
    *cnt = count ? device_counters() : nullptr;
    return count && !*cnt ? fail_in(who, "counter allocation failed") : 0;
}

// After a kernel launch: counts it and returns its error
int launched()
{
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

// The parameter errors of a projection mode and of a display window, reported as those of `who`
int check_mode(const char* who, int mode)
{
    if (mode < SVR_PROJECT_MAX || mode > SVR_PROJECT_MEAN) return fail_in(who, "mode must be 0 (max), 1 (min) or 2 (mean)");
    return 0;
}

int check_window(const char* who, float windowCenter, float windowWidth)
{
    if (!(windowWidth > 0.f) || !std::isfinite(windowWidth) || !std::isfinite(windowCenter))
        return fail_in(who, "windowWidth must be positive and finite, windowCenter finite");
    return 0;
}

}  // namespace
}  // namespace svr

using namespace svr;

extern "C" int svr_render_projection(svr_u8vec4* imgOrNull, float* valueOrNull, const svr_volume* volume, const svr_camera* camera,
                                     const svr_projection_params* params, uint32_t phase, uint32_t stride, uint32_t* bandRows)
{
    HostState& st = state();
    const char* who = "svr_render_projection";
    if (!volume || !camera || !params) return fail_msg("svr_render_projection: null volume, camera or params");
    if (!imgOrNull && !valueOrNull) return fail_msg("svr_render_projection: both outputs are null");
    const svr_projection_params p = *params;
    if (int rc = check_mode(who, p.mode)) return rc;
    if (!(p.stepSize > 0.f) || !std::isfinite(p.stepSize)) return fail_msg("svr_render_projection: stepSize must be positive and finite");
    if (int rc = check_window(who, p.windowCenter, p.windowWidth)) return rc;
    if (phase >= stride) return fail_msg("svr_render_projection: band phase must be below the band stride");
    const LaunchOptions o = launch_options();
    if (bandRows) *bandRows = o.tileH;

    ProjScene sc;
    if (int rc = make_scene(&sc, *volume, camera, o.skip)) return rc;
    dim3 grid;
    if (!band_grid(*camera, o.tileH, phase, stride, &grid)) return 0;
    Counters* cnt;
    if (int rc = launch_counters(who, o.count, &cnt)) return rc;
    const uint32_t H = camera->imageH;
    with_variant(p.mode, o.skip, o.count, [&](auto op, auto sk, auto ct) {
        project_kernel<op, sk, ct><<<grid, o.block, 0, st.stream>>>(sc, p.stepSize, p.windowCenter, p.windowWidth, (uint32_t*)imgOrNull,
                                                                    valueOrNull, 0u, H, phase, stride, cnt);
    });
    return launched();
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
    const LaunchOptions o = launch_options();
    if (bandRows) *bandRows = o.tileH;

    ProjScene sc;
    if (int rc = make_scene(&sc, *volume, camera, o.skip)) return rc;
    dim3 grid;
    if (!band_grid(*camera, o.tileH, phase, stride, &grid)) return 0;
    Counters* cnt;
    if (int rc = launch_counters("svr_render_isosurface", o.count, &cnt)) return rc;
    const uint32_t H = camera->imageH;
    const float3 color = f3(p.color[0], p.color[1], p.color[2]);
    with_variant(o.skip, o.count, [&](auto sk, auto ct) {
        iso_kernel<sk, ct><<<grid, o.block, 0, st.stream>>>(sc, p.stepSize, p.isoValue, color, (uint32_t*)imgOrNull, (float4*)surfaceOrNull, H,
                                                            phase, stride, cnt);
    });
    return launched();
}

namespace {

bool finite3(const float* a) { return std::isfinite(a[0]) && std::isfinite(a[1]) && std::isfinite(a[2]); }

// The parameter errors svr_render_slices and svr_render_curved share (include/svr_render.h), reported as those of `who`: image
// size and count, mode, slab and window; no CUDA call
template <class P>
int check_stack_params(const char* who, const P& p)
{
    if (p.imageW == 0u || p.imageW > 16384u || p.imageH == 0u || p.imageH > 16384u) return fail_in(who, "imageW and imageH must be in 1..16384");
    if (p.count == 0u || p.count > 65535u) return fail_in(who, "count must be in 1..65535");
    if (int rc = check_mode(who, p.mode)) return rc;
    if (!(p.thickness >= 0.f) || !std::isfinite(p.thickness)) return fail_in(who, "thickness must be finite and not negative");
    if (p.thickness > 0.f) {
        if (!(p.sampleSpacing > 0.f) || !std::isfinite(p.sampleSpacing)) return fail_in(who, "sampleSpacing must be positive and finite for a slab");
        if (!(p.thickness / p.sampleSpacing <= 65536.f)) return fail_in(who, "thickness / sampleSpacing must be at most 65536");
    }
    return check_window(who, p.windowCenter, p.windowWidth);
}

// svr_render_slices' parameter errors (include/svr_render.h), reported as those of `who`; no CUDA call
int check_slice_params(const char* who, const svr_slice_params& p)
{
    if (!finite3(p.axisU) || !finite3(p.axisV)) return fail_in(who, "axisU and axisV must be finite");
    const float3 nc = cross(f3(p.axisU[0], p.axisU[1], p.axisU[2]), f3(p.axisV[0], p.axisV[1], p.axisV[2]));
    const float nn = dot(nc, nc);
    if (!(nn > 0.f) || !std::isfinite(nn)) return fail_in(who, "cross(axisU, axisV) must be nonzero and finite");
    if (p.count > 1u && !finite3(p.axisW)) return fail_in(who, "axisW must be finite when count > 1");
    return check_stack_params(who, p);
}

// The slab rule of include/svr_render.h (svr_render_slices, svr_render_curved): K samples h apart, the first at t0 + h / 2; a
// thin image (thickness 0) is one sample at 0
struct Slab {
    uint32_t K;
    float t0, h;
};

Slab slab_rule(float thickness, float sampleSpacing)
{
    const float h = thickness > 0.f ? sampleSpacing : 0.f;
    const uint32_t K = thickness > 0.f ? (uint32_t)std::max(1.f, std::floor(thickness / h + 0.5f)) : 1u;
    return {K, -((float)K * h) * 0.5f, h};
}

// The volume's box clipped by its clip planes, [cmin, cmax] (include/svr_render.h, svr_render_slices)
void clipped_box(const svr_volume& v, float3* cmin, float3* cmax)
{
    *cmin = f3(v.bbox.vmin.x * -v.x_clip.x, v.bbox.vmin.y * -v.y_clip.x, v.bbox.vmin.z * -v.z_clip.x);
    *cmax = f3(v.bbox.vmax.x * v.x_clip.y, v.bbox.vmax.y * v.y_clip.y, v.bbox.vmax.z * v.z_clip.y);
}

}  // namespace

extern "C" int svr_render_slices(svr_u8vec4* imgOrNull, float* valueOrNull, const svr_volume* volume, const svr_slice_params* params)
{
    HostState& st = state();
    const char* who = "svr_render_slices";
    if (!volume || !params) return fail_msg("svr_render_slices: null volume or params");
    if (!imgOrNull && !valueOrNull) return fail_msg("svr_render_slices: both outputs are null");
    const svr_slice_params p = *params;
    if (int rc = check_slice_params(who, p)) return rc;
    const float3 u = f3(p.axisU[0], p.axisU[1], p.axisU[2]), v = f3(p.axisV[0], p.axisV[1], p.axisV[2]);
    const float3 nc = cross(u, v);
    const float nn = dot(nc, nc);

    SliceGeom g;
    g.center = f3(p.center[0], p.center[1], p.center[2]);
    g.u = u;
    g.v = v;
    g.w = p.count > 1u ? f3(p.axisW[0], p.axisW[1], p.axisW[2]) : f3(0.f);
    g.n = nc / std::sqrt(nn);
    g.W = p.imageW;
    g.H = p.imageH;
    const Slab slab = slab_rule(p.thickness, p.sampleSpacing);
    g.K = slab.K;
    g.t0 = slab.t0;
    g.h = slab.h;
    float3 cmin, cmax;
    clipped_box(*volume, &cmin, &cmax);
    g.box = turn_box(g.n, cmin, cmax);

    const LaunchOptions o = launch_options();
    ProjScene sc;
    const bool skip = o.skip && g.K > 1u;  // a thin slice takes its one fetch and never walks
    if (int rc = make_scene(&sc, *volume, nullptr, skip)) return rc;
    Counters* cnt;
    if (int rc = launch_counters(who, o.count, &cnt)) return rc;
    const dim3 grid((p.imageW + 15u) / 16u, (p.imageH + o.tileH - 1u) / o.tileH, p.count);
    with_variant(p.mode, skip, o.count, [&](auto op, auto sk, auto ct) {
        slice_kernel<op, sk, ct><<<grid, o.block, 0, st.stream>>>(sc, g, p.windowCenter, p.windowWidth, (uint32_t*)imgOrNull, valueOrNull, cnt);
    });
    return launched();
}

namespace {

struct D3 {
    double x, y, z;
};
D3 operator+(D3 a, D3 b) { return {a.x + b.x, a.y + b.y, a.z + b.z}; }
D3 operator-(D3 a, D3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
D3 operator*(double s, D3 a) { return {s * a.x, s * a.y, s * a.z}; }
double dot(D3 a, D3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
D3 cross(D3 a, D3 b) { return {a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x}; }
D3 normalize(D3 a) { return (1.0 / std::sqrt(dot(a, a))) * a; }
bool is_zero(D3 a) { return a.x == 0.0 && a.y == 0.0 && a.z == 0.0; }
svr_vec4 v4(D3 a, float w) { return {(float)a.x, (float)a.y, (float)a.z, w}; }

// The frame rule of include/svr_render.h: nStations frames, 4 svr_vec4 each, into out; `who` names the entry point in an error.
// No CUDA call.
int curve_frames(const char* who, const float* points, uint32_t nPoints, const float* up, float stationSpacing, uint32_t nStations,
                 svr_vec4* out)
{
    auto err = [&](const char* what) { return fail_msg((std::string(who) + ": " + what).c_str()); };
    if (!points || !up) return err("null points or up");
    if (nPoints < 2u || nPoints > (1u << 20)) return err("nPoints must be in 2..2^20");
    if (!(stationSpacing > 0.f) || !std::isfinite(stationSpacing)) return err("stationSpacing must be positive and finite");
    if (nStations == 0u) return err("nStations must be at least 1");
    for (size_t i = 0; i < 3 * (size_t)nPoints; ++i)
        if (!std::isfinite(points[i])) return err("every point must be finite");
    // 1. drop repeats; cumulative arc length
    std::vector<D3> P;
    std::vector<double> S;
    P.reserve(nPoints);
    S.reserve(nPoints);
    for (uint32_t i = 0; i < nPoints; ++i) {
        const D3 q = {points[3 * i], points[3 * i + 1], points[3 * i + 2]};
        if (!P.empty() && q.x == P.back().x && q.y == P.back().y && q.z == P.back().z) continue;
        S.push_back(P.empty() ? 0.0 : S.back() + std::sqrt(dot(q - P.back(), q - P.back())));
        P.push_back(q);
    }
    if (P.size() < 2) return err("the curve needs at least 2 distinct points");
    if (!std::isfinite(up[0]) || !std::isfinite(up[1]) || !std::isfinite(up[2])) return err("up must be finite");
    const D3 upv = {up[0], up[1], up[2]};
    if (is_zero(upv)) return err("up must not be zero");
    const double L = S.back(), D = stationSpacing;
    if (0.5 * D > L) return err("no valid station: the curve is shorter than half a station");
    // 2. c(s) on segment m, the last m <= M - 2 with S_m <= s
    const size_t M = P.size();
    auto seg = [&](double s) {
        const size_t m = (size_t)(std::upper_bound(S.begin(), S.end(), s) - S.begin());
        return std::min(m == 0 ? 0 : m - 1, M - 2);
    };
    auto at = [&](double s) {
        const size_t m = seg(s);
        return P[m] + ((s - S[m]) / (S[m + 1] - S[m])) * (P[m + 1] - P[m]);
    };
    // 3., 4. station position and tangent
    auto station = [&](uint32_t i, D3* c, D3* t) {
        const double s = ((double)i + 0.5) * D;
        *c = at(s);
        D3 d = at(std::min(s + D, L)) - at(std::max(s - D, 0.0));
        if (is_zero(d)) {
            const size_t m = seg(s);
            d = P[m + 1] - P[m];
        }
        *t = normalize(d);
    };
    D3 c, t;
    station(0, &c, &t);
    const D3 r0 = upv - dot(upv, t) * t;
    if (std::sqrt(dot(r0, r0)) <= 1e-6 * std::sqrt(dot(upv, upv))) return err("up must not be parallel to the tangent at station 0");
    // 5. double reflection from station to station
    D3 r = normalize(r0);
    for (uint32_t i = 0; i < nStations; ++i) {
        svr_vec4* o = out + 4 * (size_t)i;
        if (((double)i + 0.5) * D > L) {  // 6.
            o[0] = o[1] = o[2] = o[3] = svr_vec4{0.f, 0.f, 0.f, 0.f};
            continue;
        }
        if (i > 0) {
            D3 cn, tn;
            station(i, &cn, &tn);
            const D3 v1 = cn - c;
            const double c1 = dot(v1, v1);
            D3 rL = r, tL = t;
            if (c1 != 0.0) {
                rL = r - (2.0 / c1 * dot(v1, r)) * v1;
                tL = t - (2.0 / c1 * dot(v1, t)) * v1;
            }
            const D3 v2 = tn - tL;
            const double c2 = dot(v2, v2);
            if (c2 != 0.0) rL = rL - (2.0 / c2 * dot(v2, rL)) * v2;
            r = normalize(rL - dot(rL, tn) * tn);
            c = cn;
            t = tn;
        }
        o[0] = v4(c, 1.f);
        o[1] = v4(t, 0.f);
        o[2] = v4(r, 0.f);
        o[3] = v4(cross(t, r), 0.f);
    }
    return 0;
}

// The frame table into curveFrames through the pinned staging buffer, on the library stream.  The host waits only for the
// copy that last read the staging buffer; that copy is stream-ordered after the earlier renders.
int stage_curve_table(HostState& st, const std::vector<svr_vec4>& table)
{
    DeviceState& d = st.dev;
    const size_t n = table.size();
    if (!d.curveStageEvent) SVR_TRY(cudaEventCreateWithFlags(&d.curveStageEvent, cudaEventDisableTiming));
    SVR_TRY(cudaEventSynchronize(d.curveStageEvent));
    if (d.curveStageCap < n) {
        if (d.curveStage) cudaFreeHost(d.curveStage);
        d.curveStage = nullptr;
        d.curveStageCap = 0;
        SVR_TRY(cudaHostAlloc((void**)&d.curveStage, n * sizeof(float4), cudaHostAllocPortable));
        d.curveStageCap = n;
    }
    SVR_TRY(d.curveFrames.reserve(n));
    memcpy(d.curveStage, table.data(), n * sizeof(float4));
    SVR_TRY(cudaMemcpyAsync(d.curveFrames.p, d.curveStage, n * sizeof(float4), cudaMemcpyHostToDevice, st.stream));
    SVR_TRY(cudaEventRecord(d.curveStageEvent, st.stream));
    return 0;
}

}  // namespace

extern "C" int svr_curve_frames(const float* points, uint32_t nPoints, const float up[3], float stationSpacing, uint32_t nStations,
                                svr_vec4* hostFrames)
{
    if (!hostFrames) return fail_msg("svr_curve_frames: null hostFrames");
    return curve_frames("svr_curve_frames", points, nPoints, up, stationSpacing, nStations, hostFrames);
}

extern "C" int svr_render_curved(svr_u8vec4* imgOrNull, float* valueOrNull, const svr_volume* volume, const svr_curved_params* params,
                                 const float* points, uint32_t nPoints)
{
    HostState& st = state();
    const char* who = "svr_render_curved";
    if (!volume || !params || !points) return fail_msg("svr_render_curved: null volume, params or points");
    if (!imgOrNull && !valueOrNull) return fail_msg("svr_render_curved: both outputs are null");
    const svr_curved_params p = *params;
    if (p.layout != SVR_CURVED_STRAIGHTENED && p.layout != SVR_CURVED_CROSS)
        return fail_msg("svr_render_curved: layout must be 0 (straightened) or 1 (cross-sections)");
    if (int rc = check_stack_params(who, p)) return rc;
    if (!(p.pixelSpacing > 0.f) || !std::isfinite(p.pixelSpacing)) return fail_msg("svr_render_curved: pixelSpacing must be positive and finite");
    if (!std::isfinite(p.angle0) || !std::isfinite(p.angleStep)) return fail_msg("svr_render_curved: angle0 and angleStep must be finite");
    const bool cross = p.layout == SVR_CURVED_CROSS;
    const uint32_t nStations = cross ? p.count : p.imageH, nTrig = cross ? 1u : p.count;
    std::vector<svr_vec4> table(4 * (size_t)nStations + nTrig);
    if (int rc = curve_frames(who, points, nPoints, p.up, p.stationSpacing, nStations, table.data())) return rc;
    for (uint32_t j = 0; j < nTrig; ++j) {
        const double theta = (double)p.angle0 + (double)j * (double)p.angleStep;
        table[4 * (size_t)nStations + j] = svr_vec4{(float)std::cos(theta), (float)std::sin(theta), 0.f, 0.f};
    }

    CurveGeom g;
    clipped_box(*volume, &g.cmin, &g.cmax);
    g.W = p.imageW;
    g.H = p.imageH;
    const Slab slab = slab_rule(p.thickness, p.sampleSpacing);
    g.K = slab.K;
    g.t0 = slab.t0;
    g.h = slab.h;
    g.ps = p.pixelSpacing;
    g.trig = 4u * nStations;
    g.cross = cross ? 1 : 0;

    const LaunchOptions o = launch_options();
    ProjScene sc;
    // slabs of fewer than CURVED_WALK_MIN_K samples, and thin images, do not walk: 16-sample slabs measured slower with the walk,
    // 64-sample ones faster (DESIGN.md section 7k)
    const bool skip = o.skip && g.K >= CURVED_WALK_MIN_K;
    if (int rc = make_scene(&sc, *volume, nullptr, skip)) return rc;
    Counters* cnt;
    if (int rc = launch_counters(who, o.count, &cnt)) return rc;
    if (int rc = stage_curve_table(st, table)) return rc;
    const float4* frames = st.dev.curveFrames.p;
    const dim3 grid((p.imageW + 15u) / 16u, (p.imageH + o.tileH - 1u) / o.tileH, p.count);
    with_variant(p.mode, skip, o.count, [&](auto op, auto sk, auto ct) {
        curved_kernel<op, sk, ct><<<grid, o.block, 0, st.stream>>>(sc, g, frames, p.windowCenter, p.windowWidth, (uint32_t*)imgOrNull,
                                                                   valueOrNull, cnt);
    });
    return launched();
}

namespace svr {
namespace {

// ---- label maps (include/svr_render.h: svr_render_labels, svr_render_label_slices) ----------------------------------------

// The label table as the kernels read it, a launch parameter (4128 bytes): colours and the 256-bit visibility mask
struct LabelTable {
    float4 color[256];
    uint32_t vis[8];  // bit l: label l is visible (l != 0 and color[l].w > 0)
};

struct LabelScene {
    svr_volume vol;          // a label volume: point-filtered u8, unnormalised coordinates, border 0
    svr_camera cam;
    float3 dims;             // (nx, ny, nz)
    const uint4* presence;   // with skipping: per cell 8 words (2 uint4), the labels of the cell and its one-voxel apron
    int gx, gy, gz;
    float3 scale;            // normalised texture coordinate -> cell coordinate (CellWalk)
};

SVR_DEV uint32_t label_at(const svr_volume& v, int i, int j, int k)
{
    return tex3D<unsigned char>(v.tex, (float)i + 0.5f, (float)j + 0.5f, (float)k + 0.5f);
}

SVR_DEV bool label_visible(const LabelTable& t, uint32_t l) { return (t.vis[l >> 5] >> (l & 31u)) & 1u; }

SVR_DEV float lerp_rn(float a, float b, float f) { return __fadd_rn(__fmul_rn(__fsub_rn(1.f, f), a), __fmul_rn(f, b)); }

// The 8 corners around x: u = tex_coord(x) dims - 1/2, i = floor(u), f = u - i; v[c] = vis of corner c (x fastest), lab[c] its label
struct LabelCorners {
    float3 f;
    float v[8];
    uint32_t lab[8];
};

SVR_DEV LabelCorners label_corners(const LabelScene& s, const LabelTable& t, float3 x)
{
    const float3 tc = tex_coord(s.vol, x);
    const float ux = __fsub_rn(__fmul_rn(tc.x, s.dims.x), 0.5f), uy = __fsub_rn(__fmul_rn(tc.y, s.dims.y), 0.5f),
                uz = __fsub_rn(__fmul_rn(tc.z, s.dims.z), 0.5f);
    const float ix = floorf(ux), iy = floorf(uy), iz = floorf(uz);
    LabelCorners c;
    c.f = f3(__fsub_rn(ux, ix), __fsub_rn(uy, iy), __fsub_rn(uz, iz));
#pragma unroll
    for (int n = 0; n < 8; ++n) {
        c.lab[n] = label_at(s.vol, (int)ix + (n & 1), (int)iy + ((n >> 1) & 1), (int)iz + (n >> 2));
        c.v[n] = label_visible(t, c.lab[n]) ? 1.f : 0.f;
    }
    return c;
}

// m(x): the trilinear interpolation of the visible labels' indicator
SVR_DEV float label_indicator(const LabelScene& s, const LabelTable& t, float3 x)
{
    const LabelCorners c = label_corners(s, t, x);
    const float y0 = lerp_rn(lerp_rn(c.v[0], c.v[1], c.f.x), lerp_rn(c.v[2], c.v[3], c.f.x), c.f.y);
    const float y1 = lerp_rn(lerp_rn(c.v[4], c.v[5], c.f.x), lerp_rn(c.v[6], c.v[7], c.f.x), c.f.y);
    return lerp_rn(y0, y1, c.f.z);
}

// The visible label with the largest summed corner weight at x, ties to the smaller id (0 if no corner is visible)
SVR_DEV uint32_t label_pick(const LabelScene& s, const LabelTable& t, float3 x)
{
    const LabelCorners c = label_corners(s, t, x);
    float w[8];
#pragma unroll
    for (int n = 0; n < 8; ++n) {
        const float wx = n & 1 ? c.f.x : __fsub_rn(1.f, c.f.x), wy = (n >> 1) & 1 ? c.f.y : __fsub_rn(1.f, c.f.y),
                    wz = n >> 2 ? c.f.z : __fsub_rn(1.f, c.f.z);
        w[n] = c.v[n] != 0.f ? __fmul_rn(__fmul_rn(wx, wy), wz) : 0.f;
    }
    uint32_t best = 0u;
    float bestW = -1.f;
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        if (c.v[a] == 0.f) continue;
        float sum = 0.f;
#pragma unroll
        for (int b = 0; b < 8; ++b)
            if (c.lab[b] == c.lab[a]) sum = __fadd_rn(sum, w[b]);
        if (sum > bestW || (sum == bestW && c.lab[a] < best)) {
            best = c.lab[a];
            bestW = sum;
        }
    }
    return best;
}

// The analytic gradient of m at x in world units: the derivative of the trilinear weights times dims * invSize
SVR_DEV float3 label_gradient(const LabelScene& s, const LabelTable& t, float3 x)
{
    const LabelCorners c = label_corners(s, t, x);
    const float* v = c.v;
    const float3 f = c.f;
    const float dx = lerp_rn(lerp_rn(v[1] - v[0], v[3] - v[2], f.y), lerp_rn(v[5] - v[4], v[7] - v[6], f.y), f.z);
    const float dy = lerp_rn(lerp_rn(v[2] - v[0], v[3] - v[1], f.x), lerp_rn(v[6] - v[4], v[7] - v[5], f.x), f.z);
    const float dz = lerp_rn(lerp_rn(v[4] - v[0], v[5] - v[1], f.x), lerp_rn(v[6] - v[2], v[7] - v[3], f.x), f.y);
    return f3(__fmul_rn(dx, __fmul_rn(s.dims.x, s.vol.bbox.invSize.x)), __fmul_rn(dy, __fmul_rn(s.dims.y, s.vol.bbox.invSize.y)),
              __fmul_rn(dz, __fmul_rn(s.dims.z, s.vol.bbox.invSize.z)));
}

// 3D label surfaces (include/svr_render.h): iso_kernel's rays, samples, hit search and refinement on m with iso = 1/2.  Skipping
// drops the samples of cells whose presence mask holds no visible label (m = 0 < 1/2 on all of them); the refinement recomputes
// the sample before the hit from its index.
template <bool SKIP, bool COUNT>
__global__ void __launch_bounds__(256) label_kernel(const __grid_constant__ LabelScene s, const __grid_constant__ LabelTable t, float stepSize,
                                                    uint32_t* __restrict__ img, float4* __restrict__ surface, uint8_t* __restrict__ label,
                                                    uint32_t y1, uint32_t bandPhase, uint32_t bandStride, Counters* cnt)
{
    const uint2 pix = band_pixel(0u, y1, bandPhase, bandStride);
    const uint32_t idx = pix.x, idy = pix.y;
    const bool inside = idx < s.cam.imageW && idy < y1;
    LocalCounters<COUNT> lc;
    Ray ray;
    bool found = false;
    float2 hit = make_float2(0.f, 0.f);
    if (inside) {
        ray = camera_ray_center(s.cam, idx, idy);
        lc.add(SVR_CNT_PATHS, 1);
        float tNear, tFar;
        if (intersect_volume(s.vol, ray, &tNear, &tFar)) {
            float t0, h;
            const uint32_t K = sample_count(stepSize, tNear, tFar, &t0, &h);
            auto value = [&](float tt) { return label_indicator(s, t, ray.orig + tt * ray.dir); };
            // a cell may hold a hit if its presence mask holds a visible label
            auto mayHit = [&](size_t cell) {
                const uint4 p0 = __ldg(s.presence + 2 * cell), p1 = __ldg(s.presence + 2 * cell + 1);
                return ((p0.x & t.vis[0]) | (p0.y & t.vis[1]) | (p0.z & t.vis[2]) | (p0.w & t.vis[3]) | (p1.x & t.vis[4]) |
                        (p1.y & t.vis[5]) | (p1.z & t.vis[6]) | (p1.w & t.vis[7])) != 0u;
            };
            found = first_hit<SKIP, 1>(s, ray, t0, h, K, value, 0.5f, mayHit, lc, &hit);
        }
    }
    // as iso_kernel: the counts are complete, flushed before the shading
    lc.flush(cnt);
    if (!inside) return;
    uint32_t rgba = 0u, lab = 0u;
    float4 surf = make_float4(0.f, 0.f, 0.f, INFINITY);
    if (found) {
        lab = label_pick(s, t, ray.orig + hit.y * ray.dir);
        const float3 x = ray.orig + hit.x * ray.dir;
        const float3 camPos = f3(s.cam.pos);
        const float3 g = label_gradient(s, t, x);
        float3 n = f3(0.f);
        float cosTerm = 1.f, specularTerm = 0.f;
        if (dot(g, g) > 0.f) {
            n = normalize(g);
            if (dot(n, ray.dir) > 0.f) n = -n;
            cosTerm = fabsf(dot(n, normalize(camPos - x)));
            specularTerm = powf(cosTerm, 30.f);
        }
        const float4 color = t.color[lab];
        const float r = fminf(color.x * cosTerm * 0.8f + specularTerm * 0.2f, 1.f);
        const float gr = fminf(color.y * cosTerm * 0.8f + specularTerm * 0.2f, 1.f);
        const float b = fminf(color.z * cosTerm * 0.8f + specularTerm * 0.2f, 1.f);
        rgba = pack_u8x4(r * 255.f, gr * 255.f, b * 255.f, 255.f);
        surf = make_float4(n.x, n.y, n.z, dot(x - camPos, -f3(s.cam.w)));
    }
    const size_t offset = (size_t)idy * s.cam.imageW + idx;
    if (img) img[offset] = rgba;
    if (surface) surface[offset] = surf;
    if (label) label[offset] = (uint8_t)lab;
}

// The slice geometry of svr_render_label_slices, from the host: svr_render_slices' pixel centres and clipped box
struct LabelSliceScene {
    svr_volume vol;
    float3 center, u, v, w, cmin, cmax, dims;
    uint32_t W, H;
};

// L of pixel (x, y) of image j: the label of the voxel holding the pixel centre, 0 outside the clipped box
SVR_DEV uint32_t slice_label(const LabelSliceScene& g, uint32_t x, uint32_t y, uint32_t j)
{
    const float fx = __fsub_rn((float)x + 0.5f, 0.5f * (float)g.W), fy = __fsub_rn((float)y + 0.5f, 0.5f * (float)g.H);
    const float3 c = g.center + fx * g.u + fy * g.v + (float)j * g.w;
    if (!(c.x >= g.cmin.x && c.y >= g.cmin.y && c.z >= g.cmin.z && c.x <= g.cmax.x && c.y <= g.cmax.y && c.z <= g.cmax.z)) return 0u;
    const float3 tc = tex_coord(g.vol, c);
    return label_at(g.vol, (int)floorf(__fmul_rn(tc.x, g.dims.x)), (int)floorf(__fmul_rn(tc.y, g.dims.y)), (int)floorf(__fmul_rn(tc.z, g.dims.z)));
}

SVR_DEV uint32_t blend_channel(uint32_t in, float a, float c)
{
    return (uint32_t)__fadd_rn(__fadd_rn(__fmul_rn(__fsub_rn(1.f, a), (float)in), __fmul_rn(a, __fmul_rn(255.f, c))), 0.5f);
}

// Label overlays (include/svr_render.h): pixel (x, y) of image blockIdx.z
__global__ void __launch_bounds__(256) label_slice_kernel(const __grid_constant__ LabelSliceScene g, const __grid_constant__ LabelTable t,
                                                          uint32_t* __restrict__ img, uint8_t* __restrict__ label, int outline)
{
    const uint2 pix = band_pixel(0u, g.H, 0u, 1u);
    const uint32_t x = pix.x, y = pix.y, j = blockIdx.z;
    if (x >= g.W || y >= g.H) return;
    const uint32_t L = slice_label(g, x, y, j);
    const size_t offset = ((size_t)j * g.H + y) * g.W + x;
    if (label) label[offset] = (uint8_t)L;
    if (!img || !label_visible(t, L)) return;
    bool edge = false;
    if (outline)
        edge = (x > 0u && slice_label(g, x - 1u, y, j) != L) || (x + 1u < g.W && slice_label(g, x + 1u, y, j) != L) ||
               (y > 0u && slice_label(g, x, y - 1u, j) != L) || (y + 1u < g.H && slice_label(g, x, y + 1u, j) != L);
    const float4 col = t.color[L];
    const float a = edge ? 1.f : col.w;
    const uint32_t in = img[offset];
    img[offset] = blend_channel(in & 255u, a, col.x) | (blend_channel((in >> 8) & 255u, a, col.y) << 8) |
                  (blend_channel((in >> 16) & 255u, a, col.z) << 16) | (255u << 24);
}

// The table errors of include/svr_render.h (no CUDA call), and the table the kernels read
int make_label_table(const char* who, const svr_label_params& p, LabelTable* t)
{
    memset(t, 0, sizeof(*t));
    for (int l = 0; l < 256; ++l) {
        for (int c = 0; c < 4; ++c)
            if (!(p.color[l][c] >= 0.f && p.color[l][c] <= 1.f)) {
                char msg[160];
                snprintf(msg, sizeof(msg), "%s: table entry color[%d][%d] must be finite and in [0, 1]", who, l, c);
                return fail_msg(msg);
            }
        t->color[l] = make_float4(p.color[l][0], p.color[l][1], p.color[l][2], p.color[l][3]);
        if (l != 0 && p.color[l][3] > 0.f) t->vis[l >> 5] |= 1u << (l & 31);
    }
    return 0;
}

// A label volume is a point-filtered, unnormalised, element-type 8-bit unsigned 3-D array (svr_labels_create): its array and dims
int label_volume(const char* who, const svr_volume& v, cudaArray_t* arr, int3* dims)
{
    auto err = [&]() { return fail_msg((std::string(who) + ": the volume is not a label volume (svr_labels_create)").c_str()); };
    if (!v.tex) return err();
    cudaTextureDesc td;
    SVR_TRY(cudaGetTextureObjectTextureDesc(&td, v.tex));
    cudaResourceDesc rd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&rd, v.tex));
    if (rd.resType != cudaResourceTypeArray || td.filterMode != cudaFilterModePoint || td.readMode != cudaReadModeElementType || td.normalizedCoords)
        return err();
    cudaChannelFormatDesc ch;
    cudaExtent ext;
    unsigned int flags = 0;
    SVR_TRY(cudaArrayGetInfo(&ch, &ext, &flags, rd.res.array.array));
    if (ch.x != 8 || ch.y || ch.z || ch.w || ch.f != cudaChannelFormatKindUnsigned || ext.depth == 0) return err();
    *arr = rd.res.array.array;
    *dims = make_int3((int)ext.width, (int)ext.height, (int)ext.depth);
    return 0;
}

}  // namespace
}  // namespace svr

extern "C" int svr_render_labels(svr_u8vec4* imgOrNull, svr_vec4* surfaceOrNull, uint8_t* labelOrNull, const svr_volume* labels,
                                 const svr_camera* camera, const svr_label_params* table, float stepSize, uint32_t phase, uint32_t stride,
                                 uint32_t* bandRows)
{
    HostState& st = state();
    const char* who = "svr_render_labels";
    if (!labels || !camera || !table) return fail_msg("svr_render_labels: null labels volume, camera or table");
    if (!imgOrNull && !surfaceOrNull && !labelOrNull) return fail_msg("svr_render_labels: all three outputs are null");
    if (!(stepSize > 0.f) || !std::isfinite(stepSize)) return fail_msg("svr_render_labels: stepSize must be positive and finite");
    LabelTable t;
    if (int rc = make_label_table(who, *table, &t)) return rc;
    if (phase >= stride) return fail_msg("svr_render_labels: band phase must be below the band stride");
    cudaArray_t arr;
    int3 dims;
    if (int rc = label_volume(who, *labels, &arr, &dims)) return rc;
    const LaunchOptions o = launch_options();
    if (bandRows) *bandRows = o.tileH;

    LabelScene sc;
    memset(&sc, 0, sizeof(sc));
    sc.vol = *labels;
    sc.cam = *camera;
    sc.dims = f3((float)dims.x, (float)dims.y, (float)dims.z);
    if (o.skip) {
        if (int rc = ensure_label_grid(arr, labels->tex, dims, st.options[SVR_OPT_MACROCELL_SIZE])) return rc;
        const DeviceState& d = st.dev;
        sc.presence = (const uint4*)d.labelPresence.p;
        sc.gx = d.labelGridDims.x;
        sc.gy = d.labelGridDims.y;
        sc.gz = d.labelGridDims.z;
        sc.scale = f3((float)dims.x / (float)d.labelCell, (float)dims.y / (float)d.labelCell, (float)dims.z / (float)d.labelCell);
    }
    dim3 grid;
    if (!band_grid(*camera, o.tileH, phase, stride, &grid)) return 0;
    Counters* cnt;
    if (int rc = launch_counters(who, o.count, &cnt)) return rc;
    const uint32_t H = camera->imageH;
    with_variant(o.skip, o.count, [&](auto sk, auto ct) {
        label_kernel<sk, ct><<<grid, o.block, 0, st.stream>>>(sc, t, stepSize, (uint32_t*)imgOrNull, (float4*)surfaceOrNull, labelOrNull, H,
                                                              phase, stride, cnt);
    });
    return launched();
}

extern "C" int svr_render_label_slices(svr_u8vec4* imgOrNull, uint8_t* labelOrNull, const svr_volume* labels, const svr_slice_params* params,
                                       const svr_label_params* table, int outline)
{
    HostState& st = state();
    const char* who = "svr_render_label_slices";
    if (!labels || !params || !table) return fail_msg("svr_render_label_slices: null labels volume, params or table");
    if (!imgOrNull && !labelOrNull) return fail_msg("svr_render_label_slices: both outputs are null");
    const svr_slice_params p = *params;
    if (int rc = check_slice_params(who, p)) return rc;
    LabelTable t;
    if (int rc = make_label_table(who, *table, &t)) return rc;
    if (outline != 0 && outline != 1) return fail_msg("svr_render_label_slices: outline must be 0 or 1");
    cudaArray_t arr;
    int3 dims;
    if (int rc = label_volume(who, *labels, &arr, &dims)) return rc;

    LabelSliceScene g;
    memset(&g, 0, sizeof(g));
    g.vol = *labels;
    g.center = f3(p.center[0], p.center[1], p.center[2]);
    g.u = f3(p.axisU[0], p.axisU[1], p.axisU[2]);
    g.v = f3(p.axisV[0], p.axisV[1], p.axisV[2]);
    g.w = p.count > 1u ? f3(p.axisW[0], p.axisW[1], p.axisW[2]) : f3(0.f);
    clipped_box(*labels, &g.cmin, &g.cmax);
    g.dims = f3((float)dims.x, (float)dims.y, (float)dims.z);
    g.W = p.imageW;
    g.H = p.imageH;
    const LaunchOptions o = launch_options();
    const dim3 grid((p.imageW + 15u) / 16u, (p.imageH + o.tileH - 1u) / o.tileH, p.count);
    label_slice_kernel<<<grid, o.block, 0, st.stream>>>(g, t, (uint32_t*)imgOrNull, labelOrNull, outline);
    return launched();
}
