// svr_scene.cuh -- the scene as the kernels see it, and the small device functions of the path.
//
// The reference keeps five __constant__ PODs in pathtracer.cu's translation unit
// (pathtracer.cu:34-68).  Here the same PODs plus the derived acceleration data travel as ONE
// kernel parameter block (DevScene, < 1 KB; kernel parameters live in the constant bank), so every
// kernel in every translation unit sees a consistent snapshot and launches on different streams
// cannot race on a global symbol.
#pragma once

#include "svr_math.cuh"

namespace svr {

// Macrocell majorant grid: cell (i,j,k) covers voxels [i*C, (i+1)*C) per axis in texel-index space.
// `cells` holds one float per cell: > 0 the majorant (max TF opacity reachable inside the cell);
// < 0 the cell is empty and so is the cube of radius (-value - 1) cells around it.  The array has a
// one-cell empty border, so indices -1 .. g are valid on every axis; `cells` points at cell (0,0,0).
struct DevGrid {
    const float* cells;
    const float2* range;     // per cell (min, max) of the filtered intensity before densityScale (no border)
    const int* occ;          // bounding box of the non-empty cells: lo x,y,z then hi x,y,z (inclusive)
    int gx, gy, gz;
    int px, pxy;             // row and slice pitch of `cells`
    int cell;                // cell edge in voxels
    float3 scale;            // normalised texture coordinate -> cell coordinate (dims / cell)
    float3 invScale;         // and back (cell / dims): a tap along a ray is taken at (g0 + t dg) * invScale
    float3 toCell, cellOff;  // world -> cell coordinate: p * toCell - cellOff  (toCell = invSize * scale, cellOff = vmin * toCell)
    float pyF;               // rows per slice of `cells` (gy + 2), as a float
    SVR_DEV float at(int cx, int cy, int cz) const { return __ldg(cells + (cz * pxy + cy * px + cx)); }
    // the same for integer-valued float coordinates; row index formed in fp32 (exact: rows * slices < 2^24)
    SVR_DEV float at(float3 cf) const { return __ldg(cells + ((int)fmaf(cf.z, pyF, cf.y) * px + (int)cf.x)); }
};

// Importance sampler of the environment light: a grid of w x h direction cells over (u, v) = (phi / 2 pi, theta / pi), cell
// probability proportional to (luminance + a floor) * sin(theta).  marg[0..h]: cumulative row probabilities;
// cond[j * (w + 1) + 0..w]: cumulative cell probabilities within row j.  Built by svr_env_io.cu: env_sampler_build.
struct DevEnvSampler {
    const float* marg;
    const float* cond;
    int w, h;
};

struct DevScene {
    svr_volume vol;
    svr_transfer_function tf;
    svr_camera cam;
    svr_env_light env;
    svr_area_light lights[SVR_MAX_LIGHT_SOURCES];
    uint32_t numLights;
    int32_t envEnabled;
    int32_t shadowEstimator;  // 0 binary delta tracking (transmittance.h:10-17), 1 ratio tracking
    uint32_t seedKey;
    int3 volDim;
    DevGrid grid;
    int32_t envNee;           // 1 = the environment light is a next-event target (SVR_OPT_ENV_NEE); escaped bounce rays then add nothing
    DevEnvSampler envS;
};

// ---- counters (SVR_OPT_COUNTERS) -------------------------------------------------------------
struct Counters {
    unsigned long long v[16];
};

template <bool ON>
struct LocalCounters;
template <>
struct LocalCounters<false> {
    SVR_DEV void add(int, uint32_t) {}
    SVR_DEV void flush(Counters*) {}
};
template <>
struct LocalCounters<true> {
    uint32_t c[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    SVR_DEV void add(int slot, uint32_t n) { c[slot] += n; }
    SVR_DEV void flush(Counters* g)
    {
#pragma unroll
        for (int i = 0; i < 9; ++i) {
            uint32_t x = c[i];
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
            if ((threadIdx.x & 31) == 0 && x) atomicAdd(&g->v[i], (unsigned long long)x);
        }
    }
};

// ---- volume (core/cuda_volume.h) ---------------------------------------------------------------
// cuda_volume.h:87-90
SVR_DEV float3 tex_coord(const svr_volume& v, float3 p) { return (p - f3(v.bbox.vmin)) * f3(v.bbox.invSize); }

// cuda_volume.h:92-100: hardware trilinear fetch (1.8 fixed-point weights, border = 0) times densityScale
SVR_DEV float intensity_at(const svr_volume& v, float3 p)
{
    float3 tc = tex_coord(v, p);
    return tex3D<float>(v.tex, tc.x, tc.y, tc.z) * v.densityScale;
}

// cuda_volume.h:54-61
SVR_DEV float3 gradient_at(const svr_volume& v, float3 p)
{
    float xd = intensity_at(v, p + f3(v.spacing.x, 0.f, 0.f)) - intensity_at(v, p - f3(v.spacing.x, 0.f, 0.f));
    float yd = intensity_at(v, p + f3(0.f, v.spacing.y, 0.f)) - intensity_at(v, p - f3(0.f, v.spacing.y, 0.f));
    float zd = intensity_at(v, p + f3(0.f, 0.f, v.spacing.z)) - intensity_at(v, p - f3(0.f, 0.f, v.spacing.z));
    return f3(xd, yd, zd) * 0.5f * f3(v.invSpacing);
}

// cuda_transfer_function.h:22-30
SVR_DEV float4 tf_at(const svr_transfer_function& tf, float intensity) { return tex1D<float4>(tf.tex, intensity); }

// cuda_bbox.h:33-54 through cuda_volume.h:49-52 (GLM min/max: `a < b ? a : b`)
SVR_DEV bool intersect_volume(const svr_volume& v, const Ray& ray, float* tNear, float* tFar)
{
    float3 invDir = 1.f / ray.dir;
    float3 cmin = f3(v.bbox.vmin) * f3(-v.x_clip.x, -v.y_clip.x, -v.z_clip.x);
    float3 cmax = f3(v.bbox.vmax) * f3(v.x_clip.y, v.y_clip.y, v.z_clip.y);
    float3 tbot = invDir * (cmin - ray.orig);
    float3 ttop = invDir * (cmax - ray.orig);
    float3 tmin = f3(tbot.x < ttop.x ? tbot.x : ttop.x, tbot.y < ttop.y ? tbot.y : ttop.y,
                     tbot.z < ttop.z ? tbot.z : ttop.z);
    float3 tmax = f3(tbot.x > ttop.x ? tbot.x : ttop.x, tbot.y > ttop.y ? tbot.y : ttop.y,
                     tbot.z > ttop.z ? tbot.z : ttop.z);
    float largest_tmin = fmaxf(tmin.x, fmaxf(tmin.y, tmin.z));
    float smallest_tmax = fminf(tmax.x, fminf(tmax.y, tmax.z));
    *tNear = largest_tmin;
    *tFar = smallest_tmax;
    return smallest_tmax > largest_tmin;
}

// ---- camera (core/cuda_camera.h) ---------------------------------------------------------------
// cuda_camera.h:85-95: pixel centre, pinhole
SVR_DEV Ray camera_ray_center(const svr_camera& c, uint32_t x, uint32_t y)
{
    float nx = 2.f * (((float)x + 0.5f) / ((float)c.imageW - 1.f)) - 1.f;
    float ny = 2.f * (((float)y + 0.5f) / ((float)c.imageH - 1.f)) - 1.f;
    nx = nx * c.aspectRatio * c.tanFovxOverTwo;
    ny = ny * c.tanFovxOverTwo;
    Ray r;
    r.orig = f3(c.pos);
    r.dir = normalize(nx * f3(c.u) + ny * f3(c.v) - f3(c.w));
    return r;
}

// Pixel of this thread in the image layout of the ray-marching kernels (ray caster, projection): a warp is an 8x4 pixel
// tile, a block 16 pixels wide (2 warps across) and blockDim/16 rows high.  Row bands of the block's height are dealt out
// round robin from the middle of the image outwards: this launch renders bands bandPhase, bandPhase + bandStride, ...
// (1 GPU: phase 0, stride 1).  Blocks launch in blockIdx order and the camera looks at the volume's centre
// (Canvas::ZoomToExtent), so the long rays start first and the short ones fill the tail.
SVR_DEV uint2 band_pixel(uint32_t y0, uint32_t y1, uint32_t bandPhase, uint32_t bandStride)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t idx = blockIdx.x * 16u + (warp & 1u) * 8u + (lane & 7u);
    const uint32_t nBands = ((y1 - y0) + (blockDim.x >> 4) - 1u) / (blockDim.x >> 4);
    const uint32_t k = blockIdx.y * bandStride + bandPhase;  // k-th band counted from the middle
    const uint32_t mid = nBands >> 1;
    const uint32_t band = (k & 1u) ? mid - ((k + 1u) >> 1) : mid + (k >> 1);
    const uint32_t idy = y0 + band * (blockDim.x >> 4) + (warp >> 1) * 4u + (lane >> 3);
    return make_uint2(idx, idy);
}

// sampling.h:26-32.  EXACT_PI: the reference evaluates 2.f * M_PI * u in double.
template <bool EXACT_PI>
SVR_DEV float two_pi_times(float u)
{
    if (EXACT_PI) return (float)(2.0 * SVR_PI_D * (double)u);
    return 2.f * SVR_PI_F * u;
}

template <bool EXACT_PI, class Rng>
SVR_DEV float2 uniform_sample_disk(Rng& rng, float r)
{
    r *= sqrtf(rng.next());
    float theta = two_pi_times<EXACT_PI>(rng.next());
    return make_float2(cosf(theta) * r, sinf(theta) * r);
}

// cuda_camera.h:66-83: jittered pixel, thin lens
template <bool EXACT_PI, class Rng>
SVR_DEV Ray camera_ray_jittered(const svr_camera& c, uint32_t x, uint32_t y, Rng& rng)
{
    float nx = 2.f * (((float)x + rng.next()) / ((float)c.imageW - 1.f)) - 1.f;
    float ny = 2.f * (((float)y + rng.next()) / ((float)c.imageH - 1.f)) - 1.f;
    nx = nx * c.aspectRatio * c.tanFovxOverTwo;
    ny = ny * c.tanFovxOverTwo;
    nx = nx * c.focalLength;
    ny = ny * c.focalLength;
    // EXACT_PI marks the reference-twin stream, which must consume the two lens draws even for a pinhole
    // (sampling.h:28-29 via cuda_camera.h:80); the counter-based streams skip them when the aperture is closed
    float2 a = make_float2(0.f, 0.f);
    if (EXACT_PI || c.apeture != 0.f) a = uniform_sample_disk<EXACT_PI>(rng, c.apeture);
    Ray r;
    r.orig = f3(c.pos) + a.x * f3(c.u) + a.y * f3(c.v);
    r.dir = normalize((nx - a.x) * f3(c.u) + (ny - a.y) * f3(c.v) - c.focalLength * f3(c.w));
    return r;
}

// cuda_camera.h:66-83 for a closed aperture (the lens sample is the origin itself): the direction through the pixel at
// sub-pixel position (jx, jy)
SVR_DEV float3 camera_dir_pinhole(const svr_camera& c, uint32_t x, uint32_t y, float jx, float jy)
{
    float nx = 2.f * (((float)x + jx) / ((float)c.imageW - 1.f)) - 1.f;
    float ny = 2.f * (((float)y + jy) / ((float)c.imageH - 1.f)) - 1.f;
    nx = nx * c.aspectRatio * c.tanFovxOverTwo;
    ny = ny * c.tanFovxOverTwo;
    nx = nx * c.focalLength;
    ny = ny * c.focalLength;
    return normalize(nx * f3(c.u) + ny * f3(c.v) - c.focalLength * f3(c.w));
}

// ---- lights (core/geometry/cuda_disk.h, core/lights/) ------------------------------------------
SVR_DEV float disk_area(const svr_disk& d) { return SVR_PI_F * d.radius * d.radius; }  // cuda_disk.h:53-56

// cuda_arealight.h:57
SVR_DEV float3 light_radiance(const svr_area_light& l)
{
    return 500.f * f3(l.color) * l.intensity * SVR_INV_PI_F / disk_area(l.disk);
}

// cuda_disk.h:32-51
SVR_DEV bool disk_intersect(const svr_disk& d, const Ray& ray, float* t)
{
    float denom = dot(f3(d.normal), ray.dir);
    if (fabsf(denom) > 1e-6f) {
        float3 co = f3(d.center) - ray.orig;
        *t = dot(co, f3(d.normal)) / denom;
        if (*t >= 0.f) {
            float3 p = ray.orig + *t * ray.dir;
            float3 c2 = p - f3(d.center);
            return sqrtf(dot(c2, c2)) <= d.radius;
        }
    }
    return false;
}

struct LightHit {
    float t;
    float3 normal, radiance;
};

// light_sample.h:23-49
SVR_DEV bool nearest_light(const DevScene& s, const Ray& ray, LightHit* ls)
{
    float tNear = FLT_MAX, t = FLT_MAX;
    int id = -1;
    for (uint32_t i = 0; i < s.numLights; ++i) {
        if (disk_intersect(s.lights[i].disk, ray, &t) && (t < tNear)) {
            tNear = t;
            id = (int)i;
        }
    }
    if (id != -1) {
        ls->t = tNear;
        ls->normal = f3(s.lights[id].disk.normal);
        ls->radiance = light_radiance(s.lights[id]);
        return true;
    }
    ls->t = -FLT_MAX;
    return false;
}

// light_sample.h:51-68
template <bool EXACT_PI, class Rng>
SVR_DEV float3 sample_light(const svr_area_light& light, float3 pos, Rng& rng, float3* lightPos, float3* wi, float* pdf)
{
    float2 lp = uniform_sample_disk<EXACT_PI>(rng, light.disk.radius);
    float3 ln = f3(light.disk.normal);
    Onb onb(ln);
    *lightPos = f3(light.disk.center) + onb.u * lp.x + onb.v * lp.y;
    float3 sv = *lightPos - pos;
    *wi = normalize(sv);
    float cosTerm = dot(ln, -(*wi));
    *pdf = dot(sv, sv) / (fabsf(cosTerm) * disk_area(light.disk));
    return cosTerm > 0.f ? light_radiance(light) : f3(0.f);
}

// cuda_environment_light.h:58-72 (the call the reference left commented out at pathtracer.cu:233)
SVR_DEV float3 env_radiance(const svr_env_light& e, float3 dir)
{
    if (e.tex == 0) return f3(e.defaultRadiance) * e.intensity;
    float theta = acosf(dir.y);
    float phi = atan2f(dir.x, dir.z);
    phi = phi < 0.f ? phi + 2.f * SVR_PI_F : phi;
    float u = phi * 0.5f * SVR_INV_PI_F;
    float v = theta * SVR_INV_PI_F;
    float4 val = tex2D<float4>(e.tex, u + e.offset.x, v + e.offset.y);
    return f3(val.x, val.y, val.z) * e.intensity;
}

// direction of (u, v) in the parameterisation env_radiance inverts: theta = acos(dir.y) = pi v, phi = atan2(dir.x, dir.z) = 2 pi u
SVR_DEV float3 env_direction(float u, float v)
{
    float st, ct, sp, cp;
    __sincosf(SVR_PI_F * v, &st, &ct);
    __sincosf(2.f * SVR_PI_F * u, &sp, &cp);
    return f3(st * sp, ct, st * cp);
}

// A direction with probability density *pdf (per unit solid angle) proportional to the sampler's cell weights: row by the
// marginal, cell by the row's conditional, uniform in (u, v) within the cell.
SVR_DEV float3 sample_env(const DevEnvSampler& e, float xi1, float xi2, float* pdf)
{
    int lo = 0, hi = e.h - 1;
    while (lo < hi) {  // largest row j with marg[j] <= xi1
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(e.marg + mid) <= xi1) lo = mid;
        else hi = mid - 1;
    }
    const int j = lo;
    const float m0 = __ldg(e.marg + j), m1 = __ldg(e.marg + j + 1);
    const float* row = e.cond + (size_t)j * (e.w + 1);
    lo = 0;
    hi = e.w - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(row + mid) <= xi2) lo = mid;
        else hi = mid - 1;
    }
    const int i = lo;
    const float c0 = __ldg(row + i), c1 = __ldg(row + i + 1);
    const float pRow = m1 - m0, pCell = c1 - c0;
    const float dv = pRow > 0.f ? (xi1 - m0) / pRow : 0.5f, du = pCell > 0.f ? (xi2 - c0) / pCell : 0.5f;
    const float u = ((float)i + fminf(fmaxf(du, 0.f), 0.999999f)) / (float)e.w, v = ((float)j + fminf(fmaxf(dv, 0.f), 0.999999f)) / (float)e.h;
    const float sinTheta = __sinf(SVR_PI_F * v);
    // density in (u, v): pRow * pCell * w * h; d omega = 2 pi^2 sin(theta) du dv
    *pdf = sinTheta > 0.f ? pRow * pCell * (float)e.w * (float)e.h / (2.f * SVR_PI_F * SVR_PI_F * sinTheta) : 0.f;
    return env_direction(u, v);
}

// ---- BSDFs (core/bsdf/) ------------------------------------------------------------------------
#define SVR_IOR (2.5f)    // pathtracer.cu:30
#define SVR_ALPHA (0.15f) // pathtracer.cu:31

SVR_DEV float schlick_fresnel(float ni, float no, float cosin)  // fresnel.h:10-15
{
    float R0 = (ni - no) * (ni - no) / ((ni + no) * (ni + no));
    float c = 1.f - cosin;
    return R0 + (1.f - R0) * c * c * c * c * c;
}

// henyey_greenstein.h:15-22 with g == PHASE_FUNC_G == 0 (pathtracer.cu:29): isotropic, 1/(4 pi)
SVR_DEV float hg_phase_f() { return SVR_INV_PI_F * 0.25f; }

// henyey_greenstein.h:29-51, g == 0
template <bool EXACT_PI, class Rng>
SVR_DEV void hg_phase_sample(float3 wo, float3* wi, float* pdf, Rng& rng)
{
    float phi = two_pi_times<EXACT_PI>(rng.next());
    float cosTheta = 1.f - 2.f * rng.next();
    float sinTheta = sqrtf(fmaxf(0.f, 1.f - cosTheta * cosTheta));
    Onb onb(wo);
    *wi = normalize(onb.local(sinTheta * cosf(phi), sinTheta * sinf(phi), cosTheta));
    *pdf = hg_phase_f();
}

SVR_DEV float lambert_f() { return 1.f / SVR_PI_F; }  // lambert.h:15-18

// sampling.h:47-56 + lambert.h:20-24
template <bool EXACT_PI, class Rng>
SVR_DEV void lambert_sample(float3 normal, float3* wi, float* pdf, Rng& rng)
{
    Onb onb(normal);
    float phi = two_pi_times<EXACT_PI>(rng.next());
    float sinTheta = sqrtf(rng.next());
    float cosTheta = sqrtf(fmaxf(0.f, 1.f - sinTheta * sinTheta));
    *wi = normalize(onb.local(sinTheta * cosf(phi), sinTheta * sinf(phi), cosTheta));
    *pdf = fabsf(dot(*wi, normal)) / SVR_PI_F;
}

SVR_DEV float beckmann_d(float3 normal, float3 wh, float alpha)  // microfacet.h:18-25
{
    float c2 = dot(normal, wh);
    c2 *= c2;
    return expf((c2 - 1.f) / (alpha * alpha * c2)) / (SVR_PI_F * alpha * alpha * c2 * c2);
}

SVR_DEV float geometry_cook_torrance(float3 wi, float3 wo, float3 normal, float3 wh)  // microfacet.h:42-50
{
    float cosO = dot(wo, wh);
    float cosTerm = dot(normal, wh);
    float g1 = 2.f * cosTerm * dot(normal, wo) / cosO;
    float g2 = 2.f * cosTerm * dot(normal, wi) / cosO;
    return fminf(1.f, fminf(g1, g2));
}

SVR_DEV float microfacet_f(float3 wi, float3 wo, float3 normal, float ior, float alpha)  // microfacet.h:52-68
{
    if (dot(wi, normal) * dot(wo, normal) < 0.f) return 0.f;
    float3 wh = normalize(wi + wo);
    float F = schlick_fresnel(1.f, ior, fabsf(dot(wh, wo)));
    float G = geometry_cook_torrance(wi, wo, normal, wh);
    float D = beckmann_d(normal, wh, alpha);
    return F * G * D / (4.f * fabsf(dot(normal, wi)) * fabsf(dot(normal, wo)));
}

// microfacet.h:70-79 + 95-111
template <class Rng>
SVR_DEV void microfacet_sample(float3 wo, float3 normal, float alpha, float3* wi, float* pdf, Rng& rng)
{
    Onb onb(normal);
    float phi = 2.f * SVR_PI_F * rng.next();
    float cosTheta = 1.f / (1.f - alpha * alpha * logf(rng.next_one_minus()));
    float sinTheta = sqrtf(fmaxf(0.f, 1.f - cosTheta * cosTheta));
    float3 wh = normalize(onb.local(sinTheta * cosf(phi), sinTheta * sinf(phi), cosTheta));
    wh = dot(wo, wh) >= 0.f ? wh : -wh;
    *wi = reflect(-wo, wh);
    *pdf = beckmann_d(normal, wh, alpha) / (4.f * fabsf(dot(wo, wh)));
}

// tonemapping.h:13-27.  The default argument gamma = 1/2.2 makes the exponent 1/gamma = 2.2;
// reproduced as written.
SVR_DEV float3 tone_map(float3 L, float exposure)
{
    float3 l = L * 16.f;
    l.x = 1.f - expf(-l.x * exposure);
    l.y = 1.f - expf(-l.y * exposure);
    l.z = 1.f - expf(-l.z * exposure);
    float invGamma = 1.f / (1.f / 2.2f);
    l.x = powf(l.x, invGamma);
    l.y = powf(l.y, invGamma);
    l.z = powf(l.z, invGamma);
    return l;
}

SVR_DEV uint32_t pack_u8x4(float r, float g, float b, float a)
{
    // glm::u8vec4(float...) converts by truncation (static_cast<uint8_t>)
    uint32_t R = (uint32_t)(uint8_t)(int)r, G = (uint32_t)(uint8_t)(int)g, B = (uint32_t)(uint8_t)(int)b,
             A = (uint32_t)(uint8_t)(int)a;
    return R | (G << 8) | (B << 16) | (A << 24);
}

}  // namespace svr
