// svr_pathtrace.cu -- Monte Carlo volumetric path tracer behind render_pathtracer
// (pathtracer.h:17; kernel_pathtracer / hdr_to_ldr / clear_hdr_buffer, pathtracer.cu:86-94, 200-304).
//
// One launch renders a BATCH of samples per pixel: each lane owns a pixel, walks its samples one
// after the other, keeps the radiance sum in registers, and at the end merges once into the
// caller's accumulator and writes the tone-mapped pixel -- the reference's three launches per
// sample (clear, trace + 12-byte RMW, tone map; pathtracer.cu:297-303) collapse into one launch
// per batch.
//
// Estimator modes (SVR_OPT_PT_MODE):
//   0  reference twin: global majorant tf.maxOpacity (woodcock_tracking.h:28-30), XORWOW stream
//      seeded wangHash(frameNo) + pixel with the reference's draw order -> path-for-path the same
//      walk as kernel_pathtracer up to fast-math / FMA-contraction rounding.
//   1  global majorant + Philox counter RNG (same estimator, different random stream).
//   2  local majorants: a walk over the macrocell grid (svr_macrocell.cu); within a cell the free
//      path is sampled against the cell's majorant, optical depth carries across cell faces, cells
//      with majorant 0 cost no fetch and are leapt over several at a time.  Delta tracking with any
//      valid majorant samples the same free-path distribution, so the expectation is unchanged.
// Shadow rays: binary delta-tracking estimate as the reference (transmittance.h:10-17), or ratio
// tracking (SVR_OPT_SHADOW_ESTIMATOR = 1).
//
// Kernel shapes (SVR_OPT_PT_KERNEL):
//   0  phase-scheduled warp: the reference's three nested data-dependent loops (bounces x tracking
//      x shadow tracking, SURVEY.md section 3.1) are cut into five phases -- GENERATE, MARCH (walk
//      macrocells / draw a free flight), COLLIDE (fetch + accept/reject), EVENT (shade, sample the
//      light, start the shadow ray) and BOUNCE (add direct light, sample the BSDF).  Every lane
//      carries its own phase; each round the warp votes and runs the phase most lanes are waiting
//      in, so each piece of code executes with as many active lanes as the warp can muster, whatever
//      ray (camera, bounce, shadow) or sample each lane is on.
//   1  megakernel: the reference's loop nest as written, one path at a time per lane.
#include "svr_rng.cuh"
#include "svr_state.h"

#include <type_traits>

// Launch bounds of the path-tracing kernels: at most SVR_PT_MAX_THREADS threads per block and at least
// SVR_PT_MIN_BLOCKS resident blocks per SM, i.e. a register budget of 65536 / (128 * 9) = 56 per thread
// (36 warps per SM).  Chosen by measurement (DESIGN.md section 3.1, round 2, C3 per 256-spp launch): 6 blocks (80
// registers) 9.01 ms, 7 (72) 8.55, 8 (64) 8.31, 9 (56, 314 B of spills) 8.22, 10 (48) 8.40, 12 (40) 8.43 -- the kernel
// waits on dependent latencies (cell code, tap, table look-up), and resident warps hide them better than registers do.
#ifndef SVR_PT_MIN_BLOCKS
#define SVR_PT_MIN_BLOCKS 9
#endif
#ifndef SVR_PT_MAX_THREADS
#define SVR_PT_MAX_THREADS 128
#endif
// the lane-per-pixel kernel (shape 1: render_pathtracer's one sample per call)
#ifndef SVR_PT_MEGA_BLOCKS
#define SVR_PT_MEGA_BLOCKS SVR_PT_MIN_BLOCKS
#endif
// the majorant-profile kernel (shape 4) and the scatter-queue kernel (shape 3) have budgets of their own
#ifndef SVR_PT_PROFILE_BLOCKS
#define SVR_PT_PROFILE_BLOCKS 7
#endif
// (C4, one 512-spp launch: 8 blocks 431 ms, 9 blocks 419 ms, 10 blocks 429 ms)
#ifndef SVR_PT_QUEUE_BLOCKS
#define SVR_PT_QUEUE_BLOCKS 9
#endif


namespace svr {
Counters* device_counters();

namespace {

struct PtLaunch {
    uint32_t traceDepth;
    uint32_t firstSample;  // == frameNo of the first sample in the batch
    uint32_t nSamples;
    uint32_t y0, y1;       // row range
    float* hdr;            // packed vec3 running mean (reference ABI) or null
    uint32_t* img;         // tone-mapped u8vec4 or null
    float4* sum;           // rgb = sum of samples, w = sample count (multi-GPU partials) or null
    int32_t clearSum;
    int32_t marchBurst;    // phase-scheduled kernel: macrocell visits per MARCH round
    int32_t entryCache;    // 1 = per-pixel camera-ray entry cache (mode 2)
    int32_t warpPixels;    // sample-parallel kernel: pixels one warp renders one after the other
    int32_t lightCull;     // 1 = classify_pixel may rule out camera-ray light hits (SVR_OPT_PT_LIGHT_CULL)
    int32_t clipped;       // some clip plane is active: the volume's box is smaller than its texture
    uint32_t bandRows;               // (out) rows per band of the kernel shape chosen
    int32_t pixelCache;              // shapes 1-3: 2 = pixelInfo holds the classification of every pixel (classify_pixels_kernel); others 0
    float2* pixelInfo;               // (tSkip, flags: bit 0 lights, bit 1 empty) per pixel
    int32_t blockSplit;              // shape 2: the warps of a block split the samples of one row's pixels (SVR_OPT_PT_BLOCK_SPLIT)
    uint32_t bandPhase, bandStride;  // this launch renders the row bands (block rows) phase, phase + stride, ... (1 GPU: 0, 1)
    float* perSample;                // look-ahead launch (shape 2, nSamples <= 32): component c of sample j of pixel p -> perSample[p * 3 * nSamples + 3 * j + c], nothing else is written
    uint8_t* constantPixel;          // look-ahead launch: 1 for a pixel whose every sample is the constant sky (no record written), else 0
};

template <int MODE>
struct RngOf {
    typedef Philox type;
};
template <>
struct RngOf<0> {
    typedef XorwowCompat type;
};

// ---------------------------------------------------------------------------------------------
// free-path sampling, split into visit() (advance to the next tentative collision or out of the
// volume; no volume fetch) and collide() (fetch + accept/reject) so that a warp can run each half
// convergently.
// ---------------------------------------------------------------------------------------------
enum VisitResult { VISIT_CONTINUE = 0, VISIT_COLLIDE = 1, VISIT_ESCAPED = 2 };

// woodcock_tracking.h:20-51, global majorant tf.GetMaxOpacity()
struct TrackGlobal {
    float t, tMin, tMax;

    template <class Rng>
    SVR_DEV bool begin(const DevScene& s, const Ray& ray, Rng&, float)
    {
        float tNear, tFar;
        if (!intersect_volume(s.vol, ray, &tNear, &tFar)) return false;
        tMin = tNear < 0.f ? 1e-6f : tNear;
        tMax = tFar;
        t = tMin;
        return true;
    }
    template <bool COUNT, class Rng>
    SVR_DEV VisitResult visit(const DevScene& s, const Ray&, Rng& rng, LocalCounters<COUNT>&)
    {
        const float invSigmaMaxSampleInterval = 1.f / (s.tf.maxOpacity * 1.f);  // BASE_SAMPLE_STEP_SIZE 1
        t += -logf(rng.next_one_minus()) * invSigmaMaxSampleInterval;
        return t > tMax ? VISIT_ESCAPED : VISIT_COLLIDE;
    }
    // true = real collision at t
    template <bool COUNT, class Rng>
    SVR_DEV bool collide(const DevScene& s, const Ray& ray, Rng& rng, LocalCounters<COUNT>& lc, int slot, float* ratioT)
    {
        const float invSigmaMax = 1.f / s.tf.maxOpacity;
        float intensity = intensity_at(s.vol, ray.orig + t * ray.dir);
        float sigma_t = tf_at(s.tf, intensity).w;
        lc.add(slot, 1);
        lc.add(SVR_CNT_TF_LOOKUPS, 1);
        if (ratioT) {
            *ratioT *= 1.f - sigma_t * invSigmaMax;
            return false;
        }
        return rng.next() < sigma_t * invSigmaMax || t > tMax;
    }
};

// Cell-space description of a ray: g(t) = g0 + t * dg is the position in macrocell coordinates.
struct CellRay {
    float3 g0, dg;
    float3 invDg;  // 1 / dg; FLT_MAX on an axis the ray does not move along (clip(): no constraint inside the slab)
    // exit_t(): the far face of the cube of r cells around cell c lies at f + 1/2 with f = c +- (r - 1/2) and
    // is crossed at (f + 1/2 - g0) / dg = f * k + h, one FMA.  An axis the ray does not move along has
    // k = 0, h = FLT_MAX: its faces are never reached.
    float3 k, h;
    SVR_DEV void init(const DevScene& s, const Ray& ray)
    {
        const float3 toCell = s.grid.toCell;
        g0 = ray.orig * toCell - s.grid.cellOff;
        dg = ray.dir * toCell;
        invDg.x = dg.x != 0.f ? 1.f / dg.x : FLT_MAX;
        invDg.y = dg.y != 0.f ? 1.f / dg.y : FLT_MAX;
        invDg.z = dg.z != 0.f ? 1.f / dg.z : FLT_MAX;
        k.x = dg.x != 0.f ? invDg.x : 0.f;
        k.y = dg.y != 0.f ? invDg.y : 0.f;
        k.z = dg.z != 0.f ? invDg.z : 0.f;
        h.x = dg.x != 0.f ? (0.5f - g0.x) * invDg.x : FLT_MAX;
        h.y = dg.y != 0.f ? (0.5f - g0.y) * invDg.y : FLT_MAX;
        h.z = dg.z != 0.f ? (0.5f - g0.z) * invDg.z : FLT_MAX;
    }
    // ray-parameter step that moves 1e-3 cell along the fastest axis
    SVR_DEV float eps() const { return 1e-3f * fminf(fminf(fabsf(invDg.x), fabsf(invDg.y)), fabsf(invDg.z)); }
    // parameter interval inside the slab [lo, hi] (cell coordinates) on every axis.  On a static axis
    // both products are +-huge with the same sign outside the slab (empty interval) and opposite signs
    // inside it (no constraint).
    SVR_DEV void clip(float3 lo, float3 hi, float* tA, float* tB) const
    {
        const float ax = (lo.x - g0.x) * invDg.x, bx = (hi.x - g0.x) * invDg.x;
        const float ay = (lo.y - g0.y) * invDg.y, by = (hi.y - g0.y) * invDg.y;
        const float az = (lo.z - g0.z) * invDg.z, bz = (hi.z - g0.z) * invDg.z;
        *tA = fmaxf(fmaxf(fminf(ax, bx), fminf(ay, by)), fminf(az, bz));
        *tB = fminf(fminf(fmaxf(ax, bx), fmaxf(ay, by)), fmaxf(az, bz));
    }
    // cell (as floats) containing the ray at parameter te
    SVR_DEV float3 locate(float te) const
    {
        return f3(floorf(fmaf(te, dg.x, g0.x)), floorf(fmaf(te, dg.y, g0.y)), floorf(fmaf(te, dg.z, g0.z)));
    }
    // parameter at which the ray leaves the cube of `r` cells beyond cell cf on the far side (r = 1: the
    // cell itself) and r - 1 cells on the near side.  A function of the face alone, not of how the ray got
    // here, so walks that start at different parameters (entry cache on / off) visit identical positions.
    SVR_DEV float exit_t(float3 cf, float r) const
    {
        // the face's coordinate minus 1/2, exact (an integer plus or minus a half-integer)
        const float rr = r - 0.5f;
        const float fx = cf.x + copysignf(rr, k.x), fy = cf.y + copysignf(rr, k.y), fz = cf.z + copysignf(rr, k.z);
        return fminf(fminf(fmaf(fx, k.x, h.x), fmaf(fy, k.y, h.y)), fmaf(fz, k.z, h.z));
    }
};

// Delta tracking against per-macrocell majorants with empty-space leaping.  The walk is position
// based: each visit looks up the cell under the ray just past the current parameter, spends the
// cell's optical depth (or leaps over the empty cube an empty cell records) and moves to the far
// face.  Occupied and empty cells run the same instructions, so lanes do not diverge inside the walk,
// and no per-axis DDA state has to live in registers.
struct TrackLocal {
    float t, tMax;
    float tau;  // optical depth still to travel before the next tentative collision
    float sig;  // majorant of the cell the tentative collision lies in
    CellRay cr;
    float epsT;  // cr.eps(): the step that carries the walk across a cell face, computed once per ray (-1 % on C3)

    SVR_DEV bool begin(const DevScene& s, const Ray& ray, Philox& rng, float tSkip)
    {
        float tNear, tFar;
        if (!intersect_volume(s.vol, ray, &tNear, &tFar)) return false;
        // a NaN direction component slips through the slab test (fminf/fmaxf drop NaNs); it must not index the grid
        if (!(fabsf(ray.dir.x) + fabsf(ray.dir.y) + fabsf(ray.dir.z) < 4.f)) return false;
        const float tMin = tNear < 0.f ? 1e-6f : tNear;
        cr.init(s, ray);
        // nothing can collide outside the box of non-empty cells, nor before the pixel's cached entry
        const int* occ = s.grid.occ;
        float tA, tB;
        cr.clip(f3((float)__ldg(occ + 0), (float)__ldg(occ + 1), (float)__ldg(occ + 2)),
                f3((float)(__ldg(occ + 3) + 1), (float)(__ldg(occ + 4) + 1), (float)(__ldg(occ + 5) + 1)), &tA, &tB);
        t = fmaxf(fmaxf(tMin, tA), tSkip);
        tMax = fminf(tFar, tB);
        if (!(t < tMax)) return false;
        tau = -logf(rng.next_one_minus());
        epsT = cr.eps();
        return true;
    }
    template <bool COUNT>
    SVR_DEV VisitResult visit(const DevScene& s, const Ray& ray, Philox&, LocalCounters<COUNT>& lc)
    {
        const float te = t + epsT;
        const float3 cf = cr.locate(te);
        const float m = s.grid.at(cf);
        lc.add(SVR_CNT_CELLS, 1);
        // m > 0: majorant of this cell.  m < 0: empty, and so is the cube of radius -m-1 around it.
        const float sg = fmaxf(m, 0.f);
        const float tE = cr.exit_t(cf, fmaxf(-m, 1.f));
        const float dd = fmaxf(fminf(tE, tMax) - t, 0.f) * sg;
        if (tau < dd) {
            t += tau / sg;
            sig = sg;
            return VISIT_COLLIDE;
        }
        tau -= dd;
        if (tE >= tMax) return VISIT_ESCAPED;
        t = fmaxf(tE, te);
        return VISIT_CONTINUE;
    }
    template <bool COUNT>
    SVR_DEV bool collide(const DevScene& s, const Ray& ray, Philox& rng, LocalCounters<COUNT>& lc, int slot, float* ratioT)
    {
        // the tap's texture coordinate from the ray in cell coordinates (already in registers for the walk): (g0 + t dg) / scale is
        // (orig + t dir - vmin) * invSize up to rounding, three operations fewer, and the loop does not touch the world-space ray
        const float3 tc = f3(fmaf(t, cr.dg.x, cr.g0.x), fmaf(t, cr.dg.y, cr.g0.y), fmaf(t, cr.dg.z, cr.g0.z)) * s.grid.invScale;
        float intensity = tex3D<float>(s.vol.tex, tc.x, tc.y, tc.z) * s.vol.densityScale;
        float sigma_t = tf_at(s.tf, intensity).w;
        lc.add(slot, 1);
        lc.add(SVR_CNT_TF_LOOKUPS, 1);
        float ua, ub;
        rng.next2(ua, ub);  // one Philox block: the accept draw and the next free-flight draw
        tau = -logf(1.f - ub);
        if (ratioT) {
            *ratioT *= 1.f - sigma_t / sig;
            return false;
        }
        return ua * sig < sigma_t;
    }
};

template <int MODE>
struct TrackOf {
    typedef TrackGlobal type;
};
template <>
struct TrackOf<2> {
    typedef TrackLocal type;
};
// MODE 3 (internal): mode 2 with the environment light as a next-event target (SVR_OPT_ENV_NEE).  An estimator of its own
// so that the code it adds costs the other modes' kernels no registers.
template <>
struct TrackOf<3> {
    typedef TrackLocal type;
};

// What is known about ALL camera rays of a pixel before any sample is drawn.  With a pinhole
// (aperture 0) the samples of a pixel share the origin and differ by at most half a pixel diagonal in
// direction, so one look along the pixel's centre ray bounds what every jittered ray can meet:
//   lights : some camera ray of the pixel may hit an area-light disk (get_nearest_light_sample,
//            pathtracer.cu:214-215, has to be evaluated);
//   empty  : no camera ray of the pixel can reach a non-empty macrocell (mode 2): every sample escapes;
//   tSkip  : parameter up to which every camera ray of the pixel runs through empty macrocells
//            (mode 2; 0 when nothing can be said).
// Only empty space is skipped and no random number is consumed, so images do not change.
struct PixelInfo {
    float tSkip;
    bool lights, empty;
};

SVR_DEV PixelInfo classify_pixel(const DevScene& s, uint32_t idx, uint32_t idy, bool haveGrid, bool walk, bool lightCull)
{
    PixelInfo pi;
    pi.tSkip = 0.f;
    pi.lights = s.numLights != 0;
    pi.empty = false;
    const svr_camera& c = s.cam;
    if (c.apeture != 0.f) return pi;
    Ray ray;
    {
        float nx = 2.f * (((float)idx + 0.5f) / ((float)c.imageW - 1.f)) - 1.f;
        float ny = 2.f * (((float)idy + 0.5f) / ((float)c.imageH - 1.f)) - 1.f;
        nx = nx * c.aspectRatio * c.tanFovxOverTwo;
        ny = ny * c.tanFovxOverTwo;
        ray.orig = f3(c.pos);
        ray.dir = normalize(nx * f3(c.u) + ny * f3(c.v) - f3(c.w));
    }
    // largest angle (radians, small) between the centre ray and any jittered ray of the pixel
    const float hx = c.aspectRatio * c.tanFovxOverTwo / ((float)c.imageW - 1.f), hy = c.tanFovxOverTwo / ((float)c.imageH - 1.f);
    const float alpha = sqrtf(hx * hx + hy * hy) * 1.05f;

    // ---- lights: a ray hits a disk only if it passes within `radius` of the centre, in front of the origin
    bool lights = !lightCull && s.numLights != 0;
    for (uint32_t i = 0; i < s.numLights; ++i) {
        const float3 v = f3(s.lights[i].disk.center) - ray.orig;
        const float dist = sqrtf(dot(v, v)), along = dot(v, ray.dir);
        const float3 off = v - along * ray.dir;
        const float reach = s.lights[i].disk.radius + dist * alpha * 1.1f;
        // (NaN-safe: any comparison that fails keeps the light)
        if (!(dot(off, off) > reach * reach) && !(along < -reach)) lights = true;
    }
    pi.lights = lights;
    if (!haveGrid) return pi;

    // ---- the macrocell grid along the centre ray
    CellRay cr;
    cr.init(s, ray);
    const int* occ = s.grid.occ;
    const float3 lo = f3((float)__ldg(occ + 0), (float)__ldg(occ + 1), (float)__ldg(occ + 2));
    const float3 hi = f3((float)(__ldg(occ + 3) + 1), (float)(__ldg(occ + 4) + 1), (float)(__ldg(occ + 5) + 1));
    if (!(lo.x < hi.x)) {  // no occupied cell at all
        pi.empty = true;
        pi.tSkip = FLT_MAX;
        return pi;
    }
    // sideways spread of the pixel's rays, in world units, at the farthest point of the occupied box
    const float3 cellWorld = f3((float)s.grid.cell) * f3(s.vol.spacing);
    const float minCell = fminf(fminf(cellWorld.x, cellWorld.y), cellWorld.z);
    const float3 bc = f3(s.vol.bbox.vmin) + 0.5f * (lo + hi) * cellWorld - ray.orig;
    const float3 bh = 0.5f * (hi - lo) * cellWorld;
    const float farthest = sqrtf(dot(bc, bc)) + sqrtf(dot(bh, bh));
    if (!(farthest * alpha < 0.9f * minCell)) return pi;
    // occupied box grown by one cell: a jittered ray inside the occupied box keeps the centre ray inside this one
    float tA, tB;
    cr.clip(lo - f3(1.f), hi + f3(1.f), &tA, &tB);
    tA = fmaxf(tA, 0.f);
    if (!(tA < tB)) {
        pi.empty = true;
        pi.tSkip = FLT_MAX;
        return pi;
    }
    if (!walk) return pi;
    // walk the centre ray with every empty cube shrunk by one cell; as long as it stays in empty space,
    // every jittered ray of the pixel is in empty space too
    float t = tA;
    for (int guard = 0; guard < 4096; ++guard) {
        const float te = t + cr.eps();
        float3 cf = cr.locate(te);
        cf.x = fminf(fmaxf(cf.x, -1.f), (float)s.grid.gx);
        cf.y = fminf(fmaxf(cf.y, -1.f), (float)s.grid.gy);
        cf.z = fminf(fmaxf(cf.z, -1.f), (float)s.grid.gz);
        const float m = s.grid.at(cf);
        if (!(m <= -2.f)) break;  // a non-empty cell is at most one cell away from the centre ray
        const float tE = cr.exit_t(cf, -m - 1.f);  // cube of radius d-2: the sideways cell stays inside the empty cube of radius d-1
        if (tE >= tB) {
            pi.empty = true;
            pi.tSkip = FLT_MAX;
            return pi;
        }
        t = fmaxf(tE, te);
    }
    pi.tSkip = t;
    return pi;
}

// The classification of every pixel, made once per scene by a kernel of its own (classify_pixels_kernel: one lane per pixel,
// 32 different pixels per warp) and read by the render kernels -- inside the sample-parallel kernel a warp classifies the two
// pixels of its run with two lanes while thirty wait, 0.3 ms per C3 launch against 0.03 ms for the whole image here.
SVR_DEV PixelInfo load_pixel_info(const float2* info, uint32_t offset)
{
    const float2 c = info[offset];
    const uint32_t f = __float_as_uint(c.y);
    PixelInfo pi;
    pi.tSkip = c.x;
    pi.lights = (f & 1u) != 0u;
    pi.empty = (f & 2u) != 0u;
    return pi;
}

__global__ void __launch_bounds__(128) classify_pixels_kernel(const __grid_constant__ DevScene s, float2* info, int haveGrid, int walk, int lightCull)
{
    // 8 x 4 pixels per warp, 16 x 8 per block: neighbouring centre rays walk the same macrocells
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t idx = blockIdx.x * 16u + (warp & 1u) * 8u + (lane & 7u);
    const uint32_t idy = blockIdx.y * 8u + (warp >> 1) * 4u + (lane >> 3);
    if (idx >= s.cam.imageW || idy >= s.cam.imageH) return;
    const PixelInfo pi = classify_pixel(s, idx, idy, haveGrid != 0, walk != 0, lightCull != 0);
    info[idy * s.cam.imageW + idx] = make_float2(pi.tSkip, __uint_as_float((pi.lights ? 1u : 0u) | (pi.empty ? 2u : 0u)));
}

// ---------------------------------------------------------------------------------------------
// shading (pathtracer.cu:96-198)
// ---------------------------------------------------------------------------------------------
struct VolumeSample {  // cuda_volume.h:124-132
    float3 ptInWorld, wo;
    float3 gradient;
    float4 color_opacity;
};

enum ShadingType { ISOTROPIC, BRDF };

// pathtracer.cu:106-131
SVR_DEV float3 bsdf(const VolumeSample& vs, float3 wi, ShadingType st)
{
    float3 diffuseColor = f3(vs.color_opacity.x, vs.color_opacity.y, vs.color_opacity.z);
    if (st == ISOTROPIC) return diffuseColor * hg_phase_f();
    float3 normal = normalize(vs.gradient);
    normal = dot(vs.wo, normal) < 0.f ? -normal : normal;
    float cosTerm = fmaxf(0.f, dot(wi, normal));
    float ks = schlick_fresnel(1.0f, SVR_IOR, cosTerm);
    float kd = 1.f - ks;
    float3 diffuse = diffuseColor * lambert_f();
    float3 specular = f3(1.f) * microfacet_f(wi, vs.wo, normal, SVR_IOR, SVR_ALPHA);
    return (kd * diffuse + ks * specular) * cosTerm;
}

// pathtracer.cu:133-169
template <bool EXACT_PI, class Rng>
SVR_DEV float3 sample_bsdf(const VolumeSample& vs, float3* wi, float* pdf, Rng& rng, ShadingType st)
{
    float3 color = f3(vs.color_opacity.x, vs.color_opacity.y, vs.color_opacity.z);
    if (st == ISOTROPIC) {
        hg_phase_sample<EXACT_PI>(vs.wo, wi, pdf, rng);
        return color * hg_phase_f();
    }
    float3 normal = normalize(vs.gradient);
    float cosTerm = dot(vs.wo, normal);
    if (cosTerm < 0.f) {
        cosTerm = -cosTerm;
        normal = -normal;
    }
    float ks = schlick_fresnel(1.f, SVR_IOR, cosTerm);
    float kd = 1.f - ks;
    float p = 0.25f + 0.5f * ks;
    if (rng.next() < p) {
        microfacet_sample(vs.wo, normal, SVR_ALPHA, wi, pdf, rng);
        float f = microfacet_f(*wi, vs.wo, normal, SVR_IOR, SVR_ALPHA);
        return f3(1.f) * f * ks / p;
    }
    lambert_sample<EXACT_PI>(normal, wi, pdf, rng);
    return color * lambert_f() * kd / (1.f - p);
}

// What a bounce collects per unit radiance arriving from wi, in expectation over sample_bsdf and the lobe choice of
// pathtracer.cu:250-267: the lobes the bounce can take -- the phase function unless Pbrdf is 1, the BRDF with its cosine
// unless Pbrdf is 0 -- weighted as sample_bsdf weights them (Fresnel of the OUTGOING direction, pathtracer.cu:143-153;
// bsdf(), which the area lights use, takes the Fresnel term of the incoming one, :118-121).  Used by the environment
// light's next-event estimation, which replaces exactly that collection.
SVR_DEV float3 lobes_as_sampled(const VolumeSample& vs, float3 wi, float Pbrdf)
{
    const float3 color = f3(vs.color_opacity.x, vs.color_opacity.y, vs.color_opacity.z);
    float3 f = f3(0.f);
    if (Pbrdf < 1.f) f += color * hg_phase_f();
    if (Pbrdf > 0.f) {
        float3 normal = normalize(vs.gradient);
        float cosO = dot(vs.wo, normal);
        if (cosO < 0.f) {
            cosO = -cosO;
            normal = -normal;
        }
        const float cosI = dot(wi, normal);
        if (cosI > 0.f) {
            const float ks = schlick_fresnel(1.f, SVR_IOR, cosO), kd = 1.f - ks;
            f += (kd * lambert_f() * color + f3(ks * microfacet_f(wi, vs.wo, normal, SVR_IOR, SVR_ALPHA))) * cosI;
        }
    }
    return f;
}

// pathtracer.cu:96-103 (the 0.0722 term is a double product in the reference)
template <bool EXACT, class Rng>
SVR_DEV bool russian_roulette(float3* T, Rng& rng)
{
    float illum;
    if (EXACT) illum = (float)((double)(0.2126f * T->x + 0.7152f * T->y) + 0.0722 * (double)T->z);
    else illum = 0.2126f * T->x + 0.7152f * T->y + 0.0722f * T->z;
    if (rng.next() > illum) return true;
    *T = *T / illum;
    return false;
}

// Per-lane path state shared by both kernel shapes.
template <int MODE>
struct PathState {
    typename RngOf<MODE>::type rng;
    typename TrackOf<MODE>::type trk;
    Ray ray;          // the ray being tracked (camera / bounce ray, or the shadow ray)
    // L: radiance.  The reference-twin mode keeps the reference's order of additions -- L per path, paths
    // summed (pathtracer.cu:208, 279) -- so L restarts with every path and `sum` collects the paths; the
    // other modes add every contribution of every path of the pixel straight into L.
    float3 L, sum, T;
    uint32_t k;
    // stash across the shadow ray
    VolumeSample vs;
    float3 pending;   // numLights * bsdf * Li / pdf, to be multiplied by the transmittance
    float Pbrdf;
    float ratioT;     // ratio-tracking running transmittance
    ShadingType st;
    bool shadow;      // the tracked ray is a shadow ray
    bool camLights;   // a camera ray of this pixel may hit a light (PixelInfo::lights)
    bool envEsc;      // the ray being tracked adds the environment light if it escapes (always, unless the environment is a
                      // next-event target and this is a bounce ray whose vertex has already been lit by it)
};

// what a lane does next
enum Next { NEXT_TRACK = 0, NEXT_PATH_DONE = 1, NEXT_FLIGHT_MISSED = 2, NEXT_BOUNCE = 3, NEXT_EVENT_AT_T = 4 /* scatter queue: a collision popped from the queue */ };

// pathtracer.cu:204-213: seed, camera ray; then start tracking it.  Returns false when the ray
// cannot collide (misses the volume): an immediate "escaped" event.
template <int MODE>
SVR_DEV bool path_begin(const DevScene& s, PathState<MODE>& ps, uint32_t idx, uint32_t idy, uint32_t offset, uint32_t sample,
                        float tSkip)
{
    constexpr bool EXACT_PI = MODE == 0;
    ps.rng.init(s.seedKey, offset, sample);
    if (MODE == 0) ps.L = f3(0.f);
    ps.T = f3(1.f);
    ps.k = 0;
    ps.shadow = false;
    if (MODE == 3) ps.envEsc = true;
    ps.ray = camera_ray_jittered<EXACT_PI>(s.cam, idx, idy, ps.rng);
    return ps.trk.begin(s, ps.ray, ps.rng, tSkip);
}

// A camera / bounce flight ended at distance t (or left the volume: t = -FLT_MAX):
// pathtracer.cu:214-255 plus estimate_direct_light up to the shadow ray (:171-191).
template <int MODE, bool COUNT>
SVR_DEV Next event_flight_end(const DevScene& s, PathState<MODE>& ps, float t, uint32_t traceDepth, LocalCounters<COUNT>& lc)
{
    constexpr bool EXACT_PI = MODE == 0;
    if (ps.k == 0) {
        // get_nearest_light_sample on the camera ray (pathtracer.cu:214-215, 220-229); the ray is still
        // the camera ray here, so the hit is evaluated at the event instead of living in registers
        LightHit ls;
        if (ps.camLights && nearest_light(s, ps.ray, &ls)) {
            float tt = t < 0.f ? FLT_MAX : t;
            if (ls.t < tt) {
                float cosTerm = dot(ls.normal, -ps.ray.dir);
                ps.L += ps.T * ls.radiance * (cosTerm <= 0.f ? 0.f : 1.f);
                return NEXT_PATH_DONE;
            }
        }
    }
    if (t < 0.f) {
        if (s.envEnabled && (MODE != 3 || ps.envEsc)) ps.L += ps.T * env_radiance(s.env, ps.ray.dir);  // the line commented out at pathtracer.cu:233
        return NEXT_PATH_DONE;
    }
    VolumeSample& vs = ps.vs;
    vs.wo = -ps.ray.dir;
    vs.ptInWorld = ps.ray.orig + t * ps.ray.dir;
    float intensity = intensity_at(s.vol, vs.ptInWorld);
    vs.color_opacity = tf_at(s.tf, intensity);
    vs.gradient = gradient_at(s.vol, vs.ptInWorld);
    float gradientMagnitude = sqrtf(dot(vs.gradient, vs.gradient));
    lc.add(SVR_CNT_SHADE_TAPS, 7);
    lc.add(SVR_CNT_TF_LOOKUPS, 1);
    lc.add(SVR_CNT_SCATTERS, 1);
    const float gf = s.vol.gradientFactor;
    ps.Pbrdf = vs.color_opacity.w * (1.f - expf(-25.f * gf * gf * gf * gradientMagnitude * 65535.f * s.vol.invMaxMagnitude));
    ps.st = (ps.rng.next() < ps.Pbrdf) ? BRDF : ISOTROPIC;

    // estimate_direct_light, pathtracer.cu:171-198
    ps.shadow = true;
    ps.pending = f3(0.f);
    ps.ratioT = 1.f;
    // One light is picked uniformly (pathtracer.cu:179).  With SVR_OPT_ENV_NEE the environment light is one more candidate:
    // sampled by importance from its luminance (sample_env) and weighted with BOTH lobes of the hybrid model -- exactly what
    // the bounce ray would have collected from the sky on leaving the medium (it no longer does: event_bounce clears envEsc).
    // (the sky reaches a vertex through the ray that leaves it, and the reference traces that ray only if another iteration
    // of its bounce loop follows, pathtracer.cu:216: the last vertex of a path gets no environment light)
    const bool envNee = MODE == 3 && ps.k + 1 < traceDepth;
    const uint32_t nPick = s.numLights + (envNee ? 1u : 0u);
    if (nPick != 0) {
        int lightId = (int)((float)nPick * ps.rng.next());
        lightId = lightId < (int)nPick ? lightId : (int)nPick - 1;
        if (lightId < (int)s.numLights) {
            float3 lightPos, wi;
            float pdf;
            float3 Li = sample_light<EXACT_PI>(s.lights[lightId], vs.ptInWorld, ps.rng, &lightPos, &wi, &pdf);
            if (pdf > 0.f && max3(Li) > 0.f) {
                ps.pending = (float)nPick * bsdf(vs, wi, ps.st) * Li / pdf;
                // transmittance.h:10-17: track from the sample toward the light through the whole box
                ps.ray.orig = vs.ptInWorld;
                ps.ray.dir = normalize(lightPos - vs.ptInWorld);
                return ps.trk.begin(s, ps.ray, ps.rng, 0.f) ? NEXT_TRACK : NEXT_FLIGHT_MISSED;
            }
        } else if (envNee) {
            float pdf;
            const float xi1 = ps.rng.next(), xi2 = ps.rng.next();
            const float3 wi = sample_env(s.envS, xi1, xi2, &pdf);
            const float3 Li = env_radiance(s.env, wi);
            if (pdf > 0.f && max3(Li) > 0.f) {
                ps.pending = (float)nPick * lobes_as_sampled(vs, wi, ps.Pbrdf) * Li / pdf;
                ps.ray.orig = vs.ptInWorld;
                ps.ray.dir = wi;
                return ps.trk.begin(s, ps.ray, ps.rng, 0.f) ? NEXT_TRACK : NEXT_FLIGHT_MISSED;
            }
        }
    }
    return NEXT_BOUNCE;  // no shadow ray to fly: bounce with nothing pending
}

// The shadow flight ended (or there was none): add the direct light, then bounce (pathtracer.cu:257-276).
// `occluded` is the binary estimator's verdict (transmittance.h:14-16).
template <int MODE, bool COUNT>
SVR_DEV Next event_bounce(const DevScene& s, PathState<MODE>& ps, bool occluded, uint32_t traceDepth, LocalCounters<COUNT>&)
{
    constexpr bool EXACT_PI = MODE == 0;
    const float Tr = s.shadowEstimator ? ps.ratioT : (occluded ? 0.f : 1.f);
    ps.L += ps.T * (Tr * ps.pending);
    ps.shadow = false;
    const VolumeSample& vs = ps.vs;
    // the last bounce's BSDF sample is never used: skip it unless reproducing the reference's draws
    if (MODE != 0 && ps.k + 1 >= traceDepth) return NEXT_PATH_DONE;
    float3 wi = f3(0.f);
    float pdf = 0.f;
    float3 f = sample_bsdf<EXACT_PI>(vs, &wi, &pdf, ps.rng, ps.st);
    float cosTerm = fabsf(dot(normalize(vs.gradient), wi));
    const bool sampled = max3(f) > 0.f && pdf > 0.f;
    if (sampled) {
        if (ps.st == ISOTROPIC)
            ps.T *= f / (pdf * (1.f - ps.Pbrdf));
        else
            ps.T *= f * cosTerm / (pdf * ps.Pbrdf);
    }
    // With the environment as a next-event target this vertex has been lit by it through both lobes; the bounce ray must not
    // collect it again.  A bounce whose BSDF sample was void keeps its throughput in the reference (the `if` above): that part
    // of the reference's estimator is not covered by the lobes, so such a ray still collects the sky on leaving.
    if (MODE == 3) ps.envEsc = !sampled;
    ps.ray.orig = vs.ptInWorld;
    ps.ray.dir = wi;
    if (ps.k >= 3) {
        if (russian_roulette<EXACT_PI>(&ps.T, ps.rng)) return NEXT_PATH_DONE;
    }
    ps.k += 1;
    if (ps.k >= traceDepth) return NEXT_PATH_DONE;
    return ps.trk.begin(s, ps.ray, ps.rng, 0.f) ? NEXT_TRACK : NEXT_FLIGHT_MISSED;
}

// Russian roulette for ratio tracking on a nearly opaque segment; true = terminate with T = 0
template <class Rng>
SVR_DEV bool ratio_roulette(float& T, Rng& rng)
{
    if (T >= 0.02f) return false;
    if (rng.next() * 0.02f >= T) {
        T = 0.f;
        return true;
    }
    T = 0.02f;
    return false;
}

SVR_DEV void write_pixel(const DevScene& s, const PtLaunch& a, uint32_t offset, float3 sum)
{
    if (a.sum) {
        float4 prev = a.clearSum ? make_float4(0.f, 0.f, 0.f, 0.f) : a.sum[offset];
        a.sum[offset] = make_float4(prev.x + sum.x, prev.y + sum.y, prev.z + sum.z, prev.w + (float)a.nSamples);
    }
    if (a.hdr) {
        // running_estimate (pathtracer.cu:81-84) for one sample; its closed form for a batch
        float* h = a.hdr + 3 * (size_t)offset;
        const float N0 = (float)a.firstSample;
        float3 acc = a.firstSample == 0 ? f3(0.f) : f3(h[0], h[1], h[2]);  // frameNo==0 clears (pathtracer.cu:297-300)
        if (a.nSamples == 1)
            acc = acc + (sum - acc) / (N0 + 1.f);
        else
            acc = (acc * N0 + sum) / (N0 + (float)a.nSamples);
        h[0] = acc.x;
        h[1] = acc.y;
        h[2] = acc.z;
        if (a.img) {
            float3 l = tone_map(acc, s.cam.exposure);  // hdr_to_ldr, pathtracer.cu:282-290
            a.img[offset] = pack_u8x4(l.x * 255.f, l.y * 255.f, l.z * 255.f, 255.f);
        }
    }
}

// The same for a pixel a whole warp has rendered (every lane holds the reduced sum): lanes 0..2 read-modify-write one
// component each of the packed vec3 accumulator -- one coalesced 12-byte access instead of three scalar ones by one lane --
// and tone-map it; lane 0 packs the three bytes and writes the u8vec4, and the float4 of the multi-GPU partial sums.
SVR_DEV void write_pixel_warp(const DevScene& s, const PtLaunch& a, uint32_t offset, float3 sum, uint32_t lane)
{
    if (a.sum && lane == 0) {
        float4 prev = a.clearSum ? make_float4(0.f, 0.f, 0.f, 0.f) : a.sum[offset];
        a.sum[offset] = make_float4(prev.x + sum.x, prev.y + sum.y, prev.z + sum.z, prev.w + (float)a.nSamples);
    }
    if (a.hdr) {
        float byteF = 0.f;
        if (lane < 3) {
            float* h = a.hdr + 3 * (size_t)offset + lane;
            const float mine = lane == 0 ? sum.x : (lane == 1 ? sum.y : sum.z);
            const float N0 = (float)a.firstSample;
            float acc = a.firstSample == 0 ? 0.f : *h;  // frameNo==0 clears (pathtracer.cu:297-300)
            if (a.nSamples == 1) acc = acc + (mine - acc) / (N0 + 1.f);  // running_estimate (pathtracer.cu:81-84); its closed form for a batch
            else acc = (acc * N0 + mine) / (N0 + (float)a.nSamples);
            *h = acc;
            // hdr_to_ldr, pathtracer.cu:282-290 (component-wise: tone_map)
            byteF = powf(1.f - expf(-(acc * 16.f) * s.cam.exposure), 1.f / (1.f / 2.2f)) * 255.f;
        }
        if (a.img) {
            const float g = __shfl_sync(0xffffffffu, byteF, 1), b = __shfl_sync(0xffffffffu, byteF, 2);
            if (lane == 0) a.img[offset] = pack_u8x4(byteF, g, b, 255.f);
        }
    }
}

// the flight's verdict for the binary transmittance estimator, transmittance.h:14-15
SVR_DEV bool occluded_at(const TrackGlobal& trk, float t) { return (t > trk.tMin) && (t < trk.tMax); }
// local-majorant flights report either a collision strictly inside (tMin, tMax) or -FLT_MAX
SVR_DEV bool occluded_at(const TrackLocal&, float t) { return t > -FLT_MAX; }

// ---------------------------------------------------------------------------------------------
// kernel shape 1: megakernel (the reference's loop nest)
// ---------------------------------------------------------------------------------------------
// Radiance accumulators of a pixel (see PathState::L)
template <int MODE>
SVR_DEV void pixel_begin(PathState<MODE>& ps)
{
    ps.L = f3(0.f);
    ps.sum = f3(0.f);
}
template <int MODE>
SVR_DEV void path_end(PathState<MODE>& ps)
{
    if (MODE == 0) ps.sum += ps.L;
}
template <int MODE>
SVR_DEV float3 pixel_sum(const PathState<MODE>& ps) { return MODE == 0 ? ps.sum : ps.L; }

// One flight: the tracking loop of the ray in ps.ray (started with ps.trk.begin).  Returns the parameter of the
// real collision that ended it, or -FLT_MAX (the ray left the medium; a ratio-tracked shadow ray always does).
template <int MODE, bool COUNT>
SVR_DEV float fly(const DevScene& s, PathState<MODE>& ps, LocalCounters<COUNT>& lc)
{
    const int slot = ps.shadow ? SVR_CNT_SHADOW_TAPS : SVR_CNT_TRACK_TAPS;
    float* ratio = (ps.shadow && s.shadowEstimator) ? &ps.ratioT : nullptr;
    while (true) {
        VisitResult v = ps.trk.template visit<COUNT>(s, ps.ray, ps.rng, lc);
        if (v == VISIT_CONTINUE) continue;
        if (v == VISIT_ESCAPED) break;
        if (ps.trk.template collide<COUNT>(s, ps.ray, ps.rng, lc, slot, ratio)) return ps.trk.t;
        if (ratio && ratio_roulette(ps.ratioT, ps.rng)) break;
    }
    return -FLT_MAX;
}

// One path: the reference's loop nest for one (pixel, sample), added to the pixel's accumulators.
template <int MODE, bool COUNT>
SVR_DEV void trace_sample(const DevScene& s, const PtLaunch& a, PathState<MODE>& ps, uint32_t idx, uint32_t idy, uint32_t offset,
                            uint32_t sample, const PixelInfo& pi, LocalCounters<COUNT>& lc)
{
    lc.add(SVR_CNT_PATHS, 1);
    if (pi.empty && !pi.lights && (!s.envEnabled || s.env.tex == 0)) {
        // every camera ray of this pixel escapes without meeting anything: the sample is the (constant) sky
        if (a.traceDepth != 0 && s.envEnabled) {
            if (MODE == 0) ps.sum += f3(s.env.defaultRadiance) * s.env.intensity;
            else ps.L += f3(s.env.defaultRadiance) * s.env.intensity;
        }
        return;
    }
    ps.camLights = pi.lights;
    Next next = path_begin<MODE>(s, ps, idx, idy, offset, sample, pi.tSkip) ? NEXT_TRACK : NEXT_FLIGHT_MISSED;
    if (a.traceDepth == 0) next = NEXT_PATH_DONE;  // the bounce loop never runs (pathtracer.cu:216): the sample is black
    while (next != NEXT_PATH_DONE) {
        float t = -FLT_MAX;
        if (next == NEXT_TRACK) t = fly<MODE, COUNT>(s, ps, lc);
        if (next == NEXT_BOUNCE || ps.shadow)
            next = event_bounce<MODE, COUNT>(s, ps, occluded_at(ps.trk, t), a.traceDepth, lc);
        else
            next = event_flight_end<MODE, COUNT>(s, ps, t, a.traceDepth, lc);
    }
    path_end<MODE>(ps);
}

template <int MODE, bool COUNT>
__global__ void __launch_bounds__(SVR_PT_MAX_THREADS, SVR_PT_MEGA_BLOCKS) pathtrace_mega_kernel(const __grid_constant__ DevScene s, const PtLaunch a, Counters* cnt)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t idx = blockIdx.x * 16u + (warp & 1u) * 8u + (lane & 7u);
    const uint32_t idy = a.y0 + (blockIdx.y * a.bandStride + a.bandPhase) * (blockDim.x >> 4) + (warp >> 1) * 4u + (lane >> 3);
    const bool inside = idx < s.cam.imageW && idy < a.y1;
    LocalCounters<COUNT> lc;
    if (inside) {
        const uint32_t offset = idy * s.cam.imageW + idx;
        PixelInfo pi;
        pi = load_pixel_info(a.pixelInfo, offset);
        PathState<MODE> ps;
        pixel_begin<MODE>(ps);
        for (uint32_t n = 0; n < a.nSamples; ++n) trace_sample<MODE, COUNT>(s, a, ps, idx, idy, offset, a.firstSample + n, pi, lc);
        write_pixel(s, a, offset, pixel_sum<MODE>(ps));
    }
    lc.flush(cnt);
}

// ---------------------------------------------------------------------------------------------
// kernel shape 2: sample-parallel warp.  The 32 lanes of a warp take 32 different SAMPLES of the
// same pixel (sample = lane, lane + 32, ...), one pixel after the other over a short run of pixels.
// All lanes shoot (nearly) the same camera ray: they walk the same macrocells in lockstep and their
// fetches fall into the same texels, every lane has the same expected work, and the unit of
// scheduling is a few pixels instead of a 16 x 8 tile x all samples, so expensive image regions
// spread over all SMs.  The pixel's sum is a fixed-order butterfly over the lanes: deterministic.
// ---------------------------------------------------------------------------------------------
// SPLIT (SVR_OPT_PT_BLOCK_SPLIT): the warps of a block share ONE row of pixels and split every pixel's samples between them
// (warp w takes the rounds w, w + nWarps, ...; their sums meet in shared memory in a fixed order) instead of taking a row
// each.  A pixel then occupies a warp for a quarter of the time, which shortens the end of a launch -- the last blocks of a
// frame run with the machine half empty -- and matters when a frame is short (one frame divided over 8 GPUs).
// AHEAD (SVR_OPT_PT_LOOKAHEAD): at most 32 samples, one per lane, and instead of a pixel's sum every sample's radiance is stored
// for render_pathtracer's later calls.
template <int MODE, bool COUNT, bool SPLIT, bool AHEAD = false>
__global__ void __launch_bounds__(SVR_PT_MAX_THREADS, SVR_PT_MIN_BLOCKS) pathtrace_warp_kernel(const __grid_constant__ DevScene s, const PtLaunch a, Counters* cnt)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nWarps = blockDim.x >> 5;
    const uint32_t idy = a.y0 + (blockIdx.y * a.bandStride + a.bandPhase) * (SPLIT ? 1u : nWarps) + (SPLIT ? 0u : warp);
    __shared__ float part[SPLIT ? SVR_PT_MAX_THREADS / 32 : 1][3];
    LocalCounters<COUNT> lc;
    if (idy < a.y1) {
        PathState<MODE> ps;
        for (uint32_t i = 0; i < (uint32_t)a.warpPixels; ++i) {
            const uint32_t idx = blockIdx.x * (uint32_t)a.warpPixels + i;
            if (idx >= s.cam.imageW) break;
            const uint32_t offset = idy * s.cam.imageW + idx;
            const PixelInfo pi = load_pixel_info(a.pixelInfo, offset);  // classify_pixels_kernel, once per scene
            pixel_begin<MODE>(ps);
            if (pi.empty && !pi.lights && (!s.envEnabled || s.env.tex == 0)) {
                // every sample of this pixel is the constant sky (see trace_sample): nSamples times the same value, written by one lane
                const float3 sky = (a.traceDepth != 0 && s.envEnabled) ? f3(s.env.defaultRadiance) * s.env.intensity : f3(0.f);
                if (AHEAD) {
                    if (lane == 0) a.constantPixel[offset] = 1;
                    continue;
                }
                if (lane == 0 && (!SPLIT || warp == 0)) {
                    lc.add(SVR_CNT_PATHS, a.nSamples);
                    write_pixel(s, a, offset, sky * (float)a.nSamples);
                }
                continue;
            }
            for (uint32_t n = lane + (SPLIT ? 32u * warp : 0u); n < a.nSamples; n += (SPLIT ? 32u * nWarps : 32u))
                trace_sample<MODE, COUNT>(s, a, ps, idx, idy, offset, a.firstSample + n, pi, lc);
            float3 sum = pixel_sum<MODE>(ps);
            __syncwarp();
            if (AHEAD) {
                // lane j traced exactly sample j: `sum` is that sample's radiance.  The pixel's record is 3 * nSamples consecutive
                // floats (x, y, z of sample 0, of sample 1, ...): transposed through shuffles so that every store is one coalesced
                // row of the record (one 4-byte store per lane into 32 slices 25 MB apart took 4 ms per 32-sample batch).
                float* rec = a.perSample + (size_t)offset * (3u * a.nSamples);
#pragma unroll
                for (uint32_t r = 0; r < 3u; ++r) {
                    const uint32_t i = r * 32u + lane, src = i / 3u, c = i - 3u * src;
                    const float vx = __shfl_sync(0xffffffffu, sum.x, (int)src), vy = __shfl_sync(0xffffffffu, sum.y, (int)src),
                                vz = __shfl_sync(0xffffffffu, sum.z, (int)src);
                    if (i < 3u * a.nSamples) rec[i] = c == 0u ? vx : (c == 1u ? vy : vz);
                }
                if (lane == 0) a.constantPixel[offset] = 0;
                continue;
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                sum.x += __shfl_xor_sync(0xffffffffu, sum.x, o);
                sum.y += __shfl_xor_sync(0xffffffffu, sum.y, o);
                sum.z += __shfl_xor_sync(0xffffffffu, sum.z, o);
            }
            if (SPLIT) {
                if (lane == 0) {
                    part[warp][0] = sum.x;
                    part[warp][1] = sum.y;
                    part[warp][2] = sum.z;
                }
                __syncthreads();
                if (warp == 0) {
                    sum = f3(part[0][0], part[0][1], part[0][2]);
                    for (uint32_t w = 1; w < nWarps; ++w) sum += f3(part[w][0], part[w][1], part[w][2]);  // fixed order: deterministic
                    write_pixel_warp(s, a, offset, sum, lane);
                }
                __syncthreads();  // `part` is free for the next pixel
            } else {
                write_pixel_warp(s, a, offset, sum, lane);
            }
        }
    }
    lc.flush(cnt);
}

// Adaptive sampling (svr_pathtracer_accumulate_adaptive): shape 2 over a list of pixels.  Warp w of the grid renders the pixel
// list[w] exactly as pathtrace_warp_kernel does -- same samples per lane, same butterfly, so `sum` receives the same bits -- and
// also adds the sum of the samples with an odd offset from firstSample to `half` (rgb, w = nSamples / 2).  Lane j traces the
// offsets j, j + 32, ...: odd lanes hold odd offsets, and before the butterfly's last step (xor 1) every even lane holds the
// even lanes' sum and receives the odd lanes' sum from its neighbour.  nSamples is a multiple of 32; no counters.
template <int MODE>
__global__ void __launch_bounds__(SVR_PT_MAX_THREADS, SVR_PT_MIN_BLOCKS) pathtrace_list_kernel(const __grid_constant__ DevScene s, const PtLaunch a,
                                                                                           const uint32_t* __restrict__ list, uint32_t count, float4* half)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t item = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (item >= count) return;  // whole warps
    const uint32_t offset = list[item];
    const uint32_t idy = offset / s.cam.imageW, idx = offset - idy * s.cam.imageW;
    const PixelInfo pi = load_pixel_info(a.pixelInfo, offset);
    LocalCounters<false> lc;
    if (pi.empty && !pi.lights && (!s.envEnabled || s.env.tex == 0)) {
        // the constant sky, as pathtrace_warp_kernel writes it; half of it is the odd samples' share (exactly half the sum)
        if (lane == 0) {
            const float3 sky = (a.traceDepth != 0 && s.envEnabled) ? f3(s.env.defaultRadiance) * s.env.intensity : f3(0.f);
            write_pixel(s, a, offset, sky * (float)a.nSamples);
            const float3 o = sky * (float)(a.nSamples / 2u);
            const float4 prev = half[offset];
            half[offset] = make_float4(prev.x + o.x, prev.y + o.y, prev.z + o.z, prev.w + (float)(a.nSamples / 2u));
        }
        return;
    }
    PathState<MODE> ps;
    pixel_begin<MODE>(ps);
    for (uint32_t n = lane; n < a.nSamples; n += 32u) trace_sample<MODE, false>(s, a, ps, idx, idy, offset, a.firstSample + n, pi, lc);
    float3 sum = pixel_sum<MODE>(ps);
    __syncwarp();
#pragma unroll
    for (int o = 16; o > 1; o >>= 1) {
        sum.x += __shfl_xor_sync(0xffffffffu, sum.x, o);
        sum.y += __shfl_xor_sync(0xffffffffu, sum.y, o);
        sum.z += __shfl_xor_sync(0xffffffffu, sum.z, o);
    }
    const float3 other = f3(__shfl_xor_sync(0xffffffffu, sum.x, 1), __shfl_xor_sync(0xffffffffu, sum.y, 1), __shfl_xor_sync(0xffffffffu, sum.z, 1));
    sum.x += other.x;
    sum.y += other.y;
    sum.z += other.z;
    write_pixel_warp(s, a, offset, sum, lane);
    if (lane == 0) {  // an even lane: `other` is the odd lanes' sum
        const float4 prev = half[offset];
        half[offset] = make_float4(prev.x + other.x, prev.y + other.y, prev.z + other.z, prev.w + (float)(a.nSamples / 2u));
    }
}

// ---------------------------------------------------------------------------------------------
// kernel shape 3: sample-parallel warp with a scatter queue (deep paths).  In a high-albedo medium most
// samples of a pixel leave after no or one scatter event and a few bounce traceDepth times; with the loop
// nest of shape 2 the warp waits for its longest path (ncu on C4: 6 of 32 lanes active).  Here a warp
// alternates between two kinds of rounds:
//   A  32 camera rays of the pixel (coherent: same origin, neighbouring directions).  A sample whose camera
//      ray leaves the medium is finished on the spot; one that collides is pushed on the warp's queue in
//      shared memory as (ray, collision parameter, throughput, bounce count, random-stream position);
//   B  when 32 queued collisions are waiting (or no camera ray is left): 32 lanes pop one each and run ONE
//      scatter event -- shade, sample the light, fly the shadow ray, add the direct light, sample the BSDF,
//      fly the bounce ray -- and push the collision that flight ends in, if any.
// Both kinds run the same loop (trace_sample's), entered at different points and left at the first collision
// that is not the lane's own, so every device function is instantiated once.
// Every round starts with all lanes busy, whatever the depth of the paths they serve.  A path is still a
// pure function of (seed, pixel, sample): the counter of its Philox stream travels with the queue entry.
// The image equals shape 2 up to float summation order (the lanes add into per-lane partial sums).
// ---------------------------------------------------------------------------------------------
constexpr int SVR_QUEUE_CAP = 64;    // entries per warp: a round pushes at most 32 onto fewer than 32
constexpr int SVR_QUEUE_WORDS = 14;  // orig 3, dir 3, t, T 3, k | have << 31, c0, c1, r1

template <bool COUNT>
SVR_DEV void queue_push(float* q, int idx, const PathState<2>& ps, float t)
{
    q[0 * SVR_QUEUE_CAP + idx] = ps.ray.orig.x;
    q[1 * SVR_QUEUE_CAP + idx] = ps.ray.orig.y;
    q[2 * SVR_QUEUE_CAP + idx] = ps.ray.orig.z;
    q[3 * SVR_QUEUE_CAP + idx] = ps.ray.dir.x;
    q[4 * SVR_QUEUE_CAP + idx] = ps.ray.dir.y;
    q[5 * SVR_QUEUE_CAP + idx] = ps.ray.dir.z;
    q[6 * SVR_QUEUE_CAP + idx] = t;
    q[7 * SVR_QUEUE_CAP + idx] = ps.T.x;
    q[8 * SVR_QUEUE_CAP + idx] = ps.T.y;
    q[9 * SVR_QUEUE_CAP + idx] = ps.T.z;
    q[10 * SVR_QUEUE_CAP + idx] = __uint_as_float(ps.k | (ps.rng.have << 31));  // k <= traceDepth < 2^31
    q[11 * SVR_QUEUE_CAP + idx] = __uint_as_float(ps.rng.c0);
    q[12 * SVR_QUEUE_CAP + idx] = __uint_as_float(ps.rng.c1);
    q[13 * SVR_QUEUE_CAP + idx] = __uint_as_float(ps.rng.r1);
}

SVR_DEV float queue_pop(const float* q, int idx, PathState<2>& ps)
{
    ps.ray.orig = f3(q[0 * SVR_QUEUE_CAP + idx], q[1 * SVR_QUEUE_CAP + idx], q[2 * SVR_QUEUE_CAP + idx]);
    ps.ray.dir = f3(q[3 * SVR_QUEUE_CAP + idx], q[4 * SVR_QUEUE_CAP + idx], q[5 * SVR_QUEUE_CAP + idx]);
    ps.T = f3(q[7 * SVR_QUEUE_CAP + idx], q[8 * SVR_QUEUE_CAP + idx], q[9 * SVR_QUEUE_CAP + idx]);
    const uint32_t kh = __float_as_uint(q[10 * SVR_QUEUE_CAP + idx]);
    ps.k = kh & 0x7fffffffu;
    ps.rng.have = kh >> 31;
    ps.rng.c0 = __float_as_uint(q[11 * SVR_QUEUE_CAP + idx]);
    ps.rng.c1 = __float_as_uint(q[12 * SVR_QUEUE_CAP + idx]);
    ps.rng.r1 = __float_as_uint(q[13 * SVR_QUEUE_CAP + idx]);
    ps.shadow = false;
    return q[6 * SVR_QUEUE_CAP + idx];
}

// ---- work items, the scatter event as a function and paired flights (shared by shapes 3 and 5) -------------------------------
// Capacities: every ray in the pool can become one event, so nEv + nPool <= SVR_EVQ_CAP is kept at all times (a flight
// phase can then always empty the pool); an event phase turns up to 32 events into up to 64 rays, a camera batch adds 32.
// The more rays a flight phase starts with, the better its lanes stay packed (rays per lane), at the price of shared memory.
// Measured on C4 (128 spp per launch, round 2): 64 / 64 at 6 blocks per SM 153.6 ms, 96 / 128 at 4 blocks 185 ms, 128 / 160 at
// 3 blocks 211 ms, 192 / 224 at 2 blocks 259 ms -- the kernel is bound by memory latency, and resident warps buy more than
// packed lanes (shape 3 at 8 blocks per SM: 120.8 ms).
#ifndef SVR_POOL_CAP
#define SVR_POOL_CAP 64
#endif
#ifndef SVR_EVQ_CAP
#define SVR_EVQ_CAP 64
#endif
constexpr int SVR_ITEM_WORDS = 13;   // orig 3, dir 3, a 3 (throughput / contribution), x (optical depth left | collision parameter), meta, c0, c1
constexpr int SVR_POOL_SLOTS = 16;   // pixels of a warp's run
#ifndef SVR_POOL_CHUNK
#define SVR_POOL_CHUNK 24
#endif
#ifndef SVR_PT_POOL_BLOCKS
#define SVR_PT_POOL_BLOCKS 6
#endif
enum RayKind { RAY_CAMERA = 0, RAY_BOUNCE = 1, RAY_SHADOW = 2 };

struct WorkItem {
    float3 o, d, a;
    float x;
    uint32_t meta, c0, c1;  // meta: bounce count (20 bits) | pixel slot << 20 | kind << 26
    SVR_DEV uint32_t k() const { return meta & 0xfffffu; }
    SVR_DEV uint32_t slot() const { return (meta >> 20) & 63u; }
    SVR_DEV uint32_t kind() const { return meta >> 26; }
    static SVR_DEV uint32_t pack(uint32_t k, uint32_t slot, uint32_t kind) { return k | (slot << 20) | (kind << 26); }
};

template <int CAP>
SVR_DEV void item_store(float* q, int idx, const WorkItem& it)
{
    q[0 * CAP + idx] = it.o.x;
    q[1 * CAP + idx] = it.o.y;
    q[2 * CAP + idx] = it.o.z;
    q[3 * CAP + idx] = it.d.x;
    q[4 * CAP + idx] = it.d.y;
    q[5 * CAP + idx] = it.d.z;
    q[6 * CAP + idx] = it.a.x;
    q[7 * CAP + idx] = it.a.y;
    q[8 * CAP + idx] = it.a.z;
    q[9 * CAP + idx] = it.x;
    q[10 * CAP + idx] = __uint_as_float(it.meta);
    q[11 * CAP + idx] = __uint_as_float(it.c0);
    q[12 * CAP + idx] = __uint_as_float(it.c1);
}

template <int CAP>
SVR_DEV WorkItem item_load(const float* q, int idx)
{
    WorkItem it;
    it.o = f3(q[0 * CAP + idx], q[1 * CAP + idx], q[2 * CAP + idx]);
    it.d = f3(q[3 * CAP + idx], q[4 * CAP + idx], q[5 * CAP + idx]);
    it.a = f3(q[6 * CAP + idx], q[7 * CAP + idx], q[8 * CAP + idx]);
    it.x = q[9 * CAP + idx];
    it.meta = __float_as_uint(q[10 * CAP + idx]);
    it.c0 = __float_as_uint(q[11 * CAP + idx]);
    it.c1 = __float_as_uint(q[12 * CAP + idx]);
    return it;
}

// radiance into the pixel's fixed-point sum (2^-32; contributions are non-negative)
SVR_DEV void accum_add(unsigned long long* acc, uint32_t slot, float3 v)
{
    const float sc = 4294967296.f, top = 4.0e9f;
    if (v.x > 0.f) atomicAdd(acc + slot * 3 + 0, (unsigned long long)(fminf(v.x, top) * sc));
    if (v.y > 0.f) atomicAdd(acc + slot * 3 + 1, (unsigned long long)(fminf(v.y, top) * sc));
    if (v.z > 0.f) atomicAdd(acc + slot * 3 + 2, (unsigned long long)(fminf(v.z, top) * sc));
}


// One scatter event as a function of the collision alone (pathtracer.cu:214-276): the camera ray's light hit, shading, the
// light sample -- which becomes a SHADOW ray that carries its whole contribution T * nLights * bsdf * Li / pdf and a random
// stream of its own, and owes the path nothing afterwards -- and the BSDF sample with Russian roulette, which becomes the
// BOUNCE ray.  `direct`: radiance to add at once (a camera ray that meets a light before its collision ends there).
template <bool COUNT>
SVR_DEV void scatter_event(const DevScene& s, uint32_t traceDepth, bool camLights, const WorkItem& ev, WorkItem& sh, bool& haveShadow, WorkItem& bo,
                           bool& haveBounce, float3& direct, LocalCounters<COUNT>& lc)
{
    const uint32_t k = ev.k(), slot = ev.slot();
    const float t = ev.x;
    haveShadow = haveBounce = false;
    if (k == 0 && camLights) {
        // the camera ray may hit a light before its collision (pathtracer.cu:214-229)
        Ray cr;
        cr.orig = ev.o;
        cr.dir = ev.d;
        LightHit ls;
        if (nearest_light(s, cr, &ls) && ls.t < t) {
            const float cosTerm = dot(ls.normal, -ev.d);
            direct = ev.a * ls.radiance * (cosTerm <= 0.f ? 0.f : 1.f);
            return;
        }
    }
    Philox rng;
    rng.c0 = ev.c0;
    rng.c1 = ev.c1;
    rng.r1 = 0;
    rng.have = 0;
    VolumeSample vs;
    vs.wo = -ev.d;
    vs.ptInWorld = ev.o + t * ev.d;
    const float intensity = intensity_at(s.vol, vs.ptInWorld);
    vs.color_opacity = tf_at(s.tf, intensity);
    vs.gradient = gradient_at(s.vol, vs.ptInWorld);
    const float gradientMagnitude = sqrtf(dot(vs.gradient, vs.gradient));
    lc.add(SVR_CNT_SHADE_TAPS, 7);
    lc.add(SVR_CNT_TF_LOOKUPS, 1);
    lc.add(SVR_CNT_SCATTERS, 1);
    const float gf = s.vol.gradientFactor;
    const float Pbrdf = vs.color_opacity.w * (1.f - expf(-25.f * gf * gf * gf * gradientMagnitude * 65535.f * s.vol.invMaxMagnitude));
    const ShadingType st = (rng.next() < Pbrdf) ? BRDF : ISOTROPIC;
    // estimate_direct_light (pathtracer.cu:171-198)
    if (s.numLights != 0) {
        int lightId = (int)((float)s.numLights * rng.next());
        lightId = lightId < (int)s.numLights ? lightId : (int)s.numLights - 1;
        float3 lightPos, wi;
        float pdf;
        const float3 Li = sample_light<false>(s.lights[lightId], vs.ptInWorld, rng, &lightPos, &wi, &pdf);
        if (pdf > 0.f && max3(Li) > 0.f) {
            sh.o = vs.ptInWorld;
            sh.d = normalize(lightPos - vs.ptInWorld);
            sh.a = ev.a * ((float)s.numLights * bsdf(vs, wi, st) * Li / pdf);
            sh.x = -1.f;
            sh.meta = WorkItem::pack(k, slot, RAY_SHADOW);
            sh.c0 = rng.c0;
            sh.c1 = ev.c1 ^ 0xA511E9B3u;  // a stream of its own: it flies beside the bounce ray
            haveShadow = max3(sh.a) > 0.f;
        }
    }
    // the bounce (pathtracer.cu:257-276); the last bounce's BSDF sample would never be used
    if (k + 1 < traceDepth) {
        float3 wi = f3(0.f);
        float pdf = 0.f;
        const float3 f = sample_bsdf<false>(vs, &wi, &pdf, rng, st);
        const float cosTerm = fabsf(dot(normalize(vs.gradient), wi));
        float3 T = ev.a;
        if (max3(f) > 0.f && pdf > 0.f) {
            if (st == ISOTROPIC) T *= f / (pdf * (1.f - Pbrdf));
            else T *= f * cosTerm / (pdf * Pbrdf);
        }
        bool alive = true;
        if (k >= 3) alive = !russian_roulette<false>(&T, rng);
        if (alive) {
            bo.o = vs.ptInWorld;
            bo.d = wi;
            bo.a = T;
            bo.x = -1.f;
            bo.meta = WorkItem::pack(k + 1, slot, RAY_BOUNCE);
            bo.c0 = rng.c0;
            bo.c1 = ev.c1;
            haveBounce = true;
        }
    }
}

// One more block per SM than the other shapes (64 registers, some spills): this kernel serves incoherent deep
// paths in volumes that miss the caches, where more warps in flight pay (C4: 130 -> 125 ms per 128 spp).
// (Round 2 also tried flying the shadow ray and the bounce ray of a scatter event in ONE loop, their cell loads and taps issued
// side by side -- two outstanding fetches per lane: 216 ms per 128 spp on C4 against 117; both halves of the loop run with
// the lanes of either ray, 51 % more warp instructions, and two walks' state spills: profiles/r02/pt_c4_paired_flights_experiment.summary.txt.)
template <bool COUNT>
__global__ void __launch_bounds__(SVR_PT_MAX_THREADS, SVR_PT_QUEUE_BLOCKS) pathtrace_queue_kernel(const __grid_constant__ DevScene s, const PtLaunch a, Counters* cnt)
{
    constexpr int MODE = 2;
    __shared__ float queues[SVR_PT_MAX_THREADS / 32][SVR_QUEUE_WORDS * SVR_QUEUE_CAP];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t idy = a.y0 + (blockIdx.y * a.bandStride + a.bandPhase) * (blockDim.x >> 5) + warp;
    float* q = queues[warp];
    LocalCounters<COUNT> lc;
    if (idy < a.y1) {
        PathState<MODE> ps;
        for (uint32_t i = 0; i < (uint32_t)a.warpPixels; ++i) {
            const uint32_t idx = blockIdx.x * (uint32_t)a.warpPixels + i;
            if (idx >= s.cam.imageW) break;
            const uint32_t offset = idy * s.cam.imageW + idx;
            const PixelInfo pi = load_pixel_info(a.pixelInfo, offset);
            pixel_begin<MODE>(ps);
            ps.camLights = pi.lights;
            if (pi.empty && !pi.lights && (!s.envEnabled || s.env.tex == 0)) {
                // every sample of this pixel is the constant sky (see trace_sample): the same additions, nothing else
                const float3 sky = (a.traceDepth != 0 && s.envEnabled) ? f3(s.env.defaultRadiance) * s.env.intensity : f3(0.f);
                for (uint32_t n = lane; n < a.nSamples; n += 32u) {
                    lc.add(SVR_CNT_PATHS, 1);
                    ps.L += sky;
                }
            } else if (a.traceDepth == 0) {
                for (uint32_t n = lane; n < a.nSamples; n += 32u) lc.add(SVR_CNT_PATHS, 1);  // black (pathtracer.cu:216)
            } else {
                uint32_t nextN = 0;  // camera rays issued so far (warp-uniform)
                int queued = 0;      // entries on the queue (warp-uniform)
                while (nextN < a.nSamples || queued > 0) {
                    // what this lane does in the round: a popped collision (round B) or a fresh camera ray (round A)
                    bool active, own = false;  // own: the flight-end event at hand is the popped entry's own collision
                    Next next = NEXT_PATH_DONE;
                    float t = -FLT_MAX;
                    if (queued >= 32 || nextN >= a.nSamples) {
                        const int take = queued < 32 ? queued : 32;
                        queued -= take;
                        active = (int)lane < take;
                        if (active) {
                            t = queue_pop(q, queued + (int)lane, ps);
                            next = NEXT_EVENT_AT_T;
                            own = true;
                        }
                    } else {
                        const uint32_t n = nextN + lane;
                        nextN += 32u;
                        active = n < a.nSamples;
                        if (active) {
                            lc.add(SVR_CNT_PATHS, 1);
                            next = path_begin<MODE>(s, ps, idx, idy, offset, a.firstSample + n, pi.tSkip) ? NEXT_TRACK : NEXT_FLIGHT_MISSED;
                        }
                    }
                    __syncwarp();  // every pop of the round precedes every push
                    // trace_sample's loop, left at the first collision that is not the lane's own: that one is queued
                    bool push = false;
                    while (active) {
                        if (next == NEXT_TRACK) t = fly<MODE, COUNT>(s, ps, lc);
                        else if (next != NEXT_EVENT_AT_T) t = -FLT_MAX;
                        if (next == NEXT_BOUNCE || ps.shadow) {
                            next = event_bounce<MODE, COUNT>(s, ps, occluded_at(ps.trk, t), a.traceDepth, lc);
                        } else {
                            if (t >= 0.f && !own) {
                                push = true;
                                break;
                            }
                            own = false;
                            next = event_flight_end<MODE, COUNT>(s, ps, t, a.traceDepth, lc);
                        }
                        if (next == NEXT_PATH_DONE) break;
                    }
                    const unsigned m = __ballot_sync(0xffffffffu, push);
                    if (push) queue_push<COUNT>(q, queued + __popc(m & ((1u << lane) - 1u)), ps, t);
                    queued += __popc(m);
                    __syncwarp();  // this round's pushes precede the next round's pops (other lanes read them)
                }
            }
            float3 sum = ps.L;
            __syncwarp();
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                sum.x += __shfl_xor_sync(0xffffffffu, sum.x, o);
                sum.y += __shfl_xor_sync(0xffffffffu, sum.y, o);
                sum.z += __shfl_xor_sync(0xffffffffu, sum.z, o);
            }
            write_pixel_warp(s, a, offset, sum, lane);
        }
    }
    lc.flush(cnt);
}

// ---------------------------------------------------------------------------------------------
// kernel shape 4: sample-parallel warp, camera rays tracked against a per-pixel MAJORANT PROFILE, scatter queue.
//
// In shapes 2 and 3 every lane walks the macrocells of its own camera ray although the 32 lanes of a warp shoot
// (nearly) the same ray: on C3 that is 14.7 dependent cell visits per scattered sample, repeated by every lane, and the
// tentative collisions on the way execute with a third of the lanes (ncu, profiles/r01).  Here the walk is done ONCE per
// pixel, by the warp together, and no lane ever walks a camera ray:
//   1. profile.  The pixel's centre ray is cut into slabs by the macrocell planes of its fastest axis; lane k looks up
//      the cells slab k crosses and keeps their largest majorant M_k (32 slabs per round, one per lane).  A jittered
//      ray of the pixel has the same origin and, at equal ray parameter t, lies within dev = t * alpha of the centre ray
//      (alpha: half the pixel's angular diagonal).  Every macrocell majorant already bounds the medium up to half a
//      voxel outside its cell (svr_macrocell.cu stage 1); whatever dev exceeds that is covered by widening the looked-up
//      cell box sideways by r = dev - 0.45 voxel and by giving each slab plane a transition interval of +-r in which the
//      larger of the two neighbouring slab majorants applies.  So M(t), piecewise constant in t, is a valid majorant
//      for EVERY camera ray of the pixel.  A shuffle scan turns it into cumulative optical depth C(t), kept in shared
//      memory (2 intervals per slab, at most 128 slabs; longer rays use slabs several cells thick).
//   2. camera rounds.  A lane holds one sample: it adds an exponential draw to its optical-depth target, inverts C
//      (galloping search from where it stands; t follows in closed form), fetches the medium at its OWN ray's point and
//      accepts with probability sigma / M(t) -- delta tracking against M(t).  One iteration is one tentative collision
//      for every lane: the same instructions for all, whatever each ray has met so far.  A lane whose sample collides
//      pushes it on the scatter queue (shape 3's), a lane whose sample leaves the medium adds light / sky; both take the
//      pixel's next sample and go on, so lanes do not wait for each other's samples.
//   3. scatter rounds: shape 3's round B, unchanged (shade, light sample, shadow flight, BSDF, bounce flight).
// Any valid majorant gives the same free-path distribution, so the estimator is the reference's; the random walk of a
// sample is still a pure function of (seed, pixel, sample), but it is not the walk shapes 1-3 make (other tentative
// collisions): images agree statistically, not bit for bit.  Needs a pinhole camera (one origin per pixel).
// ---------------------------------------------------------------------------------------------
constexpr int SVR_PROF_SLABS = 128;

struct PixelProfile {  // warp-uniform
    float t0, dT, rho;  // parameter of the first slab plane, parameter length of a slab, half-width of a transition interval
    float tA;           // where the profile begins (intervals are cut off there)
    float total;        // optical depth of the whole profile
    int n;              // slabs
    int iStart;         // first interval that can hold a collision
};

SVR_DEV float axis_of(float3 v, int a) { return a == 0 ? v.x : (a == 1 ? v.y : v.z); }

// Builds the profile of the pixel whose centre ray is `ray` (all lanes call it with the same arguments).
// C[0 .. 2n]: cumulative optical depth at the start of interval i; interval 2k = transition around plane k
// ([t_k - rho, t_k + rho], majorant max(M[k-1], M[k])), interval 2k+1 = slab k proper ([t_k + rho, t_k+1 - rho], M[k]).
template <bool COUNT>
SVR_DEV void build_profile(const DevScene& s, const Ray& ray, float alpha, float* C, float* M, PixelProfile& pp, uint32_t lane,
                           LocalCounters<COUNT>& lc)
{
    pp.total = 0.f;
    pp.n = 0;
    pp.iStart = 0;
    pp.t0 = pp.dT = pp.rho = pp.tA = 0.f;
    const DevGrid& g = s.grid;
    const float3 g0 = ray.orig * g.toCell - g.cellOff, dg = ray.dir * g.toCell;
    const int* occ = g.occ;
    const float3 lo = f3((float)__ldg(occ + 0), (float)__ldg(occ + 1), (float)__ldg(occ + 2));
    const float3 hi = f3((float)(__ldg(occ + 3) + 1), (float)(__ldg(occ + 4) + 1), (float)(__ldg(occ + 5) + 1));
    if (!(lo.x < hi.x)) return;  // no occupied cell at all
    // sideways spread of the pixel's rays at the far end of the occupied box, in cells per axis, beyond the 0.45 voxel
    // every majorant already covers
    const float3 cellWorld = f3((float)g.cell) * f3(s.vol.spacing);
    const float3 bc = f3(s.vol.bbox.vmin) + 0.5f * (lo + hi) * cellWorld - ray.orig;
    const float3 bh = 0.5f * (hi - lo) * cellWorld;
    const float devWorld = (sqrtf(dot(bc, bc)) + sqrtf(dot(bh, bh))) * alpha;
    const float slack = 0.45f / (float)g.cell;
    const float3 r = f3(fmaxf(devWorld * fabsf(g.toCell.x) - slack, 0.f), fmaxf(devWorld * fabsf(g.toCell.y) - slack, 0.f),
                        fmaxf(devWorld * fabsf(g.toCell.z) - slack, 0.f));
    // parameter interval in which some ray of the pixel can be inside the occupied box
    float tA, tB;
    {
        const float3 inv = f3(dg.x != 0.f ? 1.f / dg.x : FLT_MAX, dg.y != 0.f ? 1.f / dg.y : FLT_MAX, dg.z != 0.f ? 1.f / dg.z : FLT_MAX);
        const float3 a0 = (lo - r - f3(1.f) - g0) * inv, a1 = (hi + r + f3(1.f) - g0) * inv;
        tA = fmaxf(fmaxf(fminf(a0.x, a1.x), fminf(a0.y, a1.y)), fminf(a0.z, a1.z));
        tB = fminf(fminf(fmaxf(a0.x, a1.x), fmaxf(a0.y, a1.y)), fmaxf(a0.z, a1.z));
    }
    tA = fmaxf(tA, 0.f);
    if (!(tA < tB)) return;
    if (!(fabsf(ray.dir.x) + fabsf(ray.dir.y) + fabsf(ray.dir.z) < 4.f)) return;  // NaN direction: nothing to index the grid with
    // slabs along the fastest axis, in the forward coordinate u = sign * g_axis (increasing with t)
    const float ax = fabsf(dg.x), ay = fabsf(dg.y), az = fabsf(dg.z);
    const int axis = (ax >= ay && ax >= az) ? 0 : (ay >= az ? 1 : 2);
    const float dga = axis_of(dg, axis), g0a = axis_of(g0, axis), ra = axis_of(r, axis);
    const float sgn = dga > 0.f ? 1.f : -1.f, invA = 1.f / fabsf(dga);
    const float uA = sgn * fmaf(tA, dga, g0a), uB = sgn * fmaf(tB, dga, g0a);
    const float u0 = floorf(uA);
    const float span = fmaxf(uB - u0, 0.f);
    // cells per slab: at most SVR_PROF_SLABS slabs, and a slab at least as thick as two transition half-widths
    const float S = fmaxf(floorf(span / (float)(SVR_PROF_SLABS - 1)) + 1.f, ceilf(2.f * ra));
    const int n = (int)floorf(span / S) + 2;  // the last slab lies wholly beyond tB
    const float t0 = (u0 - sgn * g0a) * invA;
    const float dT = S * invA, rho = ra * invA;
    float carryC = 0.f, carryM = 0.f;
    int firstK = n;
    for (int base = 0; base < n; base += 32) {
        const int k = base + (int)lane;
        float Mk = 0.f;
        if (k < n) {
            for (float c = 0.f; c < S; c += 1.f) {
                const float layer = u0 + (float)k * S + c;  // forward index of this layer of cells
                // the centre ray's stretch through this layer, plus the transition zones on both sides (a ray of the pixel can be
                // in this layer while the centre ray is still up to rho before / beyond it)
                const float t1 = (layer - sgn * g0a) * invA - rho, t2 = (layer + 1.f - sgn * g0a) * invA + rho;
                const float3 e = f3(fmaf(t1, dg.x, g0.x), fmaf(t1, dg.y, g0.y), fmaf(t1, dg.z, g0.z));
                const float3 x = f3(fmaf(t2, dg.x, g0.x), fmaf(t2, dg.y, g0.y), fmaf(t2, dg.z, g0.z));
                const float ia = sgn > 0.f ? layer : -layer - 1.f;
                float3 bl = f3(floorf(fminf(e.x, x.x) - r.x), floorf(fminf(e.y, x.y) - r.y), floorf(fminf(e.z, x.z) - r.z));
                float3 bu = f3(floorf(fmaxf(e.x, x.x) + r.x), floorf(fmaxf(e.y, x.y) + r.y), floorf(fmaxf(e.z, x.z) + r.z));
                if (axis == 0) bl.x = bu.x = ia;
                else if (axis == 1) bl.y = bu.y = ia;
                else bl.z = bu.z = ia;
                // cells outside the grid are empty (one-cell empty border at -1 and g): clamping onto the border keeps that
                const int x0 = (int)fminf(fmaxf(bl.x, -1.f), (float)g.gx), x1 = (int)fminf(fmaxf(bu.x, -1.f), (float)g.gx);
                const int y0 = (int)fminf(fmaxf(bl.y, -1.f), (float)g.gy), y1 = (int)fminf(fmaxf(bu.y, -1.f), (float)g.gy);
                const int z0 = (int)fminf(fmaxf(bl.z, -1.f), (float)g.gz), z1 = (int)fminf(fmaxf(bu.z, -1.f), (float)g.gz);
                for (int cz = z0; cz <= z1; ++cz)
                    for (int cy = y0; cy <= y1; ++cy)
                        for (int cx = x0; cx <= x1; ++cx) {
                            Mk = fmaxf(Mk, g.at(cx, cy, cz));
                            lc.add(SVR_CNT_CELLS, 1);
                        }
            }
        }
        float Mprev = __shfl_up_sync(0xffffffffu, Mk, 1);
        if (lane == 0) Mprev = carryM;
        // interval lengths, cut off at tA: nothing collides before the pixel's rays can be inside the occupied box (nor behind
        // the eye: tA >= 0)
        const float tk = fmaf((float)k, dT, t0);
        const float len0 = fmaxf(tk + rho - fmaxf(tk - rho, tA), 0.f), len1 = fmaxf(tk + dT - rho - fmaxf(tk + rho, tA), 0.f);
        const float d0 = k < n ? fmaxf(Mprev, Mk) * len0 : 0.f;
        const float d1 = k < n ? Mk * len1 : 0.f;
        const float pair = d0 + d1;
        float incl = pair;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const float v = __shfl_up_sync(0xffffffffu, incl, o);
            if ((int)lane >= o) incl += v;
        }
        if (k < n) {
            const float c0 = carryC + (incl - pair);
            C[2 * k] = c0;
            C[2 * k + 1] = c0 + d0;
            M[k] = Mk;
        }
        const unsigned some = __ballot_sync(0xffffffffu, pair > 0.f);
        if (some && firstK == n) firstK = base + __ffs(some) - 1;
        carryC += __shfl_sync(0xffffffffu, incl, 31);
        carryM = __shfl_sync(0xffffffffu, Mk, 31);
    }
    if (lane == 0) C[2 * n] = carryC;
    __syncwarp();
    pp.t0 = t0;
    pp.dT = dT;
    pp.rho = rho;
    pp.tA = tA;
    pp.n = n;
    pp.total = carryC;
    pp.iStart = firstK < n ? 2 * firstK : 0;
}

SVR_DEV void queue_push_raw(float* q, int idx, float3 orig, float3 dir, float t, float3 T, uint32_t k, uint32_t c0, uint32_t c1)
{
    q[0 * SVR_QUEUE_CAP + idx] = orig.x;
    q[1 * SVR_QUEUE_CAP + idx] = orig.y;
    q[2 * SVR_QUEUE_CAP + idx] = orig.z;
    q[3 * SVR_QUEUE_CAP + idx] = dir.x;
    q[4 * SVR_QUEUE_CAP + idx] = dir.y;
    q[5 * SVR_QUEUE_CAP + idx] = dir.z;
    q[6 * SVR_QUEUE_CAP + idx] = t;
    q[7 * SVR_QUEUE_CAP + idx] = T.x;
    q[8 * SVR_QUEUE_CAP + idx] = T.y;
    q[9 * SVR_QUEUE_CAP + idx] = T.z;
    q[10 * SVR_QUEUE_CAP + idx] = __uint_as_float(k);  // no buffered random word travels with the entry
    q[11 * SVR_QUEUE_CAP + idx] = __uint_as_float(c0);
    q[12 * SVR_QUEUE_CAP + idx] = __uint_as_float(c1);
    q[13 * SVR_QUEUE_CAP + idx] = 0.f;
}

// Per-warp shared memory of shape 4: the profile, an inverse table over it, the pixel's camera basis.
//   C[0 .. 2n]   cumulative optical depth at the start of interval i            (2 * SLABS + 1 floats)
//   M[0 .. n-1]  slab majorants                                                 (SLABS floats)
//   inv[0..BINS] for optical depth b * total / BINS: the interval that holds it (BINS + 1 uint16)
//   cam[0..8]    D0, du, dv: direction through sub-pixel (jx, jy) = normalize(D0 + jx du + jy dv)
constexpr int SVR_PROF_BINS = 128;
//   stash        the camera samples the lanes hold, parked while a scatter round uses the registers (7 x 32 words)
constexpr int SVR_PROF_C = 0, SVR_PROF_M = 2 * SVR_PROF_SLABS + 4, SVR_PROF_CAM = SVR_PROF_M + SVR_PROF_SLABS,
              SVR_PROF_INV = SVR_PROF_CAM + 16, SVR_PROF_STASH = SVR_PROF_INV + (SVR_PROF_BINS + 2) / 2 + 1,
              SVR_PROF_FLOATS = SVR_PROF_STASH + 7 * 32;

enum LaneStatus { LANE_IDLE = 0, LANE_FLY = 1, LANE_HIT = 2, LANE_ESC = 3 };

template <bool COUNT>
__global__ void __launch_bounds__(SVR_PT_MAX_THREADS, SVR_PT_PROFILE_BLOCKS) pathtrace_profile_kernel(const __grid_constant__ DevScene s, const PtLaunch a, Counters* cnt)
{
    constexpr int MODE = 2;
    constexpr unsigned FULL = 0xffffffffu;
    __shared__ float queues[SVR_PT_MAX_THREADS / 32][SVR_QUEUE_WORDS * SVR_QUEUE_CAP];
    __shared__ float profiles[SVR_PT_MAX_THREADS / 32][SVR_PROF_FLOATS];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t idy = a.y0 + (blockIdx.y * a.bandStride + a.bandPhase) * (blockDim.x >> 5) + warp;
    float* q = queues[warp];
    float* C = profiles[warp] + SVR_PROF_C;
    float* M = profiles[warp] + SVR_PROF_M;
    float* camv = profiles[warp] + SVR_PROF_CAM;
    unsigned short* inv = (unsigned short*)(profiles[warp] + SVR_PROF_INV);
    float* stash = profiles[warp] + SVR_PROF_STASH + lane;
    LocalCounters<COUNT> lc;
    if (idy < a.y1) {
        PathState<MODE> ps;
        const svr_camera& cam = s.cam;
        // half the pixel's angular diagonal (see classify_pixel)
        const float hx = cam.aspectRatio * cam.tanFovxOverTwo / ((float)cam.imageW - 1.f), hy = cam.tanFovxOverTwo / ((float)cam.imageH - 1.f);
        const float alpha = sqrtf(hx * hx + hy * hy) * 1.05f;
        for (uint32_t i = 0; i < (uint32_t)a.warpPixels; ++i) {
            const uint32_t idx = blockIdx.x * (uint32_t)a.warpPixels + i;
            if (idx >= cam.imageW) break;
            const uint32_t offset = idy * cam.imageW + idx;
            const PixelInfo pi = classify_pixel(s, idx, idy, false, false, a.lightCull != 0);  // lights only
            pixel_begin<MODE>(ps);
            ps.camLights = pi.lights;
            PixelProfile pp;
            pp.total = 0.f;
            if (a.traceDepth != 0) {
                __syncwarp();  // the previous pixel's profile is no longer read
                build_profile<COUNT>(s, camera_ray_center(cam, idx, idy), alpha, C, M, pp, lane, lc);
            }
            if (a.traceDepth == 0) {
                for (uint32_t n = lane; n < a.nSamples; n += 32u) lc.add(SVR_CNT_PATHS, 1);  // black (pathtracer.cu:216)
            } else if (!(pp.total > 0.f) && !pi.lights && (!s.envEnabled || s.env.tex == 0)) {
                // no camera ray of the pixel can collide and none can hit a light: every sample is the constant sky
                const float3 sky = s.envEnabled ? f3(s.env.defaultRadiance) * s.env.intensity : f3(0.f);
                for (uint32_t n = lane; n < a.nSamples; n += 32u) {
                    lc.add(SVR_CNT_PATHS, 1);
                    ps.L += sky;
                }
            } else {
                const int nI = 2 * pp.n;
                const float invDTau = pp.total > 0.f ? (float)SVR_PROF_BINS / pp.total : 0.f;
                {
                    // inverse table: inv[b] = largest interval index i with C[i] <= b * total / BINS (then the interval of any
                    // optical depth in bin b lies in inv[b] .. inv[b + 1]); and the camera basis of the pixel
                    for (int bin = (int)lane; bin <= SVR_PROF_BINS; bin += 32) {
                        const float tau = (float)bin * (pp.total * (1.f / (float)SVR_PROF_BINS));
                        int lo = 0, hi = nI > 0 ? nI - 1 : 0;
                        while (lo < hi) {
                            const int mid = (lo + hi + 1) >> 1;
                            if (C[mid] <= tau) lo = mid;
                            else hi = mid - 1;
                        }
                        inv[bin] = (unsigned short)(bin == SVR_PROF_BINS ? (nI > 0 ? nI - 1 : 0) : lo);
                    }
                    if (lane < 9) {
                        // cuda_camera.h:66-83 with a closed aperture: dir = normalize(nx u + ny v - f w), nx = (2 (x + jx) / (W - 1) - 1) aspect tan f
                        const float kx = cam.aspectRatio * cam.tanFovxOverTwo * cam.focalLength, ky = cam.tanFovxOverTwo * cam.focalLength;
                        const float sx = 2.f / ((float)cam.imageW - 1.f), sy = 2.f / ((float)cam.imageH - 1.f);
                        const float nx0 = ((float)idx * sx - 1.f) * kx, ny0 = ((float)idy * sy - 1.f) * ky;
                        const int c3 = (int)lane % 3;
                        const float u = c3 == 0 ? cam.u.x : (c3 == 1 ? cam.u.y : cam.u.z), v = c3 == 0 ? cam.v.x : (c3 == 1 ? cam.v.y : cam.v.z),
                                    w = c3 == 0 ? cam.w.x : (c3 == 1 ? cam.w.y : cam.w.z);
                        camv[lane] = lane < 3 ? nx0 * u + ny0 * v - cam.focalLength * w : (lane < 6 ? sx * kx * u : sy * ky * v);
                    }
                    if (lane == 9) {
                        camv[9] = pp.t0;
                        camv[10] = pp.dT;
                        camv[11] = pp.rho;
                        camv[12] = pp.tA;
                    }
                    __syncwarp();
                }
                const float3 camPos = f3(cam.pos);
                uint32_t nextN = 0;  // camera samples handed out so far (warp-uniform)
                int queued = 0;      // entries on the scatter queue (warp-uniform)
                // the camera sample this lane holds
                int status = LANE_IDLE;
                float3 dir = f3(0.f);
                float target = 0.f;  // LANE_FLY: optical depth of the next tentative collision; LANE_HIT: parameter of the collision
                uint32_t c0 = 0, c1 = 0;
                while (true) {
                    // ---- scatter round (shape 3's round B) whenever 32 collisions wait: one scatter event each
                    const unsigned notFlying = __ballot_sync(FULL, status != LANE_FLY);
                    const unsigned pending = __ballot_sync(FULL, status == LANE_HIT || status == LANE_ESC);
                    const bool camDone = nextN >= a.nSamples && notFlying == FULL && pending == 0u;
                    if (queued >= 32 || (camDone && queued > 0)) {
                        const int take = queued < 32 ? queued : 32;
                        queued -= take;
                        bool active = (int)lane < take, own = false;
                        Next next = NEXT_PATH_DONE;
                        float t = -FLT_MAX;
                        // the camera sample this lane holds is parked in shared memory: the scatter round needs the registers
                        stash[0 * 32] = __int_as_float(status);
                        stash[1 * 32] = dir.x;
                        stash[2 * 32] = dir.y;
                        stash[3 * 32] = dir.z;
                        stash[4 * 32] = target;
                        stash[5 * 32] = __uint_as_float(c0);
                        stash[6 * 32] = __uint_as_float(c1);
                        __syncwarp();  // the pushes of the camera rounds precede the pops
                        if (active) {
                            t = queue_pop(q, queued + (int)lane, ps);
                            next = NEXT_EVENT_AT_T;
                            own = true;
                        }
                        __syncwarp();  // every pop of the round precedes every push
                        bool push = false;
                        while (active) {
                            if (next == NEXT_TRACK) t = fly<MODE, COUNT>(s, ps, lc);
                            else if (next != NEXT_EVENT_AT_T) t = -FLT_MAX;
                            if (next == NEXT_BOUNCE || ps.shadow) {
                                next = event_bounce<MODE, COUNT>(s, ps, occluded_at(ps.trk, t), a.traceDepth, lc);
                            } else {
                                if (t >= 0.f && !own) {
                                    push = true;
                                    break;
                                }
                                own = false;
                                next = event_flight_end<MODE, COUNT>(s, ps, t, a.traceDepth, lc);
                            }
                            if (next == NEXT_PATH_DONE) break;
                        }
                        const unsigned m = __ballot_sync(FULL, push);
                        if (push) queue_push<COUNT>(q, queued + __popc(m & ((1u << lane) - 1u)), ps, t);
                        queued += __popc(m);
                        status = __float_as_int(stash[0 * 32]);
                        dir = f3(stash[1 * 32], stash[2 * 32], stash[3 * 32]);
                        target = stash[4 * 32];
                        c0 = __float_as_uint(stash[5 * 32]);
                        c1 = __float_as_uint(stash[6 * 32]);
                        continue;
                    }
                    if (camDone) break;
                    // ---- finish section: lanes whose sample collided push it, lanes whose sample left the medium add light or
                    // sky, and all of them take the pixel's next samples -- together, once enough lanes have come to rest
                    if (__popc(notFlying) >= a.marchBurst || notFlying == FULL) {
                        const unsigned hit = __ballot_sync(FULL, status == LANE_HIT);
                        if (status == LANE_HIT)
                            queue_push_raw(q, queued + __popc(hit & ((1u << lane) - 1u)), camPos, dir, target, f3(1.f), 0u, c0, c1);
                        queued += __popc(hit);
                        if (status == LANE_ESC) {
                            // the ray left the medium: pathtracer.cu:214-234 with t < 0
                            LightHit ls;
                            Ray rj;
                            rj.orig = camPos;
                            rj.dir = dir;
                            if (ps.camLights && nearest_light(s, rj, &ls)) {
                                const float cosTerm = dot(ls.normal, -dir);
                                ps.L += ls.radiance * (cosTerm <= 0.f ? 0.f : 1.f);
                            } else if (s.envEnabled) {
                                ps.L += env_radiance(s.env, dir);
                            }
                        }
                        if (status != LANE_FLY) status = LANE_IDLE;
                        if (nextN < a.nSamples) {
                            const uint32_t n = nextN + (uint32_t)__popc(notFlying & ((1u << lane) - 1u));
                            if (status == LANE_IDLE && n < a.nSamples) {
                                lc.add(SVR_CNT_PATHS, 1);
                                Philox rng;
                                rng.init(s.seedKey, offset, a.firstSample + n);
                                uint32_t w0, w1;
                                rng.generate(w0, w1);  // block 0: pixel jitter (16 bits each) and the first free flight
                                c0 = rng.c0;
                                c1 = rng.c1;
                                const float jx = (float)(w0 >> 16) * (1.f / 65536.f), jy = (float)(w0 & 0xffffu) * (1.f / 65536.f);
                                dir = normalize(f3(fmaf(jx, camv[3], fmaf(jy, camv[6], camv[0])), fmaf(jx, camv[4], fmaf(jy, camv[7], camv[1])),
                                                   fmaf(jx, camv[5], fmaf(jy, camv[8], camv[2]))));
                                target = -logf(1.f - (float)(w1 >> 8) * 5.9604645e-8f);
                                status = LANE_FLY;
                            }
                            const uint32_t handed = (uint32_t)__popc(notFlying);
                            nextN = nextN + handed < a.nSamples ? nextN + handed : a.nSamples;
                        }
                        if (queued >= 32) continue;  // (at most 63 entries: a scatter round comes before the next push)
                    }
                    // ---- camera round: every lane that holds a sample makes ONE tentative collision
                    if (status == LANE_FLY) {
                        if (!(target < pp.total)) {
                            status = LANE_ESC;
                        } else {
                            // the interval that holds `target`: largest i with C[i] <= target, between the table's bounds
                            const int bin = min((int)(target * invDTau), SVR_PROF_BINS - 1);
                            int lo = inv[bin], hi = inv[bin + 1];
                            while (lo < hi) {
                                const int mid = (lo + hi + 1) >> 1;
                                if (C[mid] <= target) lo = mid;
                                else hi = mid - 1;
                            }
                            const int k = lo >> 1;
                            const bool slab = (lo & 1) != 0;
                            const float Mk = M[k];
                            const float Mi = slab ? Mk : fmaxf(Mk, k > 0 ? M[k - 1] : 0.f);
                            const float tStart = fmaxf(fmaf((float)k, camv[10], camv[9]) + (slab ? camv[11] : -camv[11]), camv[12]);
                            const float t = tStart + (target - C[lo]) / Mi;
                            const float3 pos = camPos + t * dir;
                            float sigma = tf_at(s.tf, intensity_at(s.vol, pos)).w;
                            lc.add(SVR_CNT_TRACK_TAPS, 1);
                            lc.add(SVR_CNT_TF_LOOKUPS, 1);
                            if (COUNT && sigma > Mi) lc.add(SVR_CNT_SKIPPED, 1);  // a profile that is not a majorant (tests assert 0)
                            if (a.clipped) {
                                // collisions count inside this ray's own clipped box only (woodcock_tracking.h:24-26, 43); without clip
                                // planes the box is the volume, outside of which the texture reads 0 (border addressing)
                                Ray rj;
                                rj.orig = camPos;
                                rj.dir = dir;
                                float tNear, tFar;
                                const bool in = intersect_volume(s.vol, rj, &tNear, &tFar);
                                if (!(in && t >= (tNear < 0.f ? 1e-6f : tNear) && t <= tFar)) sigma = 0.f;
                            }
                            Philox rng;
                            rng.c0 = c0;
                            rng.c1 = c1;
                            uint32_t w0, w1;
                            rng.generate(w0, w1);  // the accept draw and the next free flight
                            c0 = rng.c0;
                            if ((float)(w0 >> 8) * 5.9604645e-8f * Mi < sigma) {
                                status = LANE_HIT;
                                target = t;
                            } else {
                                target += -logf(1.f - (float)(w1 >> 8) * 5.9604645e-8f);
                            }
                        }
                    }
                }
            }
            float3 sum = ps.L;
            __syncwarp();
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                sum.x += __shfl_xor_sync(FULL, sum.x, o);
                sum.y += __shfl_xor_sync(FULL, sum.y, o);
                sum.z += __shfl_xor_sync(FULL, sum.z, o);
            }
            write_pixel_warp(s, a, offset, sum, lane);
        }
    }
    lc.flush(cnt);
}

// ---------------------------------------------------------------------------------------------
// kernel shape 5: ray pool + event queue per warp (deep paths in media that scatter many times).
//
// ncu on C4 (1024^3 cloud, traceDepth 32) with shape 3: 6.9 of 32 lanes active per instruction (profiles/r02).  Shape 3
// starts every round with 32 busy lanes, but a round is "one scatter event, then one shadow flight, then one bounce
// flight" per lane, and flights last anything from one cell to hundreds: the warp waits for its longest flight twice per
// round, and at the end of every pixel for the last few paths that are still bouncing.  Here the unit of work is smaller
// and lanes are not tied to paths:
//   * a RAY (camera ray, bounce ray or shadow ray) is an item in a per-warp pool in shared memory; a scatter EVENT (a
//     collision waiting to be shaded) is an item in a per-warp queue;
//   * the flight phase: lanes take rays from the pool and walk them; a lane whose ray has ended takes the next one (lanes
//     re-fill together once a few are idle, so the re-fill code runs with several lanes); a ray that is not done after
//     SVR_POOL_CHUNK cell visits goes back into the pool with its remaining optical depth, so no lane holds the others up
//     for longer than a chunk.  A bounce or camera ray that collides becomes an event; a shadow ray that escapes adds its
//     contribution;
//   * the event phase: 32 events at a time, all lanes: shade, sample the light (-> a shadow ray, which carries its
//     contribution and owes nothing to the path afterwards), sample the BSDF (-> the bounce ray);
//   * the warp renders a RUN of pixels, not one pixel after the other: rays of different pixels share the pool, so the few
//     long paths of one pixel bounce on while the next pixels' camera rays keep the lanes busy.  Radiance is summed per
//     pixel in 64-bit fixed point (2^-32) with shared-memory atomics: integer sums do not depend on the order of the
//     additions, so the image is deterministic and independent of how the lanes happened to be scheduled.
// A path is still a pure function of (seed, pixel, sample); the shadow ray draws from a stream of its own (it flies
// concurrently with the bounce ray), so walks differ from shapes 1-3: parity is statistical.
// ---------------------------------------------------------------------------------------------
template <bool COUNT>
__global__ void __launch_bounds__(SVR_PT_MAX_THREADS, SVR_PT_POOL_BLOCKS) pathtrace_pool_kernel(const __grid_constant__ DevScene s, const PtLaunch a, Counters* cnt)
{
    constexpr unsigned FULL = 0xffffffffu;
    constexpr int NW = SVR_PT_MAX_THREADS / 32;
    extern __shared__ float poolMem[];  // per warp: the ray pool, then the event queue (dynamic: above 48 KB per block)
    __shared__ unsigned long long accums[NW][SVR_POOL_SLOTS * 3];
    __shared__ float tskips[NW][SVR_POOL_SLOTS];
    __shared__ uint32_t pflags[NW][SVR_POOL_SLOTS];  // bit 0: a camera ray of the pixel may hit a light; bit 1: every sample is the constant sky
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t idy = a.y0 + (blockIdx.y * a.bandStride + a.bandPhase) * (blockDim.x >> 5) + warp;
    float* pool = poolMem + warp * (SVR_ITEM_WORDS * (SVR_POOL_CAP + SVR_EVQ_CAP));
    float* evq = pool + SVR_ITEM_WORDS * SVR_POOL_CAP;
    unsigned long long* acc = accums[warp];
    float* tskip = tskips[warp];
    uint32_t* pflag = pflags[warp];
    LocalCounters<COUNT> lc;
    if (idy < a.y1) {
        const svr_camera& cam = s.cam;
        const uint32_t runPixels = min((uint32_t)a.warpPixels, (uint32_t)SVR_POOL_SLOTS);
        const uint32_t x0 = blockIdx.x * runPixels;
        const uint32_t nPix = x0 < cam.imageW ? min(runPixels, cam.imageW - x0) : 0u;
        // ---- the run's pixels: classification (one lane per pixel), sums cleared; all-sky pixels are finished on the spot
        if (lane < SVR_POOL_SLOTS * 3) acc[lane] = 0ull;
        if (lane + 32 < SVR_POOL_SLOTS * 3) acc[lane + 32] = 0ull;
        __syncwarp();
        if (lane < nPix) {
            const PixelInfo pi = classify_pixel(s, x0 + lane, idy, true, a.entryCache != 0, a.lightCull != 0);
            const bool sky = pi.empty && !pi.lights && (!s.envEnabled || s.env.tex == 0);
            tskip[lane] = pi.tSkip;
            pflag[lane] = (pi.lights ? 1u : 0u) | ((sky || a.traceDepth == 0) ? 2u : 0u);
            if (sky && a.traceDepth != 0 && s.envEnabled) {
                const float3 v = f3(s.env.defaultRadiance) * (s.env.intensity * (float)a.nSamples);
                const double sc = 4294967296.0;
                acc[lane * 3 + 0] = (unsigned long long)((double)v.x * sc);
                acc[lane * 3 + 1] = (unsigned long long)((double)v.y * sc);
                acc[lane * 3 + 2] = (unsigned long long)((double)v.z * sc);
            }
            if (COUNT && (sky || a.traceDepth == 0)) lc.add(SVR_CNT_PATHS, a.nSamples);
        }
        __syncwarp();
        uint32_t curSlot = 0, curSample = 0;  // next camera sample to hand out (warp-uniform)
        while (curSlot < nPix && (pflag[curSlot] & 2u)) ++curSlot;
        int nPool = 0, nEv = 0;               // items in the pool / the event queue (warp-uniform)
        const float3 camPos = f3(cam.pos);
        while (true) {
            const bool camLeft = curSlot < nPix;
            // what next: events (if their rays fit), else camera rays (if they fit), else fly what is in the pool
            const bool roomEv = nPool + 64 <= SVR_POOL_CAP && nEv + nPool + 32 <= SVR_EVQ_CAP;
            const bool roomCam = camLeft && nPool + 32 <= SVR_POOL_CAP && nEv + nPool + 32 <= SVR_EVQ_CAP;
            if ((nEv >= 32 && roomEv) || (nEv > 0 && nPool == 0 && !roomCam)) {
                // ================= event phase: up to 32 collisions, one scatter event each (pathtracer.cu:214-276) =================
                const int take = nEv < 32 ? nEv : 32;
                nEv -= take;
                const bool active = (int)lane < take;
                bool haveShadow = false, haveBounce = false;
                WorkItem sh, bo;
                if (active) {
                    const WorkItem ev = item_load<SVR_EVQ_CAP>(evq, nEv + (int)lane);
                    float3 direct = f3(0.f);
                    scatter_event<COUNT>(s, a.traceDepth, (pflag[ev.slot()] & 1u) != 0u, ev, sh, haveShadow, bo, haveBounce, direct, lc);
                    accum_add(acc, ev.slot(), direct);
                }
                __syncwarp();  // every load of the phase precedes every store
                const unsigned mS = __ballot_sync(FULL, haveShadow), mB = __ballot_sync(FULL, haveBounce);
                const unsigned below = (1u << lane) - 1u;
                if (haveShadow) item_store<SVR_POOL_CAP>(pool, nPool + __popc(mS & below), sh);
                nPool += __popc(mS);
                if (haveBounce) item_store<SVR_POOL_CAP>(pool, nPool + __popc(mB & below), bo);
                nPool += __popc(mB);
                __syncwarp();
                continue;
            }
            if (roomCam) {
                // ================= camera rays: the next (up to 32) samples of the current pixel go into the pool =================
                const uint32_t left = a.nSamples - curSample;
                const uint32_t n = left < 32u ? left : 32u;
                if (lane < n) {
                    lc.add(SVR_CNT_PATHS, 1);
                    Philox rng;
                    rng.init(s.seedKey, idy * cam.imageW + x0 + curSlot, a.firstSample + curSample + lane);
                    const Ray cr = camera_ray_jittered<false>(cam, x0 + curSlot, idy, rng);
                    WorkItem it;
                    it.o = cr.orig;
                    it.d = cr.dir;
                    it.a = f3(1.f);
                    it.x = -1.f;
                    it.meta = WorkItem::pack(0, curSlot, RAY_CAMERA);
                    it.c0 = rng.c0;
                    it.c1 = rng.c1;
                    item_store<SVR_POOL_CAP>(pool, nPool + (int)lane, it);
                }
                nPool += (int)n;
                curSample += n;
                if (curSample >= a.nSamples) {
                    curSample = 0;
                    ++curSlot;
                    while (curSlot < nPix && (pflag[curSlot] & 2u)) ++curSlot;
                }
                __syncwarp();
                continue;
            }
            if (nPool == 0) break;  // (no events, no rays, no camera samples left)
            // ================= flight phase: the pool is emptied; collisions of camera / bounce rays become events =================
            {
                bool flying = false;
                TrackLocal trk;
                Philox rng;
                Ray ray;
                float3 av = f3(0.f);
                uint32_t meta = 0;
                int steps = 0;
                float ratioAcc = 1.f;  // ratio tracking: transmittance of the stretch this lane has flown
                ray.orig = ray.dir = f3(0.f);
                rng.c0 = rng.c1 = rng.r1 = rng.have = 0;
                while (true) {
                    // ---- idle lanes take rays, together
                    const unsigned idle = __ballot_sync(FULL, !flying);
                    if (idle == FULL && nPool == 0) break;
                    if (nPool > 0 && (__popc(idle) >= a.marchBurst || idle == FULL)) {
                        const int rank = __popc(idle & ((1u << lane) - 1u));
                        if (!flying && rank < nPool) {
                            const WorkItem it = item_load<SVR_POOL_CAP>(pool, nPool - 1 - rank);
                            ray.orig = it.o;
                            ray.dir = it.d;
                            av = it.a;
                            meta = it.meta;
                            rng.c0 = it.c0;
                            rng.c1 = it.c1;
                            rng.r1 = 0;
                            rng.have = 0;
                            steps = 0;
                            ratioAcc = 1.f;
                            flying = true;
                            const bool ok = trk.begin(s, ray, rng, it.kind() == RAY_CAMERA ? tskip[it.slot()] : 0.f);
                            if (ok && it.x >= 0.f) trk.tau = it.x;  // a ray that went back into the pool keeps its optical depth
                            if (!ok) trk.t = FLT_MAX;               // cannot collide: it escapes at the first look
                        }
                        const int taken = __popc(idle) < nPool ? __popc(idle) : nPool;
                        nPool -= taken;
                    }
                    __syncwarp();  // pops before pushes
                    // ---- one cell visit (and the collision it may end in) for every lane that holds a ray
                    int fin = 0;  // 1: collided (camera / bounce: an event), 2: escaped, 3: back into the pool
                    if (flying) {
                        const uint32_t kind = meta >> 26;
                        VisitResult v = trk.t == FLT_MAX ? VISIT_ESCAPED : trk.template visit<COUNT>(s, ray, rng, lc);
                        if (v == VISIT_COLLIDE) {
                            const bool ratio = kind == RAY_SHADOW && s.shadowEstimator != 0;
                            float Tr = 1.f;
                            const bool real = trk.template collide<COUNT>(s, ray, rng, lc, kind == RAY_SHADOW ? SVR_CNT_SHADOW_TAPS : SVR_CNT_TRACK_TAPS,
                                                                          ratio ? &Tr : nullptr);
                            if (ratio) {
                                // ratio tracking: the contribution is attenuated and the ray flies on; Russian roulette once the
                                // transmittance of this stretch has fallen below 2 % (ratio_roulette)
                                av = av * Tr;
                                ratioAcc *= Tr;
                                if (ratioAcc < 0.02f) {
                                    if (rng.next() * 0.02f >= ratioAcc) {
                                        fin = 1;  // terminated with nothing to add
                                    } else {
                                        av = av * (0.02f / ratioAcc);
                                        ratioAcc = 0.02f;
                                    }
                                }
                            } else if (real) {
                                fin = 1;
                            }
                        } else if (v == VISIT_ESCAPED) {
                            fin = 2;
                        }
                        if (fin == 0 && ++steps >= SVR_POOL_CHUNK && kind != RAY_CAMERA) fin = 3;
                    }
                    // ---- what the finished rays leave behind
                    const unsigned below = (1u << lane) - 1u;
                    const bool toEvent = fin == 1 && (meta >> 26) != RAY_SHADOW;
                    const unsigned mE = __ballot_sync(FULL, toEvent), mR = __ballot_sync(FULL, fin == 3);
                    if (toEvent) {
                        WorkItem ev;
                        ev.o = ray.orig;
                        ev.d = ray.dir;
                        ev.a = av;
                        ev.x = trk.t;
                        ev.meta = WorkItem::pack(meta & 0xfffffu, (meta >> 20) & 63u, RAY_BOUNCE);
                        ev.c0 = rng.c0;
                        ev.c1 = rng.c1;
                        item_store<SVR_EVQ_CAP>(evq, nEv + __popc(mE & below), ev);
                    }
                    nEv += __popc(mE);
                    if (fin == 3) {
                        WorkItem it;
                        it.o = ray.orig + trk.t * ray.dir;
                        it.d = ray.dir;
                        it.a = av;
                        it.x = trk.tau;
                        it.meta = meta;
                        it.c0 = rng.c0;
                        it.c1 = rng.c1;
                        item_store<SVR_POOL_CAP>(pool, nPool + __popc(mR & below), it);
                    }
                    nPool += __popc(mR);
                    if (fin == 2) {
                        const uint32_t kind = meta >> 26, slot = (meta >> 20) & 63u;
                        if (kind == RAY_SHADOW) {
                            accum_add(acc, slot, av);  // unoccluded (binary estimator) / what ratio tracking left of it
                        } else {
                            // a camera / bounce ray left the medium: pathtracer.cu:214-234 with t < 0
                            LightHit ls;
                            if (kind == RAY_CAMERA && (pflag[slot] & 1u) && nearest_light(s, ray, &ls)) {
                                const float cosTerm = dot(ls.normal, -ray.dir);
                                accum_add(acc, slot, av * ls.radiance * (cosTerm <= 0.f ? 0.f : 1.f));
                            } else if (s.envEnabled) {
                                accum_add(acc, slot, av * env_radiance(s.env, ray.dir));
                            }
                        }
                    }
                    if (fin != 0) flying = false;
                }
            }
            __syncwarp();
        }
        // ---- the run's pixels: merge into the caller's accumulator, tone map
        __syncwarp();
        if (lane < nPix) {
            const double inv = 1.0 / 4294967296.0;
            const float3 sum = f3((float)((double)acc[lane * 3 + 0] * inv), (float)((double)acc[lane * 3 + 1] * inv), (float)((double)acc[lane * 3 + 2] * inv));
            write_pixel(s, a, idy * cam.imageW + x0 + lane, sum);
        }
    }
    lc.flush(cnt);
}

// ---------------------------------------------------------------------------------------------
// kernel shape 0: phase-scheduled warp
// ---------------------------------------------------------------------------------------------
enum Phase { PH_GEN = 0, PH_MARCH = 1, PH_COLLIDE = 2, PH_EVENT = 3, PH_BOUNCE = 4, PH_DONE = 5 };

template <int MODE, bool COUNT>
__global__ void __launch_bounds__(SVR_PT_MAX_THREADS, SVR_PT_MIN_BLOCKS) pathtrace_sched_kernel(const __grid_constant__ DevScene s, const PtLaunch a, Counters* cnt)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t idx = blockIdx.x * 16u + (warp & 1u) * 8u + (lane & 7u);
    const uint32_t idy = a.y0 + (blockIdx.y * a.bandStride + a.bandPhase) * (blockDim.x >> 4) + (warp >> 1) * 4u + (lane >> 3);
    const bool inside = idx < s.cam.imageW && idy < a.y1;
    const uint32_t offset = idy * s.cam.imageW + idx;
    LocalCounters<COUNT> lc;

    PathState<MODE> ps;
    pixel_begin<MODE>(ps);
    uint32_t n = 0;
    int phase = inside ? PH_GEN : PH_DONE;
    float tEvent = -FLT_MAX;   // flight result handed to EVENT / BOUNCE
    PixelInfo pi;
    pi.tSkip = 0.f;
    pi.lights = true;
    pi.empty = false;
    if (inside) pi = classify_pixel(s, idx, idy, MODE >= 2, a.entryCache != 0, a.lightCull != 0);
    ps.camLights = pi.lights;
    const float tSkip = pi.tSkip;

    while (true) {
        const unsigned mG = __ballot_sync(0xffffffffu, phase == PH_GEN);
        const unsigned mM = __ballot_sync(0xffffffffu, phase == PH_MARCH);
        const unsigned mC = __ballot_sync(0xffffffffu, phase == PH_COLLIDE);
        const unsigned mE = __ballot_sync(0xffffffffu, phase == PH_EVENT);
        const unsigned mB = __ballot_sync(0xffffffffu, phase == PH_BOUNCE);
        if (!(mG | mM | mC | mE | mB)) break;
        // run the phase most lanes are waiting in (ties go to the cheaper phase)
        int pick = PH_MARCH, best = __popc(mM);
        if (__popc(mC) > best) { pick = PH_COLLIDE; best = __popc(mC); }
        if (__popc(mG) > best) { pick = PH_GEN; best = __popc(mG); }
        if (__popc(mB) > best) { pick = PH_BOUNCE; best = __popc(mB); }
        if (__popc(mE) > best) { pick = PH_EVENT; best = __popc(mE); }

        if (pick == PH_MARCH) {
            // a burst of macrocell visits (mode 2) / one free-flight draw (modes 0, 1)
            const int burst = MODE >= 2 ? a.marchBurst : 1;
            for (int i = 0; i < burst; ++i) {
                if (phase == PH_MARCH) {
                    VisitResult v = ps.trk.template visit<COUNT>(s, ps.ray, ps.rng, lc);
                    if (v == VISIT_COLLIDE) phase = PH_COLLIDE;
                    else if (v == VISIT_ESCAPED) {
                        tEvent = -FLT_MAX;
                        phase = ps.shadow ? PH_BOUNCE : PH_EVENT;
                    }
                }
                if (!__any_sync(0xffffffffu, phase == PH_MARCH)) break;
            }
        } else if (pick == PH_COLLIDE) {
            if (phase == PH_COLLIDE) {
                const int slot = ps.shadow ? SVR_CNT_SHADOW_TAPS : SVR_CNT_TRACK_TAPS;
                float* ratio = (ps.shadow && s.shadowEstimator) ? &ps.ratioT : nullptr;
                if (ps.trk.template collide<COUNT>(s, ps.ray, ps.rng, lc, slot, ratio)) {
                    tEvent = ps.trk.t;
                    phase = ps.shadow ? PH_BOUNCE : PH_EVENT;
                } else if (ratio && ratio_roulette(ps.ratioT, ps.rng)) {
                    tEvent = -FLT_MAX;
                    phase = PH_BOUNCE;
                } else {
                    phase = PH_MARCH;
                }
            }
        } else if (pick == PH_GEN) {
            if (phase == PH_GEN) {
                if (n == a.nSamples) {
                    phase = PH_DONE;
                } else {
                    lc.add(SVR_CNT_PATHS, 1);
                    const bool tracking = path_begin<MODE>(s, ps, idx, idy, offset, a.firstSample + n, tSkip);
                    ++n;
                    tEvent = -FLT_MAX;
                    phase = tracking ? PH_MARCH : PH_EVENT;
                    if (a.traceDepth == 0) phase = PH_GEN;  // the bounce loop never runs (pathtracer.cu:216): the sample is black
                }
            }
        } else if (pick == PH_EVENT) {
            if (phase == PH_EVENT) {
                Next nx = event_flight_end<MODE, COUNT>(s, ps, tEvent, a.traceDepth, lc);
                if (nx == NEXT_TRACK) phase = PH_MARCH;
                else if (nx == NEXT_PATH_DONE) {
                    path_end<MODE>(ps);
                    phase = PH_GEN;
                } else {
                    // NEXT_BOUNCE: no shadow ray; NEXT_FLIGHT_MISSED: the shadow ray cannot collide
                    tEvent = -FLT_MAX;
                    phase = PH_BOUNCE;
                }
            }
        } else {
            if (phase == PH_BOUNCE) {
                Next nx = event_bounce<MODE, COUNT>(s, ps, occluded_at(ps.trk, tEvent), a.traceDepth, lc);
                if (nx == NEXT_TRACK) phase = PH_MARCH;
                else if (nx == NEXT_PATH_DONE) {
                    path_end<MODE>(ps);
                    phase = PH_GEN;
                } else {
                    tEvent = -FLT_MAX;  // the bounce ray misses the (clipped) box
                    phase = PH_EVENT;
                }
            }
        }
    }
    if (inside) write_pixel(s, a, offset, pixel_sum<MODE>(ps));
    lc.flush(cnt);
}

// A later call of the look-ahead protocol: fold the kept sample of frame a.firstSample into the running mean and tone-map --
// write_pixel itself, on the value the sample-parallel launch stored.
__global__ void __launch_bounds__(256) lookahead_consume_kernel(const __grid_constant__ DevScene s, const PtLaunch a, const float* __restrict__ records,
                                                                const uint8_t* __restrict__ constantPixel, uint32_t batch, uint32_t j)
{
    const uint32_t offset = blockIdx.x * blockDim.x + threadIdx.x;
    if (offset >= s.cam.imageW * s.cam.imageH) return;
    float3 v;
    if (constantPixel[offset]) {
        v = (a.traceDepth != 0 && s.envEnabled) ? f3(s.env.defaultRadiance) * s.env.intensity : f3(0.f);  // as the kernels write it for an all-sky pixel
    } else {
        const float* rec = records + (size_t)offset * (3u * batch) + 3u * j;
        v = f3(rec[0], rec[1], rec[2]);
    }
    write_pixel(s, a, offset, v);
}

// root-side resolve of summed partials: hdr = rgb / w, tone map, both in one pass
__global__ void resolve_kernel(const float4* __restrict__ sum, float* __restrict__ hdr, uint32_t* __restrict__ img,
                               uint32_t npix, float exposure)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= npix) return;
    float4 v = sum[i];
    float inv = v.w > 0.f ? 1.f / v.w : 0.f;
    float3 acc = f3(v.x * inv, v.y * inv, v.z * inv);
    if (hdr) {
        hdr[3 * (size_t)i + 0] = acc.x;
        hdr[3 * (size_t)i + 1] = acc.y;
        hdr[3 * (size_t)i + 2] = acc.z;
    }
    if (img) {
        float3 l = tone_map(acc, exposure);
        img[i] = pack_u8x4(l.x * 255.f, l.y * 255.f, l.z * 255.f, 255.f);
    }
}

// ---------------------------------------------------------------------------------------------
// adaptive sampling: the start of a render and the convergence pass between its rounds
// ---------------------------------------------------------------------------------------------
// clears the two accumulators, lists every pixel, clears both count slots
__global__ void adaptive_start_kernel(float4* __restrict__ sum, float4* __restrict__ half, uint32_t* __restrict__ list, uint32_t* __restrict__ counts,
                                      uint32_t npix)
{
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < 4u) counts[i] = 0u;
    if (i >= npix) return;
    sum[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    half[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    list[i] = i;
}

// d = max over channels of |tone_map(even half's mean) - tone_map(odd half's mean)| / 2: the standard error of the displayed
// value, estimated from the two halves (they differ by twice the standard error of the full mean)
SVR_DEV float half_difference(const float4* __restrict__ sum, const float4* __restrict__ half, uint32_t i, float exposure)
{
    const float4 s = sum[i], h = half[i];
    const float we = s.w - h.w;
    if (!(h.w > 0.f) || !(we > 0.f)) return 0.f;
    const float3 even = tone_map(f3((s.x - h.x) / we, (s.y - h.y) / we, (s.z - h.z) / we), exposure);
    const float3 odd = tone_map(f3(h.x / h.w, h.y / h.w, h.z / h.w), exposure);
    return 0.5f * fmaxf(fmaxf(fabsf(even.x - odd.x), fabsf(even.y - odd.y)), fabsf(even.z - odd.z));
}

// One pass over the image after a round: err = RMS of d over the 3 x 3 window (coordinates clamped to the image), optionally
// stored; a pixel stays listed iff it took the last round (w == wActive), err >= threshold and w < maxSamples.  Blocks of
// 32 x 8 pixels: d of the block and its one-pixel rim goes through shared memory, and each warp (one row of 32 pixels) appends
// its active pixels to the list with one atomicAdd.  counts[slot] = {active, err >= threshold}; the other slot is cleared for
// the next pass (the previous pass's counts have been read by then).
__global__ void __launch_bounds__(256) adaptive_converge_kernel(const float4* __restrict__ sum, const float4* __restrict__ half, float* __restrict__ err,
                                                                uint32_t* __restrict__ list, uint32_t* __restrict__ counts, uint32_t slot, uint32_t W,
                                                                uint32_t H, float wActive, float maxSamples, float threshold, float exposure)
{
    __shared__ float d[10][34];
    const int x0 = (int)(blockIdx.x * 32u) - 1, y0 = (int)(blockIdx.y * 8u) - 1;
    for (uint32_t t = threadIdx.y * 32u + threadIdx.x; t < 10u * 34u; t += 256u) {
        const int ty = (int)(t / 34u), tx = (int)(t % 34u);
        const uint32_t x = (uint32_t)min(max(x0 + tx, 0), (int)W - 1), y = (uint32_t)min(max(y0 + ty, 0), (int)H - 1);
        d[ty][tx] = half_difference(sum, half, y * W + x, exposure);
    }
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.y == 0 && threadIdx.x < 2u) counts[2u * (slot ^ 1u) + threadIdx.x] = 0u;
    __syncthreads();
    const uint32_t x = blockIdx.x * 32u + threadIdx.x, y = blockIdx.y * 8u + threadIdx.y;
    bool active = false, unconverged = false;
    if (x < W && y < H) {
        float e2 = 0.f;
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const float v = d[threadIdx.y + j][threadIdx.x + i];
                e2 += v * v;
            }
        const float e = sqrtf(e2 * (1.f / 9.f));
        const uint32_t offset = y * W + x;
        if (err) err[offset] = e;
        const float w = sum[offset].w;
        unconverged = e >= threshold;
        active = unconverged && w == wActive && w < maxSamples;
    }
    const uint32_t ballot = __ballot_sync(0xffffffffu, active), late = __ballot_sync(0xffffffffu, unconverged);
    uint32_t base = 0u;
    if (threadIdx.x == 0) {
        if (ballot) base = atomicAdd(counts + 2u * slot, (uint32_t)__popc(ballot));
        if (late) atomicAdd(counts + 2u * slot + 1u, (uint32_t)__popc(late));
    }
    base = __shfl_sync(0xffffffffu, base, 0);
    if (active) list[base + (uint32_t)__popc(ballot & ((1u << threadIdx.x) - 1u))] = y * W + x;
}

// dynamic shared memory of pathtrace_pool_kernel for blocks of `threads`
constexpr size_t pool_shared_bytes(int threads) { return sizeof(float) * SVR_ITEM_WORDS * (SVR_POOL_CAP + SVR_EVQ_CAP) * (size_t)(threads / 32); }

typedef void (*PtKernel)(const DevScene, const PtLaunch, Counters*);

// the kernel's COUNT = true instance with counters, its COUNT = false instance without
void launch_counted(PtKernel counted, PtKernel plain, dim3 grid, int block, size_t shm, cudaStream_t stream, const DevScene& sc, const PtLaunch& a,
                    Counters* cnt)
{
    (cnt ? counted : plain)<<<grid, block, shm, stream>>>(sc, a, cnt);
}

template <int MODE>
void launch_mode(int shape, dim3 grid, int block, cudaStream_t stream, const DevScene& sc, const PtLaunch& a, Counters* cnt)
{
    if (shape == 5) {  // choose_shape() only picks it for MODE 2
        static bool attr = false;
        if (!attr) {
            for (PtKernel k : {pathtrace_pool_kernel<true>, pathtrace_pool_kernel<false>})
                cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pool_shared_bytes(SVR_PT_MAX_THREADS));
            attr = true;
        }
        launch_counted(pathtrace_pool_kernel<true>, pathtrace_pool_kernel<false>, grid, block, pool_shared_bytes(block), stream, sc, a, cnt);
    } else if (shape == 4) {  // choose_shape() only picks it for MODE 2 with a pinhole camera
        launch_counted(pathtrace_profile_kernel<true>, pathtrace_profile_kernel<false>, grid, block, 0, stream, sc, a, cnt);
    } else if (shape == 3) {  // choose_shape() only picks it for MODE 2
        launch_counted(pathtrace_queue_kernel<true>, pathtrace_queue_kernel<false>, grid, block, 0, stream, sc, a, cnt);
    } else if (shape == 2 && a.perSample) {  // launch_pathtrace() only sets it without counters and without the block split
        pathtrace_warp_kernel<MODE, false, false, true><<<grid, block, 0, stream>>>(sc, a, cnt);
    } else if (shape == 2 && a.blockSplit) {
        launch_counted(pathtrace_warp_kernel<MODE, true, true>, pathtrace_warp_kernel<MODE, false, true>, grid, block, 0, stream, sc, a, cnt);
    } else if (shape == 2) {
        launch_counted(pathtrace_warp_kernel<MODE, true, false>, pathtrace_warp_kernel<MODE, false, false>, grid, block, 0, stream, sc, a, cnt);
    } else if (shape == 1) {
        launch_counted(pathtrace_mega_kernel<MODE, true>, pathtrace_mega_kernel<MODE, false>, grid, block, 0, stream, sc, a, cnt);
    } else {
        launch_counted(pathtrace_sched_kernel<MODE, true>, pathtrace_sched_kernel<MODE, false>, grid, block, 0, stream, sc, a, cnt);
    }
}

// f(std::integral_constant<int, MODE>()) for the kernels' MODE: SVR_OPT_PT_MODE, or 3 for local majorants with environment NEE
template <class F>
void with_mode(int mode, F&& f)
{
    switch (mode) {
        case 0: f(std::integral_constant<int, 0>()); break;
        case 1: f(std::integral_constant<int, 1>()); break;
        case 2: f(std::integral_constant<int, 2>()); break;
        default: f(std::integral_constant<int, 3>()); break;
    }
}

// The pixels an adaptive render still samples (svr_pathtracer_accumulate_adaptive): offsets list[0 .. count), odd samples' sums into half
struct PixelList {
    const uint32_t* list;
    uint32_t count;
    float4* half;
};

// The kernel shape a launch runs: SVR_OPT_PT_KERNEL (`requested`) where the estimator, the camera and the launch allow it.
int choose_shape(int requested, int mode, uint32_t traceDepth, int queueMinDepth, bool profile, bool pinhole, bool envNee, uint32_t nSamples,
                 uint32_t warpMinSpp, bool perSample, bool list)
{
    if (list) return 2;  // the adaptive entry point's list kernel is a sample-parallel sibling (it has ruled out counters)
    int shape = requested;
    if (mode != 2 || envNee) {
        // shapes 3-5 serve local-majorant Philox paths, and environment next-event estimation lives in the shared event code
        // of shapes 0-2: the plain sample-parallel shape stands in for them
        shape = std::min(shape, 2);
    } else if (shape == 2 || shape == 3) {
        // camera rays against the pixel's majorant profile (shape 4) when the camera is a pinhole (one origin per pixel); it has
        // shape 3's scatter queue built in.  Otherwise deep paths get the scatter queue (DESIGN.md section 3.1)
        const bool deep = shape == 3 || (queueMinDepth > 0 && traceDepth >= (uint32_t)queueMinDepth);
        shape = profile && pinhole ? 4 : (deep ? 3 : 2);
    } else if (shape == 4 && !pinhole) {
        shape = 2;
    }
    // the sample-parallel shapes need a warp's worth of samples per pixel; below that one lane per pixel
    if (shape >= 2 && nSamples < warpMinSpp && !perSample) shape = 1;
    return shape;
}

// Per-pixel classification for shapes 1-3: made for the whole image by a kernel of its own and, with SVR_OPT_PT_PIXEL_CACHE,
// kept until something a pixel can see changes (sceneEpoch); without it, made again for every launch.  The render kernels only
// read it.  A kept classification includes the entry walk whenever the option allows one: its cost is paid once, so it also
// serves single-sample launches, for which a walk per launch does not pay (images are bit-identical either way: only empty
// space is skipped).
int ensure_pixel_classification(HostState& st, const DevScene& sc, int mode, PtLaunch& a)
{
    DeviceState& d = st.dev;
    const bool keep = st.options[SVR_OPT_PT_PIXEL_CACHE] != 0;
    const int walk = keep ? (st.options[SVR_OPT_PT_ENTRY_CACHE] != 0) : a.entryCache;
    const size_t npix = (size_t)sc.cam.imageW * sc.cam.imageH;
    if (d.pixelCache.cap < npix) d.pixelCacheEpoch = 0;  // new memory holds no classification
    SVR_TRY(d.pixelCache.reserve(npix));
    const int key = (sc.envNee ? 3 : mode) * 2 + walk;
    const bool valid = keep && d.pixelCacheEpoch == st.sceneEpoch && d.pixelCacheW == sc.cam.imageW && d.pixelCacheH == sc.cam.imageH &&
                       d.pixelCacheMode == key;
    if (!valid) {
        dim3 cg((sc.cam.imageW + 15u) / 16u, (sc.cam.imageH + 7u) / 8u);
        classify_pixels_kernel<<<cg, 128, 0, st.stream>>>(sc, d.pixelCache.p, mode >= 2 ? 1 : 0, walk, a.lightCull);
        count_launch();
        SVR_TRY(cudaGetLastError());
        d.pixelCacheEpoch = keep ? st.sceneEpoch : 0;
        d.pixelCacheW = sc.cam.imageW;
        d.pixelCacheH = sc.cam.imageH;
        d.pixelCacheMode = key;
    }
    a.pixelCache = 2;
    a.pixelInfo = d.pixelCache.p;
    return 0;
}

// A launch over every row of the image, everything else zero
PtLaunch full_frame(uint32_t traceDepth, uint32_t firstSample, uint32_t nSamples)
{
    PtLaunch a;
    memset(&a, 0, sizeof(a));
    a.traceDepth = traceDepth;
    a.firstSample = firstSample;
    a.nSamples = nSamples;
    a.y0 = 0;
    a.y1 = 0xffffffffu;
    return a;
}

// pl != null: the sample-parallel shape over the listed pixels (pathtrace_list_kernel), whatever the options would pick
int launch_pathtrace(PtLaunch& a, const PixelList* pl = nullptr)
{
    HostState& st = state();
    DevScene sc = st.scene;
    if (!sc.vol.tex || !sc.tf.tex) return fail_msg("render_pathtracer: setup_volume / setup_transferfunction not called");
    if (sc.cam.imageW == 0 || sc.cam.imageH == 0) return fail_msg("render_pathtracer: setup_camera not called");
    const int mode = st.options[SVR_OPT_PT_MODE];
    sc.envEnabled = st.options[SVR_OPT_ENV_ENABLED];
    sc.envNee = 0;
    memset(&sc.envS, 0, sizeof(sc.envS));
    if (sc.envEnabled && st.options[SVR_OPT_ENV_NEE] && mode == 2) {
        int rc = ensure_env_sampler(&sc);
        if (rc) return rc;
        sc.envNee = 1;
    }
    sc.shadowEstimator = st.options[SVR_OPT_SHADOW_ESTIMATOR];
    sc.seedKey = wang_hash((uint32_t)st.options[SVR_OPT_SEED]);
    if (mode == 2) {
        int rc = ensure_grid(&sc, false);
        if (rc) return rc;
    } else {
        memset(&sc.grid, 0, sizeof(sc.grid));
    }
    if (a.y1 > sc.cam.imageH) a.y1 = sc.cam.imageH;
    if (a.y0 >= a.y1 || a.nSamples == 0) return 0;
    a.marchBurst = st.options[SVR_OPT_PT_ROUNDS] > 0 ? st.options[SVR_OPT_PT_ROUNDS] : 4;
    a.entryCache = st.options[SVR_OPT_PT_ENTRY_CACHE] && a.nSamples >= 2;
    a.lightCull = st.options[SVR_OPT_PT_LIGHT_CULL];
    a.clipped = !(sc.vol.x_clip.x == -1.f && sc.vol.x_clip.y == 1.f && sc.vol.y_clip.x == -1.f && sc.vol.y_clip.y == 1.f && sc.vol.z_clip.x == -1.f &&
                  sc.vol.z_clip.y == 1.f);
    Counters* cnt = nullptr;
    if (st.options[SVR_OPT_COUNTERS]) {
        cnt = device_counters();
        if (!cnt) return fail_msg("render_pathtracer: counter allocation failed");
    }
    const int block = st.options[SVR_OPT_PT_BLOCK];
    const int shape = choose_shape(st.options[SVR_OPT_PT_KERNEL], mode, a.traceDepth, st.options[SVR_OPT_PT_QUEUE_MIN_DEPTH], st.options[SVR_OPT_PT_PROFILE] != 0,
                                   sc.cam.apeture == 0.f, sc.envNee != 0, a.nSamples, (uint32_t)st.options[SVR_OPT_PT_WARP_MIN_SPP], a.perSample != nullptr,
                                   pl != nullptr);
    if (a.perSample && (shape != 2 || cnt || a.nSamples > 32u)) {
        a.perSample = nullptr;  // look-ahead is for the plain sample-parallel shape: the caller renders this frame the ordinary way
        return 0;
    }
    hdr_written_outside(st.dev, a.hdr, true);
    // shapes 4 and 5: idle lanes take new camera samples together, once this many wait (SVR_OPT_PT_REFILL)
    if (shape >= 4) a.marchBurst = st.options[SVR_OPT_PT_REFILL] > 0 ? st.options[SVR_OPT_PT_REFILL] : 8;
    a.warpPixels = st.options[SVR_OPT_PT_WARP_PIXELS];
    if (a.warpPixels <= 0) a.warpPixels = a.nSamples >= 128u ? 1 : 2;  // automatic: see the option's default (svr_api.cu)
    if (shape == 5) a.warpPixels = st.options[SVR_OPT_PT_POOL_PIXELS] > 0 ? st.options[SVR_OPT_PT_POOL_PIXELS] : 16;
    uint32_t tileW = 16u, tileH = (uint32_t)block / 16u;
    if (shape >= 2) {
        tileW = (uint32_t)a.warpPixels;
        tileH = (uint32_t)block / 32u;
    }
    a.pixelCache = 0;
    a.pixelInfo = nullptr;
    if (shape >= 1 && shape <= 3) {
        if (int rc = ensure_pixel_classification(st, sc, mode, a)) return rc;
    }
    const int kernelMode = sc.envNee ? 3 : mode;
    if (pl) {
        if (pl->count == 0) return 0;
        const dim3 lg((pl->count + (uint32_t)block / 32u - 1u) / ((uint32_t)block / 32u));
        with_mode(kernelMode, [&](auto m) { pathtrace_list_kernel<decltype(m)::value><<<lg, block, 0, st.stream>>>(sc, a, pl->list, pl->count, pl->half); });
        count_launch();
        SVR_TRY(cudaGetLastError());
        return 0;
    }
    a.blockSplit = shape == 2 && st.options[SVR_OPT_PT_BLOCK_SPLIT] != 0 && a.nSamples >= 32u * ((uint32_t)block / 32u);
    if (a.blockSplit) tileH = 1u;
    if (a.bandStride == 0) a.bandStride = 1;
    if (a.bandPhase >= a.bandStride) return fail_msg("render_pathtracer: band phase must be below the band stride");
    const uint32_t bands = ((a.y1 - a.y0) + tileH - 1u) / tileH;
    if (a.bandPhase >= bands) return 0;
    a.bandRows = tileH;
    dim3 grid((sc.cam.imageW + tileW - 1u) / tileW, (bands - a.bandPhase + a.bandStride - 1u) / a.bandStride);
    with_mode(kernelMode, [&](auto m) { launch_mode<decltype(m)::value>(shape, grid, block, st.stream, sc, a, cnt); });
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

}  // namespace
}  // namespace svr

using namespace svr;

// pathtracer.h:17 / pathtracer.cu:292-304.  One call = one sample per pixel; asynchronous.
// SVR_OPT_PT_LOOKAHEAD > 0: whether batches pay is MEASURED once per scene (events around one single-sample launch, the first
// batch and one fold; read when the next batch is due, never waited for).  Where nearly every pixel is sky a 32-sample batch of
// the sample-parallel kernel plus 32 folds take 0.55 of 32 single launches (C3: 26.3 -> 16.8 ms per 256 frames); with the body
// filling the frame a 32-sample launch is no better per sample than the lane-per-pixel kernel (68.0 against 64.5 ms), and
// look-ahead switches itself off until the scene changes.  Images do not depend on the decision (the two paths are bit-equal).
static bool lookahead_events(HostState& st)
{
    if (!st.dev.aheadEvReady) {
        for (int i = 0; i < 6; ++i)
            if (cudaEventCreate(&st.dev.aheadEv[i]) != cudaSuccess) {
                cudaGetLastError();
                return false;
            }
        st.dev.aheadEvReady = true;
    }
    return true;
}

// true = measured, and batches do not pay for the current scene
static bool lookahead_does_not_pay(HostState& st)
{
    if (st.dev.aheadTimedEpoch != st.sceneEpoch || st.dev.aheadSingleEpoch != st.sceneEpoch || st.dev.aheadTimeFold || !st.dev.aheadTimedBatch) return false;
    for (int i = 1; i < 6; i += 2)
        if (cudaEventQuery(st.dev.aheadEv[i]) != cudaSuccess) {
            cudaGetLastError();
            return false;  // not there yet: ask again at the next batch
        }
    float single = 0.f, batch = 0.f, fold = 0.f;
    if (cudaEventElapsedTime(&single, st.dev.aheadEv[0], st.dev.aheadEv[1]) != cudaSuccess || cudaEventElapsedTime(&batch, st.dev.aheadEv[2], st.dev.aheadEv[3]) != cudaSuccess ||
        cudaEventElapsedTime(&fold, st.dev.aheadEv[4], st.dev.aheadEv[5]) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return batch / (float)st.dev.aheadTimedBatch + fold > 0.97f * single;
}

// *done = the frame has been produced (from samples kept by an earlier call, or by a batch launched now).
static int lookahead_frame(uint32_t* img, float* hdr, uint32_t traceDepth, uint32_t frameNo, bool* done)
{
    HostState& st = state();
    *done = false;
    const uint32_t W = st.scene.cam.imageW, H = st.scene.cam.imageH;
    const int opt = st.options[SVR_OPT_PT_LOOKAHEAD];
    const bool adaptive = opt > 0;
    const uint32_t maxBatch = (uint32_t)std::min(opt < 0 ? -opt : opt, 32);
    if (maxBatch < 2u || !hdr || !W || !H || st.options[SVR_OPT_COUNTERS] || (adaptive && st.dev.aheadOffEpoch == st.sceneEpoch)) {
        st.dev.aheadCount = 0;
        return 0;
    }
    const size_t npix = (size_t)W * H;
    const bool kept = st.dev.aheadCount != 0 && st.dev.aheadEpoch == st.sceneEpoch && st.dev.aheadRender.continues(frameNo, hdr, W, H, traceDepth) &&
                      frameNo < st.dev.aheadFirst + st.dev.aheadCount;
    if (!kept) {
        st.dev.aheadCount = 0;
        // a render that has come this far without a change is likely to go on (whoever moves the camera every few frames never
        // gets here and pays nothing)
        if (frameNo < 16u) return 0;
        if (adaptive && lookahead_does_not_pay(st)) {
            st.dev.aheadOffEpoch = st.sceneEpoch;
            return 0;
        }
        uint32_t batch = maxBatch;
        while (batch >= 2u && (size_t)batch * npix * 3 * sizeof(float) > ((size_t)1 << 30)) batch >>= 1;
        if (batch < 2u) return 0;
        const size_t need = (size_t)batch * npix * 3 + (npix + 3) / 4;  // records, then one flag byte per pixel
        if (st.dev.ahead.reserve(need) != cudaSuccess) {
            cudaGetLastError();
            return 0;  // no memory for it: one sample per call as before
        }
        PtLaunch a = full_frame(traceDepth, frameNo, batch);
        a.perSample = st.dev.ahead.p;
        a.constantPixel = (uint8_t*)(st.dev.ahead.p + (size_t)batch * npix * 3);
        const bool timeIt = adaptive && st.dev.aheadTimedEpoch != st.sceneEpoch && lookahead_events(st);
        if (timeIt) SVR_TRY(cudaEventRecord(st.dev.aheadEv[2], st.stream));
        int rc = launch_pathtrace(a);
        if (rc) return rc;
        if (!a.perSample) return 0;  // another kernel shape serves this scene
        if (timeIt) {
            SVR_TRY(cudaEventRecord(st.dev.aheadEv[3], st.stream));
            st.dev.aheadTimedEpoch = st.sceneEpoch;
            st.dev.aheadTimedBatch = batch;
            st.dev.aheadTimeFold = true;
        }
        st.dev.aheadFirst = frameNo;
        st.dev.aheadCount = batch;
        st.dev.aheadEpoch = st.sceneEpoch;  // after the launch: refreshing the majorants moves the epoch
        st.aheadBatches++;
    }
    PtLaunch c;
    memset(&c, 0, sizeof(c));
    c.traceDepth = traceDepth;
    c.firstSample = frameNo;
    c.nSamples = 1;
    c.hdr = hdr;
    c.img = img;
    DevScene sc = st.scene;
    sc.envEnabled = st.options[SVR_OPT_ENV_ENABLED];  // as launch_pathtrace sets it
    const bool timeFold = st.dev.aheadTimeFold && st.dev.aheadTimedEpoch == st.sceneEpoch;
    if (timeFold) SVR_TRY(cudaEventRecord(st.dev.aheadEv[4], st.stream));
    lookahead_consume_kernel<<<(unsigned)((npix + 255) / 256), 256, 0, st.stream>>>(sc, c, st.dev.ahead.p, (const uint8_t*)(st.dev.ahead.p + (size_t)st.dev.aheadCount * npix * 3),
                                                                                   st.dev.aheadCount, frameNo - st.dev.aheadFirst);
    count_launch();
    SVR_TRY(cudaGetLastError());
    if (timeFold) {
        SVR_TRY(cudaEventRecord(st.dev.aheadEv[5], st.stream));
        st.dev.aheadTimeFold = false;
    }
    st.dev.aheadRender.follow(frameNo, hdr, W, H, traceDepth);
    *done = true;
    return 0;
}

// SVR_OPT_PT_DENOISE (include/svr_render.h).  *done = the call was a denoised frame: one sample traced by the ordinary launch into
// hdr (bit-identical to the option-off call) and into the even or odd sum by the parity of frameNo, then guides and filter into
// img (svr_denoise.cu).  A call that does not continue the followed render drops it; so does a failed allocation, and the call
// then renders as with the option off.
static int denoised_frame(uint32_t* img, float* hdr, uint32_t traceDepth, uint32_t frameNo, bool* done)
{
    HostState& st = state();
    *done = false;
    const uint32_t W = st.scene.cam.imageW, H = st.scene.cam.imageH;
    const bool follows = frameNo == 0u || st.dev.progRender.continues(frameNo, hdr, W, H, traceDepth);
    st.dev.progRender = FollowedRender();
    if (!st.options[SVR_OPT_PT_DENOISE] || st.options[SVR_OPT_COUNTERS] || !follows || !img || !hdr || !W || !H) return 0;
    const size_t npix = (size_t)W * H;
    if (!ensure_progressive_buffers(st, npix)) return 0;
    float4* const sums = st.dev.prog.p;  // even, odd
    if (frameNo == 0u) SVR_TRY(cudaMemsetAsync(sums + npix, 0, npix * sizeof(float4), st.stream));
    PtLaunch a = full_frame(traceDepth, frameNo, 1);
    a.hdr = hdr;
    a.sum = sums + (frameNo & 1u) * npix;
    a.clearSum = frameNo == 0u;
    if (int rc = launch_pathtrace(a)) return rc;
    if (int rc = progressive_denoise(img, frameNo)) return rc;
    st.dev.progRender.follow(frameNo, hdr, W, H, traceDepth);
    *done = true;
    return 0;
}

extern "C" void render_pathtracer(svr_u8vec4* img, const svr_render_params* renderParams)
{
    bool done = false;
    int rc = denoised_frame((uint32_t*)img, (float*)renderParams->hdrBuffer, renderParams->traceDepth, renderParams->frameNo, &done);
    if (!rc && !done) rc = lookahead_frame((uint32_t*)img, (float*)renderParams->hdrBuffer, renderParams->traceDepth, renderParams->frameNo, &done);
    if (!rc && !done) {
        PtLaunch a = full_frame(renderParams->traceDepth, renderParams->frameNo, 1);
        a.hdr = (float*)renderParams->hdrBuffer;
        a.img = (uint32_t*)img;
        // look-ahead's yardstick: one steady-state single-sample launch per scene (classification cached, nothing to refresh)
        HostState& st = state();
        const bool timeIt = st.options[SVR_OPT_PT_LOOKAHEAD] > 1 && a.firstSample >= 8u && a.firstSample < 16u && st.dev.aheadSingleEpoch != st.sceneEpoch &&
                            st.dev.pixelCacheEpoch == st.sceneEpoch && lookahead_events(st);
        if (timeIt) cudaEventRecord(st.dev.aheadEv[0], st.stream);
        rc = launch_pathtrace(a);
        if (timeIt && !rc) {
            cudaEventRecord(st.dev.aheadEv[1], st.stream);
            st.dev.aheadSingleEpoch = st.sceneEpoch;
        }
    }
    if (rc) {
        fprintf(stderr, "CUDA error at %s:%d code=%d \"%s\" \n", __FILE__, __LINE__, rc, svr_last_error());
        cudaDeviceReset();
        exit(EXIT_FAILURE);
    }
}

extern "C" int svr_render_pathtracer_spp(svr_u8vec4* img, const svr_render_params* renderParams, uint32_t spp)
{
    if (!renderParams || !renderParams->hdrBuffer) return fail_msg("svr_render_pathtracer_spp: hdrBuffer is null");
    state().dev.progRender = FollowedRender();  // SVR_OPT_PT_DENOISE does not apply: the render it followed has moved on without its sums
    PtLaunch a = full_frame(renderParams->traceDepth, renderParams->frameNo, spp);
    a.hdr = (float*)renderParams->hdrBuffer;
    a.img = (uint32_t*)img;
    return launch_pathtrace(a);
}

extern "C" int svr_pathtracer_accumulate(svr_vec4* sum, uint32_t traceDepth, uint32_t firstSample, uint32_t nSamples, int clear)
{
    if (!sum) return fail_msg("svr_pathtracer_accumulate: sum is null");
    PtLaunch a = full_frame(traceDepth, firstSample, nSamples);
    a.sum = (float4*)sum;
    a.clearSum = clear;
    return launch_pathtrace(a);
}

extern "C" int svr_pathtracer_accumulate_bands(svr_vec4* sum, uint32_t traceDepth, uint32_t firstSample, uint32_t nSamples, int clear,
                                               uint32_t phase, uint32_t stride, uint32_t* bandRows)
{
    if (!sum) return fail_msg("svr_pathtracer_accumulate_bands: sum is null");
    PtLaunch a = full_frame(traceDepth, firstSample, nSamples);
    a.sum = (float4*)sum;
    a.clearSum = clear;
    a.bandPhase = phase;
    a.bandStride = stride;
    int rc = launch_pathtrace(a);
    if (bandRows) *bandRows = a.bandRows;
    return rc;
}

// Adaptive sampling (include/svr_render.h).  Every round renders one sample range for all listed pixels -- a pixel that has
// stopped never restarts, so the listed pixels share one sample count -- and reads the pass's two counts through the mailbox:
// one stream synchronisation per round.
extern "C" int svr_pathtracer_accumulate_adaptive(svr_vec4* sum, svr_vec4* halfSum, float* errOrNull, uint32_t traceDepth, uint32_t firstSample,
                                                  uint32_t minSamples, uint32_t maxSamples, uint32_t batch, float threshold, uint32_t* roundsOut,
                                                  uint64_t* samplesOut, uint32_t* unconvergedOut)
{
    HostState& st = state();
    if (!sum || !halfSum) return fail_msg("svr_pathtracer_accumulate_adaptive: sum and halfSum must not be null");
    if (minSamples == 0 || maxSamples == 0 || batch == 0 || (minSamples | maxSamples | batch) % 32u != 0u)
        return fail_msg("svr_pathtracer_accumulate_adaptive: minSamples, maxSamples and batch must be positive multiples of 32");
    if (maxSamples < minSamples) return fail_msg("svr_pathtracer_accumulate_adaptive: maxSamples is below minSamples");
    if (maxSamples > (1u << 24)) return fail_msg("svr_pathtracer_accumulate_adaptive: maxSamples above 2^24 (sample counts are floats)");
    if (!(threshold >= 0.f)) return fail_msg("svr_pathtracer_accumulate_adaptive: threshold must be >= 0");
    if (st.options[SVR_OPT_COUNTERS]) return fail_msg("svr_pathtracer_accumulate_adaptive: SVR_OPT_COUNTERS must be 0");
    if (!st.scene.vol.tex || !st.scene.tf.tex) return fail_msg("render_pathtracer: setup_volume / setup_transferfunction not called");
    const uint32_t W = st.scene.cam.imageW, H = st.scene.cam.imageH, npix = W * H;
    if (!npix) return fail_msg("render_pathtracer: setup_camera not called");
    SVR_TRY(st.dev.adaptiveList.reserve(npix));
    SVR_TRY(st.dev.adaptiveCounts.reserve(4));
    float4* s4 = (float4*)sum;
    float4* h4 = (float4*)halfSum;
    adaptive_start_kernel<<<(npix + 255u) / 256u, 256, 0, st.stream>>>(s4, h4, st.dev.adaptiveList.p, st.dev.adaptiveCounts.p, npix);
    count_launch();
    SVR_TRY(cudaGetLastError());

    PtLaunch a = full_frame(traceDepth, 0, 0);
    a.sum = s4;
    PixelList pl = {st.dev.adaptiveList.p, npix, h4};
    uint32_t w = 0, n = minSamples, rounds = 0, unconverged = 0;
    uint64_t samples = 0;
    for (uint32_t pass = 0;; ++pass) {
        a.firstSample = firstSample + w;
        a.nSamples = n;
        if (int rc = launch_pathtrace(a, &pl)) return rc;
        rounds++;
        samples += (uint64_t)pl.count * n;
        w += n;
        const dim3 cb((W + 31u) / 32u, (H + 7u) / 8u);
        const uint32_t slot = pass & 1u;
        adaptive_converge_kernel<<<cb, dim3(32, 8), 0, st.stream>>>(s4, h4, errOrNull, st.dev.adaptiveList.p, st.dev.adaptiveCounts.p, slot, W, H, (float)w,
                                                                   (float)maxSamples, threshold, st.scene.cam.exposure);
        count_launch();
        SVR_TRY(cudaGetLastError());
        uint32_t c[2];
        if (int rc = read_small(st, c, st.dev.adaptiveCounts.p + 2u * slot, sizeof(c))) return rc;
        pl.count = c[0];
        unconverged = c[1];
        if (pl.count == 0) break;
        n = std::min(batch, maxSamples - w);
    }
    if (roundsOut) *roundsOut = rounds;
    if (samplesOut) *samplesOut = samples;
    if (unconvergedOut) *unconvergedOut = unconverged;
    return 0;
}

extern "C" int svr_pathtracer_resolve(svr_u8vec4* img, svr_vec3* hdrOut, const svr_vec4* sum)
{
    HostState& st = state();
    if (!sum) return fail_msg("svr_pathtracer_resolve: sum is null");
    uint32_t npix = st.scene.cam.imageW * st.scene.cam.imageH;
    if (!npix) return fail_msg("svr_pathtracer_resolve: setup_camera not called");
    hdr_written_outside(st.dev, hdrOut, false);
    resolve_kernel<<<(npix + 255u) / 256u, 256, 0, st.stream>>>((const float4*)sum, (float*)hdrOut, (uint32_t*)img, npix,
                                                               st.scene.cam.exposure);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}
