// svr_denoise.cu -- denoising of accumulated path-traced images (include/svr_render.h: svr_pathtracer_guides,
// svr_pathtracer_denoise, svr_denoise_defaults).
//
// Guides: a deterministic march per camera ray that records what the path tracer's first collision sees on average --
// coverage, albedo (TF colour), view-space depth and the camera-facing gradient normal -- each weighted by the
// first-collision density T(t) sigma(t) of delta tracking.  Filter: an edge-avoiding a-trous wavelet (Dammertz et al.
// 2010) on the albedo-demodulated mean, its luminance stop scaled by a per-pixel variance taken from the even/odd sample
// halves of an adaptive render (Schied et al. 2017, the spatial part of SVGF).
#include <cmath>

#include "svr_state.h"

namespace svr {

namespace {

// Shirley-Chiu concentric map of [0,1)^2 onto the unit disk
SVR_DEV float2 concentric_disk(float u1, float u2)
{
    const float ox = 2.f * u1 - 1.f, oy = 2.f * u2 - 1.f;
    if (ox == 0.f && oy == 0.f) return make_float2(0.f, 0.f);
    float r, th;
    if (fabsf(ox) > fabsf(oy)) {
        r = ox;
        th = 0.25f * SVR_PI_F * (oy / ox);
    } else {
        r = oy;
        th = 0.5f * SVR_PI_F - 0.25f * SVR_PI_F * (ox / oy);
    }
    return make_float2(r * cosf(th), r * sinf(th));
}

// Guide pass.  One lane per pixel, its side x side rays one after the other; blocks of 16 x 8 pixels, 8 x 4 per warp
// (neighbouring rays walk the same macrocells).  Per ray, samples at t0 + (k + 1/2) h up to the volume's far face or
// the nearest area-light disk; cells whose majorant is <= 0 (and the empty cube they record) are skipped by index.
__global__ void __launch_bounds__(128) guides_kernel(const __grid_constant__ DevScene s, float4* __restrict__ albedoCoverage,
                                                     float4* __restrict__ normalDepth, int side)
{
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t x = blockIdx.x * 16u + (warp & 1u) * 8u + (lane & 7u);
    const uint32_t y = blockIdx.y * 8u + (warp >> 1) * 4u + (lane >> 3);
    const svr_camera& c = s.cam;
    if (x >= c.imageW || y >= c.imageH) return;
    const float h = 0.5f * fminf(fminf(s.vol.spacing.x, s.vol.spacing.y), s.vol.spacing.z);
    const float3 camPos = f3(c.pos), back = -f3(c.w);
    const float inv = 1.f / (float)side;
    float alpha = 0.f, Z = 0.f;
    float3 A = f3(0.f), N = f3(0.f);
    for (int j = 0; j < side; ++j)
        for (int i = 0; i < side; ++i) {
            const float jx = ((float)i + 0.5f) * inv, jy = ((float)j + 0.5f) * inv;
            Ray ray;
            if (c.apeture == 0.f) {
                ray.orig = camPos;
                ray.dir = camera_dir_pinhole(c, x, y, jx, jy);
            } else {  // camera_ray_jittered with the lens sample at the same grid position
                float nx = 2.f * (((float)x + jx) / ((float)c.imageW - 1.f)) - 1.f;
                float ny = 2.f * (((float)y + jy) / ((float)c.imageH - 1.f)) - 1.f;
                nx = nx * c.aspectRatio * c.tanFovxOverTwo * c.focalLength;
                ny = ny * c.tanFovxOverTwo * c.focalLength;
                const float2 d = concentric_disk(jx, jy);
                const float ax = d.x * c.apeture, ay = d.y * c.apeture;
                ray.orig = camPos + ax * f3(c.u) + ay * f3(c.v);
                ray.dir = normalize((nx - ax) * f3(c.u) + (ny - ay) * f3(c.v) - c.focalLength * f3(c.w));
            }
            float tNear, tFar;
            if (!intersect_volume(s.vol, ray, &tNear, &tFar)) continue;
            LightHit lh;
            const float tEnd = nearest_light(s, ray, &lh) ? fminf(tFar, lh.t) : tFar;
            const float t0 = fmaxf(tNear, 0.f);
            const float3 dg = ray.dir * (f3(s.vol.bbox.invSize) * s.grid.scale);  // macrocell coordinates per unit t
            const float3 invDg = 1.f / dg;
            float T = 1.f;
            for (int k = 0;;) {
                const float t = fmaf((float)k + 0.5f, h, t0);
                if (!(t < tEnd)) break;
                const float3 p = ray.orig + t * ray.dir;
                const float3 tc = tex_coord(s.vol, p);
                const float3 g = tc * s.grid.scale;
                const int cx = min(max((int)floorf(g.x), 0), s.grid.gx - 1);
                const int cy = min(max((int)floorf(g.y), 0), s.grid.gy - 1);
                const int cz = min(max((int)floorf(g.z), 0), s.grid.gz - 1);
                const float sig = s.grid.at(cx, cy, cz);
                if (sig <= 0.f) {
                    // empty, and so is the cube of radius d - 1 around it (raycast_kernel): on to the first sample past its far faces
                    const int d = (int)(-sig) > 1 ? (int)(-sig) : 1;
                    const float ex = ((dg.x > 0.f ? (float)(cx + d) : (float)(cx - d + 1)) - g.x) * invDg.x;
                    const float ey = ((dg.y > 0.f ? (float)(cy + d) : (float)(cy - d + 1)) - g.y) * invDg.y;
                    const float ez = ((dg.z > 0.f ? (float)(cz + d) : (float)(cz - d + 1)) - g.z) * invDg.z;
                    const float tExit = t + fminf(fminf(dg.x != 0.f ? ex : FLT_MAX, dg.y != 0.f ? ey : FLT_MAX), dg.z != 0.f ? ez : FLT_MAX);
                    if (!(tExit < tEnd)) break;
                    k = max(k + 1, (int)ceilf((tExit - t0) / h - 0.5f));
                    continue;
                }
                ++k;
                const float4 co = tf_at(s.tf, tex3D<float>(s.vol.tex, tc.x, tc.y, tc.z) * s.vol.densityScale);
                if (!(co.w > 0.f)) continue;
                const float em = expm1f(-co.w * h);  // exp(-sigma h) - 1, accurate for thin steps
                const float pw = -T * em;
                alpha += pw;
                A += pw * f3(co.x, co.y, co.z);
                Z += pw * dot(p - camPos, back);
                const float3 gr = gradient_at(s.vol, p);
                const float g2 = dot(gr, gr);
                if (g2 > 0.f) {
                    float3 n = gr * rsqrtf(g2);
                    if (dot(n, ray.dir) > 0.f) n = -n;
                    N += pw * n;
                }
                T += T * em;
                if (T < 1e-3f) break;
            }
        }
    const size_t o = (size_t)y * c.imageW + x;
    if (alpha > 0.f) {
        const float ia = 1.f / alpha;
        const float n2 = dot(N, N);
        const float3 n = n2 > 0.f ? N * rsqrtf(n2) : f3(0.f);
        albedoCoverage[o] = make_float4(A.x * ia, A.y * ia, A.z * ia, alpha * inv * inv);
        normalDepth[o] = make_float4(n.x, n.y, n.z, Z * ia);
    } else {
        albedoCoverage[o] = make_float4(0.f, 0.f, 0.f, 0.f);
        normalDepth[o] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

SVR_DEV float luminance(float r, float g, float b) { return 0.2126f * r + 0.7152f * g + 0.0722f * b; }

// m = alpha albedo + (1 - alpha) per channel, at least 1e-3
SVR_DEV float3 modulation(float4 ac)
{
    return f3(fmaxf(fmaf(ac.w, ac.x, 1.f - ac.w), 1e-3f), fmaxf(fmaf(ac.w, ac.y, 1.f - ac.w), 1e-3f), fmaxf(fmaf(ac.w, ac.z, 1.f - ac.w), 1e-3f));
}

// Var = (l(even / m) - l(odd / m))^2 / 4, +inf where a half is empty
SVR_DEV float half_variance(const float4* __restrict__ sum, const float4* __restrict__ half, const float4* __restrict__ ac, uint32_t i)
{
    const float4 s = __ldg(sum + i), hs = __ldg(half + i);
    const float we = s.w - hs.w;
    if (!(hs.w > 0.f) || !(we > 0.f)) return __int_as_float(0x7f800000);
    const float3 m = modulation(__ldg(ac + i));
    const float le = luminance((s.x - hs.x) / (we * m.x), (s.y - hs.y) / (we * m.y), (s.z - hs.z) / (we * m.z));
    const float lo = luminance(hs.x / (hs.w * m.x), hs.y / (hs.w * m.y), hs.z / (hs.w * m.z));
    return 0.25f * (le - lo) * (le - lo);
}

// Demodulation and the variance's 3 x 3 binomial prefilter (coordinates clamped): out = (c / m, Var).  Blocks of 32 x 8
// pixels; the variance of the block and its one-pixel rim goes through shared memory.
__global__ void __launch_bounds__(256) denoise_prep_kernel(const float4* __restrict__ sum, const float4* __restrict__ half, const float4* __restrict__ ac,
                                                           float4* __restrict__ out, uint32_t W, uint32_t H)
{
    __shared__ float v[10][34];
    const int x0 = (int)(blockIdx.x * 32u) - 1, y0 = (int)(blockIdx.y * 8u) - 1;
    for (uint32_t t = threadIdx.y * 32u + threadIdx.x; t < 10u * 34u; t += 256u) {
        const int ty = (int)(t / 34u), tx = (int)(t % 34u);
        const uint32_t x = (uint32_t)min(max(x0 + tx, 0), (int)W - 1), y = (uint32_t)min(max(y0 + ty, 0), (int)H - 1);
        v[ty][tx] = half_variance(sum, half, ac, y * W + x);
    }
    __syncthreads();
    const uint32_t x = blockIdx.x * 32u + threadIdx.x, y = blockIdx.y * 8u + threadIdx.y;
    if (x >= W || y >= H) return;
    const float b[3] = {0.25f, 0.5f, 0.25f};
    float var = 0.f;
#pragma unroll
    for (int j = 0; j < 3; ++j)
#pragma unroll
        for (int i = 0; i < 3; ++i) var += b[j] * b[i] * v[threadIdx.y + j][threadIdx.x + i];
    const uint32_t o = y * W + x;
    const float4 s = __ldg(sum + o);
    const float invW = s.w > 0.f ? 1.f / s.w : 0.f;  // resolve_kernel's mean
    const float3 m = modulation(__ldg(ac + o));
    out[o] = make_float4(s.x * invW / m.x, s.y * invW / m.y, s.z * invW / m.z, var);
}

struct DenoiseStops {
    float sigmaL, sigmaN, sigmaZ, invSigmaA;
    float pixelAngle;  // 2 tan(fovx / 2) / (imageH - 1): one pixel's height per unit depth
};

// One a-trous iteration at step s: 5 x 5 B3-spline taps at p + s (dx, dy), each weighted by the four stops; taps outside
// the image are dropped and the weights renormalised.  e' = e_p + sum w (e_q - e_p) / sum w (exactly e_p where every
// other tap has weight 0 or the same value), Var' = sum w^2 Var_q / (sum w)^2.  The last iteration remodulates and
// writes hdr / img as resolve_kernel does instead of `out`.  Blocks of 32 x 8 pixels, taps read through the read-only path.
__global__ void __launch_bounds__(256) denoise_iter_kernel(const float4* __restrict__ in, float4* __restrict__ out, const float4* __restrict__ ac,
                                                           const float4* __restrict__ nd, uint32_t W, uint32_t H, int step, DenoiseStops k,
                                                           float* __restrict__ hdr, uint32_t* __restrict__ img, float exposure)
{
    const int x = (int)(blockIdx.x * 32u + threadIdx.x), y = (int)(blockIdx.y * 8u + threadIdx.y);
    if (x >= (int)W || y >= (int)H) return;
    const float hk[5] = {1.f / 16.f, 0.25f, 0.375f, 0.25f, 1.f / 16.f};
    const uint32_t o = (uint32_t)y * W + (uint32_t)x;
    const float4 cp = __ldg(in + o), np = __ldg(nd + o);
    const float ap = __ldg(&ac[o].w);
    const float lp = luminance(cp.x, cp.y, cp.z);
    const float lumDen = k.sigmaL * sqrtf(cp.w) + 1e-10f;
    const float zDen = k.sigmaZ * (float)step * (np.w * k.pixelAngle) + 1e-10f;
    const bool np0 = np.x == 0.f && np.y == 0.f && np.z == 0.f;
    float sw = 0.f, sv = 0.f;
    float3 acc = f3(0.f);
#pragma unroll
    for (int dy = -2; dy <= 2; ++dy) {
        const int yy = y + step * dy;
        if (yy < 0 || yy >= (int)H) continue;
#pragma unroll
        for (int dx = -2; dx <= 2; ++dx) {
            const int xx = x + step * dx;
            if (xx < 0 || xx >= (int)W) continue;
            const uint32_t q = (uint32_t)yy * W + (uint32_t)xx;
            const float4 cq = __ldg(in + q), nq = __ldg(nd + q);
            const float aq = __ldg(&ac[q].w);
            float wn = 1.f;
            if (k.sigmaN > 0.f) {
                const bool nq0 = nq.x == 0.f && nq.y == 0.f && nq.z == 0.f;
                if (np0 != nq0) wn = 0.f;
                else if (!np0) {
                    const float d = np.x * nq.x + np.y * nq.y + np.z * nq.z;
                    wn = d > 0.f ? __powf(d, k.sigmaN) : 0.f;
                }
            }
            const float e = fabsf(lp - luminance(cq.x, cq.y, cq.z)) / lumDen + fabsf(np.w - nq.w) / zDen + fabsf(ap - aq) * k.invSigmaA;
            const float w = hk[dy + 2] * hk[dx + 2] * wn * __expf(-e);
            if (w > 0.f) {  // (a dropped tap's variance may be +inf: it must not enter as 0 * inf)
                sw += w;
                acc += w * f3(cq.x - cp.x, cq.y - cp.y, cq.z - cp.z);
                sv += w * (w * cq.w);  // (not (w * w) * Var: w * w may flush to 0, and 0 * inf is NaN)
            }
        }
    }
    const float inv = 1.f / sw;
    const float3 e = f3(cp.x, cp.y, cp.z) + acc * inv;
    if (!hdr && !img) {
        out[o] = make_float4(e.x, e.y, e.z, sv * inv * inv);
        return;
    }
    const float3 v = modulation(__ldg(ac + o)) * e;
    if (hdr) {
        hdr[3 * (size_t)o + 0] = v.x;
        hdr[3 * (size_t)o + 1] = v.y;
        hdr[3 * (size_t)o + 2] = v.z;
    }
    if (img) {
        const float3 l = tone_map(v, exposure);
        img[o] = pack_u8x4(l.x * 255.f, l.y * 255.f, l.z * 255.f, 255.f);
    }
}

// sum = even + odd, component by component: the full sums of a progressive render whose frames went into two halves by parity
__global__ void __launch_bounds__(256) sum_halves_kernel(const float4* __restrict__ even, const float4* __restrict__ odd, float4* __restrict__ sum,
                                                         uint32_t n)
{
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    if (i >= n) return;
    const float4 e = __ldg(even + i), o = __ldg(odd + i);
    sum[i] = make_float4(e.x + o.x, e.y + o.y, e.z + o.z, e.w + o.w);
}

}  // namespace

int check_denoise_params(const char* who, const svr_denoise_params* paramsOrNull, svr_denoise_params* out)
{
    svr_denoise_params p;
    if (paramsOrNull) p = *paramsOrNull;
    else svr_denoise_defaults(&p);
    const char* err = nullptr;
    if (p.iterations > 8u) err = "iterations above 8";
    else if (!(p.sigmaLuminance > 0.f) || !std::isfinite(p.sigmaLuminance) || !(p.sigmaDepth > 0.f) || !std::isfinite(p.sigmaDepth) ||
             !(p.sigmaCoverage > 0.f) || !std::isfinite(p.sigmaCoverage))
        err = "sigmaLuminance, sigmaDepth and sigmaCoverage must be positive and finite";
    else if (!(p.sigmaNormal >= 0.f) || !std::isfinite(p.sigmaNormal)) err = "sigmaNormal must be >= 0 and finite";
    if (err) {
        char msg[192];
        snprintf(msg, sizeof(msg), "%s: %s", who, err);
        return fail_msg(msg);
    }
    *out = p;
    return 0;
}

namespace {

// The filter for checked parameters and a camera of W x H pixels, ping-ponging between the two halves of st.dev.denoise.  `sum`
// may be the second half: the prep pass reads it before the first iteration writes there.
int run_filter(uint32_t* img, float* hdr, const float4* sum, const float4* half, const float4* ac, const float4* nd, const svr_denoise_params& p)
{
    HostState& st = state();
    const uint32_t W = st.scene.cam.imageW, H = st.scene.cam.imageH;
    if (p.iterations == 0u) return svr_pathtracer_resolve((svr_u8vec4*)img, (svr_vec3*)hdr, (const svr_vec4*)sum);  // the identity, bit for bit

    hdr_written_outside(st.dev, hdr, false);  // as svr_pathtracer_resolve
    SVR_TRY(st.dev.denoise.reserve(2 * (size_t)W * H));
    float4* const buf[2] = {st.dev.denoise.p, st.dev.denoise.p + (size_t)W * H};
    const dim3 blocks((W + 31u) / 32u, (H + 7u) / 8u), threads(32, 8);
    denoise_prep_kernel<<<blocks, threads, 0, st.stream>>>(sum, half, ac, buf[0], W, H);
    count_launch();
    SVR_TRY(cudaGetLastError());
    DenoiseStops k;
    k.sigmaL = p.sigmaLuminance;
    k.sigmaN = p.sigmaNormal;
    k.sigmaZ = p.sigmaDepth;
    k.invSigmaA = 1.f / p.sigmaCoverage;
    k.pixelAngle = 2.f * st.scene.cam.tanFovxOverTwo / ((float)H - 1.f);
    for (uint32_t i = 0; i < p.iterations; ++i) {
        const bool last = i + 1u == p.iterations;
        denoise_iter_kernel<<<blocks, threads, 0, st.stream>>>(buf[i & 1u], buf[(i + 1u) & 1u], ac, nd, W, H, 1 << i, k,
                                                               last ? hdr : nullptr, last ? img : nullptr, st.scene.cam.exposure);
        count_launch();
        SVR_TRY(cudaGetLastError());
    }
    return 0;
}

}  // namespace

// st.dev.prog (even sum, odd sum, albedoCoverage, normalDepth) and the filter's buffers; on failure the CUDA error is cleared
bool ensure_progressive_buffers(HostState& st, size_t npix)
{
    if (st.dev.prog.cap < 4 * npix) st.dev.progGuideEpoch = 0;  // new memory holds no guides
    if (st.dev.prog.reserve(4 * npix) != cudaSuccess || st.dev.denoise.reserve(2 * npix) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return true;
}

// Guides made with SVR_OPT_PT_DENOISE rays before frame 16 and with 16 from there on, kept while the scene epoch stays where it
// was after the frame that made them; then the filter of (even + odd, odd).  The caller has traced the frame's sample.
int progressive_denoise(uint32_t* img, uint32_t frameNo)
{
    HostState& st = state();
    const uint32_t rays = frameNo >= 16u ? 16u : (uint32_t)st.options[SVR_OPT_PT_DENOISE];
    const uint32_t npix = st.scene.cam.imageW * st.scene.cam.imageH;
    float4* const prog = st.dev.prog.p;
    if (st.dev.progGuideEpoch != st.sceneEpoch || st.dev.progGuideRays != rays) {
        if (int rc = svr_pathtracer_guides((svr_vec4*)(prog + 2 * npix), (svr_vec4*)(prog + 3 * npix), rays)) return rc;
        st.dev.progGuideRays = rays;
    }
    sum_halves_kernel<<<(npix + 255u) / 256u, 256, 0, st.stream>>>(prog, prog + npix, st.dev.denoise.p + npix, npix);
    count_launch();
    SVR_TRY(cudaGetLastError());
    if (int rc = run_filter(img, nullptr, st.dev.denoise.p + npix, prog + npix, prog + 2 * npix, prog + 3 * npix, st.progParams)) return rc;
    st.dev.progGuideEpoch = st.sceneEpoch;  // after the frame's launches: refreshing the majorants moves the epoch
    return 0;
}

}  // namespace svr

using namespace svr;

extern "C" int svr_pathtracer_guides(svr_vec4* albedoCoverage, svr_vec4* normalDepth, uint32_t raysPerPixel)
{
    HostState& st = state();
    if (!albedoCoverage || !normalDepth) return fail_msg("svr_pathtracer_guides: albedoCoverage and normalDepth must not be null");
    if (raysPerPixel != 1u && raysPerPixel != 4u && raysPerPixel != 16u) return fail_msg("svr_pathtracer_guides: raysPerPixel must be 1, 4 or 16");
    DevScene sc = st.scene;
    if (!sc.vol.tex || !sc.tf.tex) return fail_msg("svr_pathtracer_guides: setup_volume / setup_transferfunction not called");
    if (sc.cam.imageW == 0 || sc.cam.imageH == 0) return fail_msg("svr_pathtracer_guides: setup_camera not called");
    if (int rc = ensure_grid(&sc, false)) return rc;
    const int side = raysPerPixel == 1u ? 1 : (raysPerPixel == 4u ? 2 : 4);
    const dim3 grid((sc.cam.imageW + 15u) / 16u, (sc.cam.imageH + 7u) / 8u);
    guides_kernel<<<grid, 128, 0, st.stream>>>(sc, (float4*)albedoCoverage, (float4*)normalDepth, side);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

// The single source of the filter's defaults (DESIGN.md section 7f: the sweep they were chosen from)
extern "C" int svr_denoise_defaults(svr_denoise_params* out)
{
    if (!out) return fail_msg("svr_denoise_defaults: out is null");
    out->iterations = 5;
    out->sigmaLuminance = 4.f;
    out->sigmaNormal = 128.f;
    out->sigmaDepth = 1.f;
    out->sigmaCoverage = 0.1f;
    return 0;
}

extern "C" int svr_pathtracer_denoise(svr_u8vec4* imgOrNull, svr_vec3* hdrOutOrNull, const svr_vec4* sum, const svr_vec4* halfSum,
                                      const svr_vec4* albedoCoverage, const svr_vec4* normalDepth, const svr_denoise_params* paramsOrNull)
{
    HostState& st = state();
    if (!sum || !halfSum) return fail_msg("svr_pathtracer_denoise: sum and halfSum must not be null");
    if (!albedoCoverage || !normalDepth) return fail_msg("svr_pathtracer_denoise: the guides (albedoCoverage, normalDepth) must not be null");
    if (!imgOrNull && !hdrOutOrNull) return fail_msg("svr_pathtracer_denoise: img and hdrOut are both null");
    svr_denoise_params p;
    if (int rc = check_denoise_params("svr_pathtracer_denoise", paramsOrNull, &p)) return rc;
    if (!st.scene.cam.imageW || !st.scene.cam.imageH) return fail_msg("svr_pathtracer_denoise: setup_camera not called");
    return run_filter((uint32_t*)imgOrNull, (float*)hdrOutOrNull, (const float4*)sum, (const float4*)halfSum, (const float4*)albedoCoverage,
                      (const float4*)normalDepth, p);
}

extern "C" int svr_pathtracer_set_denoise_params(const svr_denoise_params* paramsOrNull)
{
    svr_denoise_params p;
    if (int rc = check_denoise_params("svr_pathtracer_set_denoise_params", paramsOrNull, &p)) return rc;
    state().progParams = p;  // the guides do not depend on it: the scene epoch stays
    return 0;
}
