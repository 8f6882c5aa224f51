/*
 * TEST INFRASTRUCTURE -- not product code.  CPU restatement of svr_render_curved's pixel rule (include/svr_render.h) on the CPU
 * oracle's software texture filter (tex3d: 8-bit weights, border addressing), in the oracle's IEEE, no-contraction style.  It
 * takes the frame table from svr_curve_frames (the frame rule is checked on its own against a numpy restatement), computes
 * (cos, sin) in double as the host does, does no skipping and tests every sample of the slab for inclusion.  The oracle's
 * translation unit is included, not copied.  Built on first use by tests/_curved_oracle.py.
 */
#include "../oracle/svr_oracle.cpp"
#include "../include/svr_render.h"

extern "C" {

/* frames: 4 svr_vec4 per station (svr_curve_frames) of the layout's stations (imageH straightened, count cross-sections);
 * value (count * imageH * imageW floats) and u8 (rgba per pixel) may each be NULL. */
void svr_oracle_curved(const svr_oracle_scene* scene, const svr_curved_params* p, const svr_vec4* frames, float* value, uint8_t* u8)
{
    const svr_volume& v = scene->volume;
    const bool crossLayout = p->layout == SVR_CURVED_CROSS;
    const float h = p->thickness > 0.f ? p->sampleSpacing : 0.f;
    const uint32_t K = p->thickness > 0.f ? (uint32_t)fmaxf(1.f, floorf(p->thickness / h + 0.5f)) : 1u;
    const float t0 = -((float)K * h) * 0.5f;
    const V3 cmin = mk(v.bbox.vmin) * mk(-v.x_clip.x, -v.y_clip.x, -v.z_clip.x);
    const V3 cmax = mk(v.bbox.vmax) * mk(v.x_clip.y, v.y_clip.y, v.z_clip.y);
    const uint32_t W = p->imageW, H = p->imageH;
    const float ps = p->pixelSpacing;
#pragma omp parallel for schedule(dynamic, 1) num_threads(svr_oracle_threads())
    for (int64_t row = 0; row < (int64_t)p->count * H; ++row) {
        const uint32_t j = (uint32_t)(row / H), y = (uint32_t)(row % H);
        const svr_vec4* f = frames + 4 * (size_t)(crossLayout ? j : y);
        const double theta = (double)p->angle0 + (crossLayout ? 0.0 : (double)j * (double)p->angleStep);
        const float cs = (float)cos(theta), sn = (float)sin(theta);
        const V3 c = mk(f[0].x, f[0].y, f[0].z), t = mk(f[1].x, f[1].y, f[1].z), r = mk(f[2].x, f[2].y, f[2].z), b = mk(f[3].x, f[3].y, f[3].z);
        const V3 a = cs * r + sn * b, e = cs * b - sn * r;
        for (uint32_t x = 0; x < W; ++x) {
            float acc = p->mode == 0 ? -INFINITY : (p->mode == 1 ? INFINITY : 0.f);
            uint32_t taken = 0;
            if (f[0].w != 0.f) {
                const float fx = ((float)x + 0.5f) - 0.5f * (float)W, fy = ((float)y + 0.5f) - 0.5f * (float)H;
                const V3 pc = crossLayout ? c + (fx * ps) * a + (fy * ps) * e : c + (fx * ps) * a;
                const V3 n = crossLayout ? t : e;
                for (uint32_t k = 0; k < K; ++k) {
                    const V3 xk = pc + (t0 + ((float)k + 0.5f) * h) * n;
                    if (!(xk.x >= cmin.x && xk.y >= cmin.y && xk.z >= cmin.z && xk.x <= cmax.x && xk.y <= cmax.y && xk.z <= cmax.z)) continue;
                    const float s = vol_intensity(scene, xk);
                    acc = p->mode == 0 ? fmaxf(acc, s) : (p->mode == 1 ? fminf(acc, s) : acc + s);
                    ++taken;
                }
            }
            const float P = taken == 0 ? 0.f : (p->mode == 2 ? acc / (float)taken : acc);
            const size_t offset = ((size_t)j * H + y) * W + x;
            if (value) value[offset] = P;
            if (u8) {
                const float g = fminf(fmaxf((P - (p->windowCenter - 0.5f * p->windowWidth)) / p->windowWidth, 0.f), 1.f);
                const uint8_t q = taken ? (uint8_t)(int)(255.f * g) : 0;
                u8[4 * offset + 0] = q;
                u8[4 * offset + 1] = q;
                u8[4 * offset + 2] = q;
                u8[4 * offset + 3] = taken ? 255 : 0;
            }
        }
    }
}

}  // extern "C"
