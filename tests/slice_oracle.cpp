/*
 * TEST INFRASTRUCTURE -- not product code.  CPU restatement of svr_render_slices (include/svr_render.h) on the CPU oracle's
 * software texture filter (tex3d: 8-bit weights, border addressing), in the oracle's IEEE, no-contraction style.  It does no
 * skipping and tests every sample of the slab for inclusion (the kernel binary-searches the included range).  The oracle's
 * translation unit is included, not copied.  Built on first use by tests/_slice_oracle.py.
 */
#include "../oracle/svr_oracle.cpp"
#include "../include/svr_render.h"

extern "C" {

/* value (count * imageH * imageW floats) and u8 (rgba per pixel) may each be NULL. */
void svr_oracle_slices(const svr_oracle_scene* scene, const svr_slice_params* p, float* value, uint8_t* u8)
{
    const svr_volume& v = scene->volume;
    const V3 U = mk(p->axisU[0], p->axisU[1], p->axisU[2]), Vv = mk(p->axisV[0], p->axisV[1], p->axisV[2]);
    const V3 Wv = p->count > 1 ? mk(p->axisW[0], p->axisW[1], p->axisW[2]) : mk(0.f, 0.f, 0.f);
    const V3 center = mk(p->center[0], p->center[1], p->center[2]);
    const V3 nc = cross(U, Vv);
    const V3 n = nc / sqrtf(dot(nc, nc));
    const float h = p->thickness > 0.f ? p->sampleSpacing : 0.f;
    const uint32_t K = p->thickness > 0.f ? (uint32_t)fmaxf(1.f, floorf(p->thickness / h + 0.5f)) : 1u;
    const float t0 = -((float)K * h) * 0.5f;
    const V3 cmin = mk(v.bbox.vmin) * mk(-v.x_clip.x, -v.y_clip.x, -v.z_clip.x);
    const V3 cmax = mk(v.bbox.vmax) * mk(v.x_clip.y, v.y_clip.y, v.z_clip.y);
    const uint32_t W = p->imageW, H = p->imageH;
#pragma omp parallel for schedule(dynamic, 1) num_threads(svr_oracle_threads())
    for (int64_t row = 0; row < (int64_t)p->count * H; ++row) {
        const uint32_t j = (uint32_t)(row / H), y = (uint32_t)(row % H);
        for (uint32_t x = 0; x < W; ++x) {
            const float fx = ((float)x + 0.5f) - 0.5f * (float)W, fy = ((float)y + 0.5f) - 0.5f * (float)H;
            const V3 c = center + fx * U + fy * Vv + (float)j * Wv;
            float acc = p->mode == 0 ? -INFINITY : (p->mode == 1 ? INFINITY : 0.f);
            uint32_t taken = 0;
            for (uint32_t k = 0; k < K; ++k) {
                const V3 xk = c + (t0 + ((float)k + 0.5f) * h) * n;
                if (!(xk.x >= cmin.x && xk.y >= cmin.y && xk.z >= cmin.z && xk.x <= cmax.x && xk.y <= cmax.y && xk.z <= cmax.z)) continue;
                const float s = vol_intensity(scene, xk);
                acc = p->mode == 0 ? fmaxf(acc, s) : (p->mode == 1 ? fminf(acc, s) : acc + s);
                ++taken;
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
