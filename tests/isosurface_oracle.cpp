/*
 * TEST INFRASTRUCTURE -- not product code.  CPU restatement of svr_render_isosurface (include/svr_render.h) on the CPU oracle's
 * own ray generation (camera_generate_ray_rc), box intersection (vol_intersect), software texture filter (tex3d: 8-bit
 * weights, border addressing) and gradient (vol_gradient), in the oracle's IEEE, no-contraction style.  It does no skipping:
 * every sample is taken in k order until the first hit.  The oracle's translation unit is included, not copied.  Built on first
 * use by tests/_isosurface_oracle.py.
 */
#include "../oracle/svr_oracle.cpp"

extern "C" {

/* Rows [y0, y1); surface (float4 per pixel: normal, depth) and u8 (rgba per pixel) may each be NULL. */
void svr_oracle_isosurface(const svr_oracle_scene* scene, float isoValue, float stepSize, const float* color, uint32_t strideW,
                           uint32_t y0, uint32_t y1, float* surface, uint8_t* u8)
{
    const uint32_t W = scene->camera.imageW;
    const V3 camPos = mk(scene->camera.pos), back = -mk(scene->camera.w);
#pragma omp parallel for schedule(dynamic, 1) num_threads(svr_oracle_threads())
    for (int64_t idy = (int64_t)y0; idy < (int64_t)y1; ++idy) {
        for (uint32_t idx = 0; idx < W; ++idx) {
            Ray ray;
            camera_generate_ray_rc(scene->camera, idx, (uint32_t)idy, &ray);
            float tNear, tFar;
            float rgba[4] = {0.f, 0.f, 0.f, 0.f};
            float surf[4] = {0.f, 0.f, 0.f, INFINITY};
            if (vol_intersect(scene, ray, &tNear, &tFar)) {
                const float h = stepSize * 0.5f;
                const float t0 = fmaxf(tNear, 0.f);
                const uint32_t K = tFar > t0 ? (uint32_t)floorf((tFar - t0) / h + 0.5f) : 0u;
                auto t_of = [&](uint32_t k) { return t0 + ((float)k + 0.5f) * h; };
                auto value = [&](float t) { return vol_intensity(scene, ray.orig + t * ray.dir); };
                uint32_t hit = K;
                float vHit = 0.f;
                for (uint32_t k = 0; k < K; ++k) {
                    const float v = value(t_of(k));
                    if (v >= isoValue) {
                        hit = k;
                        vHit = v;
                        break;
                    }
                }
                if (hit < K) {
                    float tHit = t_of(hit);
                    if (hit > 0) {
                        float lo = t_of(hit - 1), hi = tHit, vLo = value(lo), vHi = vHit;
                        for (int i = 0; i < 4; ++i) {
                            const float m = (lo + hi) * 0.5f;
                            const float vm = value(m);
                            if (vm >= isoValue) {
                                hi = m;
                                vHi = vm;
                            } else {
                                lo = m;
                                vLo = vm;
                            }
                        }
                        tHit = lo + (hi - lo) * (isoValue - vLo) / (vHi - vLo);
                    }
                    const V3 x = ray.orig + tHit * ray.dir;
                    const V3 g = vol_gradient(scene, x);
                    const float gm = sqrtf(dot(g, g));
                    V3 n = mk(0.f, 0.f, 0.f);
                    float cosTerm = 1.f, specularTerm = 0.f;
                    if ((double)gm > 1e-3) {
                        n = normalize(g);
                        if (dot(n, ray.dir) > 0.f) n = -n;
                        cosTerm = fabsf(dot(n, normalize(camPos - x)));
                        specularTerm = powf(cosTerm, 30.f);
                    }
                    for (int c = 0; c < 3; ++c) rgba[c] = fminf(color[c] * cosTerm * 0.8f + specularTerm * 0.2f, 1.f);
                    rgba[3] = 1.f;
                    surf[0] = n.x;
                    surf[1] = n.y;
                    surf[2] = n.z;
                    surf[3] = dot(x - camPos, back);
                }
            }
            const size_t offset = (size_t)idy * strideW + idx;
            if (surface)
                for (int c = 0; c < 4; ++c) surface[4 * offset + c] = surf[c];
            if (u8)
                for (int c = 0; c < 4; ++c) u8[4 * offset + c] = (uint8_t)(int)(rgba[c] * 255.f);
        }
    }
}

}  // extern "C"
