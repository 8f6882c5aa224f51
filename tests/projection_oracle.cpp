/*
 * TEST INFRASTRUCTURE -- not product code.  CPU restatement of svr_render_projection (include/svr_render.h) on the CPU
 * oracle's own ray generation (camera_generate_ray_rc), box intersection (vol_intersect) and software texture filter (tex3d:
 * 8-bit weights, border addressing), in the oracle's IEEE, no-contraction style.  It does no skipping.  The oracle's
 * translation unit is included, not copied, so the restatement uses exactly the functions the other parity tests hold to
 * the reference's outputs.  Built on first use by tests/_projection_oracle.py.
 */
#include "../oracle/svr_oracle.cpp"

extern "C" {

/* mode: 0 max, 1 min, 2 mean.  Rows [y0, y1); value (float per pixel) and u8 (rgba per pixel) may each be NULL. */
void svr_oracle_project(const svr_oracle_scene* scene, int mode, float stepSize, float windowC, float windowW, uint32_t strideW,
                        uint32_t y0, uint32_t y1, float* value, uint8_t* u8)
{
    const uint32_t W = scene->camera.imageW;
#pragma omp parallel for schedule(dynamic, 1) num_threads(svr_oracle_threads())
    for (int64_t idy = (int64_t)y0; idy < (int64_t)y1; ++idy) {
        for (uint32_t idx = 0; idx < W; ++idx) {
            Ray ray;
            camera_generate_ray_rc(scene->camera, idx, (uint32_t)idy, &ray);
            float P = 0.f, tNear, tFar;
            if (vol_intersect(scene, ray, &tNear, &tFar)) {
                const float h = stepSize * 0.5f;
                const float t0 = fmaxf(tNear, 0.f);
                const uint32_t K = tFar > t0 ? (uint32_t)floorf((tFar - t0) / h + 0.5f) : 0u;
                float acc = mode == 0 ? -INFINITY : (mode == 1 ? INFINITY : 0.f);
                for (uint32_t k = 0; k < K; ++k) {
                    const float t = t0 + ((float)k + 0.5f) * h;
                    const float v = vol_intensity(scene, ray.orig + t * ray.dir);
                    acc = mode == 0 ? fmaxf(acc, v) : (mode == 1 ? fminf(acc, v) : acc + v);
                }
                if (K > 0) P = mode == 2 ? acc / (float)K : acc;
            }
            const size_t offset = (size_t)idy * strideW + idx;
            if (value) value[offset] = P;
            if (u8) {
                const float g = fminf(fmaxf((P - (windowC - 0.5f * windowW)) / windowW, 0.f), 1.f);
                const uint8_t q = (uint8_t)(int)(255.f * g);
                u8[4 * offset + 0] = q;
                u8[4 * offset + 1] = q;
                u8[4 * offset + 2] = q;
                u8[4 * offset + 3] = 255;
            }
        }
    }
}

}  // extern "C"
