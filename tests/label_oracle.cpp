/*
 * TEST INFRASTRUCTURE -- not product code.  CPU restatement of svr_render_labels and svr_render_label_slices
 * (include/svr_render.h) on the CPU oracle's own ray generation (camera_generate_ray_rc) and box intersection (vol_intersect),
 * in the oracle's IEEE, no-contraction style.  The scene's voxels are the u8 label ids (x fastest); a voxel outside the volume
 * reads 0.  It does no skipping: every sample is taken in k order until the first hit.  The oracle's translation unit is
 * included, not copied.  Built on first use by tests/_label_oracle.py.
 */
#include "../oracle/svr_oracle.cpp"
#include "../include/svr_render.h"

namespace {

uint32_t label_voxel(const svr_oracle_scene* s, int i, int j, int k)
{
    if (i < 0 || j < 0 || k < 0 || i >= (int)s->nx || j >= (int)s->ny || k >= (int)s->nz) return 0;
    return ((const uint8_t*)s->voxels)[((size_t)k * s->ny + j) * s->nx + i];
}

bool visible(const float* table, uint32_t l) { return l != 0 && table[4 * l + 3] > 0.f; }

float lerp(float a, float b, float f) { return (1.f - f) * a + f * b; }

/* the 8 corners around x: f, vis and labels, corner c = x + 2 y + 4 z offsets */
struct Corners {
    float f[3];
    float v[8];
    uint32_t lab[8];
};

Corners corners(const svr_oracle_scene* s, const float* table, V3 x)
{
    const svr_volume& vol = s->volume;
    const V3 tc = (x - mk(vol.bbox.vmin)) * mk(vol.bbox.invSize);
    const float u[3] = {tc.x * (float)s->nx - 0.5f, tc.y * (float)s->ny - 0.5f, tc.z * (float)s->nz - 0.5f};
    int i[3];
    Corners c;
    for (int a = 0; a < 3; ++a) {
        const float fl = floorf(u[a]);
        i[a] = (int)fl;
        c.f[a] = u[a] - fl;
    }
    for (int n = 0; n < 8; ++n) {
        c.lab[n] = label_voxel(s, i[0] + (n & 1), i[1] + ((n >> 1) & 1), i[2] + (n >> 2));
        c.v[n] = visible(table, c.lab[n]) ? 1.f : 0.f;
    }
    return c;
}

float indicator(const svr_oracle_scene* s, const float* table, V3 x)
{
    const Corners c = corners(s, table, x);
    const float y0 = lerp(lerp(c.v[0], c.v[1], c.f[0]), lerp(c.v[2], c.v[3], c.f[0]), c.f[1]);
    const float y1 = lerp(lerp(c.v[4], c.v[5], c.f[0]), lerp(c.v[6], c.v[7], c.f[0]), c.f[1]);
    return lerp(y0, y1, c.f[2]);
}

uint32_t pick(const svr_oracle_scene* s, const float* table, V3 x)
{
    const Corners c = corners(s, table, x);
    float w[8];
    for (int n = 0; n < 8; ++n) {
        const float wx = n & 1 ? c.f[0] : 1.f - c.f[0], wy = (n >> 1) & 1 ? c.f[1] : 1.f - c.f[1], wz = n >> 2 ? c.f[2] : 1.f - c.f[2];
        w[n] = c.v[n] != 0.f ? (wx * wy) * wz : 0.f;
    }
    uint32_t best = 0;
    float bestW = -1.f;
    for (int a = 0; a < 8; ++a) {
        if (c.v[a] == 0.f) continue;
        float sum = 0.f;
        for (int b = 0; b < 8; ++b)
            if (c.lab[b] == c.lab[a]) sum += w[b];
        if (sum > bestW || (sum == bestW && c.lab[a] < best)) {
            best = c.lab[a];
            bestW = sum;
        }
    }
    return best;
}

V3 gradient(const svr_oracle_scene* s, const float* table, V3 x)
{
    const Corners c = corners(s, table, x);
    const float* v = c.v;
    const float* f = c.f;
    const float dx = lerp(lerp(v[1] - v[0], v[3] - v[2], f[1]), lerp(v[5] - v[4], v[7] - v[6], f[1]), f[2]);
    const float dy = lerp(lerp(v[2] - v[0], v[3] - v[1], f[0]), lerp(v[6] - v[4], v[7] - v[5], f[0]), f[2]);
    const float dz = lerp(lerp(v[4] - v[0], v[5] - v[1], f[0]), lerp(v[6] - v[2], v[7] - v[3], f[0]), f[1]);
    const svr_volume& vol = s->volume;
    return mk(dx * ((float)s->nx * vol.bbox.invSize.x), dy * ((float)s->ny * vol.bbox.invSize.y), dz * ((float)s->nz * vol.bbox.invSize.z));
}

uint32_t slice_label(const svr_oracle_scene* s, const svr_slice_params* p, V3 center, V3 U, V3 Vv, V3 Wv, V3 cmin, V3 cmax, uint32_t x,
                     uint32_t y, uint32_t j)
{
    const float fx = ((float)x + 0.5f) - 0.5f * (float)p->imageW, fy = ((float)y + 0.5f) - 0.5f * (float)p->imageH;
    const V3 c = center + fx * U + fy * Vv + (float)j * Wv;
    if (!(c.x >= cmin.x && c.y >= cmin.y && c.z >= cmin.z && c.x <= cmax.x && c.y <= cmax.y && c.z <= cmax.z)) return 0;
    const svr_volume& vol = s->volume;
    const V3 tc = (c - mk(vol.bbox.vmin)) * mk(vol.bbox.invSize);
    return label_voxel(s, (int)floorf(tc.x * (float)s->nx), (int)floorf(tc.y * (float)s->ny), (int)floorf(tc.z * (float)s->nz));
}

}  // namespace

extern "C" {

/* Rows [y0, y1) of svr_render_labels; table: 256 x rgba.  surface (float4 per pixel), u8 (rgba per pixel) and label (one byte
 * per pixel) may each be NULL. */
void svr_oracle_labels(const svr_oracle_scene* scene, const float* table, float stepSize, uint32_t strideW, uint32_t y0, uint32_t y1,
                       float* surface, uint8_t* u8, uint8_t* label)
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
            uint32_t lab = 0;
            if (vol_intersect(scene, ray, &tNear, &tFar)) {
                const float h = stepSize * 0.5f;
                const float t0 = fmaxf(tNear, 0.f);
                const uint32_t K = tFar > t0 ? (uint32_t)floorf((tFar - t0) / h + 0.5f) : 0u;
                auto t_of = [&](uint32_t k) { return t0 + ((float)k + 0.5f) * h; };
                auto value = [&](float t) { return indicator(scene, table, ray.orig + t * ray.dir); };
                uint32_t hit = K;
                float vHit = 0.f;
                for (uint32_t k = 0; k < K; ++k) {
                    const float v = value(t_of(k));
                    if (v >= 0.5f) {
                        hit = k;
                        vHit = v;
                        break;
                    }
                }
                if (hit < K) {
                    float tHit = t_of(hit), tHi = tHit;
                    if (hit > 0) {
                        float lo = t_of(hit - 1), hi = tHit, vLo = value(lo), vHi = vHit;
                        for (int i = 0; i < 4; ++i) {
                            const float m = (lo + hi) * 0.5f;
                            const float vm = value(m);
                            if (vm >= 0.5f) {
                                hi = m;
                                vHi = vm;
                            } else {
                                lo = m;
                                vLo = vm;
                            }
                        }
                        tHit = lo + (hi - lo) * (0.5f - vLo) / (vHi - vLo);
                        tHi = hi;
                    }
                    lab = pick(scene, table, ray.orig + tHi * ray.dir);
                    const V3 x = ray.orig + tHit * ray.dir;
                    const V3 g = gradient(scene, table, x);
                    V3 n = mk(0.f, 0.f, 0.f);
                    float cosTerm = 1.f, specularTerm = 0.f;
                    if (dot(g, g) > 0.f) {
                        n = normalize(g);
                        if (dot(n, ray.dir) > 0.f) n = -n;
                        cosTerm = fabsf(dot(n, normalize(camPos - x)));
                        specularTerm = powf(cosTerm, 30.f);
                    }
                    for (int c = 0; c < 3; ++c) rgba[c] = fminf(table[4 * lab + c] * cosTerm * 0.8f + specularTerm * 0.2f, 1.f);
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
            if (label) label[offset] = (uint8_t)lab;
        }
    }
}

/* svr_render_label_slices: img (count * H * W rgba, composited in place) and label (count * H * W bytes) may each be NULL. */
void svr_oracle_label_slices(const svr_oracle_scene* scene, const svr_slice_params* p, const float* table, int outline, uint8_t* img,
                             uint8_t* label)
{
    const svr_volume& v = scene->volume;
    const V3 U = mk(p->axisU[0], p->axisU[1], p->axisU[2]), Vv = mk(p->axisV[0], p->axisV[1], p->axisV[2]);
    const V3 Wv = p->count > 1 ? mk(p->axisW[0], p->axisW[1], p->axisW[2]) : mk(0.f, 0.f, 0.f);
    const V3 center = mk(p->center[0], p->center[1], p->center[2]);
    const V3 cmin = mk(v.bbox.vmin) * mk(-v.x_clip.x, -v.y_clip.x, -v.z_clip.x);
    const V3 cmax = mk(v.bbox.vmax) * mk(v.x_clip.y, v.y_clip.y, v.z_clip.y);
    const uint32_t W = p->imageW, H = p->imageH;
    auto L = [&](uint32_t x, uint32_t y, uint32_t j) { return slice_label(scene, p, center, U, Vv, Wv, cmin, cmax, x, y, j); };
#pragma omp parallel for schedule(dynamic, 1) num_threads(svr_oracle_threads())
    for (int64_t row = 0; row < (int64_t)p->count * H; ++row) {
        const uint32_t j = (uint32_t)(row / H), y = (uint32_t)(row % H);
        for (uint32_t x = 0; x < W; ++x) {
            const uint32_t l = L(x, y, j);
            const size_t offset = ((size_t)j * H + y) * W + x;
            if (label) label[offset] = (uint8_t)l;
            if (!img || !visible(table, l)) continue;
            const bool edge = outline && ((x > 0 && L(x - 1, y, j) != l) || (x + 1 < W && L(x + 1, y, j) != l) ||
                                          (y > 0 && L(x, y - 1, j) != l) || (y + 1 < H && L(x, y + 1, j) != l));
            const float a = edge ? 1.f : table[4 * l + 3];
            for (int c = 0; c < 3; ++c)
                img[4 * offset + c] = (uint8_t)(uint32_t)(((1.f - a) * (float)img[4 * offset + c] + a * (255.f * table[4 * l + c])) + 0.5f);
            img[4 * offset + 3] = 255;
        }
    }
}

}  // extern "C"
