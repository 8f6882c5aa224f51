// svr_env_io.cu -- Radiance RGBE (.hdr) reader and the environment-light builder on top of it
// (include/svr_env_io.h; core/lights/lights.cpp:31-75, which calls stbi_loadf).  Host code.
#include <cmath>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/svr_env_io.h"
#include "svr_state.h"

namespace svr {
namespace {

bool read_line(FILE* f, std::string* out)
{
    out->clear();
    int c;
    while ((c = fgetc(f)) != EOF) {
        if (c == '\n') return true;
        if (out->size() < 1024) out->push_back((char)c);
    }
    return !out->empty();
}

// byte * 2^(e - 136); exponent byte 0 means black
inline void rgbe_to_float(const unsigned char* p, float* out)
{
    if (p[3] != 0) {
        const float f = ldexpf(1.0f, (int)p[3] - (128 + 8));
        out[0] = p[0] * f;
        out[1] = p[1] * f;
        out[2] = p[2] * f;
    } else {
        out[0] = out[1] = out[2] = 0.f;
    }
}

int decode(FILE* f, uint32_t w, uint32_t h, float* out)
{
    const size_t npix = (size_t)w * h;
    std::vector<unsigned char> line((size_t)w * 4);
    auto flat_from = [&](size_t firstPixel, const unsigned char* head) -> int {
        // the whole rest of the picture is uncompressed RGBE quads; `head` (if any) already holds one pixel
        size_t i = firstPixel;
        if (head) {
            rgbe_to_float(head, out + 3 * i);
            ++i;
        }
        unsigned char px[4];
        for (; i < npix; ++i) {
            if (fread(px, 1, 4, f) != 4) return fail_msg("svr_hdr_read: truncated pixel data");
            rgbe_to_float(px, out + 3 * i);
        }
        return 0;
    };
    if (w < 8 || w >= 32768) return flat_from(0, nullptr);
    for (uint32_t y = 0; y < h; ++y) {
        unsigned char hd[4];
        if (fread(hd, 1, 4, f) != 4) return fail_msg("svr_hdr_read: truncated scanline header");
        if (hd[0] != 2 || hd[1] != 2 || (hd[2] & 0x80)) {
            // not a run-length scanline: these four bytes are a pixel, and so is everything after them
            if (y != 0) return fail_msg("svr_hdr_read: mixed flat and run-length scanlines");
            return flat_from(0, hd);
        }
        if ((((uint32_t)hd[2] << 8) | hd[3]) != w) return fail_msg("svr_hdr_read: scanline length differs from the picture width");
        for (int k = 0; k < 4; ++k) {
            uint32_t x = 0;
            while (x < w) {
                int count = fgetc(f);
                if (count == EOF) return fail_msg("svr_hdr_read: truncated run");
                if (count > 128) {
                    int value = fgetc(f);
                    count -= 128;
                    if (value == EOF || x + (uint32_t)count > w) return fail_msg("svr_hdr_read: corrupt run");
                    for (int z = 0; z < count; ++z) line[(size_t)(x++) * 4 + k] = (unsigned char)value;
                } else {
                    if (count == 0 || x + (uint32_t)count > w) return fail_msg("svr_hdr_read: corrupt literal run");
                    for (int z = 0; z < count; ++z) {
                        int value = fgetc(f);
                        if (value == EOF) return fail_msg("svr_hdr_read: truncated literal run");
                        line[(size_t)(x++) * 4 + k] = (unsigned char)value;
                    }
                }
            }
        }
        for (uint32_t x = 0; x < w; ++x) rgbe_to_float(&line[(size_t)x * 4], out + 3 * ((size_t)y * w + x));
    }
    return 0;
}

}  // namespace
}  // namespace svr

using namespace svr;

// Largest accepted picture: 32768 per side and 2^27 pixels (2 GiB as float4), checked before anything is allocated.
static const uint32_t kMaxSide = 32768u;
static const uint64_t kMaxPixels = 1ull << 27;

// One parse of the file: header, size checks, then the pixels into *rgbVec (resized here) or into the caller's
// buffer, which was sized for wantW x wantH.
static int read_hdr(const char* path, std::vector<float>* rgbVec, float* rgbExt, uint32_t wantW, uint32_t wantH, uint32_t* w, uint32_t* h)
{
    FILE* f = fopen(path, "rb");
    if (!f) return fail_msg((std::string("svr_hdr_read: unable to load environment map: ") + path).c_str());
    int rc = 0;
    std::string line;
    bool format = false;
    if (!read_line(f, &line) || (line != "#?RADIANCE" && line != "#?RGBE")) rc = fail_msg("svr_hdr_read: not a Radiance HDR file");
    while (!rc) {
        if (!read_line(f, &line) && feof(f)) {
            rc = fail_msg("svr_hdr_read: header ends before the resolution line");
            break;
        }
        if (line.empty()) break;
        if (line == "FORMAT=32-bit_rle_rgbe") format = true;
    }
    if (!rc && !format) rc = fail_msg("svr_hdr_read: unsupported format (only FORMAT=32-bit_rle_rgbe)");
    if (!rc) {
        unsigned hh = 0, ww = 0;
        if (!read_line(f, &line) || sscanf(line.c_str(), "-Y %u +X %u", &hh, &ww) != 2 || !hh || !ww)
            rc = fail_msg("svr_hdr_read: unsupported data layout (only -Y h +X w)");
        else if (ww > kMaxSide || hh > kMaxSide || (uint64_t)ww * hh > kMaxPixels)
            rc = fail_msg("svr_hdr_read: picture too large (at most 32768 per side and 2^27 pixels)");
        else {
            // the pixel data must be able to hold the picture: a run-length scanline is at least 4 + 4 * 2 * ceil(w / 127)
            // bytes, a flat one 4 * w
            const long pos = ftell(f);
            fseek(f, 0, SEEK_END);
            const long end = ftell(f);
            fseek(f, pos, SEEK_SET);
            const uint64_t left = end > pos ? (uint64_t)(end - pos) : 0;
            const uint64_t minLine = (ww < 8 || ww >= 32768) ? 4ull * ww : 4ull + 8ull * ((ww + 126u) / 127u);
            if (left < minLine * hh) rc = fail_msg("svr_hdr_read: truncated pixel data (the file cannot hold the picture its header declares)");
        }
        if (!rc) {
            *w = ww;
            *h = hh;
            if (rgbVec) {
                rgbVec->resize((size_t)ww * hh * 3);
                rc = decode(f, ww, hh, rgbVec->data());
            } else if (rgbExt) {
                if (ww != wantW || hh != wantH) rc = fail_msg("svr_hdr_read: the picture's size differs from the size the buffer was made for");
                else rc = decode(f, ww, hh, rgbExt);
            }
        }
    }
    fclose(f);
    return rc;
}

// With rgb_out: *w and *h are in-out -- on entry the size the buffer was made for (from the sizing call), so a file
// that changed in between is an error, not an overrun.
extern "C" int svr_hdr_read(const char* path, float* rgb_out, uint32_t* w, uint32_t* h)
{
    if (!path || !w || !h) return fail_msg("svr_hdr_read: bad argument");
    try {
        const uint32_t wantW = *w, wantH = *h;
        return read_hdr(path, nullptr, rgb_out, wantW, wantH, w, h);
    } catch (...) {
        return fail_msg("svr_hdr_read: out of host memory");
    }
}

extern "C" int svr_env_load_hdr(const char* path, svr_env_light* out)
{
    if (!out || !path) return fail_msg("svr_env_load_hdr: bad argument");
    try {
        uint32_t w = 0, h = 0;
        std::vector<float> rgb;
        int rc = read_hdr(path, &rgb, nullptr, 0, 0, &w, &h);  // ONE parse: the buffer is sized from the header it decodes
        if (rc) return rc;
        std::vector<float> rgba((size_t)w * h * 4);
        for (size_t i = 0; i < (size_t)w * h; ++i) {  // lights.cpp:47-53
            rgba[4 * i + 0] = rgb[3 * i + 0];
            rgba[4 * i + 1] = rgb[3 * i + 1];
            rgba[4 * i + 2] = rgb[3 * i + 2];
            rgba[4 * i + 3] = 0.f;
        }
        return svr_env_create(out, rgba.data(), w, h);
    } catch (...) {
        return fail_msg("svr_env_load_hdr: out of host memory");
    }
}

// ------------------------------------------------------------------------------------------------
// Importance sampler of the environment light (SVR_OPT_ENV_NEE).  A fixed grid of direction cells over (u, v) =
// (phi / 2 pi, theta / pi); the weight of a cell is (the largest luminance GetEnvRadiance returns at four points of the
// cell -- so offset, wrap and filtering are whatever the renderer will see -- plus a floor of 5 % of the mean, so that no
// direction with radiance has probability 0) times sin(theta).  Three small launches; rebuilt only when the light changes.
// ------------------------------------------------------------------------------------------------
namespace svr {
namespace {
constexpr int ENV_W = 512, ENV_H = 256;

__device__ float cell_luminance(const svr_env_light& env, int i, int j)
{
    float m = 0.f;
    for (int a = 0; a < 2; ++a)
        for (int b = 0; b < 2; ++b) {
            const float3 d = env_direction(((float)i + 0.25f + 0.5f * (float)a) / (float)ENV_W, ((float)j + 0.25f + 0.5f * (float)b) / (float)ENV_H);
            const float3 L = env_radiance(env, d);
            m = fmaxf(m, 0.2126f * L.x + 0.7152f * L.y + 0.0722f * L.z);
        }
    return (m == m && m < 3.0e38f) ? fmaxf(m, 0.f) : 0.f;
}

// one block per row: luminance into cond (temporarily), the row's sum into marg[j + 1] (temporarily), total into *total
__global__ void env_lum_kernel(svr_env_light env, float* cond, float* marg, double* total)
{
    const int j = blockIdx.x, i = threadIdx.x;
    const float lum = cell_luminance(env, i, j);
    cond[(size_t)j * (ENV_W + 1) + i + 1] = lum;
    __shared__ float red[ENV_W];
    red[i] = lum;
    __syncthreads();
    for (int o = ENV_W / 2; o > 0; o >>= 1) {
        if (i < o) red[i] += red[i + o];
        __syncthreads();
    }
    if (i == 0) {
        marg[j + 1] = red[0];
        atomicAdd(total, (double)red[0] * (double)__sinf(SVR_PI_F * ((float)j + 0.5f) / (float)ENV_H));
    }
}

// one block per row: weights = (lum + floor) sin(theta), inclusive scan -> the row's conditional CDF; the row's weight sum -> marg[j + 1]
__global__ void env_cond_kernel(float* cond, float* marg, const double* total, double sinSum)
{
    const int j = blockIdx.x, i = threadIdx.x;
    const float mean = (float)(*total / sinSum) / (float)ENV_W;
    const float floorLum = mean > 0.f ? 0.05f * mean : 1.f;
    const float sinT = __sinf(SVR_PI_F * ((float)j + 0.5f) / (float)ENV_H);
    float* row = cond + (size_t)j * (ENV_W + 1);
    __shared__ float sc[ENV_W];
    sc[i] = (row[i + 1] + floorLum) * sinT;
    __syncthreads();
    for (int o = 1; o < ENV_W; o <<= 1) {
        const float v = i >= o ? sc[i - o] : 0.f;
        __syncthreads();
        sc[i] += v;
        __syncthreads();
    }
    const float sum = sc[ENV_W - 1];
    row[i + 1] = i == ENV_W - 1 ? 1.f : sc[i] / sum;
    if (i == 0) {
        row[0] = 0.f;
        marg[j + 1] = sum;
    }
}

__global__ void env_marg_kernel(float* marg)
{
    const int j = threadIdx.x;
    __shared__ float sc[ENV_H];
    sc[j] = marg[j + 1];
    __syncthreads();
    for (int o = 1; o < ENV_H; o <<= 1) {
        const float v = j >= o ? sc[j - o] : 0.f;
        __syncthreads();
        sc[j] += v;
        __syncthreads();
    }
    const float sum = sc[ENV_H - 1];
    marg[j + 1] = j == ENV_H - 1 ? 1.f : sc[j] / sum;
    if (j == 0) marg[0] = 0.f;
}
}  // namespace

int ensure_env_sampler(DevScene* scene)
{
    HostState& st = state();
    const svr_env_light& e = scene->env;
    if (!st.dev.envSamplerValid || memcmp(&st.dev.envSamplerKey, &e, sizeof(e)) != 0) {
        SVR_TRY(st.dev.envMarg.reserve(ENV_H + 1));
        SVR_TRY(st.dev.envCond.reserve((size_t)ENV_H * (ENV_W + 1)));
        SVR_TRY(st.dev.stats.reserve(2));
        SVR_TRY(cudaMemsetAsync(st.dev.stats.p, 0, 16, st.stream));
        double sinSum = 0.0;
        for (int j = 0; j < ENV_H; ++j) sinSum += (double)sinf(SVR_PI_F * ((float)j + 0.5f) / (float)ENV_H);
        env_lum_kernel<<<ENV_H, ENV_W, 0, st.stream>>>(e, st.dev.envCond.p, st.dev.envMarg.p, (double*)st.dev.stats.p);
        env_cond_kernel<<<ENV_H, ENV_W, 0, st.stream>>>(st.dev.envCond.p, st.dev.envMarg.p, (const double*)st.dev.stats.p, sinSum);
        env_marg_kernel<<<1, ENV_H, 0, st.stream>>>(st.dev.envMarg.p);
        count_launch(3);
        SVR_TRY(cudaGetLastError());
        st.dev.envSamplerKey = e;
        st.dev.envSamplerValid = true;
    }
    scene->envS.marg = st.dev.envMarg.p;
    scene->envS.cond = st.dev.envCond.p;
    scene->envS.w = ENV_W;
    scene->envS.h = ENV_H;
    return 0;
}
}  // namespace svr

// Inspection hook (tests): the sampler's cumulative tables for the current environment light, ENV_H + 1 and ENV_H * (ENV_W + 1) floats.
extern "C" int svr_env_sampler_copy(float* host_marg, float* host_cond, uint32_t* w, uint32_t* h)
{
    HostState& st = state();
    DevScene sc = st.scene;
    int rc = ensure_env_sampler(&sc);
    if (rc) return rc;
    SVR_TRY(cudaStreamSynchronize(st.stream));
    if (w) *w = ENV_W;
    if (h) *h = ENV_H;
    if (host_marg) SVR_TRY(cudaMemcpy(host_marg, st.dev.envMarg.p, (ENV_H + 1) * sizeof(float), cudaMemcpyDeviceToHost));
    if (host_cond) SVR_TRY(cudaMemcpy(host_cond, st.dev.envCond.p, (size_t)ENV_H * (ENV_W + 1) * sizeof(float), cudaMemcpyDeviceToHost));
    return 0;
}
