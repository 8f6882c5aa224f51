// svr_canvas.cu -- the interactive host shell without its window (include/svr_canvas.h): the camera
// manipulation of gui/canvas.cpp:119-226 as host arithmetic, and a Canvas object that drives the seven
// render entry points the way Canvas does (gui/canvas.cpp:8-117, gui/canvas.h:39-175).  Host code only.
#include <cmath>
#include <cstring>
#include <vector>

#include "../../include/svr_canvas.h"
#include "../../include/svr_env_io.h"
#include "../../include/svr_volume_io.h"
#include "svr_state.h"

using namespace svr;

namespace {

struct V3 {
    float x, y, z;
};
inline V3 operator*(V3 a, float s) { return {a.x * s, a.y * s, a.z * s}; }
inline V3 operator-(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
inline float dot3(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
inline V3 cross3(V3 a, V3 b) { return {a.y * b.z - b.y * a.z, a.z * b.x - b.z * a.x, a.x * b.y - b.x * a.y}; }
inline V3 normalize3(V3 a)
{
    const float inv = 1.f / sqrtf(dot3(a, a));
    return a * inv;
}
inline float length3(const float s[3]) { return sqrtf(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]); }

// glm::mat4 is column-major: m[c][r] = a[4 * c + r]
inline float& M(float* a, int c, int r) { return a[4 * c + r]; }
inline float Mc(const float* a, int c, int r) { return a[4 * c + r]; }

// glm::lookAt (right-handed), glm/gtc/matrix_transform.inl
void look_at(float* m, V3 eye, V3 center, V3 up)
{
    const V3 f = normalize3(center - eye);
    const V3 s = normalize3(cross3(f, up));
    const V3 u = cross3(s, f);
    for (int i = 0; i < 16; ++i) m[i] = (i % 5 == 0) ? 1.f : 0.f;
    M(m, 0, 0) = s.x;
    M(m, 1, 0) = s.y;
    M(m, 2, 0) = s.z;
    M(m, 0, 1) = u.x;
    M(m, 1, 1) = u.y;
    M(m, 2, 1) = u.z;
    M(m, 0, 2) = -f.x;
    M(m, 1, 2) = -f.y;
    M(m, 2, 2) = -f.z;
    M(m, 3, 0) = -dot3(s, eye);
    M(m, 3, 1) = -dot3(u, eye);
    M(m, 3, 2) = dot3(f, eye);
}

// glm::rotate(m, angle, axis) = m * R, glm/gtc/matrix_transform.inl
void rotate(float* m, float angle, V3 v)
{
    const float c = cosf(angle), s = sinf(angle);
    const V3 axis = normalize3(v);
    const V3 temp = axis * (1.f - c);
    float R[3][3];
    R[0][0] = c + temp.x * axis.x;
    R[0][1] = temp.x * axis.y + s * axis.z;
    R[0][2] = temp.x * axis.z - s * axis.y;
    R[1][0] = temp.y * axis.x - s * axis.z;
    R[1][1] = c + temp.y * axis.y;
    R[1][2] = temp.y * axis.z + s * axis.x;
    R[2][0] = temp.z * axis.x + s * axis.y;
    R[2][1] = temp.z * axis.y - s * axis.x;
    R[2][2] = c + temp.z * axis.z;
    float out[16];
    for (int col = 0; col < 3; ++col)
        for (int r = 0; r < 4; ++r) out[4 * col + r] = Mc(m, 0, r) * R[col][0] + Mc(m, 1, r) * R[col][1] + Mc(m, 2, r) * R[col][2];
    for (int r = 0; r < 4; ++r) out[12 + r] = Mc(m, 3, r);
    memcpy(m, out, sizeof(out));
}

inline double radians_d(double deg) { return deg * 0.01745329251994329576923690768489; }
inline float radians_f(float deg) { return deg * 0.01745329251994329576923690768489f; }

}  // namespace

// ------------------------------------------------------------------------------------------------
// svr_view_*
// ------------------------------------------------------------------------------------------------
extern "C" void svr_view_init(svr_view* v)
{
    memset(v, 0, sizeof(*v));
    for (int i = 0; i < 4; ++i) v->viewMat[5 * i] = 1.f;
    v->fov = 45.f;         // canvas.h:212-215
    v->apeture = 0.f;
    v->focalLength = 1.f;
    v->exposure = 1.f;
}

extern "C" void svr_view_zoom_to_extent(svr_view* v, const float volume_size[3])
{
    float maxSpan = fmaxf(volume_size[0], fmaxf(volume_size[1], volume_size[2]));
    maxSpan *= 1.5f;  // "enlarge it slightly"
    // `maxSpan / (2 * tan(glm::radians(fov * 0.5f)))` with a float argument: the <cmath> float overload
    v->eyeDist = maxSpan / (2 * tanf(radians_f(v->fov * 0.5f)));
}

extern "C" void svr_view_reset(svr_view* v, const float volume_size[3])
{
    svr_view_zoom_to_extent(v, volume_size);
    look_at(v->viewMat, {0.f, 0.f, v->eyeDist}, {0.f, 0.f, 0.f}, {0.f, 1.f, 0.f});
}

extern "C" void svr_view_rotate(svr_view* v, float degrees, float ax, float ay, float az)
{
    rotate(v->viewMat, radians_f(degrees), {ax, ay, az});
}

extern "C" void svr_view_pixel_to_view(uint32_t width, uint32_t height, float px, float py, float out[2])
{
    out[0] = 2.f * px / (float)width - 1.f;
    out[1] = 1.f - 2.f * py / (float)height;
}

extern "C" int svr_view_mouse_press(svr_view* v, uint32_t width, uint32_t height, float px, float py, int buttons)
{
    if (buttons & (SVR_BUTTON_LEFT | SVR_BUTTON_MID)) svr_view_pixel_to_view(width, height, px, py, v->mouseStart);
    return 0;
}

extern "C" int svr_view_mouse_move(svr_view* v, uint32_t width, uint32_t height, float px, float py, int buttons,
                                   const float volume_size[3])
{
    float now[2];
    svr_view_pixel_to_view(width, height, px, py, now);
    // QPointF holds doubles: the difference and the products below are formed in double (canvas.cpp:137-161)
    const double dx = (double)now[0] - (double)v->mouseStart[0], dy = (double)now[1] - (double)v->mouseStart[1];
    int changed = 0;
    if (buttons & SVR_BUTTON_LEFT) {
        const float baseDegree = 100.f;
        rotate(v->viewMat, (float)radians_d(dy * baseDegree), {1.f, 0.f, 0.f});
        rotate(v->viewMat, (float)radians_d(-dx * baseDegree), {0.f, 1.f, 0.f});
        changed = 1;
    }
    if (buttons & SVR_BUTTON_MID) {
        const float baseTranslate = length3(volume_size) * 0.5f;
        v->translate[0] += (float)(dx * baseTranslate);
        v->translate[1] += (float)(dy * baseTranslate);
        changed = 1;
    }
    v->mouseStart[0] = now[0];
    v->mouseStart[1] = now[1];
    return changed;
}

extern "C" int svr_view_wheel(svr_view* v, int delta, const float volume_size[3])
{
    v->eyeDist += (float)delta * length3(volume_size) * 0.001f;
    return 1;
}

extern "C" int svr_view_key(svr_view* v, int key)
{
    float deg;
    switch (key) {
        case SVR_KEY_DOWN: deg = 180.f; break;
        case SVR_KEY_LEFT: deg = 90.f; break;
        case SVR_KEY_RIGHT: deg = -90.f; break;
        default: return 0;
    }
    rotate(v->viewMat, radians_f(deg), {0.f, 1.f, 0.f});
    return 1;
}

extern "C" void svr_view_camera(const svr_view* v, uint32_t width, uint32_t height, svr_camera* out)
{
    const float* m = v->viewMat;
    const V3 u = {Mc(m, 0, 0), Mc(m, 0, 1), Mc(m, 0, 2)};
    const V3 vv = {Mc(m, 1, 0), Mc(m, 1, 1), Mc(m, 1, 2)};
    const V3 w = {Mc(m, 2, 0), Mc(m, 2, 1), Mc(m, 2, 2)};
    const V3 pos = w * v->eyeDist - u * v->translate[0] - vv * v->translate[1];
    memset(out, 0, sizeof(*out));
    out->pos = {pos.x, pos.y, pos.z};
    out->u = {u.x, u.y, u.z};
    out->v = {vv.x, vv.y, vv.z};
    out->w = {w.x, w.y, w.z};
    out->imageW = width;
    out->imageH = height;
    out->aspectRatio = (float)width / (float)height;
    out->tanFovxOverTwo = tanf((float)(v->fov * 0.5f * M_PI / 180.f));  // cuda_camera.h:43
    out->exposure = v->exposure;
    out->focalLength = v->focalLength;
    out->apeture = v->apeture;
}

// ------------------------------------------------------------------------------------------------
// svr_canvas_*
// ------------------------------------------------------------------------------------------------
struct svr_canvas {
    uint32_t width = 0, height = 0;
    svr_view view;
    svr_camera camera;
    svr_volume volume;
    bool ownsVolume = false;
    float volumeSize[3] = {0.f, 0.f, 0.f};
    float elementRadius = 0.f;
    svr_transfer_function tf;
    svr_env_light env;
    bool ownsEnvTex = false;
    std::vector<svr_area_light> lights;
    svr_render_params renderParams;
    svr_u8vec4* img = nullptr;
    int renderMode = SVR_RENDER_MODE_RAYCASTING;  // canvas.h:226
    svr_projection_params projection = {SVR_PROJECT_MAX, 0.f, 0.5f, 1.f};  // stepSize: elementRadius at paint time
    bool ready = false;
    bool immediate = true;
    uint64_t paints = 0;
};

namespace {

int paint_into(svr_canvas* c, svr_u8vec4* img)
{
    if (!c->ready) return 0;  // canvas.cpp:67
    if (c->renderMode == SVR_RENDER_MODE_PROJECTION) {
        svr_projection_params p = c->projection;
        p.stepSize = c->elementRadius;
        if (int rc = svr_render_projection(img, nullptr, &c->volume, &c->camera, &p, 0, 1, nullptr)) return rc;
    } else if (!c->tf.tex) {
        return fail_msg("svr_canvas_paint: no transfer function set");
    } else if (c->renderMode == SVR_RENDER_MODE_RAYCASTING)
        render_raycasting(img, &c->volume, &c->tf, &c->camera, c->elementRadius);  // canvas.cpp:92
    else
        render_pathtracer(img, &c->renderParams);                                 // canvas.cpp:96
    SVR_TRY(cudaDeviceSynchronize());                                              // canvas.cpp:106
    c->renderParams.frameNo++;                                                     // canvas.cpp:116
    c->paints++;
    return 0;
}

// Canvas::ReStartRender (canvas.h:43-47): updateGL(), then frameNo = 0
int restart(svr_canvas* c)
{
    int rc = c->immediate ? paint_into(c, c->img) : 0;
    c->renderParams.frameNo = 0;
    return rc;
}

// Canvas::UpdateCamera (canvas.cpp:179-188)
void update_camera(svr_canvas* c)
{
    svr_view_camera(&c->view, c->width, c->height, &c->camera);
    setup_camera(&c->camera);
}

void drop_volume(svr_canvas* c)
{
    if (c->ownsVolume) svr_volume_destroy(&c->volume);
    c->ownsVolume = false;
    memset(&c->volume, 0, sizeof(c->volume));
    c->ready = false;
}

void drop_env_tex(svr_canvas* c)
{
    if (c->ownsEnvTex) {
        svr_env_light e = c->env;
        svr_env_destroy(&e);
    }
    c->ownsEnvTex = false;
}

int adopt_volume(svr_canvas* c, const float volume_size[3], float element_radius)
{
    memcpy(c->volumeSize, volume_size, sizeof(c->volumeSize));
    c->elementRadius = element_radius;
    c->volume.x_clip = c->volume.y_clip = c->volume.z_clip = {-1.f, 1.f};  // canvas.cpp:31
    c->volume.densityScale = 1.f;                                          // canvas.cpp:32
    setup_volume(&c->volume);
    svr_view_reset(&c->view, c->volumeSize);                               // canvas.cpp:35-37
    update_camera(c);
    c->ready = true;
    return 0;
}

}  // namespace

extern "C" svr_canvas* svr_canvas_create(uint32_t width, uint32_t height)
{
    if (!width || !height) {
        fail_msg("svr_canvas_create: bad size");
        return nullptr;
    }
    svr_canvas* c = new svr_canvas();
    c->width = width;
    c->height = height;
    svr_view_init(&c->view);
    memset(&c->camera, 0, sizeof(c->camera));
    memset(&c->volume, 0, sizeof(c->volume));
    memset(&c->tf, 0, sizeof(c->tf));
    // lights.SetEnvionmentLight(vec3(1)); SetEnvironmentLightIntensity(0.5) (canvas.cpp:11-13)
    memset(&c->env, 0, sizeof(c->env));
    c->env.defaultRadiance = {1.f, 1.f, 1.f};
    c->env.intensity = 0.5f;
    // renderParams.SetupHDRBuffer(WIDTH, HEIGHT); traceDepth = 1 (canvas.cpp:16-17, render_parameters.h:17-23)
    c->renderParams.traceDepth = 1;
    c->renderParams.frameNo = 0;
    c->renderParams.hdrBuffer = nullptr;
    const size_t npix = (size_t)width * height;
    if (cudaMalloc((void**)&c->renderParams.hdrBuffer, npix * sizeof(svr_vec3)) != cudaSuccess ||
        cudaMemset(c->renderParams.hdrBuffer, 0, npix * sizeof(svr_vec3)) != cudaSuccess ||
        cudaMalloc((void**)&c->img, npix * sizeof(svr_u8vec4)) != cudaSuccess ||  // stands in for the PBO (canvas.cpp:50-53)
        cudaMemset(c->img, 0, npix * sizeof(svr_u8vec4)) != cudaSuccess) {
        fail("svr_canvas_create: buffers", cudaGetLastError());
        cudaFree(c->renderParams.hdrBuffer);
        cudaFree(c->img);
        delete c;
        return nullptr;
    }
    c->volume.gradientFactor = 0.5f;  // canvas.cpp:19
    setup_env_lights(&c->env);
    return c;
}

extern "C" void svr_canvas_destroy(svr_canvas* c)
{
    if (!c) return;
    cudaDeviceSynchronize();
    drop_volume(c);
    drop_env_tex(c);
    cudaFree(c->renderParams.hdrBuffer);  // RenderParams::Clear (canvas.cpp:24)
    cudaFree(c->img);
    delete c;
}

extern "C" int svr_canvas_load_volume(svr_canvas* c, const char* path)
{
    if (!c || !path) return fail_msg("svr_canvas_load_volume: bad argument");
    svr_volume vol;
    svr_volume_stats stats;
    int rc = svr_volume_load_metaimage(path, &vol, &stats, nullptr, 0);  // volumeReader.Read + CreateDeviceVolume
    if (rc) return rc;
    const float gradientFactor = c->volume.gradientFactor;
    drop_volume(c);
    c->volume = vol;
    c->volume.gradientFactor = gradientFactor;  // a member of Canvas::deviceVolume, not of the file
    c->ownsVolume = true;
    const float size[3] = {stats.dim[0] * stats.spacing[0], stats.dim[1] * stats.spacing[1], stats.dim[2] * stats.spacing[2]};
    return adopt_volume(c, size, length3(stats.spacing) * 0.5f);
}

extern "C" int svr_canvas_set_volume(svr_canvas* c, const svr_volume* vol, const float volume_size[3], float element_radius)
{
    if (!c) return fail_msg("svr_canvas_set_volume: null canvas");
    if (!c || !vol || !vol->tex || !volume_size) return fail_msg("svr_canvas_set_volume: bad argument");
    const float gradientFactor = c->volume.gradientFactor;
    drop_volume(c);
    c->volume = *vol;
    c->volume.gradientFactor = gradientFactor;
    return adopt_volume(c, volume_size, element_radius);
}

extern "C" int svr_canvas_set_transfer_function(svr_canvas* c, const svr_transfer_function* tf)
{
    if (!c) return fail_msg("svr_canvas_set_transfer_function: null canvas");
    if (!c || !tf) return fail_msg("svr_canvas_set_transfer_function: bad argument");
    c->tf = *tf;
    setup_transferfunction(&c->tf);
    return restart(c);
}

extern "C" int svr_canvas_set_density_scale(svr_canvas* c, double s)
{
    if (!c) return fail_msg("svr_canvas_set_density_scale: null canvas");
    c->volume.densityScale = (float)s;
    setup_volume(&c->volume);
    return restart(c);
}

extern "C" int svr_canvas_set_gradient_factor(svr_canvas* c, double g)
{
    if (!c) return fail_msg("svr_canvas_set_gradient_factor: null canvas");
    c->volume.gradientFactor = (float)g;
    setup_volume(&c->volume);
    return restart(c);
}

extern "C" int svr_canvas_set_scatter_times(svr_canvas* c, double depth)
{
    if (!c) return fail_msg("svr_canvas_set_scatter_times: null canvas");
    c->renderParams.traceDepth = (uint32_t)depth;
    return restart(c);
}

extern "C" int svr_canvas_set_render_mode(svr_canvas* c, int mode)
{
    if (!c) return fail_msg("svr_canvas_set_render_mode: null canvas");
    if (mode != SVR_RENDER_MODE_PATHTRACER && mode != SVR_RENDER_MODE_RAYCASTING && mode != SVR_RENDER_MODE_PROJECTION)
        return fail_msg("svr_canvas_set_render_mode: bad mode");
    c->renderMode = mode;  // the timer that repaints in path-tracer mode (canvas.h:80-93) is the host's paint loop
    return restart(c);
}

extern "C" int svr_canvas_set_projection(svr_canvas* c, int mode, float windowCenter, float windowWidth)
{
    if (!c) return fail_msg("svr_canvas_set_projection: null canvas");
    if (mode < SVR_PROJECT_MAX || mode > SVR_PROJECT_MEAN) return fail_msg("svr_canvas_set_projection: mode must be 0 (max), 1 (min) or 2 (mean)");
    if (!(windowWidth > 0.f) || !std::isfinite(windowWidth) || !std::isfinite(windowCenter))
        return fail_msg("svr_canvas_set_projection: windowWidth must be positive and finite, windowCenter finite");
    c->projection.mode = mode;
    c->projection.windowCenter = windowCenter;
    c->projection.windowWidth = windowWidth;
    return restart(c);
}

extern "C" int svr_canvas_set_env_background(svr_canvas* c, float r, float g, float b)
{
    if (!c) return fail_msg("svr_canvas_set_env_background: null canvas");
    // cudaEnvironmentLight::Set(radiance) also resets intensity to 1 and the offset (cuda_environment_light.h:25-31)
    drop_env_tex(c);
    c->env.tex = 0;
    c->env.defaultRadiance = {r, g, b};
    c->env.intensity = 1.f;
    c->env.offset = {0.f, 0.f};
    setup_env_lights(&c->env);
    return restart(c);
}

extern "C" int svr_canvas_set_env_map(svr_canvas* c, const char* hdr_path)
{
    if (!c) return fail_msg("svr_canvas_set_env_map: null canvas");
    svr_env_light e;
    int rc = svr_env_load_hdr(hdr_path, &e);  // Lights::SetEnvironmentLight(filename): Set(tex), intensity 1, offset 0
    if (rc) return rc;
    drop_env_tex(c);
    const svr_vec3 keep = c->env.defaultRadiance;
    c->env = e;
    c->env.defaultRadiance = keep;
    c->ownsEnvTex = true;
    setup_env_lights(&c->env);
    return restart(c);
}

extern "C" int svr_canvas_set_env_offset(svr_canvas* c, float u, float v)
{
    if (!c) return fail_msg("svr_canvas_set_env_offset: null canvas");
    c->env.offset = {u, v};
    setup_env_lights(&c->env);
    return restart(c);
}

extern "C" int svr_canvas_set_env_intensity(svr_canvas* c, float intensity)
{
    if (!c) return fail_msg("svr_canvas_set_env_intensity: null canvas");
    c->env.intensity = intensity;
    setup_env_lights(&c->env);
    return restart(c);
}

extern "C" int svr_canvas_set_area_lights(svr_canvas* c, const svr_area_light* lights, uint32_t n)
{
    if (!c) return fail_msg("svr_canvas_set_area_lights: null canvas");
    c->lights.assign(lights, lights + (lights ? n : 0));
    svr_area_light none;
    memset(&none, 0, sizeof(none));
    setup_area_lights(c->lights.empty() ? &none : c->lights.data(), (uint32_t)c->lights.size());
    return restart(c);
}

extern "C" int svr_canvas_set_fov(svr_canvas* c, float fov)
{
    if (!c) return fail_msg("svr_canvas_set_fov: null canvas");
    c->view.fov = fov;
    update_camera(c);
    return restart(c);
}

extern "C" int svr_canvas_set_apeture(svr_canvas* c, float apeture)
{
    if (!c) return fail_msg("svr_canvas_set_apeture: null canvas");
    c->view.apeture = apeture;
    update_camera(c);
    return restart(c);
}

extern "C" int svr_canvas_set_focal_length(svr_canvas* c, float focal_length)
{
    if (!c) return fail_msg("svr_canvas_set_focal_length: null canvas");
    c->view.focalLength = focal_length;
    update_camera(c);
    return restart(c);
}

extern "C" int svr_canvas_set_exposure(svr_canvas* c, float exposure)
{
    if (!c) return fail_msg("svr_canvas_set_exposure: null canvas");
    c->view.exposure = exposure;
    update_camera(c);
    return restart(c);
}

extern "C" int svr_canvas_set_clip_plane(svr_canvas* c, int axis, double lo, double hi)
{
    if (!c) return fail_msg("svr_canvas_set_clip_plane: null canvas");
    const svr_vec2 p = {(float)lo, (float)hi};
    if (axis == 0) c->volume.x_clip = p;
    else if (axis == 1) c->volume.y_clip = p;
    else if (axis == 2) c->volume.z_clip = p;
    else return fail_msg("svr_canvas_set_clip_plane: axis must be 0, 1 or 2");
    setup_volume(&c->volume);
    return restart(c);
}

extern "C" int svr_canvas_mouse_press(svr_canvas* c, float px, float py, int buttons)
{
    if (!c) return fail_msg("svr_canvas_mouse_press: null canvas");
    svr_view_mouse_press(&c->view, c->width, c->height, px, py, buttons);
    return 0;
}

extern "C" int svr_canvas_mouse_move(svr_canvas* c, float px, float py, int buttons)
{
    if (!c) return fail_msg("svr_canvas_mouse_move: null canvas");
    // one repaint per handled button (UpdateCamera(); updateGL()), then ReStartRender() (canvas.cpp:135-169)
    const int changed = svr_view_mouse_move(&c->view, c->width, c->height, px, py, buttons, c->volumeSize);
    if (changed) {
        update_camera(c);
        if (c->immediate) {
            const int repaints = ((buttons & SVR_BUTTON_LEFT) ? 1 : 0) + ((buttons & SVR_BUTTON_MID) ? 1 : 0);
            for (int i = 0; i < repaints; ++i) {
                int rc = paint_into(c, c->img);
                if (rc) return rc;
            }
        }
    }
    return restart(c);
}

extern "C" int svr_canvas_wheel(svr_canvas* c, int delta)
{
    if (!c) return fail_msg("svr_canvas_wheel: null canvas");
    svr_view_wheel(&c->view, delta, c->volumeSize);
    update_camera(c);
    return restart(c);
}

extern "C" int svr_canvas_key(svr_canvas* c, int key)
{
    if (!c) return fail_msg("svr_canvas_key: null canvas");
    if (!svr_view_key(&c->view, key)) return 0;
    update_camera(c);
    if (c->immediate) {
        int rc = paint_into(c, c->img);  // updateGL()
        if (rc) return rc;
    }
    return restart(c);
}

extern "C" int svr_canvas_paint(svr_canvas* c) { return c ? paint_into(c, c->img) : fail_msg("svr_canvas_paint: null canvas"); }

extern "C" int svr_canvas_paint_into(svr_canvas* c, svr_u8vec4* device_img)
{
    if (!c || !device_img) return fail_msg("svr_canvas_paint_into: bad argument");
    return paint_into(c, device_img);
}

extern "C" void svr_canvas_set_immediate_repaint(svr_canvas* c, int on) { c->immediate = on != 0; }

extern "C" const svr_u8vec4* svr_canvas_image(const svr_canvas* c) { return c->img; }
extern "C" const svr_vec3* svr_canvas_hdr(const svr_canvas* c) { return c->renderParams.hdrBuffer; }

extern "C" int svr_canvas_read_image(const svr_canvas* c, void* host_rgba8)
{
    if (!c || !host_rgba8) return fail_msg("svr_canvas_read_image: bad argument");
    SVR_TRY(cudaMemcpy(host_rgba8, c->img, (size_t)c->width * c->height * sizeof(svr_u8vec4), cudaMemcpyDeviceToHost));
    return 0;
}

extern "C" uint32_t svr_canvas_frame_no(const svr_canvas* c) { return c->renderParams.frameNo; }
extern "C" uint64_t svr_canvas_paint_count(const svr_canvas* c) { return c->paints; }
extern "C" void svr_canvas_get_view(const svr_canvas* c, svr_view* out) { *out = c->view; }
extern "C" void svr_canvas_get_camera(const svr_canvas* c, svr_camera* out) { *out = c->camera; }
extern "C" void svr_canvas_get_volume(const svr_canvas* c, svr_volume* out) { *out = c->volume; }
extern "C" void svr_canvas_get_env_light(const svr_canvas* c, svr_env_light* out) { *out = c->env; }
