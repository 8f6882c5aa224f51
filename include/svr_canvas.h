/*
 * svr_canvas.h -- C ABI of the interactive host shell without its window: what gui/canvas.{h,cpp} does
 * between the Qt events and the seven render entry points (SURVEY.md section 8f, rank 4).
 *
 * Two layers:
 *   svr_view_*    the camera manipulation of Canvas as pure host arithmetic (no CUDA, no window): the view
 *                 matrix (glm::lookAt / glm::rotate semantics -- GLM is the reference's un-vendored vector
 *                 library, CMakeLists.txt:37; its published column-major formulas are restated), mouse
 *                 rotate / translate, wheel zoom, arrow keys, ZoomToExtent, UpdateCamera
 *                 (gui/canvas.cpp:119-226, gui/canvas.h:183-187).
 *   svr_canvas_*  a Canvas object: owns the accumulation buffer (RenderParams::SetupHDRBuffer) and an
 *                 image buffer in device memory that stands in for the GL pixel-buffer object
 *                 (canvas.cpp:43-55), keeps the scene PODs, forwards every setter to setup_* and restarts
 *                 the progressive render the way Canvas::ReStartRender does (canvas.h:43-47), and paints
 *                 one frame per call (Canvas::paintGL, canvas.cpp:63-117).  What is NOT here: the window,
 *                 the GL context and cudaGraphicsGLRegisterBuffer / glDrawPixels -- a windowed host maps
 *                 its PBO and passes that pointer to svr_canvas_paint_into instead.
 * Functions returning int return 0 on success; svr_last_error() has the text otherwise.
 */
#ifndef SVR_CANVAS_H
#define SVR_CANVAS_H

#include "svr_types.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ---- view state: the camera-related members of Canvas (canvas.h:210-217) ---- */
typedef struct svr_view {
    float viewMat[16];        /* glm::mat4, column-major: viewMat[4*c + r] = m[c][r] */
    float eyeDist;
    float translate[2];       /* cameraTranslate */
    float fov, apeture, focalLength, exposure;   /* 45, 0, 1, 1 */
    float mouseStart[2];      /* mouseStartPoint, in view coordinates */
} svr_view;

enum svr_mouse_button { SVR_BUTTON_LEFT = 1, SVR_BUTTON_MID = 4 };   /* Qt::LeftButton, Qt::MidButton */
enum svr_key { SVR_KEY_LEFT = 0, SVR_KEY_RIGHT = 1, SVR_KEY_DOWN = 2 };

/* members as Canvas initialises them: identity matrix, eyeDist 0, translate 0, fov 45, apeture 0,
 * focalLength 1, exposure 1 */
void svr_view_init(svr_view* v);
/* Canvas::ZoomToExtent (canvas.cpp:191-197): eyeDist = 1.5 * max(extent) / (2 tan(fov / 2)) */
void svr_view_zoom_to_extent(svr_view* v, const float volume_size[3]);
/* the view half of Canvas::LoadVolume (canvas.cpp:35-38): ZoomToExtent, viewMat = lookAt((0,0,eyeDist), 0, +y) */
void svr_view_reset(svr_view* v, const float volume_size[3]);
/* viewMat = glm::rotate(viewMat, radians(degrees), axis) */
void svr_view_rotate(svr_view* v, float degrees, float ax, float ay, float az);
/* Canvas::PixelPosToViewPos (canvas.h:160-164) */
void svr_view_pixel_to_view(uint32_t width, uint32_t height, float px, float py, float out[2]);
/* mousePressEvent / mouseMoveEvent / wheelEvent / keyPressEvent (canvas.cpp:119-177, 198-226); positions in
 * pixels, `buttons` an OR of svr_mouse_button, `delta` as QWheelEvent::delta().  Return 1 when the camera
 * changed (the caller publishes it and restarts the render), 0 otherwise. */
int svr_view_mouse_press(svr_view* v, uint32_t width, uint32_t height, float px, float py, int buttons);
int svr_view_mouse_move(svr_view* v, uint32_t width, uint32_t height, float px, float py, int buttons, const float volume_size[3]);
int svr_view_wheel(svr_view* v, int delta, const float volume_size[3]);
int svr_view_key(svr_view* v, int key);
/* Canvas::UpdateCamera (canvas.cpp:179-188) + cudaCamera::Setup (core/cuda_camera.h:34-47) */
void svr_view_camera(const svr_view* v, uint32_t width, uint32_t height, svr_camera* out);

/* ---- the canvas ---- */
typedef struct svr_canvas svr_canvas;
/* canvas.h:30, plus the intensity projection (svr_render_projection), which the reference lacks */
enum svr_render_mode { SVR_RENDER_MODE_PATHTRACER = 0, SVR_RENDER_MODE_RAYCASTING = 1, SVR_RENDER_MODE_PROJECTION = 2 };

/* Canvas::Canvas (canvas.cpp:8-20): white environment at intensity 0.5, traceDepth 1, gradient factor 0.5,
 * ray-casting mode; buffers for a width x height image (the reference's WIDTH x HEIGHT, common.h:8-9). */
svr_canvas* svr_canvas_create(uint32_t width, uint32_t height);
void svr_canvas_destroy(svr_canvas* c);

/* Canvas::LoadVolume (canvas.cpp:27-41) on a MetaImage file; the canvas owns the volume. */
int svr_canvas_load_volume(svr_canvas* c, const char* metaimage_path);
/* The same for a volume built elsewhere (not owned): clip planes (-1,1), density scale 1, setup_volume,
 * ZoomToExtent, view reset.  volume_size = dim * spacing (VolumeReader::GetVolumeSize), element_radius =
 * |spacing| / 2 (GetElementBoundingSphereRadius, the ray caster's step size). */
int svr_canvas_set_volume(svr_canvas* c, const svr_volume* vol, const float volume_size[3], float element_radius);

/* setters of canvas.h:49-156; each publishes with setup_* and restarts the render */
int svr_canvas_set_transfer_function(svr_canvas* c, const svr_transfer_function* tf);
int svr_canvas_set_density_scale(svr_canvas* c, double s);
int svr_canvas_set_gradient_factor(svr_canvas* c, double g);
int svr_canvas_set_scatter_times(svr_canvas* c, double depth);
int svr_canvas_set_render_mode(svr_canvas* c, int mode);
int svr_canvas_set_env_background(svr_canvas* c, float r, float g, float b);
int svr_canvas_set_env_map(svr_canvas* c, const char* hdr_path);
int svr_canvas_set_env_offset(svr_canvas* c, float u, float v);
int svr_canvas_set_env_intensity(svr_canvas* c, float intensity);
int svr_canvas_set_area_lights(svr_canvas* c, const svr_area_light* lights, uint32_t n);
int svr_canvas_set_fov(svr_canvas* c, float fov);
int svr_canvas_set_apeture(svr_canvas* c, float apeture);
int svr_canvas_set_focal_length(svr_canvas* c, float focal_length);
int svr_canvas_set_exposure(svr_canvas* c, float exposure);
int svr_canvas_set_clip_plane(svr_canvas* c, int axis, double lo, double hi);
/* Projection mode (SVR_RENDER_MODE_PROJECTION): the svr_projection_mode and the display window.  Checked as
 * svr_render_projection checks them; restarts the render like the other setters.  Defaults: MAX, window (0.5, 1). */
int svr_canvas_set_projection(svr_canvas* c, int mode, float windowCenter, float windowWidth);

/* events, positions in pixels */
int svr_canvas_mouse_press(svr_canvas* c, float px, float py, int buttons);
int svr_canvas_mouse_move(svr_canvas* c, float px, float py, int buttons);
int svr_canvas_wheel(svr_canvas* c, int delta);
int svr_canvas_key(svr_canvas* c, int key);

/* Canvas::paintGL: one ray-cast frame, or one more path-traced sample per pixel, or in projection mode one projection of
 * the canvas's camera with element_radius as stepSize (no transfer function needed); synchronises and advances
 * the frame counter.  A canvas without a volume paints nothing (`ready`, canvas.cpp:67).  _paint renders into
 * the canvas's own image buffer, _paint_into into the caller's (a mapped GL pixel-buffer object). */
int svr_canvas_paint(svr_canvas* c);
int svr_canvas_paint_into(svr_canvas* c, svr_u8vec4* device_img);
/* The reference repaints inside every setter and event (updateGL in ReStartRender, canvas.h:43-47).  A batch
 * host that only looks at the frames it asks for can turn those immediate repaints off; the frame counter is
 * reset either way. */
void svr_canvas_set_immediate_repaint(svr_canvas* c, int on);

/* state */
const svr_u8vec4* svr_canvas_image(const svr_canvas* c);      /* device memory, width * height */
const svr_vec3* svr_canvas_hdr(const svr_canvas* c);          /* device memory, the running mean */
int svr_canvas_read_image(const svr_canvas* c, void* host_rgba8);
uint32_t svr_canvas_frame_no(const svr_canvas* c);
uint64_t svr_canvas_paint_count(const svr_canvas* c);
void svr_canvas_get_view(const svr_canvas* c, svr_view* out);
void svr_canvas_get_camera(const svr_canvas* c, svr_camera* out);
void svr_canvas_get_volume(const svr_canvas* c, svr_volume* out);
void svr_canvas_get_env_light(const svr_canvas* c, svr_env_light* out);

#ifdef __cplusplus
}
#endif
#endif /* SVR_CANVAS_H */
