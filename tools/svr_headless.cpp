// svr_headless.cpp -- headless C++ driver for libsvr_b200.so (the benchmark host north_star asks
// for next to the Qt canvas).  It does what gui/canvas.cpp does with the seven entry points --
// build the scene structs, setup_*, then render_pathtracer once per frame (canvas.cpp:63-117) or
// render_raycasting -- on the synthetic configurations of SURVEY.md section 8d, times the loop with
// CUDA events and writes the image as PPM (tone-mapped u8) and PFM (float accumulator).
//
//   svr_headless [--config C1|C2|C3|C4] [--mode pt|rc|mip|minip|aip|iso|slice|cpr|labels] [--window C,W] [--iso V]
//                [--axis x|y|z --index I --slab N] [--curve FILE] [--up x,y,z] [--labels FILE [--outline]]
//                [--spp N] [--depth D] [--batched 0|1]
//                [--pt-mode 0|1|2] [--n N --w W --h H] [--out prefix] [--reps R] [--volume file.mhd|.mha] [--tf file.tf|app]
//                [--interact script.txt]
// --interact replays an interaction script through the windowless Canvas (include/svr_canvas.h: gui/canvas.cpp's
// event handlers, setters and frame protocol) instead of timing a render loop.  One command per line:
//   press X Y BUTTONS | move X Y BUTTONS | wheel DELTA | key left|right|down      (BUTTONS: 1 left, 4 middle)
//   mode pt|rc | depth D | density S | gradient G | fov F | exposure E | apeture A | focal L | clip x|y|z LO HI
//   envcolor R G B | envintensity I | envmap file.hdr | repaint 0|1 | paint N | save prefix
//   denoise 0|1|4|16      (SVR_OPT_PT_DENOISE: the denoised progressive display from the next restart of the render on)
// The whole script is parsed before the device is touched: a malformed line fails with exit code 2.
//
// --mode mip|minip|aip renders the maximum / minimum / average intensity projection (svr_render_projection) with the ray
// caster's step size, grey through the display window --window C,W (default 0.5,1); the .pfm then holds the projected values.
// --mode iso renders the white isosurface at --iso V (default 0.5; svr_render_isosurface) with the ray caster's step size.
// --mode slice renders the --w x --h slice (svr_render_slices) normal to --axis (default z: axial; y coronal, x sagittal) through
// voxel --index (default the middle one), one voxel per pixel, centred on the volume in the plane and oriented as
// scene.axis_slice; --slab N makes it the MIP of a slab of N voxels (one sample per voxel), grey through --window.
// --mode cpr renders the --w x --h straightened curved planar reformation (svr_render_curved) along the polyline of --curve FILE
// (whitespace-separated world xyz triples), the frame's roll fixed by --up (default 0,0,1), pixel and station spacing the
// smallest voxel spacing; --slab N and --window as for slices.
// --labels FILE loads a MetaImage label map (svr_labels_load_metaimage); it lines up with the volume when dims and spacing match.
// --mode labels renders its label surfaces (svr_render_labels) with the ray caster's step size, every label 1..max drawn in
// label_palette's colour (below; scene.label_palette in Python).  --mode slice with --labels overlays the labels on the grey slice
// (svr_render_label_slices) at half opacity, --outline drawing the outline pixels opaque.
// --volume loads a MetaImage file the way Canvas::LoadVolume does (core/VolumeReader.cpp:13-94) instead of
// generating the configuration's synthetic volume; camera and light are framed on its extent.
// --tf loads a transfer function saved by the application (gui/transferfunction.cpp:55-88); `app` is the
// application's start-up transfer function (gui/mainwindow.cpp:46-62).
//
// --batched 1 (default) renders the N samples in one svr_render_pathtracer_spp call; --batched 0
// calls the reference entry point render_pathtracer N times with frameNo = 0..N-1, exactly the
// frame protocol of Canvas::paintGL.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include <fstream>
#include <sstream>

#include "svr_canvas.h"
#include "svr_render.h"
#include "svr_tf_io.h"
#include "svr_volume_io.h"

#define CK(x)                                                                                   \
    do {                                                                                        \
        cudaError_t e_ = (x);                                                                   \
        if (e_ != cudaSuccess) {                                                                \
            fprintf(stderr, "CUDA error %s at %s:%d\n", cudaGetErrorString(e_), __FILE__, __LINE__); \
            return 1;                                                                           \
        }                                                                                       \
    } while (0)
#define SVR(x)                                                                   \
    do {                                                                         \
        if ((x) != 0) {                                                          \
            fprintf(stderr, "%s failed: %s\n", #x, svr_last_error());            \
            return 1;                                                            \
        }                                                                        \
    } while (0)

struct Config {
    const char* name;
    int n, format, kind, w, h;
    const char* tf;
    int depth, spp, env;
    unsigned seed;
};
static const Config kConfigs[] = {
    {"C1", 128, SVR_VOXEL_U8, SVR_GEN_SPHERE, 512, 512, "default", 1, 16, 0, 1234},
    {"C2", 256, SVR_VOXEL_U8, SVR_GEN_CT, 1024, 1024, "thin", 1, 1, 0, 1234},
    {"C3", 512, SVR_VOXEL_U16, SVR_GEN_CT, 1920, 1080, "default", 1, 256, 1, 1234},
    {"C4", 1024, SVR_VOXEL_F16, SVR_GEN_CLOUD, 1920, 1080, "cloud", 32, 512, 0, 42},
};

// colour nodes of the default transfer function, gui/mainwindow.cpp:57-62
static void tf_table(const std::string& kind, std::vector<float>& t)
{
    static const float xs[6] = {0.f, 0.2f, 0.4f, 0.6f, 0.8f, 1.f};
    static const float cs[6][3] = {{69, 199, 186}, {172, 3, 57}, {169, 83, 58}, {43, 32, 161}, {247, 158, 97}, {183, 7, 140}};
    const int n = SVR_TF_TABLE_SIZE;
    t.resize(4 * n);
    for (int i = 0; i < n; ++i) {
        double x = (double)i / (n - 1);
        int k = 0;
        while (k < 4 && x > xs[k + 1]) ++k;
        double f = (x - xs[k]) / (xs[k + 1] - xs[k]);
        for (int c = 0; c < 3; ++c) t[4 * i + c] = (float)(((1 - f) * cs[k][c] + f * cs[k + 1][c]) / 255.0);
        double o;
        if (kind == "thin") o = 0.02 * fmin(fmax((x - 0.1) / 0.9, 0.0), 1.0);
        else if (kind == "cloud") { o = 0.5 * x; t[4 * i] = t[4 * i + 1] = t[4 * i + 2] = 1.f; }
        else o = 0.5 * fmin(fmax(x / 0.1, 0.0), 1.0);
        t[4 * i + 3] = (float)o;
    }
}

// One line of an --interact script.  canvas == nullptr: parse only (non-zero = malformed); otherwise run it (non-zero = a call
// failed).  Blank lines and lines starting with '#' do nothing.
static int interact_line(svr_canvas* canvas, const std::string& line, int npix, int W, int H)
{
#define RUN(x)                   \
    do {                         \
        if (canvas) SVR(x);      \
    } while (0)
    std::istringstream ls(line);
    std::string cmd;
    if (!(ls >> cmd) || cmd[0] == '#') return 0;
    float a = 0.f, b = 0.f, c3 = 0.f;
    int n = 0;
    std::string word;
    if (cmd == "press" && ls >> a >> b >> n) RUN(svr_canvas_mouse_press(canvas, a, b, n));
    else if (cmd == "move" && ls >> a >> b >> n) RUN(svr_canvas_mouse_move(canvas, a, b, n));
    else if (cmd == "wheel" && ls >> n) RUN(svr_canvas_wheel(canvas, n));
    else if (cmd == "key" && ls >> word) RUN(svr_canvas_key(canvas, word == "left" ? SVR_KEY_LEFT : word == "right" ? SVR_KEY_RIGHT : SVR_KEY_DOWN));
    else if (cmd == "mode" && ls >> word) RUN(svr_canvas_set_render_mode(canvas, word == "pt" ? SVR_RENDER_MODE_PATHTRACER : SVR_RENDER_MODE_RAYCASTING));
    else if (cmd == "depth" && ls >> a) RUN(svr_canvas_set_scatter_times(canvas, a));
    else if (cmd == "density" && ls >> a) RUN(svr_canvas_set_density_scale(canvas, a));
    else if (cmd == "gradient" && ls >> a) RUN(svr_canvas_set_gradient_factor(canvas, a));
    else if (cmd == "fov" && ls >> a) RUN(svr_canvas_set_fov(canvas, a));
    else if (cmd == "exposure" && ls >> a) RUN(svr_canvas_set_exposure(canvas, a));
    else if (cmd == "apeture" && ls >> a) RUN(svr_canvas_set_apeture(canvas, a));
    else if (cmd == "focal" && ls >> a) RUN(svr_canvas_set_focal_length(canvas, a));
    else if (cmd == "clip" && ls >> word >> a >> b) RUN(svr_canvas_set_clip_plane(canvas, word == "x" ? 0 : word == "y" ? 1 : 2, a, b));
    else if (cmd == "envcolor" && ls >> a >> b >> c3) RUN(svr_canvas_set_env_background(canvas, a, b, c3));
    else if (cmd == "envintensity" && ls >> a) RUN(svr_canvas_set_env_intensity(canvas, a));
    else if (cmd == "envmap" && ls >> word) RUN(svr_canvas_set_env_map(canvas, word.c_str()));
    else if (cmd == "denoise" && ls >> n && (n == 0 || n == 1 || n == 4 || n == 16)) RUN(svr_set_option(SVR_OPT_PT_DENOISE, n));
    else if (cmd == "repaint" && ls >> n) {
        if (canvas) svr_canvas_set_immediate_repaint(canvas, n);
    } else if (cmd == "paint" && ls >> n) {
        for (int i = 0; i < n; ++i) RUN(svr_canvas_paint(canvas));
    } else if (cmd == "save" && ls >> word) {
        if (!canvas) return 0;
        std::vector<unsigned char> px((size_t)npix * 4);
        SVR(svr_canvas_read_image(canvas, px.data()));
        FILE* f = fopen((word + ".ppm").c_str(), "wb");
        if (f) {
            fprintf(f, "P6\n%d %d\n255\n", W, H);
            for (int y = H - 1; y >= 0; --y)
                for (int x = 0; x < W; ++x) fwrite(&px[4 * ((size_t)y * W + x)], 1, 3, f);
            fclose(f);
        }
    } else {
        return 2;
    }
    return 0;
#undef RUN
}

int main(int argc, char** argv)
{
    Config cfg = kConfigs[0];
    std::string mode = "pt", out = "svr_out", volumePath, tfPath;
    std::string interactPath;
    int batched = 1, ptMode = 2, reps = 3, sppArg = -1, depthArg = -1;
    float windowC = 0.5f, windowW = 1.f, isoValue = 0.5f;
    int sliceAxis = 2, sliceIndex = -1, slab = 0;
    std::string curvePath;
    float up[3] = {0.f, 0.f, 1.f};
    std::string labelsPath;
    int outline = 0;
    for (int i = 1; i < argc;) {
        std::string k = argv[i];
        if (k == "--outline") {  // the one option without a value
            outline = 1;
            ++i;
            continue;
        }
        if (i + 1 >= argc) break;
        std::string v = argv[i + 1];
        i += 2;
        if (k == "--config") {
            bool ok = false;
            for (const Config& c : kConfigs)
                if (v == c.name) cfg = c, ok = true;
            if (!ok) { fprintf(stderr, "unknown config %s\n", v.c_str()); return 2; }
        } else if (k == "--mode") mode = v;
        else if (k == "--spp") sppArg = atoi(v.c_str());
        else if (k == "--depth") depthArg = atoi(v.c_str());
        else if (k == "--batched") batched = atoi(v.c_str());
        else if (k == "--pt-mode") ptMode = atoi(v.c_str());
        else if (k == "--n") cfg.n = atoi(v.c_str());
        else if (k == "--w") cfg.w = atoi(v.c_str());
        else if (k == "--h") cfg.h = atoi(v.c_str());
        else if (k == "--out") out = v;
        else if (k == "--volume") volumePath = v;
        else if (k == "--tf") tfPath = v;
        else if (k == "--reps") reps = atoi(v.c_str());
        else if (k == "--interact") interactPath = v;
        else if (k == "--window") {
            if (sscanf(v.c_str(), "%f,%f", &windowC, &windowW) != 2) { fprintf(stderr, "--window wants C,W\n"); return 2; }
        } else if (k == "--iso") {
            if (sscanf(v.c_str(), "%f", &isoValue) != 1) { fprintf(stderr, "--iso wants a value\n"); return 2; }
        } else if (k == "--axis") {
            if (v != "x" && v != "y" && v != "z") { fprintf(stderr, "--axis wants x, y or z\n"); return 2; }
            sliceAxis = v[0] - 'x';
        } else if (k == "--index") sliceIndex = atoi(v.c_str());
        else if (k == "--slab") slab = atoi(v.c_str());
        else if (k == "--curve") curvePath = v;
        else if (k == "--labels") labelsPath = v;
        else if (k == "--up") {
            if (sscanf(v.c_str(), "%f,%f,%f", &up[0], &up[1], &up[2]) != 3) { fprintf(stderr, "--up wants x,y,z\n"); return 2; }
        }
        else { fprintf(stderr, "unknown option %s\n", k.c_str()); return 2; }
    }
    std::vector<std::string> script;
    if (!interactPath.empty()) {
        std::ifstream in(interactPath);
        if (!in) {
            fprintf(stderr, "cannot open %s\n", interactPath.c_str());
            return 1;
        }
        std::string line;
        for (int lineNo = 1; std::getline(in, line); ++lineNo) {
            if (interact_line(nullptr, line, 0, 0, 0)) {
                fprintf(stderr, "%s:%d: cannot parse '%s'\n", interactPath.c_str(), lineNo, line.c_str());
                return 2;
            }
            script.push_back(line);
        }
    }
    const int projMode = mode == "mip" ? SVR_PROJECT_MAX : mode == "minip" ? SVR_PROJECT_MIN : mode == "aip" ? SVR_PROJECT_MEAN : -1;
    if (sppArg > 0) cfg.spp = sppArg;
    if (depthArg >= 0) cfg.depth = depthArg;
    const int W = cfg.w, H = cfg.h;
    int N = cfg.n;
    const size_t npix = (size_t)W * H;

    SVR(svr_set_device(0));
    SVR(svr_set_option(SVR_OPT_PT_MODE, ptMode));
    SVR(svr_set_option(SVR_OPT_ENV_ENABLED, cfg.env));

    // ---- Canvas::LoadVolume (gui/canvas.cpp:27-41) with a synthetic volume instead of a MetaImage file
    svr_volume vol;
    uint32_t dims[3] = {(uint32_t)N, (uint32_t)N, (uint32_t)N};
    if (!volumePath.empty()) {
        svr_volume_stats vs;
        SVR(svr_volume_load_metaimage(volumePath.c_str(), &vol, &vs, nullptr, 0));
        const float ex = vs.dim[0] * vs.spacing[0], ey = vs.dim[1] * vs.spacing[1], ez = vs.dim[2] * vs.spacing[2];
        N = (int)fmaxf(ex, fmaxf(ey, ez));  // the extent the camera and the light are framed on (gui/canvas.cpp:191-197)
        for (int a = 0; a < 3; ++a) dims[a] = vs.dim[a];
        fprintf(stderr, "loaded %s: %u x %u x %u, spacing %g %g %g, range [%g, %g], max |grad| %g, %u histogram bins\n", volumePath.c_str(),
                vs.dim[0], vs.dim[1], vs.dim[2], vs.spacing[0], vs.spacing[1], vs.spacing[2], vs.data_min, vs.data_max,
                vs.max_gradient_magnitude, vs.histogram_bins);
    } else {
        const size_t bpv = cfg.format == SVR_VOXEL_U8 ? 1 : (cfg.format == SVR_VOXEL_F32 ? 4 : 2);
        void* dVox = nullptr;
        CK(cudaMalloc(&dVox, (size_t)N * N * N * bpv));
        SVR(svr_generate_volume(dVox, cfg.kind, cfg.format, N, cfg.seed));
        SVR(svr_volume_create(&vol, dVox, 1, cfg.format, N, N, N, 1.f, 1.f, 1.f, 0.f));
        CK(cudaFree(dVox));
    }
    setup_volume(&vol);
    svr_volume labels;
    memset(&labels, 0, sizeof(labels));
    uint32_t maxLabel = 0;
    if (!labelsPath.empty()) SVR(svr_labels_load_metaimage(labelsPath.c_str(), &labels, &maxLabel));
    if (mode == "labels" && labelsPath.empty()) { fprintf(stderr, "--mode labels wants --labels FILE\n"); return 2; }
    // label_palette (scene.py): label l in ((73 l + 91) mod 256, (151 l + 17) mod 256, (29 l + 193) mod 256) / 255
    svr_label_params palette;
    memset(&palette, 0, sizeof(palette));
    for (uint32_t l = 1; l <= maxLabel; ++l) {
        palette.color[l][0] = (float)((73u * l + 91u) & 255u) / 255.f;
        palette.color[l][1] = (float)((151u * l + 17u) & 255u) / 255.f;
        palette.color[l][2] = (float)((29u * l + 193u) & 255u) / 255.f;
        palette.color[l][3] = mode == "labels" ? 1.f : 0.5f;
    }

    std::vector<float> table;
    tf_table(cfg.tf, table);
    if (!tfPath.empty()) {
        svr_tf_opacity_node on[256];
        svr_tf_color_node cn[256];
        uint32_t no = 256, nc = 256;
        if (tfPath == "app") SVR(svr_tf_default_nodes(on, &no, cn, &nc));
        else SVR(svr_tf_file_read(tfPath.c_str(), on, &no, cn, &nc));
        float maxOpacity = 0.f;
        SVR(svr_tf_build_table(on, no, cn, nc, table.data(), SVR_TF_TABLE_SIZE, &maxOpacity));
        fprintf(stderr, "transfer function %s: %u opacity nodes, %u colour nodes, max opacity %g\n", tfPath.c_str(), no, nc, maxOpacity);
    }
    svr_transfer_function tf;
    SVR(svr_tf_create(&tf, table.data(), SVR_TF_TABLE_SIZE));
    setup_transferfunction(&tf);

    // camera framed as Canvas::ZoomToExtent does (gui/canvas.cpp:191-197), cuda_camera.h:34-47
    svr_camera cam;
    memset(&cam, 0, sizeof(cam));
    const float fov = 45.f;
    cam.imageW = W;
    cam.imageH = H;
    cam.exposure = 1.f;
    cam.apeture = 0.f;
    cam.focalLength = 1.f;
    cam.aspectRatio = (float)W / (float)H;
    cam.tanFovxOverTwo = tanf((float)(fov * 0.5f * M_PI / 180.f));
    cam.pos = {0.f, 0.f, (float)(1.5 * N / (2.0 * tan(fov * 0.5 * M_PI / 180.0)))};
    cam.u = {1, 0, 0};
    cam.v = {0, 1, 0};
    cam.w = {0, 0, 1};
    setup_camera(&cam);

    // MainWindow::onAddLight (gui/mainwindow.cpp:229-240), radius scaled with the volume
    svr_area_light light;
    const float R = 0.5f * sqrtf(3.f) * (float)N;
    light.disk.radius = 10.f * (float)N / 128.f;
    light.disk.center = {0.f, 1.5f * R + 1.f, 0.f};
    light.disk.normal = {0.f, -1.f, 0.f};
    light.color = {1, 1, 1};
    light.intensity = 500.f;
    setup_area_lights(&light, 1);
    svr_env_light env;
    memset(&env, 0, sizeof(env));
    env.defaultRadiance = {0.5f, 0.5f, 0.5f};  // gui/canvas.cpp:11-12
    env.intensity = 1.f;
    setup_env_lights(&env);

    if (!interactPath.empty()) {
        // ---- the windowless Canvas driven by a script of events and setters
        svr_canvas* canvas = svr_canvas_create((uint32_t)W, (uint32_t)H);
        if (!canvas) {
            fprintf(stderr, "svr_canvas_create failed: %s\n", svr_last_error());
            return 1;
        }
        const float size[3] = {2.f * vol.bbox.vmax.x, 2.f * vol.bbox.vmax.y, 2.f * vol.bbox.vmax.z};  // VolumeReader::GetVolumeSize
        const float radius = 0.5f * sqrtf(vol.spacing.x * vol.spacing.x + vol.spacing.y * vol.spacing.y + vol.spacing.z * vol.spacing.z);
        SVR(svr_canvas_set_volume(canvas, &vol, size, radius));
        SVR(svr_canvas_set_transfer_function(canvas, &tf));
        SVR(svr_canvas_set_area_lights(canvas, &light, 1));
        for (size_t i = 0; i < script.size(); ++i) {
            const int rc = interact_line(canvas, script[i], (int)npix, W, H);
            if (rc) return rc;
        }
        svr_camera cc;
        svr_canvas_get_camera(canvas, &cc);
        printf("{\"interact\": \"%s\", \"paints\": %llu, \"frame_no\": %u, \"camera_pos\": [%.4f, %.4f, %.4f], \"launches\": %llu}\n",
               interactPath.c_str(), (unsigned long long)svr_canvas_paint_count(canvas), svr_canvas_frame_no(canvas), cc.pos.x, cc.pos.y, cc.pos.z,
               (unsigned long long)svr_launch_count());
        svr_canvas_destroy(canvas);
        svr_volume_destroy(&vol);
        svr_tf_destroy(&tf);
        return 0;
    }

    // RenderParams::SetupHDRBuffer (render_parameters.h:17-23) and the image the PBO would be
    svr_render_params rp;
    rp.traceDepth = (uint32_t)cfg.depth;
    rp.frameNo = 0;
    CK(cudaMalloc((void**)&rp.hdrBuffer, npix * sizeof(svr_vec3)));
    CK(cudaMemset(rp.hdrBuffer, 0, npix * sizeof(svr_vec3)));
    svr_u8vec4* dImg = nullptr;
    CK(cudaMalloc((void**)&dImg, npix * 4));
    float* dValue = nullptr;
    if (projMode >= 0 || mode == "slice" || mode == "cpr") CK(cudaMalloc((void**)&dValue, npix * sizeof(float)));

    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0));
    CK(cudaEventCreate(&e1));
    // VolumeReader::GetElementBoundingSphereRadius (core/VolumeReader.cpp:198-201): half the voxel diagonal
    const float stepSize = 0.5f * sqrtf(vol.spacing.x * vol.spacing.x + vol.spacing.y * vol.spacing.y + vol.spacing.z * vol.spacing.z);
    const svr_projection_params proj = {projMode, stepSize, windowC, windowW};
    const svr_isosurface_params iso = {isoValue, stepSize, {1.f, 1.f, 1.f}};
    svr_slice_params slice;
    memset(&slice, 0, sizeof(slice));
    {
        static const int kU[3] = {1, 0, 0}, kV[3] = {2, 2, 1};  // sagittal U = +y, V = +z; coronal U = +x, V = +z; axial U = +x, V = +y
        const float sp[3] = {vol.spacing.x, vol.spacing.y, vol.spacing.z};
        const int a = sliceAxis;
        const int index = sliceIndex >= 0 ? sliceIndex : (int)dims[a] / 2;
        slice.center[a] = ((float)index + 0.5f - 0.5f * (float)dims[a]) * sp[a];
        slice.axisU[kU[a]] = sp[kU[a]];
        slice.axisV[kV[a]] = sp[kV[a]];
        slice.axisW[a] = sp[a];
        slice.imageW = (uint32_t)W;
        slice.imageH = (uint32_t)H;
        slice.count = 1;
        slice.mode = SVR_PROJECT_MAX;
        slice.thickness = (float)slab * sp[a];
        slice.sampleSpacing = sp[a];
        slice.windowCenter = windowC;
        slice.windowWidth = windowW;
    }
    std::vector<float> curve;
    svr_curved_params cpr;
    memset(&cpr, 0, sizeof(cpr));
    if (mode == "cpr") {
        std::ifstream cf(curvePath);
        if (curvePath.empty() || !cf) { fprintf(stderr, "--mode cpr wants --curve FILE (whitespace-separated xyz triples)\n"); return 2; }
        for (float x; cf >> x;) curve.push_back(x);
        if (curve.size() % 3 != 0) { fprintf(stderr, "%s: the number of values is not a multiple of 3\n", curvePath.c_str()); return 2; }
        const float sp = fminf(vol.spacing.x, fminf(vol.spacing.y, vol.spacing.z));
        memcpy(cpr.up, up, sizeof(up));
        cpr.layout = SVR_CURVED_STRAIGHTENED;
        cpr.imageW = (uint32_t)W;
        cpr.imageH = (uint32_t)H;
        cpr.count = 1;
        cpr.mode = SVR_PROJECT_MAX;
        cpr.pixelSpacing = sp;
        cpr.stationSpacing = sp;
        cpr.thickness = (float)slab * sp;
        cpr.sampleSpacing = sp;
        cpr.windowCenter = windowC;
        cpr.windowWidth = windowW;
    }
    float best = 1e30f;
    for (int rep = 0; rep < reps + 1; ++rep) {  // first pass warms up (and builds the macrocell grid)
        CK(cudaEventRecord(e0, 0));
        if (mode == "rc") {
            render_raycasting(dImg, &vol, &tf, &cam, stepSize);
        } else if (projMode >= 0) {
            SVR(svr_render_projection(dImg, dValue, &vol, &cam, &proj, 0, 1, nullptr));
        } else if (mode == "iso") {
            SVR(svr_render_isosurface(dImg, nullptr, &vol, &cam, &iso, 0, 1, nullptr));
        } else if (mode == "labels") {
            SVR(svr_render_labels(dImg, nullptr, nullptr, &labels, &cam, &palette, stepSize, 0, 1, nullptr));
        } else if (mode == "slice") {
            SVR(svr_render_slices(dImg, dValue, &vol, &slice));
            if (labels.tex) SVR(svr_render_label_slices(dImg, nullptr, &labels, &slice, &palette, outline));
        } else if (mode == "cpr") {
            SVR(svr_render_curved(dImg, dValue, &vol, &cpr, curve.data(), (uint32_t)(curve.size() / 3)));
        } else if (batched) {
            rp.frameNo = 0;
            SVR(svr_render_pathtracer_spp(dImg, &rp, (uint32_t)cfg.spp));
        } else {
            for (int f = 0; f < cfg.spp; ++f) {
                rp.frameNo = (uint32_t)f;
                render_pathtracer(dImg, &rp);
            }
        }
        CK(cudaEventRecord(e1, 0));
        CK(cudaEventSynchronize(e1));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        if (rep > 0 && ms < best) best = ms;
    }
    if (mode == "rc" || mode == "iso" || mode == "labels" || mode == "slice" || mode == "cpr" || projMode >= 0)
        printf("{\"config\": \"%s\", \"mode\": \"%s\", \"ms\": %.4f, \"mrays_per_s\": %.2f, \"launches\": %llu}\n", cfg.name, mode.c_str(),
               best, npix / (best * 1e-3) / 1e6, (unsigned long long)svr_launch_count());
    else
        printf("{\"config\": \"%s\", \"mode\": \"pt\", \"pt_mode\": %d, \"batched\": %d, \"spp\": %d, \"depth\": %d, \"ms\": %.4f, "
               "\"msamples_per_s\": %.2f, \"launches\": %llu}\n",
               cfg.name, ptMode, batched, cfg.spp, cfg.depth, best, npix * (double)cfg.spp / (best * 1e-3) / 1e6,
               (unsigned long long)svr_launch_count());

    // ---- images: PPM (rows flipped so +y is up) and PFM of the accumulator
    std::vector<unsigned char> img(npix * 4);
    CK(cudaMemcpy(img.data(), dImg, npix * 4, cudaMemcpyDeviceToHost));
    {
        FILE* f = fopen((out + ".ppm").c_str(), "wb");
        if (f) {
            fprintf(f, "P6\n%d %d\n255\n", W, H);
            for (int y = H - 1; y >= 0; --y)
                for (int x = 0; x < W; ++x) fwrite(&img[4 * ((size_t)y * W + x)], 1, 3, f);
            fclose(f);
        }
    }
    if (projMode >= 0 || mode == "slice" || mode == "cpr") {
        std::vector<float> value(npix);
        CK(cudaMemcpy(value.data(), dValue, npix * sizeof(float), cudaMemcpyDeviceToHost));
        FILE* f = fopen((out + ".pfm").c_str(), "wb");
        if (f) {
            fprintf(f, "Pf\n%d %d\n-1.0\n", W, H);
            fwrite(value.data(), sizeof(float), value.size(), f);
            fclose(f);
        }
    } else if (mode != "rc" && mode != "iso" && mode != "labels" && mode != "slice" && mode != "cpr") {
        std::vector<float> hdr(npix * 3);
        CK(cudaMemcpy(hdr.data(), rp.hdrBuffer, npix * 12, cudaMemcpyDeviceToHost));
        FILE* f = fopen((out + ".pfm").c_str(), "wb");
        if (f) {
            fprintf(f, "PF\n%d %d\n-1.0\n", W, H);
            fwrite(hdr.data(), sizeof(float), hdr.size(), f);
            fclose(f);
        }
    }
    svr_volume_destroy(&vol);
    svr_volume_destroy(&labels);
    svr_tf_destroy(&tf);
    cudaFree(rp.hdrBuffer);
    cudaFree(dImg);
    cudaFree(dValue);
    return 0;
}
