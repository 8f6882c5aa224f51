/*
 * svr_render.h -- C ABI of libsvr_b200.so, the B200-native drop-in for the render hot path of
 * SunVolumeRender (pathtracer.cu + raycasting.cu).
 *
 * Part 1 is the reference's own boundary: the seven unmangled symbols a host (gui/canvas.cpp or
 * tools/svr_headless.cpp) links against.  The reference declares them `extern "C"` with C++
 * reference parameters; a reference and a pointer are the same thing at the ABI level, so the
 * prototypes below are binary-identical to pathtracer.h:17-24 and raycasting.h:8 and a host
 * compiled against the reference headers links to this library unchanged (INTEGRATION.md).
 *
 * Part 2 is the headless extension the reference lacks: batched samples-per-pixel, float
 * outputs for parity checks, sum-buffers for the multi-GPU split, resource builders that mirror
 * the reference's loaders, synthetic volume generators and tap counters.
 *
 * All pointers named `img`, `hdrBuffer`, `sum`, `out`, `dev*` are DEVICE pointers unless the name
 * says host.  No torch types, no C++ types.
 */
#ifndef SVR_RENDER_H
#define SVR_RENDER_H

#include "svr_types.h"

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------
 * Part 1 -- the reference boundary (error convention = utils/helper_cuda.h:967-981: print
 * "CUDA error at file:line ...", cudaDeviceReset(), exit(EXIT_FAILURE); no return codes).
 * ------------------------------------------------------------------------------------------ */

/* pathtracer.h:17 / pathtracer.cu:292-304.  One call = one sample per pixel with seed stream
 * `frameNo`; frameNo == 0 clears hdrBuffer; hdrBuffer holds the running mean afterwards and img
 * the tone-mapped image.  Asynchronous on the library stream (svr_set_stream). */
void render_pathtracer(svr_u8vec4* img, const svr_render_params* renderParams);

/* pathtracer.h:20-24 / pathtracer.cu:34-68.  Copy the POD into library-owned device state.
 * setup_volume / setup_transferfunction also (re)build the macrocell majorant grid. */
void setup_volume(const svr_volume* vol);
void setup_transferfunction(const svr_transfer_function* tf);
void setup_camera(const svr_camera* cam);
void setup_env_lights(const svr_env_light* light);
void setup_area_lights(svr_area_light* lights, uint32_t n); /* n is clamped to 8 */

/* raycasting.h:8 / raycasting.cu:69-75.  Deterministic front-to-back compositing; takes its
 * scene by argument, not from setup_*.  stepSize = 0.5*|spacing| in the reference caller
 * (core/VolumeReader.cpp:198-201, gui/canvas.cpp:92); the march step is stepSize*0.5. */
void render_raycasting(svr_u8vec4* img, svr_volume* volume, svr_transfer_function* transferFunction,
                       svr_camera* camera, float stepSize);

/* ------------------------------------------------------------------------------------------
 * Part 2 -- headless extension.  Functions returning int: 0 = ok, non-zero = error
 * (svr_last_error() gives the text).  They never call exit().
 * ------------------------------------------------------------------------------------------ */

#define SVR_VERSION 100

int svr_version(void);
const char* svr_last_error(void);

/* Stream all launches and copies are issued on (a cudaStream_t; NULL = legacy default stream). */
int svr_set_stream(void* cuda_stream);
/* Bind the calling thread to a device and (re)initialise library state there. */
int svr_set_device(int device);

enum svr_option {
    /* path tracer estimator:
     *   0 = reference-compatible: global majorant, XORWOW stream seeded wangHash(frameNo)+pixel
     *       in the reference's draw order (path-exact twin of kernel_pathtracer);
     *   1 = global majorant, Philox4x32-10 counter RNG keyed (seed, pixel, sample);
     *   2 = local majorants (macrocell DDA) + Philox (default, fastest; same expectation). */
    SVR_OPT_PT_MODE = 0,
    /* shadow-ray estimator: 0 = binary delta tracking (transmittance.h:10-17), 1 = ratio tracking */
    SVR_OPT_SHADOW_ESTIMATOR = 1,
    /* 0 = escaped paths add nothing (pathtracer.cu:233 is commented out); 1 = add envLight */
    SVR_OPT_ENV_ENABLED = 2,
    /* macrocell edge in voxels: 0 (default) = chosen from the scene, about twice the mean free path inside
     * the medium, re-evaluated when volume, transfer function or density scale change; or a power of two in 2..64 */
    SVR_OPT_MACROCELL_SIZE = 3,
    /* skipping in the ray-marching kernels: the ray caster's empty-space skipping through the macrocell grid, the
     * projection's skipping of cells that cannot change the projected value (svr_render_projection) and the isosurface's
     * skipping of cells below the threshold (svr_render_isosurface), and the same projection skipping across a thick slab
     * (svr_render_slices; svr_render_curved for slabs of 32 samples or more), and the label surfaces' skipping of cells
     * that hold no visible label (svr_render_labels, through a label presence grid of its own): 0 off, 1 on (default) */
    SVR_OPT_RC_SKIP = 4,
    /* Philox key */
    SVR_OPT_SEED = 5,
    /* 1 = kernels also count taps / lookups / steps (slower; used for bytes_algo) */
    SVR_OPT_COUNTERS = 6,
    /* threads per block of the path tracer / ray caster (tuning) */
    SVR_OPT_PT_BLOCK = 7,
    SVR_OPT_RC_BLOCK = 8,
    /* path-tracer kernel shape: 2 = sample-parallel warp (the lanes of a warp take different samples of
     * the same pixel), 1 = megakernel (one pixel per lane, samples one after the other),
     * 0 = phase-scheduled warp (generate / march / collide / event / bounce phases, the warp
     * votes each round and runs the phase most lanes wait in), 3 = sample-parallel warp with the scatter
     * queue at every depth (see SVR_OPT_PT_QUEUE_MIN_DEPTH), 4 = majorant-profile kernel (see SVR_OPT_PT_PROFILE),
     * 5 = ray pool + event queue per warp: lanes take rays and scatter events from per-warp queues instead of owning a path */
    SVR_OPT_PT_KERNEL = 9,
    /* phase-scheduled kernel: macrocell visits per MARCH round (0 = default 4) */
    SVR_OPT_PT_ROUNDS = 10,
    /* 1 (default) = empty macrocells record how far the empty space around them extends and rays
     * leap over it; 0 = one cell at a time.  Images are bit-identical either way. */
    SVR_OPT_LEAP = 11,
    /* 1 (default) = each pixel finds once, along its centre ray, how far the camera rays of all its
     * samples can be advanced through empty macrocells; 0 = every sample walks from the volume face.
     * Images are bit-identical either way (only empty cells are skipped). */
    SVR_OPT_PT_ENTRY_CACHE = 12,
    /* sample-parallel kernel (SVR_OPT_PT_KERNEL = 2): pixels a warp renders one after the other (1..64; 0, the
     * default, lets the library choose by launch length: 1 from 128 samples per launch on, 2 below), and the
     * smallest batch (samples per pixel per launch) the kernel is used for; smaller batches run the megakernel.
     * Images differ from the other shapes only in float summation order. */
    SVR_OPT_PT_WARP_PIXELS = 13,
    SVR_OPT_PT_WARP_MIN_SPP = 14,
    /* SVR_OPT_PT_KERNEL = 2 with local majorants (SVR_OPT_PT_MODE = 2): from this traceDepth on the
     * sample-parallel kernel runs with a per-warp queue of scatter events in shared memory (kernel shape 3:
     * camera-ray rounds and scatter-event rounds that each start with all 32 lanes busy, however unequal the
     * path lengths).  Default 8; 0 = never.  Images differ from shape 2 only in float summation order. */
    SVR_OPT_PT_QUEUE_MIN_DEPTH = 15,
    /* 1 (default) = setup_volume / _transferfunction / _camera / _env_lights return after cudaDeviceSynchronize,
     * as the reference's do (pathtracer.cu:34-55).  0 = they only store the PODs (this library passes the scene
     * as kernel parameters, there is no device copy to wait for): a streaming host whose copy streams must keep
     * running across the setup calls of the next frame turns the synchronisation off. */
    SVR_OPT_SETUP_SYNC = 16,
    /* 1 (default) = a pixel whose camera rays provably pass every area-light disk skips get_nearest_light_sample
     * (pathtracer.cu:214-215); 0 = every camera ray tests every disk, as the reference does.  Images are
     * bit-identical either way (the cull is conservative). */
    SVR_OPT_PT_LIGHT_CULL = 17,
    /* 1 = with local majorants and a pinhole camera the sample-parallel shapes track camera rays against a per-pixel
     * majorant PROFILE the warp builds once per pixel (kernel shape 4: no lane walks a camera ray, every tentative
     * collision of a camera ray runs with the lanes packed; scatter queue as shape 3).  Same estimator, other random
     * walks: images agree with shapes 1-3 statistically.  0 (default) = shapes 2 / 3 as selected: the profile kernel
     * executes fewer cell visits but measured slower on every BASELINE configuration (DESIGN.md section 3.1). */
    SVR_OPT_PT_PROFILE = 18,
    /* shape 4: idle lanes take the pixel's next camera samples together once this many lanes wait (1..32, 0 = default 8) */
    SVR_OPT_PT_REFILL = 19,
    /* kernel shape 5 (ray pool + event queue per warp, SVR_OPT_PT_KERNEL = 5): pixels in a warp's run (1..16, 0 = default 16);
     * rays of all of them share the warp's pool */
    SVR_OPT_PT_POOL_PIXELS = 20,
    /* 1 = the environment light (when SVR_OPT_ENV_ENABLED) is a NEXT-EVENT target beside the area lights: at every scatter
     * event one of (area lights + environment) is picked uniformly; the environment is sampled by importance from its
     * luminance (a 512 x 256 direction grid built from the map, its offset and intensity; rebuilt when they change) and
     * weighted with both lobes of the shading model; bounce rays that leave the medium then add nothing.  Same
     * expectation as collecting the sky on escape (0, default: what the reference's commented-out line would do), far
     * lower variance for maps with small bright features.  Ignored by the reference-twin mode and kernel shape 5. */
    SVR_OPT_ENV_NEE = 21,
    /* sample-parallel kernel (shape 2): 1 = the warps of a block share one row of pixels and split every pixel's samples
     * between them (batches of at least 32 samples per warp); 0 (default) = one row per warp.  A pixel then occupies a warp
     * for a quarter of the time: shorter blocks, a shorter end of the launch -- for short frames (one frame divided over
     * several GPUs).  The image differs from 0 only in the order of four float additions per pixel. */
    SVR_OPT_PT_BLOCK_SPLIT = 22,
    /* Every pixel's classification -- how far its camera rays can skip empty space, whether they can hit a light, whether the
     * pixel is all sky -- is made for the whole image by a kernel of its own (one lane per pixel) and read by the render kernels
     * (shapes 1-3).  1 (default) = it is kept across launches -- the frames of a progressive render, the batches of an
     * accumulation -- and made again only after something a pixel can see has changed (any setup_*, upload or option);
     * 0 = made again for every launch.  Images are bit-identical either way (only empty space is skipped). */
    SVR_OPT_PT_PIXEL_CACHE = 23,
    /* 1 (default) = svr_volume_upload from a DEVICE buffer into an array made by svr_volume_create, once the macrocell grid
     * exists for that array, runs as one kernel that stores the voxels into the array and reduces the grid's value ranges from
     * the same pass (streamed time series: a new volume per frame).  0 = copy, then rebuild the ranges from the array at the
     * next render.  Arrays, ranges and images are bit-identical either way. */
    SVR_OPT_FUSED_UPLOAD = 24,
    /* render_pathtracer (one sample per call): once a progressive render has reached frame 16 with nothing changed, the next 32
     * samples of every pixel are computed in ONE launch of the sample-parallel kernel and kept; the following calls only fold the
     * kept sample of their frame into the running mean and tone-map (the same arithmetic on the same sample values: hdrBuffer and
     * image are bit-identical, frame for frame, to computing one sample per call).  Any setup_*, upload or option, a frameNo other
     * than the next one, another hdrBuffer, size or traceDepth discards what was kept.  Value = the batch (default 32, at most
     * 32); > 0: the library times one single-sample launch, the first batch and one fold per scene and stops batching for that
     * scene when it does not pay (views in which the volume fills the frame); < 0: always batch -value samples; 0, 1, -1 = off.
     * Not used with SVR_OPT_COUNTERS, nor where the scatter-queue kernel would run (traceDepth >= SVR_OPT_PT_QUEUE_MIN_DEPTH).
     * Memory: batch x pixels x 12 bytes (at most 1 GiB; larger canvases get smaller batches). */
    SVR_OPT_PT_LOOKAHEAD = 25,
    /* Denoised progressive display (DESIGN.md section 7g).  0 (default) = off.  1, 4 or 16 = on, with that many guide rays per
     * pixel (svr_pathtracer_guides) at the start of a render; other values are rejected.  While on, a render_pathtracer call
     * produces a DENOISED FRAME when SVR_OPT_COUNTERS is 0 and the call continues the render the library follows: frameNo == 0,
     * or frameNo is the previous call's plus 1 with the same hdrBuffer, imageW x imageH and traceDepth.  A denoised frame
     *   - traces one sample as the option-off call does: hdrBuffer is bit-identical to the option-off run;
     *   - adds the sample to library-owned float4 sums, one for the even frames and one for the odd ones (both cleared at
     *     frameNo == 0);
     *   - uses library-owned guide images made by svr_pathtracer_guides with the option's ray count before frame 16 and with
     *     16 rays from frame 16 on; they are remade when the scene has changed since they were made (any setup_*, upload or
     *     option) or the frame wants another ray count (so once at the first denoised frame >= 16, one hitch);
     *   - writes img as svr_pathtracer_denoise(img, NULL, even + odd, odd, guides, params) does, bit for bit, params as set
     *     by svr_pathtracer_set_denoise_params.  At frame 0 the odd half is empty: the luminance stop is off and the first
     *     frame after a change is an edge-avoiding blur guided by the guides alone.
     * Any other call renders as with the option off, and the library follows no render until the next frameNo == 0 (so turning
     * the option on in the middle of a render takes effect at the next restart).  svr_render_pathtracer_spp also ends it.
     * If the library cannot allocate its buffers the call renders as with the option off.  Look-ahead (SVR_OPT_PT_LOOKAHEAD)
     * is not used for denoised frames.  Memory: 4 x 16 bytes per pixel, kept, besides the filter's 2 x 16 bytes. */
    SVR_OPT_PT_DENOISE = 26,
    SVR_OPT_COUNT_
};
/* Defaults can also come from the environment, read once at first use, for hosts that only know the
 * seven reference entry points: SVR_PT_MODE, SVR_SHADOW_ESTIMATOR, SVR_ENV_ENABLED, SVR_RC_SKIP,
 * SVR_SEED, SVR_PT_KERNEL, SVR_PT_DENOISE (same values as the options; SVR_PT_DENOISE=4 gives the reference GUI a
 * denoised progressive display). */
int svr_set_option(int key, int value);
int svr_get_option(int key);

/* Equivalent to `spp` consecutive render_pathtracer calls with frameNo, frameNo+1, ... but in one
 * launch: samples accumulate in registers, hdrBuffer is read and written once, the tone map
 * runs once.  frameNo == 0 clears first.  img may be NULL (no tone map).  The equivalence holds for
 * hdrBuffer always and for img while SVR_OPT_PT_DENOISE is 0: this call ignores that option and ends the
 * render it follows (the next render_pathtracer call renders as with the option off until frameNo == 0). */
int svr_render_pathtracer_spp(svr_u8vec4* img, const svr_render_params* renderParams, uint32_t spp);

/* Multi-GPU building blocks (SURVEY.md section 8e).  `sum` is imageW*imageH float4: rgb = sum of
 * radiance samples, w = number of samples.  Samples [firstSample, firstSample+nSamples) are
 * rendered; clear != 0 zeroes `sum` first.  After an NCCL sum-reduce of the per-GPU buffers the
 * root calls svr_pathtracer_resolve: hdr = rgb / w (optional packed-vec3 output) and the
 * tone-mapped image (tonemapping.h:13-27), fused in one pass. */
int svr_pathtracer_accumulate(svr_vec4* sum, uint32_t traceDepth, uint32_t firstSample, uint32_t nSamples, int clear);
/* The IMAGE split of the multi-GPU path tracer (SURVEY.md section 8e, "interleaved image tiles, no reduce needed, only a
 * gather"): as svr_pathtracer_accumulate, for the row bands phase, phase + stride, ... only (bands of *bandRows rows, the
 * chosen kernel's block height, counted from row 0); rank r of N passes (r, N).  Pixels outside the call's bands are not
 * touched, so N ranks writing into ONE buffer (peer mappings of rank 0's buffer, svr_stage_*, svr_peer_*) assemble the frame
 * without a reduce, and every pixel's samples are summed by one GPU in the single-GPU order: the frame is bit-identical to
 * a single-GPU render.  Preferable to the sample split when there are few samples per GPU (per-pixel set-up is divided
 * too). */
int svr_pathtracer_accumulate_bands(svr_vec4* sum, uint32_t traceDepth, uint32_t firstSample, uint32_t nSamples, int clear,
                                    uint32_t phase, uint32_t stride, uint32_t* bandRows);
int svr_pathtracer_resolve(svr_u8vec4* img, svr_vec3* hdrOut, const svr_vec4* sum);
/* Adaptive sampling.  Clears sum and halfSum, then renders samples [firstSample, firstSample + n_p) of every pixel p into
 * them, n_p in {minSamples, minSamples + batch, ..., maxSamples}: sum as svr_pathtracer_accumulate (rgb += samples, w += count),
 * halfSum the samples whose offset from firstSample is odd (rgb, w = n_p / 2).  Resolve sum with svr_pathtracer_resolve.
 * The loop: every pixel takes minSamples; then, after each round, a pass over the image computes per pixel
 *     d_p   = max over r, g, b of |tone_map(even mean) - tone_map(odd mean)| / 2, with exposure cam.exposure,
 *             even mean = (sum - halfSum) / (w - halfSum.w), odd mean = halfSum / halfSum.w
 *             (the two halves differ by twice the standard error of the full mean: d_p estimates the displayed value's),
 *     err_p = RMS of d over the 3 x 3 window around p, coordinates clamped to the image,
 * and a pixel keeps sampling iff it took the last round, err_p >= threshold and w_p < maxSamples; those pixels take
 * min(batch, maxSamples - w) more samples.  A pixel that has stopped never restarts, so every round renders one sample range.
 * The loop ends when no pixel is left; reading each pass's counts costs one stream synchronisation per round.
 * threshold = 0 stops no pixel before maxSamples (err >= 0 always).  A pixel's samples are a function of (seed, pixel, sample),
 * and each pixel is summed by one warp in a fixed order: sum equals, bit for bit, the uniform svr_pathtracer_accumulate
 * sequence (firstSample, minSamples, clear) + (firstSample + minSamples + k batch, batch, no clear) truncated where the
 * pixel's w stops.
 * Kernel: the sample-parallel shape over a list of pixels, for every traceDepth (deep paths pay that shape's cost: the
 * scatter queue's per-lane order does not split samples by parity); SVR_OPT_PT_KERNEL, _PROFILE, _BLOCK_SPLIT and
 * _WARP_PIXELS do not apply.  Estimator modes 0-2 and SVR_OPT_ENV_NEE as elsewhere.  hdr buffers are not touched.
 * errOrNull: err_p of the final pass (imageW*imageH floats).  *roundsOut = render launches, *samplesOut = sum of w,
 * *unconvergedOut = pixels with err_p >= threshold in the final pass (any may be NULL).
 * Errors: null sum / halfSum; minSamples, maxSamples or batch not a positive multiple of 32; maxSamples < minSamples or
 * above 2^24; threshold < 0 or NaN; SVR_OPT_COUNTERS = 1; the scene checks of the other render calls. */
int svr_pathtracer_accumulate_adaptive(svr_vec4* sum, svr_vec4* halfSum, float* errOrNull, uint32_t traceDepth,
                                       uint32_t firstSample, uint32_t minSamples, uint32_t maxSamples, uint32_t batch,
                                       float threshold, uint32_t* roundsOut, uint64_t* samplesOut, uint32_t* unconvergedOut);
/* Denoising: guide images of the bound scene, then an edge-avoiding a-trous filter of an accumulated image (DESIGN.md 7f).
 * Guides.  Writes albedoCoverage and normalDepth (imageW*imageH float4 each, row-major like sum): the noise-free mean of what
 * a camera ray's first collision sees.  Delta tracking collides at density T(t) sigma(t), sigma = TF opacity per world unit
 * (the path tracer's extinction), so each ray marches from the volume's near face (clip planes included) to its far face or
 * the nearest area-light disk, whichever comes first, with step h = 0.5 min(spacing), samples at t0 + (k + 1/2) h, cells of
 * majorant <= 0 skipped through the macrocell grid; per sample p = T (1 - exp(-sigma h)), alpha += p, A += p rgb(TF),
 * Z += p dot(x - cam.pos, -cam.w) (view-space depth), N += p n (n = normalised gradient turned to face the ray's origin;
 * a zero gradient adds nothing), T *= exp(-sigma h); a ray stops at T < 1e-3.  raysPerPixel (1, 4 or 16) rays on a
 * sqrt(k) x sqrt(k) grid of sub-pixel positions ((i + 1/2) / sqrt(k), (j + 1/2) / sqrt(k)); with apeture > 0 the same
 * grid position is mapped to the lens disk (concentric mapping) and the ray passes through the focal plane as in
 * render_pathtracer.  Summed over the pixel's rays: albedoCoverage = (A / alpha, alpha / k), normalDepth = (normalize(N),
 * Z / alpha); 0 for all eight where alpha = 0.  Estimator modes and SVR_OPT_COUNTERS do not apply; one launch.
 * Errors: null outputs; raysPerPixel not 1, 4 or 16; the scene checks of the other render calls. */
int svr_pathtracer_guides(svr_vec4* albedoCoverage, svr_vec4* normalDepth, uint32_t raysPerPixel);
/* Filter parameters (svr_denoise_defaults fills the defaults: 5, 4, 128, 1, 0.1). */
typedef struct svr_denoise_params {
    uint32_t iterations;   /* a-trous iterations, 0..8 (steps 1, 2, 4, ...) */
    float sigmaLuminance;  /* luminance stop, in standard deviations of the pixel's estimate */
    float sigmaNormal;     /* normal stop exponent (0 = off) */
    float sigmaDepth;      /* depth stop, in pixel footprints per unit step */
    float sigmaCoverage;   /* coverage stop */
} svr_denoise_params;
int svr_denoise_defaults(svr_denoise_params* out);
/* Filter.  sum / halfSum as svr_pathtracer_accumulate_adaptive leaves them (for a uniform render: that call with
 * minSamples = maxSamples and threshold 0 -- one round, bit-identical to svr_pathtracer_accumulate -- fills halfSum), the
 * guides of svr_pathtracer_guides.  Outputs as svr_pathtracer_resolve: packed vec3 HDR and / or the tone-mapped image.
 *   demodulate: c = sum.rgb / sum.w, m = alpha albedo + (1 - alpha) per channel (at least 1e-3), e = c / m;
 *   variance:   Var = (l(even / m) - l(odd / m))^2 / 4, l = Rec. 709 luminance, even = (sum - halfSum) / (w - halfSum.w),
 *               odd = halfSum / halfSum.w; +inf where either half is empty (the luminance stop is then off); then the
 *               3 x 3 binomial filter, coordinates clamped;
 *   iteration i < iterations, step s = 2^i: 5 x 5 taps q = p + s (dx, dy), kernel h = [1/16, 1/4, 3/8, 1/4, 1/16] x h,
 *               taps outside the image dropped, weight w = h w_l w_n w_z w_a with
 *                 w_l = exp(-|l(e_p) - l(e_q)| / (sigmaLuminance sqrt(Var_p) + 1e-10)),
 *                 w_n = max(0, n_p . n_q)^sigmaNormal (1 if both normals are 0, 0 if one is; 1 for sigmaNormal = 0),
 *                 w_z = exp(-|z_p - z_q| / (sigmaDepth s f_p + 1e-10)), f_p = 2 z_p tanFovxOverTwo / (imageH - 1),
 *                 w_a = exp(-|alpha_p - alpha_q| / sigmaCoverage);
 *               e' = sum w e_q / sum w, Var' = sum w^2 Var_q / (sum w)^2 (taps of weight 0 add nothing);
 *   resolve:    hdr = m e, then the tone map and u8 packing of svr_pathtracer_resolve.
 * iterations = 0 is svr_pathtracer_resolve, bit for bit (that case skips the demodulation: m (c / m) is not c in float).
 * paramsOrNull = NULL: svr_denoise_defaults.  The filter's buffers are the library's (2 x 16 bytes per pixel, kept).
 * Errors, all reported before any CUDA call: null sum, halfSum or guide; both outputs null; iterations > 8; sigmaLuminance,
 * sigmaDepth or sigmaCoverage not positive or not finite; sigmaNormal negative or not finite; setup_camera not called. */
int svr_pathtracer_denoise(svr_u8vec4* imgOrNull, svr_vec3* hdrOutOrNull, const svr_vec4* sum, const svr_vec4* halfSum,
                           const svr_vec4* albedoCoverage, const svr_vec4* normalDepth, const svr_denoise_params* paramsOrNull);
/* The filter parameters of the denoised progressive display (SVR_OPT_PT_DENOISE); NULL restores svr_denoise_defaults.  Checked
 * as svr_pathtracer_denoise checks them, before any CUDA call.  Takes effect at the next denoised frame; the guides do not
 * depend on it, so the render goes on. */
int svr_pathtracer_set_denoise_params(const svr_denoise_params* paramsOrNull);

/* Staging buffers for streaming volumes to replicated scenes (SURVEY.md section 8e: the volume is replicated
 * per GPU; the reference is single-device, main.cpp:7-33, and has no counterpart).  One process per GPU:
 * every process allocates linear staging buffers (svr_stage_alloc = cudaMalloc), exports them to the
 * process that uploads (svr_stage_export = cudaIpcGetMemHandle, 64 bytes to send over any channel), which
 * imports them from ITS device (svr_stage_import = cudaIpcOpenMemHandle with lazy peer access, so the
 * mapping is a peer mapping over NVLink) and fills them with svr_stage_copy (cudaMemcpyAsync, kind
 * default: pinned host, local or imported peer memory -- copy engines only, no SMs, so the transfer runs
 * beside a render kernel that occupies every SM).  svr_volume_upload(vol, stage, 1) then moves the staged
 * voxels into the volume's cudaArray.  `stream` is a cudaStream_t. */
int svr_stage_alloc(void** dev_ptr, uint64_t bytes);
int svr_stage_free(void* dev_ptr);
int svr_stage_export(const void* dev_ptr, unsigned char handle_out[64]);
int svr_stage_import(const unsigned char handle[64], void** peer_ptr);
int svr_stage_release(void* peer_ptr);
int svr_stage_copy(void* dst, const void* src, uint64_t bytes, void* stream);

/* Completion flags between the GPUs of one box (ray casting on N GPUs without a collective): every rank renders its
 * bands straight into rank 0's image through a peer mapping of that buffer (svr_stage_alloc / _export / _import; pass
 * the mapped pointer as `img`), then raises rank 0's flag with svr_peer_signal (a peer mapping of an 8-byte,
 * zero-initialised svr_stage_alloc buffer: word 0 counts signals, word 1 is set when a wait timed out); rank 0's stream
 * waits with svr_peer_wait until word 0 has reached `expected` (wrap-safe; gives up after timeout_ms).  Both are
 * stream-ordered launches on the library's stream: no host synchronisation, no NCCL. */
int svr_peer_signal(void* peer_flag);
int svr_peer_wait(void* flag, uint32_t expected, uint32_t timeout_ms);

/* Ray caster variants: float RGBA before quantisation (parity is checked on these), and a row
 * range [y0, y1) for the image-tile split across GPUs.  out/img are full-frame buffers. */
int svr_render_raycasting_f32(svr_vec4* out, const svr_volume* volume, const svr_transfer_function* tf,
                              const svr_camera* camera, float stepSize);
int svr_render_raycasting_rows(svr_u8vec4* img, svr_vec4* outOrNull, const svr_volume* volume,
                               const svr_transfer_function* tf, const svr_camera* camera, float stepSize,
                               uint32_t y0, uint32_t y1);

/* The balanced split: the image is cut into bands of *bandRows rows (the kernel's block height), numbered from
 * the middle of the image outwards (0 = the middle band, 1 = the one below it, 2 = the one above, ...), and this
 * call renders bands phase, phase + stride, phase + 2 stride, ... -- rank r of N passes (r, N).  Contiguous row blocks
 * give the ranks that see the body several times the work of the ranks that see its margins; interleaved bands
 * do not.  Rows outside the call's bands are left untouched (zero the image first and sum-reduce the u8 images:
 * disjoint bands make the sum a gather; or let every rank write into one image through peer mappings, svr_peer_*).
 * The headless ray-cast entry points (_f32, _rows, _bands) rebuild the empty-space majorants when the transfer function's
 * HANDLE changes or an edit was announced (setup_transferfunction, svr_tf_upload); only render_raycasting itself also
 * checks the table's CONTENT on every call (the reference's host may change it behind an unchanged handle). */
int svr_render_raycasting_bands(svr_u8vec4* img, svr_vec4* outOrNull, const svr_volume* volume,
                                const svr_transfer_function* tf, const svr_camera* camera, float stepSize,
                                uint32_t phase, uint32_t stride, uint32_t* bandRows);

/* Intensity projections (DESIGN.md section 7h): maximum (MIP), minimum (MinIP) and average (AIP) of the volume along each
 * pixel-centre ray, no transfer function and no setup_* needed.  The ray is camera_ray_center's (pinhole, as
 * render_raycasting), clipped to the volume box and its clip planes (the axis-aligned slab) and to t >= 0: with
 * t0 = max(tNear, 0), h = 0.5 * stepSize and K = floor((tFar - t0) / h + 0.5), sample k (0 <= k < K) lies at
 * t0 + (k + 0.5) h and has the value v_k = tex3D(volume, p) * densityScale (the hardware trilinear fetch).  The projected value
 *   MAX:  P = max_k v_k        MIN:  P = min_k v_k        MEAN:  P = (v_0 + v_1 + ... + v_{K-1}) / K (fp32 sum in k order)
 * and P = 0 when K = 0 (a ray that misses the box, or a box behind the camera).  The divisions in K and g are fp32 with
 * fast-math rounding (within 2 ulp).  valueOrNull receives P (imageW*imageH floats);
 * imgOrNull the grey image g = clamp((P - (windowCenter - windowWidth / 2)) / windowWidth, 0, 1), packed as trunc(255 g) in
 * r, g and b with alpha 255.  Both are full-frame buffers; phase 0, stride 1 renders the frame, other values the bands of
 * svr_render_raycasting_bands (*bandRows = the band height; pixels outside the call's bands are not touched).
 * SVR_OPT_RC_SKIP = 1 (default) skips the samples of macrocells that cannot change P (MAX: cell maximum at or below the running
 * maximum; MIN: cell minimum at or above the running minimum; MEAN: a cell of zero voxels), from a range grid kept per volume
 * array (SVR_OPT_MACROCELL_SIZE, else the edge already built for that array, else 8); P is bit-identical either way.
 * Errors, all reported before any CUDA call: a null volume, camera or params; both outputs null; a mode out of range;
 * stepSize or windowWidth not positive or not finite; windowCenter not finite; phase >= stride. */
enum svr_projection_mode { SVR_PROJECT_MAX = 0, SVR_PROJECT_MIN = 1, SVR_PROJECT_MEAN = 2 };
typedef struct svr_projection_params {
    int32_t mode;        /* svr_projection_mode */
    float stepSize;      /* as render_raycasting: samples 0.5 * stepSize apart */
    float windowCenter;  /* display window on the projected value */
    float windowWidth;
} svr_projection_params;
int svr_render_projection(svr_u8vec4* imgOrNull, float* valueOrNull, const svr_volume* volume, const svr_camera* camera,
                          const svr_projection_params* params, uint32_t phase, uint32_t stride, uint32_t* bandRows);

/* Isosurface (DESIGN.md section 7i): the first place along each pixel-centre ray where the volume reaches isoValue, shaded as a
 * surface with the ray caster's headlight; no transfer function and no setup_* needed.  Rays and samples are
 * svr_render_projection's: t0 = max(tNear, 0), h = 0.5 * stepSize, K = floor((tFar - t0) / h + 0.5), sample k (0 <= k < K) at
 * t_k = t0 + (k + 0.5) h with the value v(t_k), v(t) = tex3D(volume, orig + t dir) * densityScale.
 *   hit:        k* = the smallest k with v_k >= isoValue; none: the ray misses.
 *   refinement: k* = 0: t_hit = t_0 (half a step past the entry: the cap where a clip plane or the camera cuts the solid).
 *               k* > 0: lo = t_{k*-1}, hi = t_{k*} (v_lo < isoValue <= v_hi), then 4 bisection steps m = (lo + hi) / 2,
 *               hi = m if v(m) >= isoValue, else lo = m (v_lo, v_hi follow), then
 *               t_hit = lo + (hi - lo) (isoValue - v_lo) / (v_hi - v_lo).  x_hit = orig + t_hit dir.
 *   normal:     g = the ray caster's 6-tap central-difference gradient at x_hit; n = normalize(g) turned to face the ray's
 *               origin if |g| > 1e-3, else n = 0.
 *   shading:    l = normalize(cam.pos - x_hit); n != 0: c = |n . l|, s = c^30; n = 0: c = 1, s = 0;
 *               rgb = min(color c 0.8 + s 0.2, 1).
 * imgOrNull receives (trunc(255 rgb), 255) for a hit and (0, 0, 0, 0) for a miss; surfaceOrNull (imageW*imageH float4)
 * receives (n, z) with z = dot(x_hit - cam.pos, -cam.w), the view-space depth of svr_pathtracer_guides, and (0, 0, 0, +inf)
 * for a miss.  Both are full-frame buffers; phase 0, stride 1 renders the frame, other values the bands of
 * svr_render_raycasting_bands (*bandRows = the band height; pixels outside the call's bands are not touched).  The divisions
 * in K and t_hit are fp32 with fast-math rounding (within 2 ulp).
 * SVR_OPT_RC_SKIP = 1 (default) skips the samples of macrocells whose maximum is below isoValue, from the range grid of
 * svr_render_projection (SVR_OPT_MACROCELL_SIZE, else the edge already built for that array, else 8); img and surface are
 * bit-identical either way.  With SVR_OPT_COUNTERS: paths = rays, steps = samples enumerated up to and including k* (K on a
 * miss), skipped = those of them dropped, shade_taps = those taken (steps = shade_taps + skipped), cells = cell visits; the
 * 4 refinement and 6 gradient taps of each hit are not counted.
 * Errors, all reported before any CUDA call: a null volume, camera or params; both outputs null; stepSize not positive or
 * not finite; isoValue not finite; a colour component not finite or outside [0, 1]; phase >= stride. */
typedef struct svr_isosurface_params {
    float isoValue;   /* threshold on tex3D * densityScale */
    float stepSize;   /* as render_raycasting / svr_render_projection: samples 0.5 * stepSize apart */
    float color[3];   /* surface colour, each in [0, 1] */
} svr_isosurface_params;
int svr_render_isosurface(svr_u8vec4* imgOrNull, svr_vec4* surfaceOrNull, const svr_volume* volume, const svr_camera* camera,
                          const svr_isosurface_params* params, uint32_t phase, uint32_t stride, uint32_t* bandRows);

/* Slices (DESIGN.md section 7j): a stack of `count` planar images of the volume, imageW x imageH each, in parallel projection:
 * thin slices (multi-planar reformatting: axial, coronal, sagittal or oblique) or thick slabs projected along the plane's
 * normal with svr_projection_mode; no transfer function, no camera and no setup_* needed.  In fp32:
 *   pixel centre: c = center + (x + 1/2 - W/2) axisU + (y + 1/2 - H/2) axisV + j axisW   (slice j, pixel (x, y))
 *   slab:         n = normalize(cross(axisU, axisV)); h = sampleSpacing; K = thickness > 0 ? max(1, floor(thickness / h + 1/2)) : 1;
 *                 t0 = -K h / 2; sample k (0 <= k < K) at x_k = c + s_k n, s_k = t0 + (k + 1/2) h (from k, as the projection
 *                 computes its samples).  A thin slice (thickness 0) is K = 1 with s_0 = 0: x_0 = c.
 *   value:        v_k = tex3D(volume, x_k) * densityScale (the hardware trilinear fetch).
 *   inclusion:    sample k is included iff cmin <= x_k <= cmax componentwise, cmin = vmin * (-x_clip.x, -y_clip.x, -z_clip.x),
 *                 cmax = vmax * (x_clip.y, y_clip.y, z_clip.y) (the clipped box of the projection).  Each component of x_k is
 *                 monotone in k, so the included samples are one index range [kLo, kHi), found by binary search.
 *   P:            MAX: max v_k; MIN: min v_k; MEAN: (fp32 sum in k order) / (kHi - kLo), over the included samples; 0 if none.
 * valueOrNull receives P at [(j * imageH + y) * imageW + x] (count * imageH * imageW floats); imgOrNull the grey image of
 * svr_render_projection (trunc(255 g) in r, g, b, alpha 255), and (0, 0, 0, 0) for a pixel with no included sample, so
 * "outside the volume" differs from "below the window".  The divisions in MEAN and g are svr_render_projection's.
 * SVR_OPT_RC_SKIP = 1 (default) walks slabs with K > 1 through svr_render_projection's range grid and drops samples by its
 * per-mode rules; P is bit-identical either way.  A thin slice takes its one fetch and never walks.  With SVR_OPT_COUNTERS:
 * paths = pixels * slices, steps = included samples, skipped = those dropped, shade_taps = those fetched
 * (steps = shade_taps + skipped), cells = cell visits.  SVR_OPT_RC_BLOCK sets the threads per block.
 * Errors, all reported before any CUDA call: a null volume or params; both outputs null; axisU or axisV not finite, or
 * cross(axisU, axisV) zero or not finite; axisW not finite when count > 1; imageW or imageH 0 or above 16384; count 0 or above
 * 65535; a mode out of range; thickness negative or not finite; sampleSpacing not positive or not finite while thickness > 0;
 * thickness / sampleSpacing above 65536; windowWidth not positive or not finite; windowCenter not finite. */
typedef struct svr_slice_params {
    float center[3];        /* world position of the centre of slice 0 */
    float axisU[3];         /* world step from a pixel to the next one in its row (x + 1) */
    float axisV[3];         /* world step from a row to the next (y + 1) */
    float axisW[3];         /* world step from a slice to the next (j + 1); ignored when count == 1 */
    uint32_t imageW, imageH, count;
    int32_t mode;           /* svr_projection_mode across the slab */
    float thickness;        /* slab thickness along n = normalize(cross(axisU, axisV)), world units; 0 = a thin slice */
    float sampleSpacing;    /* world distance between slab samples; used when thickness > 0 */
    float windowCenter, windowWidth;
} svr_slice_params;
int svr_render_slices(svr_u8vec4* imgOrNull, float* valueOrNull, const svr_volume* volume, const svr_slice_params* params);

/* Curved planar reformation (DESIGN.md section 7k): images of the volume along a centerline, for tubular structures (vessels,
 * airways, colon, spinal canal, dental arch).  `points` is a host array of nPoints xyz triples in world coordinates, a
 * polyline (callers pass a dense one: no spline is fitted).
 * Frame rule, on the host in double precision, the results rounded to float:
 *   1. every point equal to its predecessor is dropped; at least 2 points must remain, P_0 .. P_{M-1}.  S_0 = 0,
 *      S_{m+1} = S_m + |P_{m+1} - P_m|, L = S_{M-1}.
 *   2. c(s), s in [0, L], is linear on segment m, the last m <= M - 2 with S_m <= s: P_m + ((s - S_m) / (S_{m+1} - S_m)) (P_{m+1} - P_m).
 *   3. station i lies at s_i = (i + 1/2) stationSpacing, c_i = c(s_i); it is valid iff s_i <= L.  The valid stations are a prefix.
 *   4. t_i = normalize(c(min(s_i + D, L)) - c(max(s_i - D, 0))), D = stationSpacing; where that difference is zero (a curve
 *      that doubles back), the direction of the segment of s_i (rule 2).
 *   5. the rotation-minimising frame by double reflection (Wang, Juttler, Zheng and Liu 2008): r_0 = normalize(up - (up.t_0) t_0);
 *      r_{i+1} from r_i: v1 = c_{i+1} - c_i, r^L = r_i - (2 / v1.v1)(v1.r_i) v1, t^L = t_i - (2 / v1.v1)(v1.t_i) v1;
 *      v2 = t_{i+1} - t^L, r' = r^L - (2 / v2.v2)(v2.r^L) v2 (a zero v1 or v2 skips its reflection); r_{i+1} =
 *      normalize(r' - (r'.t_{i+1}) t_{i+1}).  b_i = t_i x r_i.
 *   6. an invalid station has zero vectors and valid = 0.
 * svr_curve_frames writes, per station, 4 svr_vec4: (c, valid), (t, 0), (r, 0), (b, 0).  It makes no CUDA call: a viewer maps
 * a CPR pixel back to a world position with it.
 * Pixel rule, fp32 on the device (fx = (x + 1/2) - W/2, fy = (y + 1/2) - H/2, ps = pixelSpacing):
 *   straightened (SVR_CURVED_STRAIGHTENED): N = imageH stations, row y is station y; image j (0 <= j < count) has
 *     theta_j = angle0 + j angleStep, (cos theta_j, sin theta_j) computed in double on the host and rounded to float.
 *     a = cos r + sin b, n = cos b - sin r (= t x a); pixel (x, y) of image j is at p = c_y + (fx ps) a; the slab runs along n.
 *     count > 1 is the rotational CPR stack.
 *   cross-sections (SVR_CURVED_CROSS): N = count stations, image j is station j, theta = angle0 (angleStep is ignored);
 *     a = cos r + sin b, e = cos b - sin r (= t x a); p = c_j + (fx ps) a + (fy ps) e; the slab runs along t (= a x e).
 *   slab, inclusion, fold and outputs: those of svr_render_slices on the ray (p, n) or (p, t): K, t0, s_k from k, the clipped
 *     box, the one index range [kLo, kHi), MAX / MIN / MEAN, the window, value[(j * imageH + y) * imageW + x], and alpha 0 for
 *     a pixel with no included sample.  A pixel of an invalid station gets P = 0 and alpha 0.
 * Counters as for svr_render_slices.  SVR_OPT_RC_SKIP = 1 (default) walks slabs with K >= 32 through the range grid with
 * svr_render_slices' rules (shorter slabs are faster without the walk, DESIGN.md section 7k); thin images and shorter slabs
 * never walk.  P is bit-identical with skipping on and off.  The frames and the (cos, sin) table go to the device through a library-owned
 * pinned staging buffer; a call waits on the host only for the copy that last read that buffer.
 * Errors, all reported before any CUDA call: a null volume, params or points; both outputs null; nPoints below 2 or above
 * 2^20; a point not finite; fewer than 2 distinct points; up not finite, zero, or parallel to t_0
 * (|up - (up.t_0) t_0| <= 1e-6 |up|); no valid station (the curve is shorter than half a station); layout out of range;
 * imageW or imageH 0 or above 16384; count 0 or above 65535; mode out of range; pixelSpacing or stationSpacing not positive or
 * not finite; angle0 or angleStep not finite; and the thickness, sampleSpacing and window errors of svr_render_slices.
 * svr_curve_frames makes the same checks on its arguments (a null up or hostFrames, or nStations 0, is an error). */
enum svr_curved_layout { SVR_CURVED_STRAIGHTENED = 0, SVR_CURVED_CROSS = 1 };
typedef struct svr_curved_params {
    float up[3];             /* fixes the roll of the frame at station 0 */
    int32_t layout;          /* svr_curved_layout */
    uint32_t imageW, imageH, count;
    int32_t mode;            /* svr_projection_mode across the slab */
    float pixelSpacing;      /* world distance between neighbouring pixels across the curve */
    float stationSpacing;    /* arc length between stations */
    float angle0, angleStep; /* radians, about the tangent */
    float thickness;         /* slab thickness, world units; 0 = thin */
    float sampleSpacing;     /* used when thickness > 0 */
    float windowCenter, windowWidth;
} svr_curved_params;

/* host only, no CUDA call: the frames of nStations stations, 4 svr_vec4 each: (c, valid), (t, 0), (r, 0), (b, 0) */
int svr_curve_frames(const float* points, uint32_t nPoints, const float up[3], float stationSpacing, uint32_t nStations,
                     svr_vec4* hostFrames);
int svr_render_curved(svr_u8vec4* imgOrNull, float* valueOrNull, const svr_volume* volume, const svr_curved_params* params,
                      const float* points, uint32_t nPoints);

/* Label maps (DESIGN.md section 7l): a segmentation, one u8 label id per voxel (0 = background), made by svr_labels_create or
 * svr_labels_load_metaimage on the grid of its image, drawn as shaded 3D surfaces (svr_render_labels) or as coloured overlays
 * on slices (svr_render_label_slices).  Only these two entry points read a label volume: the grey renderers do not check for
 * one and read its texture as if it were an image.  Both reject a volume whose texture is not a point-filtered, unnormalised,
 * element-type 8-bit unsigned array.
 * The table: label l is visible iff l != 0 and color[l][3] > 0; label 0 is never drawn.  Every entry, label 0's included, must
 * be finite and in [0, 1].  The table and its 256-bit visibility mask reach the kernels as a launch parameter: a change of
 * colours or visibility costs no copy and rebuilds nothing. */
typedef struct svr_label_params {
    float color[256][4];  /* per label id: r, g, b in [0, 1]; a in [0, 1], a = 0 hides the label */
} svr_label_params;

/* 3D label surfaces: the first place along each pixel-centre ray where the visible labels' indicator reaches 1/2, shaded with
 * the isosurface's headlight in the colour of the label found there.  Rays and samples are svr_render_projection's on the label
 * volume's box and clip planes: t0 = max(tNear, 0), h = 0.5 * stepSize, K = floor((tFar - t0) / h + 0.5), sample k at
 * t_k = t0 + (k + 0.5) h.  In fp32:
 *   indicator:  u = tex_coord(x) * (nx, ny, nz) - 1/2, i = floor(u), f = u - i per axis; vis(i, j, k) = 1 if voxel (i, j, k)
 *               lies inside the volume and holds a visible label, else 0; m(x) = the trilinear interpolation of vis over the 8
 *               corners i .. i + 1, lerp(a, b, f) = (1 - f) a + f b along x, then y, then z (8 point fetches; the hardware
 *               filter's 8-bit weights are not used).
 *   hit:        k* = the smallest k with m(t_k) >= 1/2; none: the ray misses.
 *   refinement: svr_render_isosurface's with v = m and isoValue = 1/2: k* = 0: t_hit = t_0; k* > 0: 4 bisection steps between
 *               t_{k*-1} and t_{k*}, then the linear interpolation.  t_hi = the final bisection upper bound (t_0 when k* = 0).
 *   label:      the visible label with the largest summed corner weight w = wx wy wz (wx = 1 - f.x or f.x, ...; summed in corner
 *               order, x fastest) at t_hi, ties to the smaller id.
 *   normal:     g = the analytic gradient of m at x_hit (the derivative of the trilinear weights) times
 *               (nx invSize.x, ny invSize.y, nz invSize.z), in world units; n = normalize(g) turned to face the ray's origin if
 *               |g|^2 > 0, else n = 0.
 *   shading:    svr_render_isosurface's headlight with color = color[label].rgb.
 * imgOrNull receives (trunc(255 rgb), 255) for a hit and (0, 0, 0, 0) for a miss; surfaceOrNull (n, view-space depth) as
 * svr_render_isosurface writes it, (0, 0, 0, +inf) for a miss; labelOrNull (imageW*imageH bytes) the label, 0 for a miss (for
 * picking).  phase, stride and *bandRows as for svr_render_isosurface.
 * SVR_OPT_RC_SKIP = 1 (default) drops the samples of macrocells whose label presence mask (the labels of the cell's voxels and
 * a one-voxel apron, every corner a sample of the cell can read) holds no visible label: m = 0 on all of them.  img, surface
 * and label are bit-identical either way.  The presence grid is kept per label array and cell edge (SVR_OPT_MACROCELL_SIZE,
 * else 8), apart from the grey volumes' range grid; svr_volume_upload into the array rebuilds it at the next call,
 * svr_volume_destroy releases it, and a new table never rebuilds it.  Counters as for svr_render_isosurface (shade_taps counts
 * indicator evaluations; the refinement, label and gradient work is not counted).
 * Errors, all reported before any launch or allocation: a null labels volume, camera or table; all three outputs null;
 * stepSize not positive or not finite; a table entry not finite or outside [0, 1]; phase >= stride; a volume that is not a
 * label volume (the only check that makes CUDA calls). */
int svr_render_labels(svr_u8vec4* imgOrNull, svr_vec4* surfaceOrNull, uint8_t* labelOrNull, const svr_volume* labels,
                      const svr_camera* camera, const svr_label_params* table, float stepSize, uint32_t phase, uint32_t stride,
                      uint32_t* bandRows);

/* Label overlays on slices: the labels of the pixels of svr_render_slices with the same params, so that the overlay lands on
 * the grey slice's pixels.  In fp32:
 *   pixel centre: c = svr_render_slices' (the slab's centre plane).
 *   label:        L = the label of voxel floor(tex_coord(c) * (nx, ny, nz)) (0 outside the volume), and L = 0 when c lies
 *                 outside the label volume's clipped box (svr_render_slices' inclusion rule applied to c alone).
 *   outline:      with outline = 1, a pixel with a visible L is an outline pixel when one of its 4 neighbours in the same image
 *                 has a different label; neighbours outside the image do not count.
 * labelOrNull receives L for every pixel at [(j * imageH + y) * imageW + x].  imgOrNull (the grey image of svr_render_slices,
 * count * imageH * imageW rgba) is composited in place: where L is visible, with a = color[L][3] (1 on an outline pixel), each
 * colour channel becomes trunc((1 - a) in + a (255 color) + 1/2) in correctly rounded fp32 operations and alpha 255; every other
 * pixel is left as it was.  No skipping: one fetch per pixel, and four more with outline.
 * Errors, all reported before any launch: a null labels volume, params or table; both outputs null; every parameter error of
 * svr_render_slices; a table entry not finite or outside [0, 1]; outline not 0 or 1; a volume that is not a label volume. */
int svr_render_label_slices(svr_u8vec4* imgOrNull, uint8_t* labelOrNull, const svr_volume* labels, const svr_slice_params* params,
                            const svr_label_params* table, int outline);

/* ---- resource builders (the input contract of the path) ---- */
enum svr_voxel_format { SVR_VOXEL_U8 = 0, SVR_VOXEL_U16 = 1, SVR_VOXEL_F16 = 2, SVR_VOXEL_F32 = 3 };

/* Mirrors VolumeReader::CreateTextures + CreateDeviceVolume (core/VolumeReader.cpp:138-185):
 * 3-D cudaArray, border addressing, linear filter, normalised-float reads (element reads for
 * f16/f32), normalised coordinates; bbox = +-0.5*dim*spacing; invMaxMagnitude = 1/maxGradMag
 * (maxGradMag <= 0: computed on the device by central differences on the raw values, f16/f32
 * scaled by 65535).  Clip planes (-1,1), densityScale 1, gradientFactor 0.5 (gui/canvas.cpp:19,31-32).
 * `data` is x-fastest; data_on_device selects the memcpy kind. */
int svr_volume_create(svr_volume* out, const void* data, int data_on_device, int format,
                      uint32_t nx, uint32_t ny, uint32_t nz, float sx, float sy, float sz, float maxGradMag);
int svr_volume_destroy(svr_volume* vol);
/* A label volume (svr_render_labels, svr_render_label_slices): nx*ny*nz u8 label ids, x fastest, into a 3-D u8 cudaArray
 * (surface load/store allowed, as svr_volume_create makes it) behind a texture with point filtering, element-type reads,
 * unnormalised coordinates and border addressing (a voxel outside the volume reads 0, the background).  bbox, spacing,
 * invSpacing and the clip planes are svr_volume_create's (a centred box), so a segmentation with the dims and spacing of its
 * image lines up with it; densityScale and gradientFactor are unused.  svr_volume_destroy, svr_volume_upload and
 * svr_volume_download take it as they take any volume. */
int svr_labels_create(svr_volume* out, const void* data, int data_on_device, uint32_t nx, uint32_t ny, uint32_t nz, float sx,
                      float sy, float sz);
/* Re-uploads voxels (same dims and format, x-fastest) into the array behind vol->tex -- the second
 * half of VolumeReader::CreateTextures (core/VolumeReader.cpp:146-161) for a volume that is already
 * bound -- and drops the macrocell cache built from the old contents.  Asynchronous on the library
 * stream when `data` is device or pinned host memory. */
int svr_volume_upload(const svr_volume* vol, const void* data, int data_on_device);
/* Drop cached macrocell data (keyed on the cudaArray handle); call after re-uploading voxels
 * into an existing array. */
int svr_volume_invalidate_cache(void);

/* Mirrors TransferFunction::TransferFunction (gui/transferfunction.cpp:17-44): 1024 float4
 * (r,g,b,opacity) -> 1-D cudaArray texture, linear, clamp, normalised; maxOpacity = max opacity. */
int svr_tf_create(svr_transfer_function* out, const float* host_rgba, uint32_t n);
int svr_tf_destroy(svr_transfer_function* tf);
/* New table contents (same size) into the array behind tf->tex; updates tf->maxOpacity.  The caller
 * then publishes the struct with setup_transferfunction, as after any edit. */
int svr_tf_upload(svr_transfer_function* tf, const float* host_rgba, uint32_t n);

/* Mirrors Lights::SetEnvironmentLight (core/lights/lights.cpp:31-75): w x h float4 lat-long map. */
int svr_env_create(svr_env_light* out, const float* host_rgba, uint32_t w, uint32_t h);
int svr_env_destroy(svr_env_light* env);

/* ---- synthetic volumes (SURVEY.md section 8d), written x-fastest into device memory ---- */
enum svr_volume_kind { SVR_GEN_SPHERE = 0, SVR_GEN_CT = 1, SVR_GEN_CLOUD = 2 };
int svr_generate_volume(void* dev_out, int kind, int format, uint32_t n, uint32_t seed);
/* max over voxels of the central-difference gradient magnitude (VolumeReader.cpp:70-76 semantics) */
int svr_max_gradient_magnitude(const void* dev_data, int format, uint32_t nx, uint32_t ny, uint32_t nz,
                               float sx, float sy, float sz, float* host_out);

/* ---- counters (valid while SVR_OPT_COUNTERS = 1) ---- */
enum svr_counter {
    SVR_CNT_TRACK_TAPS = 0,   /* volume taps in primary/secondary tracking loops */
    SVR_CNT_SHADOW_TAPS = 1,  /* volume taps in shadow-ray tracking */
    SVR_CNT_SHADE_TAPS = 2,   /* volume taps at scatter events / ray-cast steps (1 + 6 gradient) */
    SVR_CNT_TF_LOOKUPS = 3,   /* transfer-function lookups */
    SVR_CNT_SCATTERS = 4,     /* scatter events */
    SVR_CNT_PATHS = 5,        /* paths (pixel samples) or rays */
    SVR_CNT_CELLS = 6,        /* macrocells visited */
    SVR_CNT_STEPS = 7,        /* ray-cast steps executed (incl. skipped: see SKIPPED) */
    SVR_CNT_SKIPPED = 8,      /* ray-cast steps skipped as provably empty */
    SVR_CNT_COUNT_ = 16
};
int svr_counters_reset(void);
int svr_counters_read(uint64_t* host_out, uint32_t n);

/* Number of kernel launches issued by this library since load (bench.py's gpu_launches). */
uint64_t svr_launch_count(void);
/* How many svr_volume_upload calls took the one-pass path (SVR_OPT_FUSED_UPLOAD) since the library was loaded. */
uint64_t svr_fused_upload_count(void);
/* How many look-ahead batches (SVR_OPT_PT_LOOKAHEAD) render_pathtracer has launched since the library was loaded. */
uint64_t svr_lookahead_batch_count(void);

/* Gather-roofline microbenchmarks: `taps_per_thread` dependent-free tex3D taps per thread over
 * the bound volume, coherent (ray-like) or random.  Returns taps issued via *host_taps. */
int svr_microbench_taps(const svr_volume* vol, int random, uint32_t threads, uint32_t taps_per_thread,
                        float* dev_sink, uint64_t* host_taps);

/* Layout study behind the choice of voxel storage (DESIGN.md section 2): the same taps as svr_microbench_taps done in
 * software -- eight loads + the trilinear filter in the SM -- from a linear copy of n^3 16-bit voxels (layout 1, x fastest) or
 * from a bricked copy (layout 2: 8^3-voxel bricks, each contiguous, bricks in Morton order; svr_layout_brick makes it, n a
 * multiple of 8).  Not used by any render path. */
int svr_layout_brick(const void* dev_linear, void* dev_bricked, uint32_t n);
int svr_microbench_soft_taps(const void* dev_voxels16, uint32_t n, int layout, int random, uint32_t threads,
                             uint32_t taps_per_thread, float* dev_sink, uint64_t* host_taps);

/* ---- inspection hooks (used by the parity tests; cheap, never on the render path) ---- */
/* Raw fetches through the caller's texture objects, exactly as the kernels issue them:
 * out[i] = tex3D<float>(vol->tex, uvw[3i], uvw[3i+1], uvw[3i+2]) (normalised coordinates, before
 * densityScale); rgba[4i..] = tex1D<float4>(tf->tex, x[i]).  All pointers are device pointers. */
int svr_debug_sample_volume(const svr_volume* vol, const float* dev_uvw, uint32_t n, float* dev_out);
int svr_debug_sample_tf(const svr_transfer_function* tf, const float* dev_x, uint32_t n, float* dev_rgba);
/* Macrocell grid built for the scene of the last render call: dims[3] = cells per axis, *cell = edge
 * in voxels.  svr_grid_copy copies majorants (dims[0]*dims[1]*dims[2] floats, x fastest) and/or
 * the (min,max) intensity ranges (2 floats per cell) to HOST memory; either may be NULL. */
int svr_grid_info(int32_t* dims, int32_t* cell);
int svr_grid_copy(float* host_majorant, float* host_range);

#ifdef __cplusplus
}
#endif

#endif /* SVR_RENDER_H */
