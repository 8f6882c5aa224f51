// svr_state.h -- host-side state shared by the translation units of libsvr_b200.so.
//
// Like the reference (one set of __constant__ scene PODs per process, pathtracer.cu:34-68) the
// library holds ONE scene per process and is not re-entrant; all work is issued on one stream.
#pragma once

#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <string>
#include <utility>

#include "../../include/svr_render.h"
#include "svr_scene.cuh"

namespace svr {

// A device allocation that only grows.  reserve(n) keeps the buffer when it holds n elements already, and otherwise replaces
// it; a failed allocation leaves {nullptr, 0} and returns the error.  A DevBuf of function scope frees its buffer on return.
template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t cap = 0;  // elements
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf& operator=(DevBuf&& o) noexcept
    {
        std::swap(p, o.p);
        std::swap(cap, o.cap);
        return *this;
    }
    ~DevBuf() { release(); }
    cudaError_t reserve(size_t n)
    {
        if (cap >= n) return cudaSuccess;
        release();
        const cudaError_t e = cudaMalloc(&p, n * sizeof(T));
        if (e != cudaSuccess) {
            p = nullptr;
            return e;
        }
        cap = n;
        return cudaSuccess;
    }
    void release()
    {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

// The render a sequence of render_pathtracer calls builds in one running mean: the next frame, the hdrBuffer, the image size
// and traceDepth.  A default record follows nothing.
struct FollowedRender {
    uint32_t next = 0, W = 0, H = 0, depth = 0;
    const void* hdr = nullptr;
    bool continues(uint32_t frameNo, const void* hdr_, uint32_t W_, uint32_t H_, uint32_t depth_) const
    {
        return hdr && frameNo == next && hdr_ == hdr && W_ == W && H_ == H && depth_ == depth;
    }
    void follow(uint32_t frameNo, const void* hdr_, uint32_t W_, uint32_t H_, uint32_t depth_)
    {
        next = frameNo + 1u;
        hdr = hdr_;
        W = W_;
        H = H_;
        depth = depth_;
    }
};

// Everything bound to the current device: its allocations, events and views, and the keys and flags that say what they hold
// (svr_set_device resets it)
struct DeviceState {
    // macrocell cache -- callee-owned derived data, keyed on the caller's cudaArray handle
    cudaArray_t gridArray = nullptr;      // volume array the range grid was built from
    int gridCell = 0;
    int3 gridDims = {0, 0, 0};
    int3 volDims = {0, 0, 0};
    DevBuf<float2> range;
    DevBuf<float> majorant;                // padded: (gx+2)(gy+2)(gz+2), one empty cell around the grid
    DevBuf<uint8_t> dist[2];               // ping-pong Chebyshev distance to the nearest non-empty cell
    DevBuf<int> occ;                       // bounding box of the non-empty cells: lo xyz, hi xyz
    int majorantLeap = -1;
    DevBuf<float> tfSparse;               // range-max sparse table over the TF opacity
    DevBuf<float4> tfTable;               // linear copy of the TF array
    int tfEntries = 0;
    cudaTextureObject_t volPointTex = 0;  // point-sampled view of gridArray
    cudaSurfaceObject_t uploadSurf = 0;   // store view of uploadSurfArray (svr_volume_upload from a device buffer, svr_macrocell.cu)
    cudaArray_t uploadSurfArray = nullptr;
    void* hMailbox = nullptr;             // 64 bytes of mapped pinned memory: small results reach the host without a copy engine
    void* dMailbox = nullptr;
    bool rangeValid = false;              // false until the range grid reflects the array's current voxels
    bool fingerprintDue = false;          // setup_volume was called since the voxels were last looked at
    DevBuf<unsigned long long> fingerprint;  // [0] sampled hash of the voxels the ranges were built from, [1] scratch
    bool majorantValid = false;           // false after setup_volume/setup_transferfunction
    float majorantDensityScale = 0.f;
    cudaArray_t majorantTfArray = nullptr;
    DevBuf<unsigned long long> tfHash;    // [0] hash of the TF table the majorants were built from, [1] of the live table, [2] stale flag
    cudaEvent_t tfCheckEvent = nullptr;   // behind the ray caster's per-call hash of the live table (svr_macrocell.cu: tf_check_*)
    bool tfCheckPending = false;

    // automatic macrocell size (SVR_OPT_MACROCELL_SIZE = 0): the choice and the scene it was made for
    int autoCell = 0;
    cudaArray_t autoArray = nullptr, autoTfArray = nullptr;
    float autoDensityScale = 0.f;
    unsigned autoEpoch = 0, uploadEpoch = 0;  // uploadEpoch counts svr_volume_upload / svr_tf_upload calls
    DevBuf<unsigned long long> stats;

    // importance sampler of the environment light (svr_env_io.cu), keyed on what it was built from
    DevBuf<float> envMarg;
    DevBuf<float> envCond;
    svr_env_light envSamplerKey = {};
    bool envSamplerValid = false;

    // Per-pixel classification (classify_pixel: entry skip, light cull, all-sky flag) kept across the 1-sample-per-call frames
    // of a progressive render: valid while sceneEpoch has not moved since it was stored
    DevBuf<float2> pixelCache;
    unsigned long long pixelCacheEpoch = 0;
    uint32_t pixelCacheW = 0, pixelCacheH = 0;
    int pixelCacheMode = -1;

    // Sample look-ahead of the 1-sample-per-call protocol (SVR_OPT_PT_LOOKAHEAD, svr_pathtrace.cu): the radiance of the samples
    // [aheadFirst, aheadFirst + aheadCount) of every pixel of aheadRender, computed in one sample-parallel launch
    DevBuf<float> ahead;
    FollowedRender aheadRender;
    uint32_t aheadFirst = 0, aheadCount = 0;
    unsigned long long aheadEpoch = 0;
    // does it pay for this scene?  timed once per scene epoch: a single-sample launch [0,1], the first batch [2,3], one fold [4,5]
    cudaEvent_t aheadEv[6] = {};
    bool aheadEvReady = false, aheadTimeFold = false;
    unsigned long long aheadSingleEpoch = 0, aheadTimedEpoch = 0, aheadOffEpoch = 0;
    uint32_t aheadTimedBatch = 0;

    // Adaptive sampling (svr_pathtracer_accumulate_adaptive): the offsets of the pixels still taking samples, and the counts
    // of the convergence pass (two slots of {active, unconverged}: a pass fills one and clears the other)
    DevBuf<uint32_t> adaptiveList;
    DevBuf<uint32_t> adaptiveCounts;

    // Denoising (svr_pathtracer_denoise, svr_denoise.cu): the filter's two ping-pong buffers of npix float4 (demodulated rgb,
    // variance), one after the other
    DevBuf<float4> denoise;

    // Denoised progressive display (SVR_OPT_PT_DENOISE, render_pathtracer): the even and odd frames' sample sums and the guides
    // (albedoCoverage, normalDepth) of progRender, four blocks of npix float4
    DevBuf<float4> prog;
    FollowedRender progRender;
    unsigned long long progGuideEpoch = 0;  // sceneEpoch after the frame that made the guides; 0 = none
    uint32_t progGuideRays = 0;

    DevBuf<Counters> counters;

    // Frees every allocation, event, view and the mailbox, and returns every key and flag to its default (svr_api.cu)
    void reset();
};

// The running mean `hdr` (null: none) was written outside the render look-ahead follows: the samples kept for that render no
// longer follow it.  anyHdr: whichever running mean it was (an ordinary path-tracing launch moves the one it writes on).
inline void hdr_written_outside(DeviceState& d, const void* hdr, bool anyHdr)
{
    if (hdr && (anyHdr || hdr == d.aheadRender.hdr)) d.aheadCount = 0;
}

struct HostState {
    cudaStream_t stream = nullptr;
    DevScene scene;  // what setup_* stored (zero-initialised in state())
    int options[SVR_OPT_COUNT_];
    DeviceState dev;
    unsigned long long sceneEpoch = 1;  // bumped by everything that can change what a pixel sees
    svr_denoise_params progParams;      // svr_pathtracer_set_denoise_params (state(): the defaults)
    unsigned long long launches = 0, fusedUploads = 0, aheadBatches = 0;
    std::string lastError;
};

HostState& state();

// largest empty-space leap, in cells, a macrocell can record (svr_macrocell.cu stage 3)
#define SVR_LEAP_CAP 15

// drops the macrocell cache (range grid, majorants, distances, point-sampled view)
void release_grid(HostState& st);

// Part-1 error convention, utils/helper_cuda.h:967-981: print, cudaDeviceReset, exit(EXIT_FAILURE)
inline void check_fatal(cudaError_t e, const char* what, const char* file, int line)
{
    if (e != cudaSuccess) {
        fprintf(stderr, "CUDA error at %s:%d code=%d(%s) \"%s\" \n", file, line, (int)e, cudaGetErrorName(e), what);
        cudaDeviceReset();
        exit(EXIT_FAILURE);
    }
}
#define SVR_FATAL(x) ::svr::check_fatal((x), #x, __FILE__, __LINE__)

// Part-2 error convention: record the text, return non-zero
int fail(const char* where, cudaError_t e);
int fail_msg(const char* msg);
#define SVR_TRY(x)                                             \
    do {                                                       \
        cudaError_t e_ = (x);                                  \
        if (e_ != cudaSuccess) return ::svr::fail(#x, e_);     \
    } while (0)

// Builds / refreshes the macrocell grid for (vol, tf) and fills scene->grid, scene->volDim.
// `force` rebuilds the majorants even when the cache key matches (ray caster: the TF content can
// change behind an unchanged handle, gui/transferfunction.cpp:128-151).
// `maxAutoCell` caps the automatic cell size: delta tracking through a thin medium wants large cells, the
// ray caster (which only skips empty space with the grid) never gains from cells above 8 voxels.
int ensure_grid(DevScene* scene, bool force, int maxAutoCell = 32);

// Stage 1 of the macrocell grid alone: the range grid of `vol`'s voxels (dev.range, dev.gridDims, dev.gridCell), which needs
// no transfer function.  cell = 0: the edge the cache holds for this array, else 8.  A new array or edge releases the whole
// grid; new voxels (svr_volume_upload, a setup_volume whose array holds other voxels) rebuild the ranges.
int ensure_ranges(const svr_volume& vol, int cell);

// true when the transfer-function table behind `tf` differs from the one the majorants were built from (one small
// launch + an 16-byte read-back; the ray caster's drop-in entry point, whose host may edit the table behind an unchanged
// handle, gui/transferfunction.cpp:128-151).  Also true when no majorants exist yet.
int tf_check_collect(bool* changed);
int tf_check_launch(const svr_transfer_function& tf, const unsigned int** staleFlag);
int upload_with_ranges(cudaArray_t arr, const cudaChannelFormatDesc& ch, const cudaExtent& ext, unsigned int flags, const void* devData, bool* done);

// Builds / refreshes the environment light's importance sampler for scene->env and fills scene->envS.
int ensure_env_sampler(DevScene* scene);

// Small results for the host through the mapped mailbox (svr_macrocell.cu): at most 32 bytes, synchronous with respect to
// the library's stream
int ensure_mailbox(HostState& st);
int read_small(HostState& st, void* host, const void* dev, size_t bytes);

// Denoising (svr_denoise.cu).  check_denoise_params: 0, or the error of `who` (before any CUDA call).  progressive_denoise: the
// guides and the filter of one denoised frame of render_pathtracer (SVR_OPT_PT_DENOISE) into img, after its sample has gone
// into the even or odd sum of dev.prog (frameNo & 1); ensure_progressive_buffers: false when they cannot be allocated.
int check_denoise_params(const char* who, const svr_denoise_params* paramsOrNull, svr_denoise_params* out);
bool ensure_progressive_buffers(HostState& st, size_t npix);
int progressive_denoise(uint32_t* img, uint32_t frameNo);

inline void count_launch(int n = 1) { state().launches += (unsigned long long)n; }

}  // namespace svr
