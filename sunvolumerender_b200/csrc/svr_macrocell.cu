// svr_macrocell.cu -- macrocell majorant grid (callee-owned derived data; the reference has none:
// woodcock_tracking.h:28-30 uses the single global majorant tf.GetMaxOpacity()).
//
// Stages, so that the expensive one runs once per volume and the cheap ones on every
// transfer-function / density-scale edit:
//   1. range grid : per cell, min/max of every texel a trilinear fetch positioned inside the cell can
//      touch.  A fetch at texel-space coordinate xb = u*N - 0.5 reads texels floor(xb) and
//      floor(xb)+1, so positions inside cell c (u*N in [cC, (c+1)C)) read texels cC-1 .. (c+1)C.
//      The same texels cover every position up to HALF A VOXEL outside the cell (u*N in
//      [cC - 0.5, (c+1)C + 0.5)), which is orders of magnitude more slack than the float rounding of
//      world -> cell and world -> texture coordinates needs (1e-5 voxel), so no further apron.
//      Texels outside the array read 0 (border addressing, VolumeReader.cpp:164-166), and the
//      fixed-point filter weights are a convex combination, so every filtered value lies in
//      [min, max] of that footprint.
//   2. majorant grid: per cell, max TF opacity over the intensity interval [min,max]*densityScale
//      (cuda_volume.h:96, cuda_transfer_function.h:22-30; clamp addressing), answered in O(1) from a
//      sparse range-max table over the TF's opacity column.
//   3. empty-space distances: every cell whose majorant is 0 stores -(Chebyshev distance, in cells,
//      to the nearest cell with a non-zero majorant), capped at SVR_LEAP_CAP+1.  A ray inside such a
//      cell can leap to the boundary of the cube of radius distance-1 around it without a single
//      fetch (proximity clouds on the macrocell grid).  One float per cell carries both:
//      > 0 majorant, < 0 minus the leap distance.
//   4. occupied box: the bounding box, in cells, of the cells with a non-zero majorant; rays are
//      clipped to it.
// The majorant grid is stored with a one-cell empty border on every side so that a position-based
// walk needs no clamping at the volume faces.
// The boundary passes only a texture handle (cuda_volume.h:111-121); dims, format and voxels are
// recovered with cudaGetTextureObjectResourceDesc -> cudaArrayGetInfo.
#include <cuda_fp16.h>

#include <algorithm>
#include <climits>
#include <cstring>
#include <vector>

#include "svr_state.h"

namespace svr {
namespace {

__global__ void range_kernel(cudaTextureObject_t pointTex, int3 vol, int3 grid, int cell, float2* out)
{
    int cx = blockIdx.x, cy = blockIdx.y, cz = blockIdx.z;
    int R = cell + 2;  // [cC-1, (c+1)C]
    int x0 = cx * cell - 1, y0 = cy * cell - 1, z0 = cz * cell - 1;
    float mn = FLT_MAX, mx = -FLT_MAX;
    int total = R * R * R;
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
        int x = i % R, y = (i / R) % R, z = i / (R * R);
        // unnormalised point fetch at the texel centre; out-of-range reads the border value 0
        float v = tex3D<float>(pointTex, (float)(x0 + x) + 0.5f, (float)(y0 + y) + 0.5f, (float)(z0 + z) + 0.5f);
        mn = fminf(mn, v);
        mx = fmaxf(mx, v);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = fminf(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    __shared__ float smn[8], smx[8];
    int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        smn[w] = mn;
        smx[w] = mx;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int nw = blockDim.x >> 5;
        for (int i = 1; i < nw; ++i) {
            mn = fminf(mn, smn[i]);
            mx = fmaxf(mx, smx[i]);
        }
        out[((size_t)cz * grid.y + cy) * grid.x + cx] = make_float2(mn, mx);
    }
}

// The separable min/max reduction of a brick's texels (tile with its one-texel apron in shared memory) into the cells of
// the brick: along x, then y, then z.  Shared by the kernel that reads the array and the one that fills it (below).
struct RangeAsIs {
    static __device__ float finish(float x) { return x; }
};
// FIN::finish maps the reduced min / max to the value the volume texture returns (monotonic, so it commutes with min / max)
template <int CELL, class FIN>
__device__ __forceinline__ void reduce_brick(const float* tex, float2* rx, float2* ry, int cx0, int cy0, int cz0, int3 grid, float2* out)
{
    constexpr int BX = 32 / CELL, BY = CELL <= 8 ? 8 / CELL : 1, BZ = BY;
    constexpr int TX = BX * CELL + 2, TY = BY * CELL + 2, TZ = BZ * CELL + 2;
    for (int i = threadIdx.x; i < BX * TY * TZ; i += 256) {
        const int c = i % BX, y = (i / BX) % TY, z = i / (BX * TY);
        const float* row = tex + (z * TY + y) * TX + c * CELL;
        float mn = row[0], mx = row[0];
#pragma unroll
        for (int k = 1; k < CELL + 2; ++k) {
            mn = fminf(mn, row[k]);
            mx = fmaxf(mx, row[k]);
        }
        rx[(z * TY + y) * BX + c] = make_float2(mn, mx);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < BX * BY * TZ; i += 256) {
        const int c = i % BX, cy = (i / BX) % BY, z = i / (BX * BY);
        float2 r = rx[(z * TY + cy * CELL) * BX + c];
#pragma unroll
        for (int k = 1; k < CELL + 2; ++k) {
            const float2 v = rx[(z * TY + cy * CELL + k) * BX + c];
            r.x = fminf(r.x, v.x);
            r.y = fmaxf(r.y, v.y);
        }
        ry[(z * BY + cy) * BX + c] = r;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < BX * BY * BZ; i += 256) {
        const int c = i % BX, cy = (i / BX) % BY, cz = i / (BX * BY);
        float2 r = ry[((cz * CELL) * BY + cy) * BX + c];
#pragma unroll
        for (int k = 1; k < CELL + 2; ++k) {
            const float2 v = ry[((cz * CELL + k) * BY + cy) * BX + c];
            r.x = fminf(r.x, v.x);
            r.y = fmaxf(r.y, v.y);
        }
        const int gx = cx0 + c, gy = cy0 + cy, gz = cz0 + cz;
        if (gx < grid.x && gy < grid.y && gz < grid.z)
            out[((size_t)gz * grid.y + gy) * grid.x + gx] = make_float2(FIN::finish(r.x), FIN::finish(r.y));
    }
}

// The brick kernel below reads the caller's cudaArray through a point-sampled view (the boundary passes only
// a texture handle).  (Measured alternative: the same kernel fed from the linear device buffer an upload
// copies from -- coalesced 2-byte loads, bounds checks and 64-bit addressing per texel -- takes 0.83 ms at
// 512^3 against 0.37 ms for the texture path, whose address arithmetic and border handling are free.)
struct TexFetch {
    cudaTextureObject_t tex;
    // unnormalised point fetch at the texel centre; out-of-range reads the border value 0
    __device__ float operator()(int x, int y, int z) const { return tex3D<float>(tex, (float)x + 0.5f, (float)y + 0.5f, (float)z + 0.5f); }
};

// The same range grid for cell edges <= 16, a brick of cells per block: the brick's texels (plus the
// one-texel apron) are fetched ONCE into shared memory -- 1.3-1.7 fetches per voxel instead of
// (1 + 2/C)^3 -- and reduced separably (x, then y, then z).  The cell edge is a template parameter: every
// index decode is a division by a constant and the reductions unroll (the kernel is instruction-bound).
// brick = 32 x 8 x 8 voxels (32 x 16 x 16 for 16-voxel cells)
template <class Fetch, int CELL>
__global__ void __launch_bounds__(256) range_brick_kernel(Fetch fetch, int3 grid, float2* out)
{
    constexpr int BX = 32 / CELL, BY = CELL <= 8 ? 8 / CELL : 1, BZ = BY;
    constexpr int TX = BX * CELL + 2, TY = BY * CELL + 2, TZ = BZ * CELL + 2;
    constexpr int TOTAL = TX * TY * TZ;
    extern __shared__ float smem[];
    float* tex = smem;                      // TX * TY * TZ texels
    float2* rx = (float2*)(smem + TOTAL);   // BX * TY * TZ  (reduced along x)
    float2* ry = rx + BX * TY * TZ;         // BX * BY * TZ  (reduced along x, y)
    const int cx0 = blockIdx.x * BX, cy0 = blockIdx.y * BY, cz0 = blockIdx.z * BZ;
    const int x0 = cx0 * CELL - 1, y0 = cy0 * CELL - 1, z0 = cz0 * CELL - 1;
    // consecutive threads read consecutive texels of a row; four independent fetches are in flight before
    // the first result is stored
    for (int base = threadIdx.x; base < TOTAL; base += 4 * 256) {
        float v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * 256;
            if (i < TOTAL) {
                const int x = i % TX, y = (i / TX) % TY, z = i / (TX * TY);
                v[u] = fetch(x0 + x, y0 + y, z0 + z);
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = base + u * 256;
            if (i < TOTAL) tex[i] = v[u];
        }
    }
    __syncthreads();
    reduce_brick<CELL, RangeAsIs>(tex, rx, ry, cx0, cy0, cz0, grid, out);
}

template <class Fetch, int CELL>
int launch_range_brick_cell(HostState& st, Fetch fetch)
{
    constexpr int BX = 32 / CELL, BY = CELL <= 8 ? 8 / CELL : 1, BZ = BY;
    constexpr int TX = BX * CELL + 2, TY = BY * CELL + 2, TZ = BZ * CELL + 2;
    constexpr size_t shm = sizeof(float) * ((size_t)TX * TY * TZ + 2 * (size_t)BX * TY * TZ + 2 * (size_t)BX * BY * TZ);
    dim3 g((st.dev.gridDims.x + BX - 1) / BX, (st.dev.gridDims.y + BY - 1) / BY, (st.dev.gridDims.z + BZ - 1) / BZ);
    if (shm > 48 * 1024)
        SVR_TRY(cudaFuncSetAttribute(range_brick_kernel<Fetch, CELL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
    range_brick_kernel<Fetch, CELL><<<g, 256, shm, st.stream>>>(fetch, st.dev.gridDims, st.dev.range.p);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

template <class Fetch>
int launch_range_brick(HostState& st, Fetch fetch)
{
    switch (st.dev.gridCell) {
        case 2: return launch_range_brick_cell<Fetch, 2>(st, fetch);
        case 4: return launch_range_brick_cell<Fetch, 4>(st, fetch);
        case 8: return launch_range_brick_cell<Fetch, 8>(st, fetch);
        case 16: return launch_range_brick_cell<Fetch, 16>(st, fetch);
        default: return fail_msg("range grid: brick kernel needs a cell edge of 2, 4, 8 or 16");
    }
}

// ---- svr_volume_upload from a linear device buffer (a staged frame of a streamed time series): ONE pass reads the
// voxels, stores them into the cudaArray through a surface object and reduces the range grid from the same shared-memory
// tile, instead of a driver copy into the array followed by range_brick_kernel reading the array back (measured at 512^3
// u16 inside the streamed pipeline: 0.52 ms + 0.37 ms).  Row-wise: the 32 interior texels of a tile row are one
// coalesced warp load and one surface store, lanes 0 and 1 fetch the row's two apron texels; a row's address is computed
// once per warp.  Needs an array created with cudaArraySurfaceLoadStore (svr_volume_create does; a foreign array takes the
// copy + texture path).
// What a voxel reads as through the point-sampled view: normalised float for the integer formats (the texture unit
// returns the correctly rounded v / (2^n - 1); tests/test_gpu_resources.py holds the two paths bit-equal), the stored
// value for the float formats.  The division is monotonic, so the tile holds the integers (as exact floats) and only each
// cell's min and max are divided (the first version divided every texel: 60 % of the kernel's instructions).
struct VoxU8 {
    typedef unsigned char raw;
    static __device__ float value(raw v) { return (float)v; }
    static __device__ float finish(float x) { return __fdiv_rn(x, 255.f); }
};
struct VoxU16 {
    typedef unsigned short raw;
    static __device__ float value(raw v) { return (float)v; }
    static __device__ float finish(float x) { return __fdiv_rn(x, 65535.f); }
};
struct VoxF16 {
    typedef unsigned short raw;
    static __device__ float value(raw v) { return __half2float(__ushort_as_half(v)); }
    static __device__ float finish(float x) { return x; }
};
struct VoxF32 {
    typedef float raw;
    static __device__ float value(raw v) { return v; }
    static __device__ float finish(float x) { return x; }
};

template <class V, int CELL>
__global__ void __launch_bounds__(256) upload_range_kernel(const typename V::raw* __restrict__ src, cudaSurfaceObject_t surf, int3 dims,
                                                           int3 grid, float2* out)
{
    typedef typename V::raw raw;
    constexpr int BX = 32 / CELL, BY = CELL <= 8 ? 8 / CELL : 1, BZ = BY;
    constexpr int TX = BX * CELL + 2, TY = BY * CELL + 2, TZ = BZ * CELL + 2;
    static_assert(TX == 34, "a tile row is one warp of interior texels plus two apron texels");
    constexpr int TOTAL = TX * TY * TZ, ROWS = TY * TZ;
    extern __shared__ float smem[];
    float* tex = smem;
    float2* rx = (float2*)(smem + TOTAL);
    float2* ry = rx + BX * TY * TZ;
    const int cx0 = blockIdx.x * BX, cy0 = blockIdx.y * BY, cz0 = blockIdx.z * BZ;
    const int x0 = cx0 * CELL - 1, y0 = cy0 * CELL - 1, z0 = cz0 * CELL - 1;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int gx = x0 + 1 + lane;                    // this lane's interior texel
    const int ax = lane == 0 ? x0 : x0 + TX - 1;     // lanes 0, 1: the row's apron texels
    const bool inX = gx < dims.x, apX = lane < 2 && ax >= 0 && ax < dims.x;
    for (int r0 = warp; r0 < ROWS; r0 += 8 * 4) {
        raw v[4], e[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int r = r0 + u * 8;
            v[u] = 0;
            e[u] = 0;
            if (r < ROWS) {
                const int gy = y0 + r % TY, gz = z0 + r / TY;
                if (gy >= 0 && gy < dims.y && gz >= 0 && gz < dims.z) {  // outside the array: the border value 0
                    const raw* row = src + ((size_t)gz * dims.y + gy) * dims.x;
                    if (inX) v[u] = __ldg(row + gx);
                    if (apX) e[u] = __ldg(row + ax);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int r = r0 + u * 8;
            if (r < ROWS) {
                const int y = r % TY, z = r / TY;
                float* trow = tex + r * TX;
                trow[1 + lane] = V::value(v[u]);
                if (lane < 2) trow[lane == 0 ? 0 : TX - 1] = V::value(e[u]);
                const int gy = y0 + y, gz = z0 + z;
                // the brick's own texels (not the apron, which belongs to the neighbouring bricks) go into the array
                if (y >= 1 && y < TY - 1 && z >= 1 && z < TZ - 1 && inX && gy < dims.y && gz < dims.z)
                    surf3Dwrite(v[u], surf, gx * (int)sizeof(raw), gy, gz);
            }
        }
    }
    __syncthreads();
    reduce_brick<CELL, V>(tex, rx, ry, cx0, cy0, cz0, grid, out);
}

// The same pass for the common case -- rows of a multiple of 32 voxels, 16-byte aligned source: every memory instruction
// moves 16 bytes (8 u16 voxels), one load and one surface store per thread for a 32 x 8 x 8 brick of 2-byte voxels instead
// of one per voxel (the 2-byte surface stores of the kernel above cost it 1.4 ms at 512^3 u16; this one takes a quarter).
template <class V, int CELL>
__global__ void __launch_bounds__(256) upload_range_vec_kernel(const typename V::raw* __restrict__ src, cudaSurfaceObject_t surf, int3 dims,
                                                               int3 grid, float2* out)
{
    typedef typename V::raw raw;
    constexpr int BX = 32 / CELL, BY = CELL <= 8 ? 8 / CELL : 1, BZ = BY;
    constexpr int TX = BX * CELL + 2, TY = BY * CELL + 2, TZ = BZ * CELL + 2;
    constexpr int TOTAL = TX * TY * TZ, ROWS = TY * TZ;
    constexpr int PER = 16 / (int)sizeof(raw);  // voxels per 16-byte word
    constexpr int Q = 32 / PER;                 // words per tile row
    constexpr int ITEMS = ROWS * Q;
    extern __shared__ float smem[];
    float* tex = smem;
    float2* rx = (float2*)(smem + TOTAL);
    float2* ry = rx + BX * TY * TZ;
    const int cx0 = blockIdx.x * BX, cy0 = blockIdx.y * BY, cz0 = blockIdx.z * BZ;
    const int gx0 = cx0 * CELL, y0 = cy0 * CELL - 1, z0 = cz0 * CELL - 1;
    for (int i0 = threadIdx.x; i0 < ITEMS; i0 += 2 * 256) {
        uint4 w[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int i = i0 + u * 256;
            w[u] = make_uint4(0u, 0u, 0u, 0u);
            if (i < ITEMS) {
                const int r = i / Q, q = i % Q;
                const int gy = y0 + r % TY, gz = z0 + r / TY;
                if (gy >= 0 && gy < dims.y && gz >= 0 && gz < dims.z)  // outside the array: the border value 0
                    w[u] = __ldg((const uint4*)(src + ((size_t)gz * dims.y + gy) * dims.x + gx0) + q);
            }
        }
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int i = i0 + u * 256;
            if (i < ITEMS) {
                const int r = i / Q, q = i % Q;
                const int y = r % TY, z = r / TY;
                const int gy = y0 + y, gz = z0 + z;
                raw v[PER];
                memcpy(v, &w[u], 16);
                float* t = tex + r * TX + 1 + q * PER;
#pragma unroll
                for (int k = 0; k < PER; ++k) t[k] = V::value(v[k]);
                // the brick's own rows (not the apron rows, which belong to the neighbouring bricks) go into the array
                if (y >= 1 && y < TY - 1 && z >= 1 && z < TZ - 1 && gy < dims.y && gz < dims.z)
                    surf3Dwrite(w[u], surf, gx0 * (int)sizeof(raw) + q * 16, gy, gz);
            }
        }
    }
    // the two apron texels of every row
    for (int i = threadIdx.x; i < ROWS * 2; i += 256) {
        const int r = i >> 1, side = i & 1;
        const int gx = side ? gx0 + 32 : gx0 - 1, gy = y0 + r % TY, gz = z0 + r / TY;
        raw v = 0;
        if (gx >= 0 && gx < dims.x && gy >= 0 && gy < dims.y && gz >= 0 && gz < dims.z) v = __ldg(src + ((size_t)gz * dims.y + gy) * dims.x + gx);
        tex[r * TX + (side ? TX - 1 : 0)] = V::value(v);
    }
    __syncthreads();
    reduce_brick<CELL, V>(tex, rx, ry, cx0, cy0, cz0, grid, out);
}

template <class V, int CELL>
int launch_upload_range_cell(HostState& st, const void* src, cudaSurfaceObject_t surf)
{
    constexpr int BX = 32 / CELL, BY = CELL <= 8 ? 8 / CELL : 1, BZ = BY;
    constexpr int TX = BX * CELL + 2, TY = BY * CELL + 2, TZ = BZ * CELL + 2;
    constexpr size_t shm = sizeof(float) * ((size_t)TX * TY * TZ + 2 * (size_t)BX * TY * TZ + 2 * (size_t)BX * BY * TZ);
    dim3 g((st.dev.gridDims.x + BX - 1) / BX, (st.dev.gridDims.y + BY - 1) / BY, (st.dev.gridDims.z + BZ - 1) / BZ);
    if (st.dev.volDims.x % 32 == 0 && ((uintptr_t)src & 15u) == 0) {
        if (shm > 48 * 1024)
            SVR_TRY(cudaFuncSetAttribute(upload_range_vec_kernel<V, CELL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
        upload_range_vec_kernel<V, CELL><<<g, 256, shm, st.stream>>>((const typename V::raw*)src, surf, st.dev.volDims, st.dev.gridDims, st.dev.range.p);
    } else {
        if (shm > 48 * 1024)
            SVR_TRY(cudaFuncSetAttribute(upload_range_kernel<V, CELL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)shm));
        upload_range_kernel<V, CELL><<<g, 256, shm, st.stream>>>((const typename V::raw*)src, surf, st.dev.volDims, st.dev.gridDims, st.dev.range.p);
    }
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

template <class V>
int launch_upload_range(HostState& st, const void* src, cudaSurfaceObject_t surf)
{
    switch (st.dev.gridCell) {
        case 2: return launch_upload_range_cell<V, 2>(st, src, surf);
        case 4: return launch_upload_range_cell<V, 4>(st, src, surf);
        case 8: return launch_upload_range_cell<V, 8>(st, src, surf);
        case 16: return launch_upload_range_cell<V, 16>(st, src, surf);
        default: return fail_msg("range grid: brick kernel needs a cell edge of 2, 4, 8 or 16");
    }
}

// level l, entry i: max(opacity[i .. min(i + 2^l, n) - 1])
__global__ void tf_sparse_kernel(const float4* table, int n, int levels, float* sparse)
{
    for (int i = threadIdx.x; i < n; i += blockDim.x) sparse[i] = table[i].w;
    __syncthreads();
    for (int l = 1; l < levels; ++l) {
        int half = 1 << (l - 1);
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            float a = sparse[(l - 1) * n + i];
            int j = i + half;
            float b = j < n ? sparse[(l - 1) * n + j] : a;
            sparse[l * n + i] = fmaxf(a, b);
        }
        __syncthreads();
    }
}

// padded majorant grid <- max TF opacity over each cell's intensity range; also grows the occupied box
__global__ void majorant_kernel(const float2* range, int3 grid, const float* sparse, int n, float densityScale,
                                float* padded, int* occ)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, z = blockIdx.z;
    const bool inside = x < grid.x && y < grid.y;
    float m = 0.f;
    if (inside) {
        float2 r = range[((size_t)z * grid.y + y) * grid.x + x];
        float a = r.x * densityScale, b = r.y * densityScale;
        if (a > b) {
            float t = a;
            a = b;
            b = t;
        }
        // linear-filter footprint of tex1D at x: entries floor(x*n - 0.5) and +1 (clamped).  The unit
        // converts x*n - 0.5 to fixed point with 8 fractional bits, so widen the interval by 2/256 of an
        // entry; a coordinate rounded onto an entry boundary gives the entry beyond it weight 0.
        // (Widening by whole entries would make air, intensity exactly 0, inherit the opacity of
        // entry 1 and never be empty.)
        float fa = floorf(a * (float)n - 0.5f - 0.0078125f), fb = floorf(b * (float)n - 0.5f + 0.0078125f) + 1.f;
        if (!(fa == fa)) fa = 0.f;  // NaN voxels: cover the whole table
        if (!(fb == fb)) fb = (float)(n - 1);
        int lo = (int)fminf(fmaxf(fa, 0.f), (float)(n - 1));
        int hi = (int)fminf(fmaxf(fb, 0.f), (float)(n - 1));
        int len = hi - lo + 1;
        int k = 31 - __clz(len);
        m = fmaxf(fmaxf(sparse[k * n + lo], sparse[k * n + hi - (1 << k) + 1]), 0.f);
        int px = grid.x + 2, py = grid.y + 2;
        padded[((size_t)(z + 1) * py + (y + 1)) * px + (x + 1)] = m;
    }
    // occupied box: reduced over the warp first (a warp is one row of 32 cells), six atomics per warp with an occupied cell
    // instead of six per occupied cell (they all hit the same six words: the kernel took 0.085 ms at 128^3 cells, most of it here)
    const bool occupied = m > 0.f;
    const unsigned any = __ballot_sync(0xffffffffu, occupied);
    if (any) {
        const int xlo = __reduce_min_sync(0xffffffffu, occupied ? x : INT_MAX), xhi = __reduce_max_sync(0xffffffffu, occupied ? x : -1);
        const int ylo = __reduce_min_sync(0xffffffffu, occupied ? y : INT_MAX), yhi = __reduce_max_sync(0xffffffffu, occupied ? y : -1);
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&occ[0], xlo);
            atomicMin(&occ[1], ylo);
            atomicMin(&occ[2], z);
            atomicMax(&occ[3], xhi);
            atomicMax(&occ[4], yhi);
            atomicMax(&occ[5], z);
        }
    }
}

__global__ void occ_init_kernel(int* occ)
{
    if (threadIdx.x < 3) occ[threadIdx.x] = INT_MAX;
    else if (threadIdx.x < 6) occ[threadIdx.x] = -1;
}

// Chebyshev distance, in cells, from every cell to the nearest cell with a non-zero majorant, capped at
// cap + 1.  d(c) = min over occupied c' of max(|dx|, |dy|, |dz|), and max distributes over min, so the
// transform separates into three 1-D passes out[i] = min_j max(|i - j|, in[j]): 3 launches and <= 93
// reads per cell instead of `cap` dilation passes of 27 reads each.
//   FIRST: the input is the majorant grid itself (occupied = majorant > 0); LAST: the result is written back
//   into the majorant grid as -(distance) for the empty cells.
template <bool FIRST, bool LAST>
__global__ void dist_axis_kernel(const uint8_t* __restrict__ src, uint8_t* __restrict__ dst, float* __restrict__ majorant, int gx, int gy,
                                 int gz, int axis, int cap)
{
    int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y, z = blockIdx.z;
    if (x >= gx || y >= gy) return;
    const size_t i = ((size_t)z * gy + y) * gx + x;
    const int pos = axis == 0 ? x : (axis == 1 ? y : z), len = axis == 0 ? gx : (axis == 1 ? gy : gz);
    const ptrdiff_t stride = axis == 0 ? 1 : (axis == 1 ? gx : (ptrdiff_t)gx * gy);
    auto at = [&](ptrdiff_t j) -> int { return FIRST ? (majorant[j] > 0.f ? 0 : 255) : (int)src[j]; };
    int best = at((ptrdiff_t)i);
    for (int k = 1; k < best && k <= cap; ++k) {
        int a = pos - k >= 0 ? at((ptrdiff_t)i - k * stride) : 255;
        int b = pos + k < len ? at((ptrdiff_t)i + k * stride) : 255;
        best = min(best, max(k, min(a, b)));
    }
    best = min(best, cap + 1);
    if (LAST) {
        if (best > 0) majorant[i] = -(float)best;
    } else {
        dst[i] = (uint8_t)best;
    }
}

// Sampled hash of the voxels: 8192 point fetches at hashed positions (plus nothing else: a full checksum would cost
// what rebuilding the ranges costs).  Detects that the array behind an unchanged handle holds another volume.
__global__ void fingerprint_kernel(cudaTextureObject_t pointTex, int3 vol, unsigned long long* out)
{
    const uint32_t tid = blockIdx.x * blockDim.x + threadIdx.x;
    uint32_t h = tid * 0x9E3779B1u + 0x7F4A7C15u;
    h ^= h >> 15;
    h *= 0x2C1B3C6Du;
    h ^= h >> 12;
    const uint32_t x = h % (uint32_t)vol.x;
    h = h * 0x297A2D39u + 1u;
    h ^= h >> 15;
    const uint32_t y = h % (uint32_t)vol.y;
    h = h * 0x85EBCA6Bu + 1u;
    h ^= h >> 13;
    const uint32_t z = h % (uint32_t)vol.z;
    const float v = tex3D<float>(pointTex, (float)x + 0.5f, (float)y + 0.5f, (float)z + 0.5f);
    unsigned long long c = ((unsigned long long)__float_as_uint(v) + 1ull) * ((unsigned long long)tid * 0x9E3779B97F4A7C15ull + 0x632BE59BD9B4E019ull);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(out, c);
}

// Small control traffic stays off the copy engines.  A frame pipeline reads its images back with bulk device-to-host copies
// on another stream; a 16-byte cudaMemcpyAsync or an 8-byte cudaMemsetAsync issued meanwhile queues behind them on the same
// engine (measured: 0.3 ms per call beside a 33 MB read-back; the grid refresh of a streamed frame took 0.62 ms, most of it
// waiting).  So: words are zeroed by a kernel, and results travel to the host through a mapped pinned mailbox that a kernel
// writes, followed by a stream synchronize.
__global__ void zero_words_kernel(unsigned int* p, size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = 0u;
}

int zero_words(HostState& st, void* p, size_t bytes)
{
    const size_t n = bytes / 4;
    const unsigned blocks = n <= 1024 ? 1u : (unsigned)std::min<size_t>((n + 1023) / 1024, 148 * 8);
    zero_words_kernel<<<blocks, n <= 32 ? 32 : 256, 0, st.stream>>>((unsigned int*)p, n);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

__global__ void mailbox_kernel(const unsigned int* src, unsigned int* mailbox, int words)
{
    if ((int)threadIdx.x < words) mailbox[threadIdx.x] = src[threadIdx.x];
    __threadfence_system();
}

int launch_fingerprint(HostState& st, int slot)
{
    SVR_TRY(st.dev.fingerprint.reserve(2));
    if (int rc = zero_words(st, st.dev.fingerprint.p + slot, sizeof(unsigned long long))) return rc;
    fingerprint_kernel<<<64, 128, 0, st.stream>>>(st.dev.volPointTex, st.dev.volDims, st.dev.fingerprint.p + slot);
    count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

// 64-bit hash of a transfer-function table: of the linear copy the majorants are built from (tex == 0), or of the live
// array read through its texture object at the texel centres (where the linear filter returns the texel itself)
__global__ void tf_hash_kernel(const float4* table, cudaTextureObject_t tex, int n, unsigned long long* out, const unsigned long long* ref,
                               unsigned long long* mailbox, unsigned int* staleFlag)
{
    unsigned long long h = 0ull;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float4 v = table ? table[i] : tex1D<float4>(tex, ((float)i + 0.5f) / (float)n);
        unsigned long long e = ((unsigned long long)__float_as_uint(v.x) << 32 | __float_as_uint(v.y)) * 0x9E3779B97F4A7C15ull;
        e ^= ((unsigned long long)__float_as_uint(v.z) << 32 | __float_as_uint(v.w)) * 0xC2B2AE3D27D4EB4Full;
        h += (e ^ (e >> 29)) * ((unsigned long long)i * 2ull + 1ull);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) h += __shfl_xor_sync(0xffffffffu, h, o);
    // one block: the sum is written, not accumulated (no zeroing launch).  The ray caster's per-call check (ref != null): the
    // verdict goes to a device word the ray-cast kernel of the same frame reads (stale majorants -> it does not skip), and
    // both hashes to the host mailbox, which the NEXT call looks at -- no host synchronisation per frame.
    __shared__ unsigned long long part[32];
    if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = h;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (unsigned w = 1; w < (blockDim.x + 31u) / 32u; ++w) h += part[w];
        *out = h;
        if (ref) {
            const unsigned long long r = *ref;
            *staleFlag = r != h ? 1u : 0u;
            mailbox[0] = r;
            mailbox[1] = h;
            __threadfence_system();
        }
    }
}

int create_point_view(HostState& st, const cudaResourceDesc& vrd, const cudaChannelFormatDesc& ch)
{
    if (st.dev.volPointTex) cudaDestroyTextureObject(st.dev.volPointTex);
    st.dev.volPointTex = 0;
    cudaGetLastError();  // destroying a view whose array the host has freed may report an error: the view is gone either way
    cudaTextureDesc td;
    memset(&td, 0, sizeof(td));
    td.addressMode[0] = td.addressMode[1] = td.addressMode[2] = cudaAddressModeBorder;
    td.filterMode = cudaFilterModePoint;
    td.readMode = (ch.f == cudaChannelFormatKindFloat) ? cudaReadModeElementType : cudaReadModeNormalizedFloat;
    td.normalizedCoords = 0;
    SVR_TRY(cudaCreateTextureObject(&st.dev.volPointTex, &vrd, &td, nullptr));
    return 0;
}

}  // namespace

int ensure_mailbox(HostState& st)
{
    if (!st.dev.hMailbox) {
        SVR_TRY(cudaHostAlloc(&st.dev.hMailbox, 64, cudaHostAllocMapped | cudaHostAllocPortable));
        SVR_TRY(cudaHostGetDevicePointer(&st.dev.dMailbox, st.dev.hMailbox, 0));
    }
    return 0;
}

// host <- device, at most 32 bytes, synchronous with respect to the library's stream
int read_small(HostState& st, void* host, const void* dev, size_t bytes)
{
    if (bytes > 32 || (bytes & 3)) return fail_msg("read_small: at most 32 bytes, a multiple of 4");  // bytes 32..63 of the mailbox: tf_check_launch
    if (int rc = ensure_mailbox(st)) return rc;
    mailbox_kernel<<<1, 32, 0, st.stream>>>((const unsigned int*)dev, (unsigned int*)st.dev.dMailbox, (int)(bytes / 4));
    count_launch();
    SVR_TRY(cudaGetLastError());
    SVR_TRY(cudaStreamSynchronize(st.stream));
    memcpy(host, st.dev.hMailbox, bytes);
    return 0;
}

void release_grid(HostState& st)
{
    DeviceState& d = st.dev;
    if (d.volPointTex) cudaDestroyTextureObject(d.volPointTex);
    d.volPointTex = 0;
    if (d.uploadSurf) cudaDestroySurfaceObject(d.uploadSurf);
    d.uploadSurf = 0;
    d.uploadSurfArray = nullptr;
    cudaGetLastError();  // as for the view: the array behind it may be gone already
    d.range.release();
    d.majorant.release();
    d.dist[0].release();
    d.dist[1].release();
    d.occ.release();
    st.sceneEpoch++;
    d.gridArray = nullptr;
    d.autoArray = nullptr;  // the automatic cell size is re-derived for whatever volume comes next
    d.rangeValid = false;
    d.majorantValid = false;
}

// svr_volume_upload's fast path (see upload_range_kernel).  *done stays false when the array, the grid or the options do
// not allow it; the caller then copies with the driver and the ranges are rebuilt from the array at the next render.
int upload_with_ranges(cudaArray_t arr, const cudaChannelFormatDesc& ch, const cudaExtent& ext, unsigned int flags, const void* devData, bool* done)
{
    HostState& st = state();
    *done = false;
    if (!st.options[SVR_OPT_FUSED_UPLOAD] || !(flags & cudaArraySurfaceLoadStore)) return 0;
    if (arr != st.dev.gridArray || !st.dev.range.p || !st.dev.volPointTex || st.dev.gridCell > 16) return 0;
    // setup_volume since the last render: the array behind the handle may be a new one (build_grid looks first)
    if (st.dev.fingerprintDue) return 0;
    if ((int)ext.width != st.dev.volDims.x || (int)ext.height != st.dev.volDims.y || (int)ext.depth != st.dev.volDims.z) return 0;
    if (ch.y || ch.z || ch.w) return 0;
    const bool isFloat = ch.f == cudaChannelFormatKindFloat, isUint = ch.f == cudaChannelFormatKindUnsigned;
    if (!((isUint && (ch.x == 8 || ch.x == 16)) || (isFloat && (ch.x == 16 || ch.x == 32)))) return 0;
    if (st.dev.uploadSurfArray != arr) {
        if (st.dev.uploadSurf) cudaDestroySurfaceObject(st.dev.uploadSurf);
        st.dev.uploadSurf = 0;
        st.dev.uploadSurfArray = nullptr;
        cudaGetLastError();
        cudaResourceDesc rd;
        memset(&rd, 0, sizeof(rd));
        rd.resType = cudaResourceTypeArray;
        rd.res.array.array = arr;
        SVR_TRY(cudaCreateSurfaceObject(&st.dev.uploadSurf, &rd));
        st.dev.uploadSurfArray = arr;
    }
    int rc;
    if (isUint && ch.x == 8) rc = launch_upload_range<VoxU8>(st, devData, st.dev.uploadSurf);
    else if (isUint) rc = launch_upload_range<VoxU16>(st, devData, st.dev.uploadSurf);
    else if (ch.x == 16) rc = launch_upload_range<VoxF16>(st, devData, st.dev.uploadSurf);
    else rc = launch_upload_range<VoxF32>(st, devData, st.dev.uploadSurf);
    if (rc) return rc;
    st.dev.rangeValid = true;
    st.dev.majorantValid = false;
    rc = launch_fingerprint(st, 0);  // of the voxels these ranges describe
    if (rc) return rc;
    st.fusedUploads++;
    *done = true;
    return 0;
}

// sum and count of the non-zero majorants (the statistic behind the automatic cell size)
__global__ void majorant_stats_kernel(const float* __restrict__ majorant, size_t cells, double* sum, unsigned long long* count)
{
    float s = 0.f;
    unsigned int c = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < cells; i += (size_t)gridDim.x * blockDim.x) {
        float m = majorant[i];
        if (m > 0.f) {
            s += m;
            ++c;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        c += __shfl_xor_sync(0xffffffffu, c, o);
    }
    if ((threadIdx.x & 31) == 0 && c) {
        atomicAdd(sum, (double)s);
        atomicAdd(count, (unsigned long long)c);
    }
}

int ensure_ranges(const svr_volume& vol, int cell)
{
    HostState& st = state();
    if (!vol.tex) return fail_msg("ensure_ranges: volume texture is not set");
    cudaResourceDesc vrd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&vrd, vol.tex));
    if (vrd.resType != cudaResourceTypeArray) return fail_msg("ensure_grid: textures must be bound to cudaArrays");
    cudaArray_t varr = vrd.res.array.array;

    cudaChannelFormatDesc ch;
    cudaExtent ext;
    unsigned int flags = 0;
    SVR_TRY(cudaArrayGetInfo(&ch, &ext, &flags, varr));
    if (ext.depth == 0) return fail_msg("ensure_grid: volume array is not 3-D");
    if (varr == st.dev.gridArray && st.dev.range.p && st.dev.fingerprintDue) {
        // setup_volume was called since the voxels were last looked at, with a struct that names the same resources
        // (svr_api.cu: setup_volume).  The array behind the handle may still be another one (freed and reallocated by
        // the host): compare its dims, take a fresh point-sampled view of it, and compare a sampled hash of its voxels
        // with the one taken when the ranges were built.
        if ((int)ext.width != st.dev.volDims.x || (int)ext.height != st.dev.volDims.y || (int)ext.depth != st.dev.volDims.z) {
            release_grid(st);
        } else {
            int rc = create_point_view(st, vrd, ch);
            if (rc) return rc;
            if (st.dev.rangeValid) {
                rc = launch_fingerprint(st, 1);
                if (rc) return rc;
                unsigned long long h[2] = {0, 1};
                rc = read_small(st, h, st.dev.fingerprint.p, sizeof(h));
                if (rc) return rc;
                if (h[0] != h[1]) st.dev.rangeValid = false;
            }
        }
    }
    st.dev.fingerprintDue = false;
    if (cell == 0) cell = varr == st.dev.gridArray && st.dev.range.p ? st.dev.gridCell : 8;
    if (varr != st.dev.gridArray || cell != st.dev.gridCell || !st.dev.range.p) {
        // ---- allocate for this (array, cell size)
        release_grid(st);
        int rcv = create_point_view(st, vrd, ch);
        if (rcv) return rcv;

        st.dev.volDims = make_int3((int)ext.width, (int)ext.height, (int)ext.depth);
        st.dev.gridDims = make_int3((st.dev.volDims.x + cell - 1) / cell, (st.dev.volDims.y + cell - 1) / cell,
                                (st.dev.volDims.z + cell - 1) / cell);
        size_t cells = (size_t)st.dev.gridDims.x * st.dev.gridDims.y * st.dev.gridDims.z;
        SVR_TRY(st.dev.range.reserve(cells));
        st.dev.gridArray = varr;
        st.dev.gridCell = cell;
        st.dev.rangeValid = false;
    }
    if (!st.dev.rangeValid) {
        // ---- stage 1: range grid (again after svr_volume_upload: same allocations, new voxels)
        if (cell <= 16) {
            int rc = launch_range_brick(st, TexFetch{st.dev.volPointTex});
            if (rc) return rc;
        } else {
            dim3 g(st.dev.gridDims.x, st.dev.gridDims.y, st.dev.gridDims.z);
            range_kernel<<<g, 128, 0, st.stream>>>(st.dev.volPointTex, st.dev.volDims, st.dev.gridDims, cell, st.dev.range.p);
            count_launch();
            SVR_TRY(cudaGetLastError());
        }
        st.dev.rangeValid = true;
        st.dev.majorantValid = false;
        int rc = launch_fingerprint(st, 0);  // of the voxels these ranges describe (stays on the device until it is needed)
        if (rc) return rc;
    }
    return 0;
}

// Label presence grid (svr_render_labels): one block per cell ORs the label bits of the cell's voxels and a one-voxel apron,
// [cC - 1, (c+1)C], in shared memory and writes the cell's 8 words once.  The apron holds every corner the indicator of a
// sample inside the cell reads (u = x - 1/2 lies in [cC - 1/2, (c+1)C - 1/2): corners floor(u) .. floor(u) + 1).  The label
// texture is point-filtered with unnormalised coordinates: a fetch at the voxel centre is the voxel, outside the border's 0.
// Label 0 is never visible and is not recorded.  A warp sets each distinct label's bit once (__match_any_sync).
__global__ void __launch_bounds__(128) label_presence_kernel(cudaTextureObject_t labelTex, int3 grid, int cell, uint32_t* __restrict__ out)
{
    __shared__ uint32_t mask[8];
    if (threadIdx.x < 8) mask[threadIdx.x] = 0u;
    __syncthreads();
    const int cx = blockIdx.x, cy = blockIdx.y, cz = blockIdx.z;
    const int R = cell + 2;
    const int x0 = cx * cell - 1, y0 = cy * cell - 1, z0 = cz * cell - 1;
    const int total = R * R * R;
    for (int base = 0; base < total; base += blockDim.x) {  // the same trip count for every lane: the match is warp-wide
        const int i = base + (int)threadIdx.x;
        uint32_t l = 0u;
        if (i < total) {
            const int x = i % R, y = (i / R) % R, z = i / (R * R);
            l = tex3D<unsigned char>(labelTex, (float)(x0 + x) + 0.5f, (float)(y0 + y) + 0.5f, (float)(z0 + z) + 0.5f);
        }
        const uint32_t peers = __match_any_sync(0xffffffffu, l);
        if (l != 0u && (threadIdx.x & 31) == (uint32_t)(__ffs(peers) - 1)) atomicOr(&mask[l >> 5], 1u << (l & 31u));
    }
    __syncthreads();
    if (threadIdx.x < 8) out[(((size_t)cz * grid.y + cy) * grid.x + cx) * 8 + threadIdx.x] = mask[threadIdx.x];
}

int ensure_label_grid(cudaArray_t arr, cudaTextureObject_t tex, int3 dims, int cell)
{
    HostState& st = state();
    DeviceState& d = st.dev;
    if (cell == 0) cell = 8;
    if (arr != d.labelArray || cell != d.labelCell || !d.labelPresence.p) {
        release_label_grid(st);
        const int3 g = make_int3((dims.x + cell - 1) / cell, (dims.y + cell - 1) / cell, (dims.z + cell - 1) / cell);
        SVR_TRY(d.labelPresence.reserve((size_t)g.x * g.y * g.z * 8));
        d.labelArray = arr;
        d.labelCell = cell;
        d.labelGridDims = g;
    }
    if (!d.labelValid) {
        const dim3 g(d.labelGridDims.x, d.labelGridDims.y, d.labelGridDims.z);
        label_presence_kernel<<<g, 128, 0, st.stream>>>(tex, d.labelGridDims, cell, d.labelPresence.p);
        count_launch();
        SVR_TRY(cudaGetLastError());
        d.labelValid = true;
    }
    return 0;
}

void release_label_grid(HostState& st)
{
    DeviceState& d = st.dev;
    d.labelPresence.release();
    d.labelArray = nullptr;
    d.labelCell = 0;
    d.labelGridDims = make_int3(0, 0, 0);
    d.labelValid = false;
}

static int build_grid(DevScene* scene, bool force, int cell, bool* majorantsRebuilt)
{
    HostState& st = state();
    const svr_volume& vol = scene->vol;
    const svr_transfer_function& tf = scene->tf;
    if (!vol.tex || !tf.tex) return fail_msg("ensure_grid: volume or transfer function texture is not set");

    cudaResourceDesc trd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&trd, tf.tex));
    if (trd.resType != cudaResourceTypeArray) return fail_msg("ensure_grid: textures must be bound to cudaArrays");
    cudaArray_t tarr = trd.res.array.array;

    if (majorantsRebuilt) *majorantsRebuilt = false;
    if (int rc = ensure_ranges(vol, cell)) return rc;
    // the majorant grid and its helpers, for the grid ensure_ranges settled on (release_grid frees them with the ranges)
    const size_t padded = (size_t)(st.dev.gridDims.x + 2) * (st.dev.gridDims.y + 2) * (st.dev.gridDims.z + 2);
    SVR_TRY(st.dev.majorant.reserve(padded));
    SVR_TRY(st.dev.dist[0].reserve(padded));
    SVR_TRY(st.dev.dist[1].reserve(padded));
    SVR_TRY(st.dev.occ.reserve(6));

    const int leap = st.options[SVR_OPT_LEAP] != 0;
    if (force || !st.dev.majorantValid || st.dev.majorantDensityScale != vol.densityScale || st.dev.majorantTfArray != tarr ||
        st.dev.majorantLeap != leap) {
        // ---- stage 2: majorants from (range, TF, densityScale), into the padded grid
        cudaChannelFormatDesc ch;
        cudaExtent ext;
        unsigned int flags = 0;
        SVR_TRY(cudaArrayGetInfo(&ch, &ext, &flags, tarr));
        int n = (int)ext.width;
        if (n < 2 || ch.x != 32 || ch.w != 32) return fail_msg("ensure_grid: transfer function must be a 1-D float4 array");
        int levels = 32 - __builtin_clz((unsigned)n);
        SVR_TRY(st.dev.tfTable.reserve((size_t)n));
        SVR_TRY(st.dev.tfSparse.reserve((size_t)levels * n));
        st.dev.tfEntries = n;
        SVR_TRY(cudaMemcpy2DFromArrayAsync(st.dev.tfTable.p, (size_t)n * sizeof(float4), tarr, 0, 0, (size_t)n * sizeof(float4), 1,
                                           cudaMemcpyDeviceToDevice, st.stream));
        tf_sparse_kernel<<<1, 1024, 0, st.stream>>>(st.dev.tfTable.p, n, levels, st.dev.tfSparse.p);
        SVR_TRY(st.dev.tfHash.reserve(4));  // [0] built-from, [1] live, [2] stale flag (32 bit)
        tf_hash_kernel<<<1, 256, 0, st.stream>>>(st.dev.tfTable.p, 0, n, st.dev.tfHash.p, nullptr, nullptr, nullptr);  // of the table these majorants come from
        const int px = st.dev.gridDims.x + 2, py = st.dev.gridDims.y + 2, pz = st.dev.gridDims.z + 2;
        const size_t padded = (size_t)px * py * pz;
        if (int rc = zero_words(st, st.dev.majorant.p, padded * sizeof(float))) return rc;
        occ_init_kernel<<<1, 32, 0, st.stream>>>(st.dev.occ.p);
        dim3 mb(32, 4, 1), mg((st.dev.gridDims.x + 31) / 32, (st.dev.gridDims.y + 3) / 4, st.dev.gridDims.z);
        majorant_kernel<<<mg, mb, 0, st.stream>>>(st.dev.range.p, st.dev.gridDims, st.dev.tfSparse.p, n, vol.densityScale, st.dev.majorant.p, st.dev.occ.p);
        // ---- stage 3: leap distances for empty cells (border cells included)
        dim3 pg((px + 31) / 32, (py + 3) / 4, pz);
        const int cap = leap ? SVR_LEAP_CAP : 0;
        dist_axis_kernel<true, false><<<pg, mb, 0, st.stream>>>(nullptr, st.dev.dist[0].p, st.dev.majorant.p, px, py, pz, 0, cap);
        dist_axis_kernel<false, false><<<pg, mb, 0, st.stream>>>(st.dev.dist[0].p, st.dev.dist[1].p, nullptr, px, py, pz, 1, cap);
        dist_axis_kernel<false, true><<<pg, mb, 0, st.stream>>>(st.dev.dist[1].p, nullptr, st.dev.majorant.p, px, py, pz, 2, cap);
        count_launch(7);
        SVR_TRY(cudaGetLastError());
        if (majorantsRebuilt) *majorantsRebuilt = true;
        st.sceneEpoch++;
        st.dev.majorantValid = true;
        st.dev.majorantDensityScale = vol.densityScale;
        st.dev.majorantTfArray = tarr;
        st.dev.majorantLeap = leap;
    }

    scene->volDim = st.dev.volDims;
    DevGrid& g = scene->grid;
    g.px = st.dev.gridDims.x + 2;
    g.pxy = g.px * (st.dev.gridDims.y + 2);
    g.pyF = (float)(st.dev.gridDims.y + 2);
    g.cells = st.dev.majorant.p + g.pxy + g.px + 1;  // interior cell (0,0,0)
    g.range = st.dev.range.p;
    g.occ = st.dev.occ.p;
    g.gx = st.dev.gridDims.x;
    g.gy = st.dev.gridDims.y;
    g.gz = st.dev.gridDims.z;
    g.cell = st.dev.gridCell;
    g.scale = f3((float)st.dev.volDims.x / (float)st.dev.gridCell, (float)st.dev.volDims.y / (float)st.dev.gridCell,
                 (float)st.dev.volDims.z / (float)st.dev.gridCell);
    g.invScale = f3((float)st.dev.gridCell / (float)st.dev.volDims.x, (float)st.dev.gridCell / (float)st.dev.volDims.y, (float)st.dev.gridCell / (float)st.dev.volDims.z);
    g.toCell = f3(vol.bbox.invSize) * g.scale;
    g.cellOff = f3(vol.bbox.vmin) * g.toCell;
    return 0;
}

// Macrocell edge from the scene (SVR_OPT_MACROCELL_SIZE = 0).  What a cell size costs is a trade between
// visits (one per cell crossed) and null collisions (loose majorants in cells that straddle a boundary);
// measured over the BASELINE configurations the fastest edge is about twice the mean free path inside
// the medium (tools/gpu_cell_probe.py: opaque CT body, mean majorant 0.5 per voxel -> 4; cloud, 0.14 -> 16;
// thin transfer function, 0.009 -> 32).  The statistic is the mean non-zero majorant of the current grid.
static int auto_cell(HostState& st, int current, int* want)
{
    const size_t padded = (size_t)(st.dev.gridDims.x + 2) * (st.dev.gridDims.y + 2) * (st.dev.gridDims.z + 2);
    SVR_TRY(st.dev.stats.reserve(2));
    if (int rc = zero_words(st, st.dev.stats.p, 16)) return rc;
    majorant_stats_kernel<<<148 * 4, 256, 0, st.stream>>>(st.dev.majorant.p, padded, (double*)st.dev.stats.p, (unsigned long long*)((char*)st.dev.stats.p + 8));
    count_launch();
    struct {
        double sum;
        unsigned long long count;
    } h;
    if (int rc = read_small(st, &h, st.dev.stats.p, 16)) return rc;
    *want = current;
    if (h.count == 0 || !(h.sum > 0.0)) return 0;  // nothing to track through: any size will do
    const double ideal = log2(2.0 / (h.sum / (double)h.count));  // log2 of twice the mean free path, in voxels
    // keep the current size unless the ideal is clearly nearer to another power of two (no flip-flopping
    // between two sizes whose grids give slightly different statistics)
    if (fabs(ideal - log2((double)current)) < 0.75) return 0;
    int e = (int)floor(ideal + 0.5);
    e = e < 2 ? 2 : (e > 5 ? 5 : e);
    *want = 1 << e;
    return 0;
}

// The ray caster's per-call check that the transfer-function table behind an unchanged handle still is the one the
// majorants were built from, without a host synchronisation per frame: a call first collects the verdict of the PREVIOUS
// call's hash (its event has long completed; tf_check_collect), rebuilds if that table had changed, and then launches
// this frame's hash (tf_check_launch), whose verdict the ray-cast kernel of this very frame reads from device memory: with
// stale majorants it does not skip (skipping is exact, so the image is the same, only slower, for that one frame).
int tf_check_collect(bool* changed)
{
    HostState& st = state();
    *changed = false;
    if (!st.dev.tfCheckPending) return 0;
    st.dev.tfCheckPending = false;
    SVR_TRY(cudaEventSynchronize(st.dev.tfCheckEvent));
    unsigned long long h[2];
    memcpy(h, (const char*)st.dev.hMailbox + 32, sizeof(h));
    *changed = h[0] != h[1];
    return 0;
}

// *staleFlag: device word for the ray-cast kernel (null when nothing could be checked: the grid was just rebuilt from this table)
int tf_check_launch(const svr_transfer_function& tf, const unsigned int** staleFlag)
{
    HostState& st = state();
    *staleFlag = nullptr;
    if (!tf.tex || !st.dev.majorantValid || !st.dev.tfHash.p || !st.dev.tfEntries) return 0;
    cudaResourceDesc trd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&trd, tf.tex));
    if (trd.resType != cudaResourceTypeArray || trd.res.array.array != st.dev.majorantTfArray) return 0;
    if (int rc = ensure_mailbox(st)) return rc;
    if (!st.dev.tfCheckEvent) SVR_TRY(cudaEventCreateWithFlags(&st.dev.tfCheckEvent, cudaEventDisableTiming));
    unsigned int* flag = (unsigned int*)(st.dev.tfHash.p + 2);
    tf_hash_kernel<<<1, 256, 0, st.stream>>>(nullptr, tf.tex, st.dev.tfEntries, st.dev.tfHash.p + 1, st.dev.tfHash.p, (unsigned long long*)((char*)st.dev.dMailbox + 32), flag);
    count_launch();
    SVR_TRY(cudaGetLastError());
    SVR_TRY(cudaEventRecord(st.dev.tfCheckEvent, st.stream));
    st.dev.tfCheckPending = true;
    *staleFlag = flag;
    return 0;
}

int ensure_grid(DevScene* scene, bool force, int maxAutoCell)
{
    HostState& st = state();
    const int opt = st.options[SVR_OPT_MACROCELL_SIZE];
    if (opt != 0) return build_grid(scene, force, opt, nullptr);
    int cell = st.dev.autoCell ? st.dev.autoCell : 8;
    if (cell > maxAutoCell) cell = maxAutoCell;
    int rc = build_grid(scene, force, cell, nullptr);
    if (rc) return rc;
    // re-evaluate when the scene behind the grid changed, not on every forced refresh (ray caster)
    const bool sceneChanged = st.dev.autoArray != st.dev.gridArray || st.dev.autoTfArray != st.dev.majorantTfArray ||
                              st.dev.autoDensityScale != scene->vol.densityScale || st.dev.autoEpoch != st.dev.uploadEpoch;
    if (st.dev.autoCell && !sceneChanged) return 0;
    // majorants grow with the cell they are taken over, so the statistic is looked at again on the grid of
    // the size it suggested (at most twice; the 0.75-octave hysteresis in auto_cell settles it)
    for (int round = 0; round < 3; ++round) {
        int want = cell;
        rc = auto_cell(st, cell, &want);
        if (rc) return rc;
        if (want > maxAutoCell) want = maxAutoCell;
        if (want == cell) break;
        cell = want;
        rc = build_grid(scene, force, cell, nullptr);
        if (rc) return rc;
    }
    st.dev.autoCell = cell;
    st.dev.autoArray = st.dev.gridArray;
    st.dev.autoTfArray = st.dev.majorantTfArray;
    st.dev.autoDensityScale = scene->vol.densityScale;
    st.dev.autoEpoch = st.dev.uploadEpoch;
    return 0;
}

}  // namespace svr

// ------------------------------------------------------------------------------------------------
// inspection hooks
// ------------------------------------------------------------------------------------------------
namespace {
__global__ void sample_volume_kernel(cudaTextureObject_t tex, const float* uvw, uint32_t n, float* out)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = tex3D<float>(tex, uvw[3 * i], uvw[3 * i + 1], uvw[3 * i + 2]);
}
__global__ void sample_tf_kernel(cudaTextureObject_t tex, const float* x, uint32_t n, float4* out)
{
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = tex1D<float4>(tex, x[i]);
}
}  // namespace

extern "C" int svr_debug_sample_volume(const svr_volume* vol, const float* dev_uvw, uint32_t n, float* dev_out)
{
    if (!vol || !vol->tex || !dev_uvw || !dev_out) return svr::fail_msg("svr_debug_sample_volume: bad argument");
    if (!n) return 0;
    sample_volume_kernel<<<(n + 255u) / 256u, 256, 0, svr::state().stream>>>(vol->tex, dev_uvw, n, dev_out);
    svr::count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

extern "C" int svr_debug_sample_tf(const svr_transfer_function* tf, const float* dev_x, uint32_t n, float* dev_rgba)
{
    if (!tf || !tf->tex || !dev_x || !dev_rgba) return svr::fail_msg("svr_debug_sample_tf: bad argument");
    if (!n) return 0;
    sample_tf_kernel<<<(n + 255u) / 256u, 256, 0, svr::state().stream>>>(tf->tex, dev_x, n, (float4*)dev_rgba);
    svr::count_launch();
    SVR_TRY(cudaGetLastError());
    return 0;
}

extern "C" int svr_grid_info(int32_t* dims, int32_t* cell)
{
    svr::HostState& st = svr::state();
    if (!st.dev.range.p) return svr::fail_msg("svr_grid_info: no grid has been built yet");
    if (dims) {
        dims[0] = st.dev.gridDims.x;
        dims[1] = st.dev.gridDims.y;
        dims[2] = st.dev.gridDims.z;
    }
    if (cell) *cell = st.dev.gridCell;
    return 0;
}

extern "C" int svr_grid_copy(float* host_majorant, float* host_range)
{
    svr::HostState& st = svr::state();
    if (!st.dev.range.p || !st.dev.majorant.p) return svr::fail_msg("svr_grid_copy: no grid has been built yet");
    const int gx = st.dev.gridDims.x, gy = st.dev.gridDims.y, gz = st.dev.gridDims.z;
    size_t cells = (size_t)gx * gy * gz;
    SVR_TRY(cudaStreamSynchronize(st.stream));
    if (host_majorant) {
        const int px = gx + 2, py = gy + 2, pz = gz + 2;
        std::vector<float> padded((size_t)px * py * pz);
        SVR_TRY(cudaMemcpy(padded.data(), st.dev.majorant.p, padded.size() * sizeof(float), cudaMemcpyDeviceToHost));
        for (int z = 0; z < gz; ++z)
            for (int y = 0; y < gy; ++y)
                memcpy(host_majorant + ((size_t)z * gy + y) * gx, &padded[((size_t)(z + 1) * py + (y + 1)) * px + 1], gx * sizeof(float));
    }
    if (host_range) SVR_TRY(cudaMemcpy(host_range, st.dev.range.p, cells * sizeof(float2), cudaMemcpyDeviceToHost));
    return 0;
}
