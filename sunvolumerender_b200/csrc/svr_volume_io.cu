// svr_volume_io.cu -- the volume input stage in front of the render path (include/svr_volume_io.h):
// a dependency-free MetaImage (.mhd / .mha) reader and, on the GPU, the preprocessing
// VolumeReader::Read does with VTK filters on the host (core/VolumeReader.cpp:13-94, 124-136):
// cast to short, scalar range, rescale to the full u16 range, histogram, maximum gradient magnitude.
//
// VTK is not part of the reference tree (find_package(VTK), CMakeLists.txt:24) and not installed here;
// the filter semantics below restate VTK 5's documented behaviour and are marked where they matter:
//   vtkImageCast (ClampOverflow off)   : C-style static_cast per voxel
//   vtkImageAccumulate (IgnoreZero on) : bin = (v - origin) / spacing, voxels equal to 0 and bins outside the
//                                        component extent are not counted
//   vtkImageGradientMagnitude (3-D, HandleBoundaries on): central differences times 0.5 / spacing in
//                                        double, one-sided (same 0.5 factor) at the faces, result cast to
//                                        the INPUT type (short)
#include <zlib.h>

#include <algorithm>
#include <cctype>
#include <climits>
#include <cstring>
#include <fstream>
#include <sstream>
#include <string>
#include <vector>

#include "../../include/svr_volume_io.h"
#include "svr_state.h"

namespace svr {
namespace {

size_t met_size(int t)
{
    switch (t) {
        case SVR_MET_UCHAR:
        case SVR_MET_CHAR: return 1;
        case SVR_MET_USHORT:
        case SVR_MET_SHORT: return 2;
        case SVR_MET_UINT:
        case SVR_MET_INT:
        case SVR_MET_FLOAT: return 4;
        case SVR_MET_DOUBLE: return 8;
        default: return 0;
    }
}

std::string trim(const std::string& s)
{
    size_t a = 0, b = s.size();
    while (a < b && isspace((unsigned char)s[a])) ++a;
    while (b > a && isspace((unsigned char)s[b - 1])) --b;
    return s.substr(a, b - a);
}

std::string lower(std::string s)
{
    for (char& c : s) c = (char)tolower((unsigned char)c);
    return s;
}

bool truthy(const std::string& v)
{
    std::string l = lower(v);
    return l == "true" || l == "1" || l == "yes";
}

int parse_element_type(const std::string& v)
{
    static const struct {
        const char* name;
        int t;
    } kTypes[] = {{"met_uchar", SVR_MET_UCHAR}, {"met_char", SVR_MET_CHAR},   {"met_ushort", SVR_MET_USHORT}, {"met_short", SVR_MET_SHORT},
                  {"met_uint", SVR_MET_UINT},   {"met_int", SVR_MET_INT},     {"met_float", SVR_MET_FLOAT},   {"met_double", SVR_MET_DOUBLE}};
    std::string l = lower(v);
    for (const auto& k : kTypes)
        if (l == k.name) return k.t;
    return -1;
}

// ---- kernels ------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T byteswap(T v)
{
    unsigned char* p = reinterpret_cast<unsigned char*>(&v);
    for (int i = 0; i < (int)sizeof(T) / 2; ++i) {
        unsigned char t = p[i];
        p[i] = p[sizeof(T) - 1 - i];
        p[sizeof(T) - 1 - i] = t;
    }
    return v;
}

// vtkImageCast to short, ClampOverflow off: static_cast<short>(v).  Integers wrap modulo 2^16; floating
// values truncate toward zero through int (out-of-int-range input is undefined in C++; here it saturates
// to int first).
template <typename T>
__device__ __forceinline__ short to_short(T v) { return (short)v; }
template <>
__device__ __forceinline__ short to_short<float>(float v) { return (short)__float2int_rz(v); }
template <>
__device__ __forceinline__ short to_short<double>(double v) { return (short)__double2int_rz(v); }

template <typename T>
__global__ void cast_minmax_kernel(const T* __restrict__ raw, int swap, size_t n, short* __restrict__ out, int* __restrict__ minmax)
{
    int mn = INT_MAX, mx = INT_MIN;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        T v = raw[i];
        if (swap) v = byteswap(v);
        short s = to_short<T>(v);
        out[i] = s;
        mn = min(mn, (int)s);
        mx = max(mx, (int)s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mn = min(mn, __shfl_xor_sync(0xffffffffu, mn, o));
        mx = max(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((threadIdx.x & 31) == 0 && mn <= mx) {
        atomicMin(&minmax[0], mn);
        atomicMax(&minmax[1], mx);
    }
}

// vtkImageAccumulate: extent [0, max-min-1], origin min, spacing 1, IgnoreZero on (VolumeReader.cpp:57-63)
__global__ void histogram_kernel(const short* __restrict__ data, size_t n, int origin, int bins, unsigned int* __restrict__ hist,
                                 unsigned long long* __restrict__ total)
{
    unsigned int counted = 0;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        int v = data[i];
        if (v == 0) continue;
        int b = v - origin;
        if (b >= 0 && b < bins) {
            atomicAdd(&hist[b], 1u);
            ++counted;
        }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) counted += __shfl_xor_sync(0xffffffffu, counted, o);
    if ((threadIdx.x & 31) == 0 && counted) atomicAdd(total, (unsigned long long)counted);
}

// vtkImageGradientMagnitude, Dimensionality 3, HandleBoundaries on; output cast to short; its maximum
__global__ void gradmag_max_kernel(const short* __restrict__ d, int nx, int ny, int nz, double rx, double ry, double rz, int* __restrict__ outMax)
{
    const size_t total = (size_t)nx * ny * nz;
    int m = INT_MIN;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        int x = (int)(i % nx), y = (int)((i / nx) % ny), z = (int)(i / ((size_t)nx * ny));
        int x0 = max(x - 1, 0), x1 = min(x + 1, nx - 1);
        int y0 = max(y - 1, 0), y1 = min(y + 1, ny - 1);
        int z0 = max(z - 1, 0), z1 = min(z + 1, nz - 1);
        size_t row = ((size_t)z * ny + y) * nx, col = (size_t)z * ny * nx + x;
        double dx = ((double)d[row + x0] - (double)d[row + x1]) * rx;
        double dy = ((double)d[col + (size_t)y0 * nx] - (double)d[col + (size_t)y1 * nx]) * ry;
        double dz = ((double)d[((size_t)z0 * ny + y) * nx + x] - (double)d[((size_t)z1 * ny + y) * nx + x]) * rz;
        double mag = sqrt(dx * dx + dy * dy + dz * dz);
        m = max(m, (int)(short)__double2int_rz(mag));  // static_cast<short>(sqrt(sum))
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(outMax, m);
}

// VolumeReader::Rescale<short, unsigned short> (VolumeReader.cpp:124-136), in place:
//   ptr2[i] = (ptr1[i] - dataMin) / extent * dataTypeExtent   -- fp32, IEEE division, truncation to u16
__global__ void rescale_kernel(short* __restrict__ data, size_t n, float dataMin, float extent)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        float v = __fsub_rn((float)data[i], dataMin);
        v = __fmul_rn(__fdiv_rn(v, extent), 65535.f);
        unsigned short u = extent > 0.f ? (unsigned short)__float2int_rz(v) : (unsigned short)0;
        reinterpret_cast<unsigned short*>(data)[i] = u;
    }
}

}  // namespace
}  // namespace svr

using namespace svr;

static int read_header(const char* path, svr_metaimage_header* out);

extern "C" int svr_metaimage_read_header(const char* path, svr_metaimage_header* out)
{
    if (!path || !out) return fail_msg("svr_metaimage_read_header: bad argument");
    try {
        return read_header(path, out);
    } catch (const std::bad_alloc&) {
        return fail_msg("svr_metaimage_read_header: out of host memory");
    } catch (...) {
        return fail_msg("svr_metaimage_read_header: unexpected exception");
    }
}

static int read_header(const char* path, svr_metaimage_header* out)
{
    std::ifstream f(path, std::ios::binary);
    if (!f) return fail_msg((std::string("svr_metaimage_read_header: cannot open ") + path).c_str());
    memset(out, 0, sizeof(*out));
    out->ndims = 3;
    out->dim[0] = out->dim[1] = out->dim[2] = 1;
    out->spacing[0] = out->spacing[1] = out->spacing[2] = 1.f;
    out->element_type = -1;
    out->channels = 1;
    out->header_size = 0;
    bool haveDim = false, haveSpacing = false, haveDataFile = false;
    std::string line, dataFile;
    while (std::getline(f, line)) {
        size_t eq = line.find('=');
        if (eq == std::string::npos) {
            if (trim(line).empty()) continue;
            return fail_msg((std::string("svr_metaimage_read_header: malformed line: ") + line.substr(0, 60)).c_str());
        }
        std::string key = lower(trim(line.substr(0, eq))), val = trim(line.substr(eq + 1));
        std::istringstream vs(val);
        if (key == "ndims") {
            vs >> out->ndims;
            if (out->ndims < 2 || out->ndims > 3) return fail_msg("svr_metaimage_read_header: NDims must be 2 or 3");
        } else if (key == "dimsize") {
            for (uint32_t i = 0; i < out->ndims && i < 3; ++i) vs >> out->dim[i];
            haveDim = true;
        } else if (key == "elementspacing" || (key == "elementsize" && !haveSpacing)) {
            for (uint32_t i = 0; i < out->ndims && i < 3; ++i) vs >> out->spacing[i];
            if (key == "elementspacing") haveSpacing = true;
        } else if (key == "elementtype") {
            out->element_type = parse_element_type(val);
            if (out->element_type < 0) return fail_msg((std::string("svr_metaimage_read_header: unsupported ElementType ") + val).c_str());
        } else if (key == "elementnumberofchannels") {
            vs >> out->channels;
        } else if (key == "binarydatabyteordermsb" || key == "elementbyteordermsb") {
            out->msb = truthy(val);
        } else if (key == "binarydata") {
            if (!truthy(val)) return fail_msg("svr_metaimage_read_header: ASCII data (BinaryData = False) is not supported");
        } else if (key == "compresseddata") {
            out->compressed = truthy(val);
        } else if (key == "compresseddatasize") {
            vs >> out->compressed_size;
        } else if (key == "headersize") {
            long long h = 0;
            vs >> h;
            out->header_size = h;
        } else if (key == "elementdatafile") {
            dataFile = val;
            haveDataFile = true;
            break;  // by definition the last header line; LOCAL data starts right after it
        }
        // ObjectType, TransformMatrix, Offset, CenterOfRotation, AnatomicalOrientation, ...: not needed
    }
    if (!haveDim || !haveDataFile || out->element_type < 0) return fail_msg("svr_metaimage_read_header: DimSize, ElementType and ElementDataFile are required");
    for (int i = 0; i < 3; ++i) {
        if (out->dim[i] == 0 || !(out->spacing[i] > 0.f)) return fail_msg("svr_metaimage_read_header: zero dimension or non-positive spacing");
        // the voxels end in a 3-D cudaArray (VolumeReader.cpp:144-150): 16384 texels per axis at most on every CUDA device,
        // which also keeps every size below (2^14)^3 * 8 = 2^45 bytes -- no size_t arithmetic can wrap
        if (out->dim[i] > SVR_MAX_VOLUME_DIM) return fail_msg("svr_metaimage_read_header: DimSize exceeds the 3-D texture limit (16384 per axis)");
    }
    if (lower(dataFile) == "local") {
        out->data_offset = (uint64_t)f.tellg();
        out->data_file[0] = 0;
    } else {
        if (lower(dataFile).rfind("list", 0) == 0 || dataFile.find('%') != std::string::npos)
            return fail_msg("svr_metaimage_read_header: multi-file data (LIST / printf patterns) is not supported");
        std::string full = dataFile;
        if (dataFile[0] != '/') {
            std::string p(path);
            size_t slash = p.find_last_of('/');
            if (slash != std::string::npos) full = p.substr(0, slash + 1) + dataFile;
        }
        if (full.size() >= sizeof(out->data_file)) return fail_msg("svr_metaimage_read_header: data file path too long");
        strcpy(out->data_file, full.c_str());
    }
    return 0;
}

extern "C" int svr_volume_from_raw(const void* host_data, int met_type, int msb, uint32_t nx, uint32_t ny, uint32_t nz, float sx,
                                   float sy, float sz, svr_volume* out, svr_volume_stats* stats, uint32_t* histogram,
                                   uint32_t histogram_capacity)
{
    const size_t es = met_size(met_type);
    if (!host_data || !out || !es || !nx || !ny || !nz || !(sx > 0.f) || !(sy > 0.f) || !(sz > 0.f))
        return fail_msg("svr_volume_from_raw: bad argument");
    if (nx > SVR_MAX_VOLUME_DIM || ny > SVR_MAX_VOLUME_DIM || nz > SVR_MAX_VOLUME_DIM)
        return fail_msg("svr_volume_from_raw: dimension exceeds the 3-D texture limit (16384 per axis)");
    HostState& st = state();
    const size_t n = (size_t)nx * ny * nz;
    DevBuf<uint8_t> raw, aux;
    DevBuf<short> data;
    DevBuf<unsigned int> hist;
    SVR_TRY(raw.reserve(n * es));
    SVR_TRY(data.reserve(n));
    SVR_TRY(aux.reserve(32));
    SVR_TRY(cudaMemcpyAsync(raw.p, host_data, n * es, cudaMemcpyHostToDevice, st.stream));
    int* dMinMax = (int*)aux.p;        // [0] min, [1] max, [2] max gradient magnitude
    unsigned long long* dTotal = (unsigned long long*)((char*)aux.p + 16);
    const int init[8] = {INT_MAX, INT_MIN, INT_MIN, 0, 0, 0, 0, 0};
    SVR_TRY(cudaMemcpyAsync(aux.p, init, sizeof(init), cudaMemcpyHostToDevice, st.stream));
    const int blocks = 148 * 8, threads = 256;
    short* d = data.p;
    const int swap = msb && es > 1;
    switch (met_type) {
        case SVR_MET_UCHAR: cast_minmax_kernel<unsigned char><<<blocks, threads, 0, st.stream>>>((const unsigned char*)raw.p, swap, n, d, dMinMax); break;
        case SVR_MET_CHAR: cast_minmax_kernel<signed char><<<blocks, threads, 0, st.stream>>>((const signed char*)raw.p, swap, n, d, dMinMax); break;
        case SVR_MET_USHORT: cast_minmax_kernel<unsigned short><<<blocks, threads, 0, st.stream>>>((const unsigned short*)raw.p, swap, n, d, dMinMax); break;
        case SVR_MET_SHORT: cast_minmax_kernel<short><<<blocks, threads, 0, st.stream>>>((const short*)raw.p, swap, n, d, dMinMax); break;
        case SVR_MET_UINT: cast_minmax_kernel<unsigned int><<<blocks, threads, 0, st.stream>>>((const unsigned int*)raw.p, swap, n, d, dMinMax); break;
        case SVR_MET_INT: cast_minmax_kernel<int><<<blocks, threads, 0, st.stream>>>((const int*)raw.p, swap, n, d, dMinMax); break;
        case SVR_MET_FLOAT: cast_minmax_kernel<float><<<blocks, threads, 0, st.stream>>>((const float*)raw.p, swap, n, d, dMinMax); break;
        default: cast_minmax_kernel<double><<<blocks, threads, 0, st.stream>>>((const double*)raw.p, swap, n, d, dMinMax); break;
    }
    gradmag_max_kernel<<<blocks, threads, 0, st.stream>>>(d, (int)nx, (int)ny, (int)nz, 0.5 / (double)sx, 0.5 / (double)sy, 0.5 / (double)sz, dMinMax + 2);
    count_launch(2);
    int h[3];
    SVR_TRY(cudaMemcpyAsync(h, aux.p, sizeof(h), cudaMemcpyDeviceToHost, st.stream));
    SVR_TRY(cudaStreamSynchronize(st.stream));
    raw.release();
    const int dataMin = h[0], dataMax = h[1];
    const int bins = dataMax - dataMin;  // SetComponentExtent(0, max - min - 1, ...)
    unsigned long long total = 0;
    if (bins > 0) {
        SVR_TRY(hist.reserve((size_t)bins));
        SVR_TRY(cudaMemsetAsync(hist.p, 0, (size_t)bins * sizeof(unsigned int), st.stream));
        histogram_kernel<<<blocks, threads, 0, st.stream>>>(d, n, dataMin, bins, hist.p, dTotal);
        count_launch();
        if (histogram && histogram_capacity)
            SVR_TRY(cudaMemcpyAsync(histogram, hist.p, sizeof(unsigned int) * std::min<size_t>((size_t)bins, histogram_capacity),
                                    cudaMemcpyDeviceToHost, st.stream));
        SVR_TRY(cudaMemcpyAsync(&total, dTotal, sizeof(total), cudaMemcpyDeviceToHost, st.stream));
    }
    rescale_kernel<<<blocks, threads, 0, st.stream>>>(d, n, (float)dataMin, (float)dataMax - (float)dataMin);
    count_launch();
    SVR_TRY(cudaGetLastError());
    SVR_TRY(cudaStreamSynchronize(st.stream));
    const float maxMag = (float)h[2];  // the reference divides by it unguarded (VolumeReader.cpp:183); svr_volume_create guards <= 0
    int rc = svr_volume_create(out, d, 1, SVR_VOXEL_U16, nx, ny, nz, sx, sy, sz, maxMag > 0.f ? maxMag : 1.f);
    if (rc) return rc;
    if (stats) {
        stats->dim[0] = nx;
        stats->dim[1] = ny;
        stats->dim[2] = nz;
        stats->spacing[0] = sx;
        stats->spacing[1] = sy;
        stats->spacing[2] = sz;
        stats->data_min = (float)dataMin;
        stats->data_max = (float)dataMax;
        stats->max_gradient_magnitude = maxMag;
        stats->histogram_bins = bins > 0 ? (uint32_t)bins : 0u;
        stats->histogram_total = total;
    }
    return 0;
}

static int load_metaimage(const char* path, svr_volume* out, svr_volume_stats* stats, uint32_t* histogram, uint32_t histogram_capacity);

// An exception must not cross the C boundary (a host whose memory is exhausted gets an error code, not std::terminate).
extern "C" int svr_volume_load_metaimage(const char* path, svr_volume* out, svr_volume_stats* stats, uint32_t* histogram,
                                         uint32_t histogram_capacity)
{
    try {
        return load_metaimage(path, out, stats, histogram, histogram_capacity);
    } catch (const std::bad_alloc&) {
        return fail_msg("svr_volume_load_metaimage: out of host memory");
    } catch (...) {
        return fail_msg("svr_volume_load_metaimage: unexpected exception");
    }
}

static int load_metaimage(const char* path, svr_volume* out, svr_volume_stats* stats, uint32_t* histogram, uint32_t histogram_capacity)
{
    svr_metaimage_header hd;
    int rc = svr_metaimage_read_header(path, &hd);
    if (rc) return rc;
    if (hd.channels != 1) return fail_msg("svr_volume_load_metaimage: only single-channel volumes are renderable");
    const size_t n = (size_t)hd.dim[0] * hd.dim[1] * hd.dim[2], bytes = n * met_size(hd.element_type);
    const char* dataPath = hd.data_file[0] ? hd.data_file : path;
    std::ifstream f(dataPath, std::ios::binary | std::ios::ate);
    if (!f) return fail_msg((std::string("svr_volume_load_metaimage: cannot open ") + dataPath).c_str());
    const uint64_t fileSize = (uint64_t)f.tellg();
    uint64_t start = hd.data_file[0] ? 0 : hd.data_offset;
    if (hd.data_file[0]) {
        if (hd.header_size > 0) start = (uint64_t)hd.header_size;
        else if (hd.header_size == -1 && !hd.compressed) start = fileSize >= bytes ? fileSize - bytes : 0;
    }
    std::vector<unsigned char> buf;
    if (start > fileSize) return fail_msg("svr_volume_load_metaimage: HeaderSize lies beyond the end of the data file");
    if (hd.compressed) {
        uint64_t csize = hd.compressed_size ? hd.compressed_size : fileSize - start;
        if (csize > fileSize - start) return fail_msg("svr_volume_load_metaimage: compressed data is truncated");
        // zlib's deflate cannot shrink data by more than about 1032 : 1: a header that promises more than the
        // compressed bytes can hold is rejected before anything of that size is allocated
        if (bytes / 1100 > csize + 64) return fail_msg("svr_volume_load_metaimage: DimSize x ElementType cannot come out of the compressed data");
        std::vector<unsigned char> cbuf(csize);
        f.seekg((std::streamoff)start);
        f.read((char*)cbuf.data(), (std::streamsize)csize);
        buf.resize(bytes);
        uLongf dlen = (uLongf)bytes;
        int z = uncompress(buf.data(), &dlen, cbuf.data(), (uLong)csize);
        if (z != Z_OK || dlen != bytes) return fail_msg("svr_volume_load_metaimage: zlib inflate failed or size mismatch");
    } else {
        if (bytes > fileSize - start) return fail_msg("svr_volume_load_metaimage: data file is shorter than DimSize x ElementType");
        buf.resize(bytes);
        f.seekg((std::streamoff)start);
        f.read((char*)buf.data(), (std::streamsize)bytes);
        if (!f) return fail_msg("svr_volume_load_metaimage: short read");
    }
    return svr_volume_from_raw(buf.data(), hd.element_type, hd.msb, hd.dim[0], hd.dim[1], hd.dim[2], hd.spacing[0], hd.spacing[1],
                               hd.spacing[2], out, stats, histogram, histogram_capacity);
}

extern "C" int svr_volume_download(const svr_volume* vol, void* host_out, uint64_t bytes)
{
    if (!vol || !vol->tex || !host_out) return fail_msg("svr_volume_download: bad argument");
    cudaResourceDesc rd;
    SVR_TRY(cudaGetTextureObjectResourceDesc(&rd, vol->tex));
    if (rd.resType != cudaResourceTypeArray) return fail_msg("svr_volume_download: texture is not bound to a cudaArray");
    cudaChannelFormatDesc ch;
    cudaExtent ext;
    unsigned int flags = 0;
    SVR_TRY(cudaArrayGetInfo(&ch, &ext, &flags, rd.res.array.array));
    const size_t bpe = (size_t)(ch.x + ch.y + ch.z + ch.w) / 8;
    if (bytes != (uint64_t)ext.width * ext.height * ext.depth * bpe) return fail_msg("svr_volume_download: size mismatch");
    SVR_TRY(cudaStreamSynchronize(state().stream));
    cudaMemcpy3DParms cp;
    memset(&cp, 0, sizeof(cp));
    cp.srcArray = rd.res.array.array;
    cp.extent = ext;
    cp.kind = cudaMemcpyDeviceToHost;
    cp.dstPtr = make_cudaPitchedPtr(host_out, ext.width * bpe, ext.width, ext.height);
    SVR_TRY(cudaMemcpy3D(&cp));
    return 0;
}
