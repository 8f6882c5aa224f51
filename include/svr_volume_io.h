/*
 * svr_volume_io.h -- C ABI of the volume input stage in front of the render path: what
 * VolumeReader::Read + CreateTextures + CreateDeviceVolume do in the reference
 * (core/VolumeReader.cpp:13-94, 124-185), without VTK or Qt.
 *
 *   reference step (core/VolumeReader.cpp)                       here
 *   vtkMetaImageReader (:16-38)                                  svr_metaimage_read_header + file read (host, C++)
 *   vtkImageCast -> short (:40-44)                               cast kernel (GPU), C-style conversion
 *   dims / spacing (:46-50)                                      from the header
 *   Rescale<short, unsigned short> to the full u16 range (:52-55, 124-136)   rescale kernel (GPU), same fp32 expression
 *   vtkImageAccumulate histogram, zero ignored (:57-68)          histogram kernel (GPU)
 *   max of vtkImageGradientMagnitude on the short data (:70-76)  gradient-magnitude kernel (GPU), fp64 like VTK
 *   CreateTextures / CreateDeviceVolume (:138-185)               as svr_volume_create
 *
 * Functions return 0 on success; svr_last_error() (svr_render.h) has the text otherwise.
 */
#ifndef SVR_VOLUME_IO_H
#define SVR_VOLUME_IO_H

#include "svr_types.h"

#ifdef __cplusplus
extern "C" {
#endif

/* MetaImage element types (ElementType = MET_...) */
enum svr_met_type {
    SVR_MET_UCHAR = 0, SVR_MET_CHAR = 1, SVR_MET_USHORT = 2, SVR_MET_SHORT = 3,
    SVR_MET_UINT = 4, SVR_MET_INT = 5, SVR_MET_FLOAT = 6, SVR_MET_DOUBLE = 7
};

/* Largest accepted DimSize per axis: the 3-D texture limit of every CUDA device (the voxels end in a 3-D cudaArray,
 * core/VolumeReader.cpp:144-150).  Headers beyond it are rejected before anything is allocated. */
#define SVR_MAX_VOLUME_DIM 16384u

typedef struct svr_metaimage_header {
    uint32_t ndims;          /* NDims (2 or 3; a 2-D image is one slice) */
    uint32_t dim[3];         /* DimSize */
    float spacing[3];        /* ElementSpacing (ElementSize when absent; 1 when both are) */
    int32_t element_type;    /* svr_met_type */
    uint32_t channels;       /* ElementNumberOfChannels (only 1 is loadable) */
    int32_t msb;             /* BinaryDataByteOrderMSB / ElementByteOrderMSB */
    int32_t compressed;      /* CompressedData (zlib) */
    int64_t header_size;     /* HeaderSize: bytes to skip in the data file; -1 = the data is the tail of the file */
    uint64_t compressed_size;/* CompressedDataSize (0 = to the end of the file) */
    uint64_t data_offset;    /* ElementDataFile = LOCAL: offset of the first data byte in the header file */
    char data_file[1024];    /* path of the element data file, resolved against the header's directory */
} svr_metaimage_header;

/* Parses a .mhd / .mha header.  Host only: needs no GPU. */
int svr_metaimage_read_header(const char* path, svr_metaimage_header* out);

typedef struct svr_volume_stats {
    uint32_t dim[3];
    float spacing[3];
    float data_min, data_max;          /* scalar range of the data after the cast to short (VolumeReader.cpp:54) */
    float max_gradient_magnitude;      /* VolumeReader.cpp:70-76 */
    uint32_t histogram_bins;           /* data_max - data_min (VolumeReader.cpp:59) */
    uint64_t histogram_total;          /* voxels counted (zero-valued voxels are ignored, :62) */
} svr_volume_stats;

/* VolumeReader::Read + CreateDeviceVolume for data already in host memory: `host_data` holds nx*ny*nz
 * elements of `met_type` (x fastest), byte-swapped if `msb`.  On return `out` is a bound volume exactly
 * as svr_volume_create leaves it (u16 array, invMaxMagnitude from the gradient pass), `stats` (optional)
 * the numbers VolumeReader keeps, and `histogram` (optional, `histogram_capacity` entries) the first
 * min(bins, capacity) bins. */
int svr_volume_from_raw(const void* host_data, int met_type, int msb, uint32_t nx, uint32_t ny, uint32_t nz,
                        float sx, float sy, float sz, svr_volume* out, svr_volume_stats* stats,
                        uint32_t* histogram, uint32_t histogram_capacity);

/* The same from a MetaImage file (.mhd with a raw / zlib data file, or .mha with LOCAL data). */
int svr_volume_load_metaimage(const char* path, svr_volume* out, svr_volume_stats* stats,
                              uint32_t* histogram, uint32_t histogram_capacity);

/* A label map from a MetaImage file (the files svr_volume_load_metaimage reads): any integer ElementType whose values all lie
 * in 0..255, converted to u8 on the host without rescaling, into a label volume as svr_labels_create makes it.  A float or
 * double ElementType, a value outside 0..255 (the error names it) and more than one channel are errors, all reported before
 * any CUDA call.  maxLabelOrNull receives the largest label id. */
int svr_labels_load_metaimage(const char* path, svr_volume* out, uint32_t* maxLabelOrNull);

/* Copies the voxels behind vol->tex back to host memory (x fastest, the array's own element type);
 * `bytes` must be the exact size.  Used by tests and tools. */
int svr_volume_download(const svr_volume* vol, void* host_out, uint64_t bytes);

#ifdef __cplusplus
}
#endif
#endif /* SVR_VOLUME_IO_H */
