/*
 * frogsurf.h -- C ABI of libfrogsurf.so, the B200 (sm_100a) SURF3D keypoint producer.
 *
 * SURVEY.md 8(f) rank 4: the step BEFORE the matching hot path.  The reference's producer is the
 * `surf3d` executable (vtkOpenSURF3D/surf3d.cxx) around vtk3DSURF::Update (vtk3DSURF.cxx:79-263);
 * like `match` it has no in-process plugin API, so this ABI is cut along Update()'s own stages:
 *
 *   fs_set_volume   vtkImageCast + vtkImageShiftScale + ComputeIntegral   vtk3DSURF.cxx:158-181, integral.cxx:11-121
 *   fs_detect       FastHessian::getIpoints                               fasthessian.cxx:142-283, 287-481, 521-612
 *   fs_select       partial_sort / sort by response, resize               vtk3DSURF.cxx:209-226
 *   fs_set_points   vtk3DSURF::ReadIPoints (surf3d -p)                    vtk3DSURF.cxx:34-77
 *   fs_describe     Surf::getDescriptors / getRawDescriptors              surf.cxx:36-243
 *
 * What is NOT here: image readers, vtkImageResample (-s / -d), mirror padding, clamping and masks
 * -- VTK filters whose algorithms live in VTK, which is absent from the reference tree.  The
 * volume handed to fs_set_volume is the one Update() would cast: single component, already at its
 * final sampling.
 *
 * Conventions as in frogmatch.h: plain C, FS_OK (0) or a negative status, never throws, input
 * pointers borrowed for the call, one context = one CUDA device = one host thread at a time.
 * There is NO CPU fallback: without a CUDA device fs_create() fails with FS_ERR_CUDA.
 */
#ifndef FROGSURF_H_
#define FROGSURF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct fs_ctx fs_ctx;

typedef enum fs_status {
  FS_OK = 0,
  FS_ERR_INVALID = -1,
  FS_ERR_CUDA = -2,
  FS_ERR_NOMEM = -3,
  FS_ERR_UNSUPPORTED = -4, /* descriptor type 2 (vtkImageResize sub-volumes), radius > 10 (type 0) or > 16 (type 1) */
  FS_ERR_STATE = -5        /* stage called before the one it depends on */
} fs_status;

/* voxel types fs_set_volume accepts (the MetaImage element types the callers' images come in) */
typedef enum fs_voxel_type {
  FS_U8 = 0,
  FS_I16 = 1,
  FS_U16 = 2,
  FS_I32 = 3,
  FS_F32 = 4,
  FS_I8 = 5,
  FS_U32 = 6,
  FS_F64 = 7
} fs_voxel_type;

/* one keypoint as FastHessian leaves it (ipoint.h:26-66): voxel units, before the writers apply spacing / origin */
typedef struct fs_point {
  float x, y, z;    /* Ipoint::x, y, z */
  float scale;      /* Ipoint::scale */
  float response;   /* Ipoint::response */
  int32_t laplacian;/* Ipoint::laplacian: 0 or 1 */
} fs_point;

/* per-stage device times of the most recent calls, CUDA events on the context's stream (milliseconds) */
typedef struct fs_stats {
  float ms_integral;     /* cast + shift + integral volume */
  float ms_response_map; /* all response layers */
  float ms_extrema;      /* extremum search + derivative records */
  float ms_describe;     /* descriptor kernel */
  uint32_t n_layers;
  uint32_t n_candidates; /* extrema found before interpolation */
  uint32_t n_points;     /* current number of keypoints */
  uint32_t n_clamped;    /* keypoints whose descriptor window left the volume (the reference reads out of bounds there) */
  uint64_t response_voxels; /* response-layer voxels computed by the last fs_detect */
} fs_stats;

int fs_device_count(int* n);
int fs_create(int device, fs_ctx** out);
void fs_destroy(fs_ctx* ctx);
/* Text of the most recent error (ctx == NULL: of the last failed fs_create on this thread).  Never NULL. */
const char* fs_last_error(const fs_ctx* ctx);
const char* fs_version(void);

/*
 * Hand over a volume of nx * ny * nz voxels, x fastest (VTK's layout).  `voxels` may be a host or a
 * device pointer (a device buffer is read in place on the context's own stream: whatever produced it must have
 * completed, e.g. by a synchronisation on the producing stream, before the call).  Does what vtk3DSURF::Update does before the detector runs: cast to int with
 * clamping, subtract the volume's minimum (vtkImageShiftScale, shift = -range[0]), integral volume
 * (unsigned 64-bit, inclusive prefix sums along x, y, z).
 */
int fs_set_volume(fs_ctx* ctx, const void* voxels, int voxel_type, int nx, int ny, int nz);

/*
 * FastHessian(integral, points, octaves 4, intervals 4, init_sample 2, threshold).getIpoints()
 * as vtk3DSURF.cxx:193-196 runs it: response layers, 3x3x3x3 extremum search, sub-voxel interpolation.
 * Keypoints are left in the reference's push_back order.
 */
int fs_detect(fs_ctx* ctx, float threshold, uint32_t* n_points);

/* vtk3DSURF.cxx:209-226: number_of_points > 0 keeps the strongest (same std::partial_sort / std::sort calls). */
int fs_select(fs_ctx* ctx, int number_of_points);

/* Replace the keypoints by n given ones (x, y, z, scale per point, voxel units; response and laplacian 0). */
int fs_set_points(fs_ctx* ctx, const float* xyzs, uint32_t n);

/*
 * Descriptors of the current keypoints.  type 0: SURF3D, 48 floats (surf.cxx:63-156); type 1: raw Haar
 * responses, 24 * radius^3 floats (surf.cxx:161-217).  radius = surf3d -r (default 5), normalize = -normalize.
 */
int fs_describe(fs_ctx* ctx, int type, int radius, int normalize);

/* Number of keypoints and floats per descriptor (0 before fs_describe). */
int fs_num_points(fs_ctx* ctx, uint32_t* n, uint32_t* descriptor_size);
/* Copy the keypoints (n fs_point) and, when desc != NULL, their descriptors (n * descriptor_size floats) to the host. */
int fs_get_points(fs_ctx* ctx, fs_point* points, float* desc);

/*
 * The current keypoints and descriptors exactly as the matcher's .csv / .csv.gz reader returns them from the file that
 * surf3d's writer formats (vtk3DSURF::WritePointsCSVGZ): head = n x 6 floats (x * spacing + origin, y.., z..,
 * scale * cbrt(spacing product), laplacian, response), desc = n x descriptor_size floats.  Every field is
 * strtof of its fixed-decimal text: six decimals for the header fields, `precision` for the descriptors (six when
 * negative).  spacing / origin: the volume's, as the MetaImage header gives them.  Converted on the device; values the
 * text needs more than 64-bit integers for (|v| * 10^decimals >= 9e18, precision > 9, inf / nan) are finished on the
 * host with snprintf + strtof.  FS_ERR_INVALID when a value's text is out of float range (the reader rejects it).
 */
int fs_get_points_as_read(fs_ctx* ctx, int precision, const double spacing[3], const double origin[3], float* head,
                          float* desc);

int fs_get_stats(fs_ctx* ctx, fs_stats* out);

/* ---- stage outputs, for the parity tests ------------------------------------------------------ */
/* the shifted int volume (vtk3DSURF::Cast; kept only after fs_debug_keep_cast_volume, frogsurf_debug.h) and the
 * integral volume, nx * ny * nz values each */
int fs_get_cast_volume(fs_ctx* ctx, int32_t* out);
int fs_get_integral(fs_ctx* ctx, uint64_t* out);
/* info: width, height, depth, step, filter (responselayer.h:26) */
int fs_num_layers(fs_ctx* ctx, uint32_t* n);
int fs_get_layer(fs_ctx* ctx, uint32_t layer, int32_t info[5], float* responses, uint8_t* laplacian, uint8_t* isblob);

#ifdef __cplusplus
}
#endif

#endif /* FROGSURF_H_ */
