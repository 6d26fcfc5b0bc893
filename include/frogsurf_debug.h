/*
 * frogsurf_debug.h -- host-side pieces of libfrogsurf.so exposed so that the CPU test suite can
 * check them without a GPU.  Not part of the drop-in surface.
 */
#ifndef FROGSURF_DEBUG_H_
#define FROGSURF_DEBUG_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* the restatement of glibc's expf the descriptor kernel uses (surf.cxx:227 calls expf), host build */
float fs_debug_expf(float x);
void fs_debug_expf_many(const float* x, float* y, size_t n);
/* interpolation step fasthessian.cxx:614-661: X = -pinv(H) dD; H10 = dxx dyy dzz dss dxy dxz dxs dyz dys dzs */
void fs_debug_solve_offsets(const double* dD, const double* H10, double* X);
/* response-layer geometry (fasthessian.cxx:53-81, 287-341, 366): per layer width, height, depth, step, filter, limit */
int fs_debug_layers(int nx, int ny, int nz, int32_t* out6, int cap);
/* vtk3DSURF.cxx:209-226: order[] receives the original indices of the points kept, strongest first */
uint32_t fs_debug_select(const float* response, uint32_t n, int number_of_points, uint32_t* order);

/* keep the shifted int volume (vtk3DSURF::Cast) of the following fs_set_volume calls so that fs_get_cast_volume can
 * return it; off by default (256 MB of extra writes for a 400^3 volume that nothing but the tests reads) */
/* the ordering fs_detect applies to its extrema (loop position keys): order[] = input indices ascending by key, ties in
 * input order */
void fs_debug_sort_keys(const uint64_t* keys, uint32_t n, uint32_t* order);
/* experiment switches; "response_tile": thread-to-voxel mapping of the response-layer kernel (0 flat, 1 32x8x1,
 * 2 32x4x2, 3 32x2x4, 4 32x1x8, 5 32x4x4 (default), 6-9 register-capped / smaller-CTA variants).  Results are identical
 * for every value. */
int fs_debug_set_option(const char* name, int value);
struct fs_ctx;
void fs_debug_keep_cast_volume(struct fs_ctx* ctx, int on);
/* fs_get_points_as_read's conversion of n given values at `precision` decimals (six when negative), on device 0 (needs a
 * GPU): out[i] = strtof of in[i]'s fixed-decimal text */
int fs_debug_as_read(const double* in, size_t n, int precision, float* out);

#ifdef __cplusplus
}
#endif

#endif
