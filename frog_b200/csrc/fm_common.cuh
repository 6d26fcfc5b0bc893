// fm_common.cuh -- shared device/host structures of libfrogmatch (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cfloat>
#include <cstdint>
#include <cstring>

#include "../../include/frogmatch.h"

namespace fm {

constexpr uint32_t kNone = 0xFFFFFFFFu;  // "row has no accepted match"

// FM_FLAG_ROW_TABLE: a decision site's record of one row (fm_row, include/frogmatch.h).  d1 < FLT_MAX iff a gated-in
// column set it, and only then does `nearest` name a column.
__device__ __forceinline__ void put_row(fm_row* rows, uint32_t i, float d1, float d2, uint32_t nearest) {
  rows[i] = fm_row{d1, d2, d1 < FLT_MAX ? nearest : kNone};
}
constexpr uint32_t kTaskSwap = 1u;       // Task::flags: -sym reverse pass (match.cpp:643-646)
constexpr uint32_t kTaskExact = 2u;      // Task::flags: task must use the exact brute-force kernel
constexpr int kD = 48;                   // SURF3D descriptor length the tensor-core path is built for
constexpr int kKPad = 64;                // K after augmentation: 48 descriptor + norm/one slots, 4 x UMMA_K
constexpr int kMaxClasses = 8;           // distinct Laplacian-sign values per image on the fast path
constexpr int kWideMaxD = 4096;          // longest descriptor the wide tensor-core path (fm_wide.cuh) takes, d != 48

// Image flags (set by the prep kernel; any non-zero value routes the image to the exact kernel).
constexpr uint32_t kImgNotFinite = 1u;    // NaN/Inf in descriptors, scales or laplacians
constexpr uint32_t kImgBadScale = 2u;     // scale <= 0: scale gate no longer an interval in sorted order
constexpr uint32_t kImgBigNorm = 4u;      // |desc| outside the range the FP16 operands are certified for
constexpr uint32_t kImgManyClasses = 8u;  // more than kMaxClasses distinct laplacian values
constexpr uint32_t kImgBadDim = 16u;      // d > kWideMaxD: no tensor-core path for this length

// Per-image statistics / class table produced on the device by the prep kernels.
struct ImageMeta {
  uint32_t flags;
  uint32_t n_classes;
  float max_norm2;                    // max squared L2 norm over the image's descriptors
  float max_delta2;                   // max squared L2 norm of (fp16(desc) - desc): actual FP16 rounding residual
  float class_lap[kMaxClasses];       // laplacian value of each class, ascending bit pattern order
  uint32_t class_begin[kMaxClasses + 1];  // class c occupies sorted positions [begin[c], begin[c+1])
  uint32_t min_norm2_inv;             // ~(bit pattern) of the min squared L2 norm, kept by atomicMax so that the zeroed
                                      // word means "no keypoint yet" (min_norm2() then reads NaN)
};

__host__ __device__ __forceinline__ float min_norm2(const ImageMeta& m) {
  const uint32_t u = ~m.min_norm2_inv;
  float f;
  memcpy(&f, &u, 4);
  return f;
}

// Device view of one image.  Arrays marked (orig) are in upload order -- the ids pairs.bin carries;
// arrays marked (sorted) are ordered by (laplacian class, scale) for the tensor-core path.
struct ImageDev {
  const float* desc;    // (orig) [n][d]      exact FP32 descriptors: rescoring + brute-force kernel
  const float* scale;   // (orig) [n]
  const float* lap;     // (orig) [n]
  uint32_t n;
  uint32_t d;
  uint32_t n_pad;       // n rounded up to a multiple of 128 (operand tile height)
  uint32_t pad_;
  const uint32_t* perm;        // (sorted) [n]   sorted position -> original index
  const float* scale_sorted;   // (sorted) [n]
  const float* norm2_sorted;   // (sorted) [n]   |desc|^2 in FP32 (early rejection in the rescoring kernel)
  const __half* rowop;  // (sorted) [n_pad/128] tiles of 128 x 64 halves, SWIZZLE_128B K-major image,
                        //          columns 0..47 = fp16(desc), 48,49 = 1, rest 0 (this image as rows)
  const __half* colop;  // same tiling; columns 48,49 = hi/lo halves of -|desc|^2/2 (image as columns)
  const ImageMeta* meta;
  const __half* wideop;  // (sorted) d != 48, d <= kWideMaxD only: [n_pad/128 tiles][wide_kpad(d)/64 k-blocks] of the
                         //          same 128 x 64-half SWIZZLE_128B tiles, fp16(desc) in slots 0..d-1, zeros after;
                         //          one operand for both roles (the norm term is added in the wide epilogue)
};

// K of the wide path: the descriptor length rounded up to whole 64-value k-blocks.
__host__ __device__ __forceinline__ uint32_t wide_kpad(uint32_t d) { return (d + 63u) & ~63u; }

// Byte offset of (row r, 16-byte chunk q) inside a 128 x 128 B SWIZZLE_128B K-major tile:
// 8-row x 128 B atoms, chunk index XORed with (row mod 8)  [cute Swizzle<3,4,3>].
__host__ __device__ __forceinline__ uint32_t sw128_offset(uint32_t r, uint32_t q) {
  return r * 128u + ((q ^ (r & 7u)) << 4);
}

// One directed ComputeMatches call: rows of `row_img` scan columns of `col_img`.
struct Task {
  uint32_t col_img;  // image `first`  (points2 in match.cpp:255) unless swap
  uint32_t row_img;  // image `second` (points1)
  uint32_t row_off;  // offset of this task's rows in the per-batch row arrays
  uint32_t flags;    // kTaskSwap: -sym reverse pass, emit (row, col); kTaskExact: brute-force kernel only
};

}  // namespace fm
