// fm_exact.cuh -- exact FP32 brute-force matcher: the reference's loop nest on CUDA cores.
//
// One thread owns one outer-loop row (a keypoint of image `second`, match.cpp:262) and walks the
// columns (keypoints of image `first`, :267) in ascending original order with the reference's
// own comparisons, so ties, the stale-d2 rules and NaN behaviour fall out identically:
//   gates      match.cpp:270 (laplacian !=) and :273-275 (scale ratios vs the double 1.3)
//   distance   match.cpp:243-251, r = fl(r + fl(fl(a-b)*fl(a-b))), k ascending, no FMA
//   top-2      match.cpp:303-313, strict '<'
//   accept     match.cpp:320-321, float sqrt/div
// It serves (a) images the tensor-core path is not certified for, (b) rows whose candidate list
// overflowed there and (c) FM_FLAG_FORCE_EXACT; descriptor lengths other than 48 go through the
// K-chunked kernel of fm_generic.cuh.
#pragma once
#include "fm_common.cuh"

namespace fm {

constexpr int kExactRows = 128;  // rows (threads) per CTA
constexpr int kExactCols = 32;   // columns staged in shared memory per step

// x > 1.3 with x a float promoted to double (match.cpp:273-274) <=> x > 1.3f, because
// 1.3f < 1.3 < nextafterf(1.3f, 2): no float lies strictly between them.
__device__ __forceinline__ bool scale_gate_fails(float s_row, float s_col) {
  return __fdiv_rn(s_row, s_col) > 1.3f || __fdiv_rn(s_col, s_row) > 1.3f;
}

__device__ __forceinline__ bool accept_rule(float d1, float d2, float thr, float ratio) {
  return (__fsqrt_rn(__fdiv_rn(d1, d2)) < ratio || d2 == FLT_MAX) && __fsqrt_rn(d1) < thr;
}

// Find the task a flat block index belongs to: largest t with blk_off[t] <= b.
__device__ __forceinline__ uint32_t find_segment(const uint32_t* __restrict__ off, uint32_t n, uint32_t b) {
  uint32_t lo = 0, hi = n;
  while (hi - lo > 1) {
    uint32_t mid = (lo + hi) >> 1;
    if (off[mid] <= b) lo = mid; else hi = mid;
  }
  return lo;
}

// The same, starting from a guess: the segments a kernel walks are nearly uniform in size (images of a group hold about
// the same number of keypoints), so proportional interpolation lands on or next to the answer and two or three loads
// replace the ~log2(n) DEPENDENT global loads of the bisection (0.5 us each: 5 us of prologue for a 1000-task batch).
// Galloping keeps the worst case logarithmic.  off[n] = total.
__device__ __forceinline__ uint32_t find_segment_near(const uint32_t* __restrict__ off, uint32_t n, uint32_t b, uint32_t total) {
  uint32_t g = (uint32_t)(((uint64_t)b * n) / (total ? total : 1u));
  g = min(g, n - 1);
  uint32_t lo, hi;  // invariant: off[lo] <= b < off[hi]
  if (off[g] <= b) {
    lo = g;
    uint32_t step = 1;
    hi = min(n, lo + step);
    while (hi < n && off[hi] <= b) { lo = hi; step <<= 1; hi = min(n, lo + step); }
  } else {
    hi = g;
    uint32_t step = 1;
    lo = hi > step ? hi - step : 0u;
    while (lo > 0 && off[lo] > b) { hi = lo; step <<= 1; lo = hi > step ? hi - step : 0u; }
  }
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if (off[mid] <= b) lo = mid; else hi = mid;
  }
  return lo;
}

// D_T: descriptor length, known at compile time; the row's descriptor lives in registers.
// require_flags: only tasks whose flags contain these bits are processed (0 = every task).
// rows: FM_FLAG_ROW_TABLE only (else null), the batch's records, indexed like rowres.
template <int D_T>
__global__ void __launch_bounds__(kExactRows)
exact_match_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks,
                   const uint32_t* __restrict__ task_blk_off, uint32_t n_tasks, float thr, float ratio,
                   uint32_t require_flags, uint32_t* __restrict__ rowres, float* __restrict__ rowdist,
                   fm_row* __restrict__ rows) {
  extern __shared__ float smem[];
  const uint32_t t = find_segment(task_blk_off, n_tasks, blockIdx.x);
  const Task task = tasks[t];
  if ((task.flags & require_flags) != require_flags) return;  // CTA-uniform
  const ImageDev A = images[task.col_img];
  const ImageDev B = images[task.row_img];
  constexpr int d = D_T;
  float* s_desc = smem;                          // [kExactCols][d]
  float* s_scale = s_desc + kExactCols * d;      // [kExactCols]
  float* s_lap = s_scale + kExactCols;           // [kExactCols]

  const uint32_t row = (blockIdx.x - task_blk_off[t]) * kExactRows + threadIdx.x;
  const bool active = row < B.n;

  float r[D_T];
  float sc = 1.f, lp = 0.f;
  if (active) {
    sc = B.scale[row];
    lp = B.lap[row];
    const float4* src = reinterpret_cast<const float4*>(B.desc + (size_t)row * D_T);
#pragma unroll
    for (int q = 0; q < D_T / 4; q++) {
      float4 v = __ldg(src + q);
      r[4 * q] = v.x; r[4 * q + 1] = v.y; r[4 * q + 2] = v.z; r[4 * q + 3] = v.w;
    }
  }

  float d1 = FLT_MAX, d2 = FLT_MAX;
  uint32_t match = 0;
  for (uint32_t c0 = 0; c0 < A.n; c0 += kExactCols) {
    const uint32_t nc = min((uint32_t)kExactCols, A.n - c0);
    __syncthreads();
    for (uint32_t idx = threadIdx.x; idx < nc * (uint32_t)d; idx += kExactRows)
      s_desc[idx] = __ldg(A.desc + (size_t)c0 * d + idx);
    if (threadIdx.x < nc) {
      s_scale[threadIdx.x] = A.scale[c0 + threadIdx.x];
      s_lap[threadIdx.x] = A.lap[c0 + threadIdx.x];
    }
    __syncthreads();
    if (!active) continue;
    for (uint32_t c = 0; c < nc; c++) {
      if (lp != s_lap[c]) continue;
      if (scale_gate_fails(sc, s_scale[c])) continue;
      float acc = 0.f;
      const float4* col = reinterpret_cast<const float4*>(s_desc + c * D_T);
#pragma unroll
      for (int q = 0; q < D_T / 4; q++) {
        float4 v = col[q];
        float e;
        e = __fsub_rn(r[4 * q], v.x);     acc = __fadd_rn(acc, __fmul_rn(e, e));
        e = __fsub_rn(r[4 * q + 1], v.y); acc = __fadd_rn(acc, __fmul_rn(e, e));
        e = __fsub_rn(r[4 * q + 2], v.z); acc = __fadd_rn(acc, __fmul_rn(e, e));
        e = __fsub_rn(r[4 * q + 3], v.w); acc = __fadd_rn(acc, __fmul_rn(e, e));
      }
      if (acc < d1) { d2 = d1; d1 = acc; match = c0 + c; }
      else if (acc < d2) { d2 = acc; }
    }
  }
  if (active) {
    rowres[task.row_off + row] = accept_rule(d1, d2, thr, ratio) ? match : kNone;
    if (rowdist) rowdist[task.row_off + row] = d1;  // FM_FLAG_DISTANCES: the reference's norm() of the emitted pair
    if (rows) put_row(rows, task.row_off + row, d1, d2, match);
  }
}

inline size_t exact_smem_bytes(int d) { return ((size_t)kExactCols * d + 2 * kExactCols) * sizeof(float); }

}  // namespace fm
