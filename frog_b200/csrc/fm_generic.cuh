// fm_generic.cuh -- exact FP32 matcher for ANY descriptor length (d != 48): the reference's loop nest
// (match.cpp:262-330, and its `-all` form :295-300) on CUDA cores, K-chunked.
//
// surf3d can write descriptors of 24 r^3 or 8 r^3 values (-type 1 / 2: 3000 or 1000 floats at the
// default radius 5, vtkOpenSURF3D/surf3d.cxx:36-39), far too long to keep a row in registers or a
// column tile in shared memory.  One thread still owns one outer-loop row, but the distance of a
// (row, column) pair is accumulated over chunks of 64 descriptor values: per chunk the CTA stages
// 32 columns x 64 values (transposed, so a thread reads four columns per LDS.128) and its own
// 128 rows x 64 values in shared memory, and every thread advances 32 register accumulators.
// Each accumulator sees its k values in ascending order with separately rounded sub / mul / add,
// so the result is the reference's `norm` (match.cpp:243-251) bit for bit; the zero padding of a
// short last chunk adds +0.0, which changes nothing.  Gates are applied when a finished column
// tile is consumed, in ascending column order, with the reference's comparisons.
#pragma once
#include "fm_common.cuh"
#include "fm_exact.cuh"

namespace fm {

constexpr int kGenCols = 32;   // columns per tile (register accumulators per thread)
constexpr int kGenChunk = 64;  // descriptor values per chunk
constexpr int kGenColStride = kGenCols + 4;  // 16-byte aligned rows, fewer bank conflicts on the transposed store

struct GenSmem {
  float colT[kGenChunk][kGenColStride];  // [k][column]
  float row[kExactRows][kGenChunk + 1];  // [row][k]
  float scale[kGenCols], lap[kGenCols];
};

// kMode 0: nearest / second-nearest + acceptance -> rowres (match.cpp:303-330), and the row's record -> rows
// (FM_FLAG_ROW_TABLE; null otherwise).
// kMode 1: -all count pass -> row_count / row_final.   kMode 2: -all emit pass (see fm_all.cuh).
template <int kMode>
__global__ void __launch_bounds__(kExactRows)
exact_generic_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks,
                     const uint32_t* __restrict__ task_blk_off, uint32_t n_tasks, float thr, float ratio,
                     uint32_t require_flags, uint32_t* __restrict__ rowres, uint32_t* __restrict__ row_count,
                     uint32_t* __restrict__ row_final, const uint32_t* __restrict__ row_carry,
                     const unsigned long long* __restrict__ row_off, const unsigned long long* __restrict__ task_base,
                     uint2* __restrict__ out, float* __restrict__ rowdist, fm_row* __restrict__ rows) {
  __shared__ GenSmem sm;
  const uint32_t t = find_segment(task_blk_off, n_tasks, blockIdx.x);
  const Task task = tasks[t];
  if ((task.flags & require_flags) != require_flags) return;  // CTA-uniform
  const ImageDev A = images[task.col_img];
  const ImageDev B = images[task.row_img];
  const uint32_t d = A.d;
  const uint32_t row0 = (blockIdx.x - task_blk_off[t]) * kExactRows;
  const uint32_t row = row0 + threadIdx.x;
  const bool active = row < B.n;
  const bool swap = task.flags & kTaskSwap;
  const float sc = active ? B.scale[row] : 1.f, lp = active ? B.lap[row] : 0.f;

  float d1 = FLT_MAX, d2 = FLT_MAX;
  uint32_t match = (kMode == 2 && active) ? row_carry[task.row_off + row] : 0u;
  uint32_t count = 0;
  uint2* o = (kMode == 2 && active) ? out + task_base[t] + row_off[task.row_off + row] : nullptr;

  for (uint32_t c0 = 0; c0 < A.n; c0 += kGenCols) {
    const uint32_t nc = min((uint32_t)kGenCols, A.n - c0);
    __syncthreads();  // the previous tile has been consumed
    if (threadIdx.x < nc) {
      sm.scale[threadIdx.x] = A.scale[c0 + threadIdx.x];
      sm.lap[threadIdx.x] = A.lap[c0 + threadIdx.x];
    }
    float acc[kGenCols];
#pragma unroll
    for (int c = 0; c < kGenCols; c++) acc[c] = 0.f;
    for (uint32_t k0 = 0; k0 < d; k0 += kGenChunk) {
      const uint32_t kc = min((uint32_t)kGenChunk, d - k0);
      __syncthreads();  // the previous chunk has been consumed
      for (uint32_t idx = threadIdx.x; idx < (uint32_t)(kGenCols * kGenChunk); idx += kExactRows) {
        const uint32_t c = idx / kGenChunk, k = idx % kGenChunk;  // consecutive threads: consecutive k (coalesced)
        sm.colT[k][c] = (c < nc && k < kc) ? __ldg(A.desc + (size_t)(c0 + c) * d + k0 + k) : 0.f;
      }
      for (uint32_t idx = threadIdx.x; idx < (uint32_t)(kExactRows * kGenChunk); idx += kExactRows) {
        const uint32_t r = idx / kGenChunk, k = idx % kGenChunk;
        sm.row[r][k] = (row0 + r < B.n && k < kc) ? __ldg(B.desc + (size_t)(row0 + r) * d + k0 + k) : 0.f;
      }
      __syncthreads();
      for (uint32_t k = 0; k < kc; k++) {
        const float rk = sm.row[threadIdx.x][k];
#pragma unroll
        for (int c4 = 0; c4 < kGenCols / 4; c4++) {
          const float4 v = *reinterpret_cast<const float4*>(&sm.colT[k][4 * c4]);
          float e;
          e = __fsub_rn(rk, v.x); acc[4 * c4 + 0] = __fadd_rn(acc[4 * c4 + 0], __fmul_rn(e, e));
          e = __fsub_rn(rk, v.y); acc[4 * c4 + 1] = __fadd_rn(acc[4 * c4 + 1], __fmul_rn(e, e));
          e = __fsub_rn(rk, v.z); acc[4 * c4 + 2] = __fadd_rn(acc[4 * c4 + 2], __fmul_rn(e, e));
          e = __fsub_rn(rk, v.w); acc[4 * c4 + 3] = __fadd_rn(acc[4 * c4 + 3], __fmul_rn(e, e));
        }
      }
    }
    if (!active) continue;
#pragma unroll
    for (int c = 0; c < kGenCols; c++) {
      if ((uint32_t)c >= nc) continue;
      if (lp != sm.lap[c]) continue;                    // match.cpp:270
      if (scale_gate_fails(sc, sm.scale[c])) continue;  // match.cpp:273-275
      const float dist = acc[c];
      if (kMode == 0) {
        if (dist < d1) { d2 = d1; d1 = dist; match = c0 + c; }
        else if (dist < d2) { d2 = dist; }
      } else if (__fsqrt_rn(dist) < thr) {  // match.cpp:295
        if (kMode == 2) o[count] = swap ? make_uint2(row, match) : make_uint2(match, row);
        count++;
      } else if (dist < d1) {
        d1 = dist;
        match = c0 + c;
      }
    }
  }
  if (!active) return;
  if (kMode == 0) {
    rowres[task.row_off + row] = accept_rule(d1, d2, thr, ratio) ? match : kNone;
    if (rowdist) rowdist[task.row_off + row] = d1;
    if (rows) put_row(rows, task.row_off + row, d1, d2, match);
  }
  if (kMode == 1) {
    row_count[task.row_off + row] = count;
    row_final[task.row_off + row] = d1 != FLT_MAX ? match : kNone;
  }
}

}  // namespace fm
