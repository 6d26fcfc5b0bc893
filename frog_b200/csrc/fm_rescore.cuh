// fm_rescore.cuh -- exact FP32 rescoring of the tensor-core candidates + the accept decision
// (replaces the tail of ComputeMatches, match.cpp:303-330, for rows scored by fm_score.cuh).
//
// Soundness.  Let t~ be the FP16-operand score and t the exact value of a.b - |b|^2/2, with
// |t~ - t| <= eps for every pair of the task.  If A2 is the second-largest t~ of a row, every
// column that can be the exact nearest or second-nearest neighbour (or tie with them) has
// t~ >= A2 - 2*eps: for such a column x and the better of the two approximate leaders y != x,
// t~(x) >= t(x) - eps >= t(y) - eps >= t~(y) - 2 eps >= A2 - 2 eps.  The scoring kernel captures
// every column above a threshold that never exceeds A2 - 2 eps, so the lists are complete unless
// one overflowed (marker) -- then the row is queued for the exact row kernel below.  Captured are
// re-evaluated with the reference's own arithmetic (gates, sequential FP32 norm, strict compares,
// lowest-original-index tie rule), so accepted pairs are bit-identical to the reference.
#pragma once
#include "fm_common.cuh"
#include "fm_exact.cuh"
#include "fm_score.cuh"

namespace fm {

struct RescoreCounters {
  unsigned long long candidates;      // exact distances evaluated
  unsigned long long redo_rows;       // rows handed to exact_rows_kernel
  unsigned long long rejected_early;  // rows proven unacceptable from their approximate scores alone
};

__device__ __forceinline__ float exact_norm48(const float (&r)[kD], const float* __restrict__ col) {
  float acc = 0.f;
  const float4* c4 = reinterpret_cast<const float4*>(col);
#pragma unroll
  for (int q = 0; q < kD / 4; q++) {
    float4 v = __ldg(c4 + q);
    float e;
    e = __fsub_rn(r[4 * q], v.x);     acc = __fadd_rn(acc, __fmul_rn(e, e));
    e = __fsub_rn(r[4 * q + 1], v.y); acc = __fadd_rn(acc, __fmul_rn(e, e));
    e = __fsub_rn(r[4 * q + 2], v.z); acc = __fadd_rn(acc, __fmul_rn(e, e));
    e = __fsub_rn(r[4 * q + 3], v.w); acc = __fadd_rn(acc, __fmul_rn(e, e));
  }
  return acc;
}

// Order-independent form of match.cpp:303-313: (d1, match, d2) = (min, lowest index attaining it,
// second smallest of the multiset).
__device__ __forceinline__ void top2_merge_one(float dist, uint32_t j, float& d1, float& d2, uint32_t& match) {
  if (dist < d1) { d2 = d1; d1 = dist; match = j; }
  else if (dist == d1) { d2 = d1; if (j < match) match = j; }
  else if (dist < d2) { d2 = dist; }
}

__device__ __forceinline__ void top2_merge_sets(float od1, float od2, uint32_t om, float& d1, float& d2, uint32_t& match) {
  const bool other_wins = od1 < d1 || (od1 == d1 && om < match);
  const float hi_d1 = fmaxf(d1, od1);  // the larger of the two minima is a second-smallest candidate
  d2 = fminf(hi_d1, fminf(d2, od2));
  if (other_wins) { d1 = od1; match = om; }
}

// One thread per sorted row of the task.
__global__ void __launch_bounds__(128, 6)
rescore_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks,
               const uint32_t* __restrict__ task_blk_off, uint32_t n_tasks, uint32_t segs,
               const Cand* __restrict__ cands, float thr, float ratio, uint32_t* __restrict__ rowres,
               uint2* __restrict__ redo_list, RescoreCounters* __restrict__ counters, float* __restrict__ rowdist,
               const uint8_t* __restrict__ rowstat, fm_row* __restrict__ rows) {
  const uint32_t t = find_segment_near(task_blk_off, n_tasks, blockIdx.x, gridDim.x);
  const Task task = tasks[t];
  if (task.flags & kTaskExact) return;
  const ImageDev A = images[task.col_img];
  const ImageDev B = images[task.row_img];
  const uint32_t s = (blockIdx.x - task_blk_off[t]) * 128 + threadIdx.x;
  if (s >= B.n) return;
  // Two-phase path: the reject pass of the scoring kernel has already proven most rows unacceptable (rowstat = 1);
  // their candidate lists were never written, and rowres was pre-filled with kNone for the whole batch, so such a
  // row costs this kernel one byte.
  const bool pre_rejected = rowstat != nullptr && rowstat[task.row_off + s] != 0;
  const uint32_t row = pre_rejected ? 0u : B.perm[s];
  const float eps = task_eps(A.meta, B.meta);

  // Candidate lists (one per column segment) hold every column whose score exceeded the list's
  // final capture threshold g2 - 2 eps <= (row's 2nd best) - 2 eps, unsorted; a +inf marker in
  // any list means that list overflowed.
  const uint32_t L = segs * kTopK;
  const Cand* c = cands + (size_t)(task.row_off + s) * L;
  float a1 = -INFINITY, a2 = -INFINITY;
  bool overflow = false;
  if (!pre_rejected) {
    for (uint32_t e = 0; e < L; e++) {
      const float v = c[e].t;
      if (v == INFINITY) overflow = true;
      else if (v > a1) { a2 = a1; a1 = v; }
      else if (v > a2) { a2 = v; }
    }
  }
  const float band = a2 - 2.f * eps;  // -inf when the row has fewer than two candidates
  // A truncated list dropped columns scoring <= its smallest kept entry: still complete iff that
  // entry is below the band.
  for (uint32_t g = 0; g < segs && !overflow && !pre_rejected; g++) {
    const Cand* l = c + g * kTopK;
    if (l[0].t > -INFINITY && (l[0].col & kCandTruncated)) {
      float lowest = l[0].t;
      for (int k = 1; k < kTopK; k++) lowest = fminf(lowest, l[k].t);
      if (lowest >= band) overflow = true;
    }
  }

  // Early rejection, certified (certified_reject, fm_score.cuh): the lists hold the row's two best approximate scores
  // a1 >= a2, and when the reference's ratio or threshold test must fail for them the row emits nothing and no exact
  // distance has to be gathered: with -d2 0.8 on unrelated images that is almost every row.
  // A row table (rows != null, never with the two-phase path) records every row's exact (d1, d2): no row is rejected
  // here.
  bool rejected = pre_rejected;
  if (!pre_rejected && !overflow && a1 > -INFINITY && !rows) rejected = certified_reject(B.norm2_sorted[s], a1, a2, eps, thr, ratio);

  uint32_t match = kNone;
  uint32_t n_eval = 0;
  float d1 = FLT_MAX, d2 = FLT_MAX;
  uint32_t best = 0;
  if (!overflow && !rejected && a1 > -INFINITY) {
    float r[kD];
    const float4* src = reinterpret_cast<const float4*>(B.desc + (size_t)row * kD);
#pragma unroll
    for (int q = 0; q < kD / 4; q++) {
      float4 v = __ldg(src + q);
      r[4 * q] = v.x; r[4 * q + 1] = v.y; r[4 * q + 2] = v.z; r[4 * q + 3] = v.w;
    }
    for (uint32_t e = 0; e < L; e++) {
      const Cand cd = c[e];
      if (!(cd.t > -INFINITY) || !(cd.t >= band)) continue;
      // Both gates (match.cpp:270, :273-275) hold for every captured column: the scoring kernel only captures inside
      // the row's interval [lo, hi), which bands_kernel built with the reference's own predicates (and which
      // tests/test_gpu_stages.py compares with the gate matrix).  Not re-reading lap / scale of the row and of each
      // column saves a fifth of this kernel's L2 sector traffic.
      const uint32_t j = A.perm[cd.col & ~kCandTruncated];
      const float dist = exact_norm48(r, A.desc + (size_t)j * kD);
      n_eval++;
      top2_merge_one(dist, j, d1, d2, best);
    }
    if (accept_rule(d1, d2, thr, ratio)) match = best;
    if (rowdist) rowdist[task.row_off + row] = d1;
  }
  if (!pre_rejected) rowres[task.row_off + row] = match;
  if (rows && !overflow) put_row(rows, task.row_off + row, d1, d2, best);  // (an overflowing row: exact_rows_kernel)
  if (overflow) {
    unsigned long long slot = atomicAdd(&counters->redo_rows, 1ull);
    redo_list[slot] = make_uint2(t, s);
  }
  // statistics: one atomic per warp
  uint32_t n_rej = rejected ? 1u : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    n_eval += __shfl_xor_sync(0xffffffffu, n_eval, o);
    n_rej += __shfl_xor_sync(0xffffffffu, n_rej, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (n_eval) atomicAdd(&counters->candidates, (unsigned long long)n_eval);
    if (n_rej) atomicAdd(&counters->rejected_early, (unsigned long long)n_rej);
  }
}

// Exact redo of queued rows: one CTA per row (queued rows are rare -- a handful per million -- so
// the parallelism has to come from inside the row).  Threads stride over the row's gate interval
// [lo, hi) of sorted columns (every column outside it fails a reference gate, fm_score.cuh
// bands_kernel), evaluate the reference's gates and FP32 distance on each, keep an
// order-independent (d1, lowest original index, d2) and merge across lanes / warps as multisets.
constexpr int kRedoThreads = 512;

__global__ void __launch_bounds__(kRedoThreads)
exact_rows_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks,
                  const uint2* __restrict__ bands, const uint2* __restrict__ redo_list,
                  const RescoreCounters* __restrict__ counters, float thr, float ratio,
                  uint32_t* __restrict__ rowres, float* __restrict__ rowdist, fm_row* __restrict__ rows) {
  __shared__ float s_d1[kRedoThreads / 32], s_d2[kRedoThreads / 32];
  __shared__ uint32_t s_m[kRedoThreads / 32];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned long long n = counters->redo_rows;
  for (unsigned long long w = blockIdx.x; w < n; w += gridDim.x) {
    const uint2 item = redo_list[w];
    const Task task = tasks[item.x];
    const ImageDev A = images[task.col_img];
    const ImageDev B = images[task.row_img];
    const uint32_t row = B.perm[item.y];
    const uint2 band = bands[task.row_off + item.y];
    float r[kD];
    const float4* src = reinterpret_cast<const float4*>(B.desc + (size_t)row * kD);
#pragma unroll
    for (int q = 0; q < kD / 4; q++) {
      float4 v = __ldg(src + q);
      r[4 * q] = v.x; r[4 * q + 1] = v.y; r[4 * q + 2] = v.z; r[4 * q + 3] = v.w;
    }
    const float sc = B.scale[row], lp = B.lap[row];
    float d1 = FLT_MAX, d2 = FLT_MAX;
    uint32_t match = 0;
    for (uint32_t c = band.x + threadIdx.x; c < band.y; c += kRedoThreads) {
      const uint32_t j = A.perm[c];
      if (lp != A.lap[j]) continue;                    // match.cpp:270
      if (scale_gate_fails(sc, A.scale[j])) continue;  // match.cpp:273-275
      const float dist = exact_norm48(r, A.desc + (size_t)j * kD);
      top2_merge_one(dist, j, d1, d2, match);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float od1 = __shfl_xor_sync(0xffffffffu, d1, o);
      const float od2 = __shfl_xor_sync(0xffffffffu, d2, o);
      const uint32_t om = __shfl_xor_sync(0xffffffffu, match, o);
      top2_merge_sets(od1, od2, om, d1, d2, match);
    }
    if (lane == 0) { s_d1[warp] = d1; s_d2[warp] = d2; s_m[warp] = match; }
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int k = 1; k < kRedoThreads / 32; k++) top2_merge_sets(s_d1[k], s_d2[k], s_m[k], d1, d2, match);
      rowres[task.row_off + row] = accept_rule(d1, d2, thr, ratio) ? match : kNone;
      if (rowdist) rowdist[task.row_off + row] = d1;
      if (rows) put_row(rows, task.row_off + row, d1, d2, match);
    }
    __syncthreads();
  }
}

}  // namespace fm
