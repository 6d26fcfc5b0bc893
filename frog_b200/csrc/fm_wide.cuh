// fm_wide.cuh -- the tensor-core path for descriptor lengths other than 48 (surf3d -type 1 raw Haar descriptors of
// 24 r^3 values, -type 2 descriptors of 8 r^3 values; any 1 <= d <= kWideMaxD): wide scoring kernel, its certified
// error bound, exact rescoring, exact redo of the rows whose lists may be incomplete, and the batch driver.
//
// Scores.  Each image carries ONE FP16 operand (ImageDev::wideop, fm_prep.cuh prep_wide_pack_kernel): fp16(desc) in
// K_pad = wide_kpad(d) slots, zeros after d, as [n_pad / 128 tiles][K_pad / 64 k-blocks] of 16 KB SWIZZLE_128B tiles.
// The MMA yields a16.b16 in FP32 and the epilogue adds -|b|^2/2 (FP32, norm2_sorted), so t~ = a16.b16 - |b|^2/2,
// larger t~ <=> smaller distance, as on the d = 48 path.
//
// Kernel (reject_kernel's skeleton, fm_reject.cuh).  One persistent CTA per SM walks units blockIdx.x, + gridDim.x, ...
// A unit is one 128-row block of a task (the blk_off prefix), so the CTAs running at the same time work on consecutive
// row blocks of one task and share its column band in L2.  A step is 256 sorted columns of the unit's band union
// (bands_kernel), 256-aligned.
//   warp 0      scheduler  : task lookup, the unit's 128 bands and step range -> a 4-slot ring in shared memory
//   warp 1      TMA        : per step and k-block, the unit's 16 KB row tile and the step's two 16 KB column tiles
//                            into a 4-stage ring (48 KB a stage)
//   warp 2      MMA        : per step K_pad / 16 tcgen05.mma M=128 x N<=256 x K=16 into one of two 256-column TMEM
//                            buffers (N trimmed to the step's columns inside the band union, in 16-column pieces),
//                            then a commit hands the buffer to the epilogue
//   warps 3..10 epilogue   : warp (lane quadrant q = warp % 4, column half c) drains its 32 rows x 128 columns of the
//                            buffer in two 64-column halves (releasing it after the second load), adds -|b|^2/2, gates
//                            each column to the row's band [lo, hi) and keeps
//                            the row's kTopK largest gated scores (one compare against the 8th per score, a sorted
//                            insertion only when it is beaten).  At unit end warp (q, 0) merges the list of warp (q, 1)
//                            and writes one Cand list per row (segs = 1), kCandTruncated when hi - lo > kTopK.
// No running threshold and no look-ahead: every MMA is issued once.  With the truncated bit the completeness rule of
// fm_rescore.cuh holds unchanged: a truncated list whose smallest kept score is >= a2 - 2 eps goes to the exact redo.
//
// Certified error bound (wide_task_eps).  With t_ref = (|a|^2 - d^2_ref) / 2, d^2_ref the reference's sequential FP32
// sum of d terms (match.cpp:243-251), and a16 = a + da, b16 = b + db the FP16 operands (|da|, |db| the measured
// residual norms, |a|, |b| <= the images' max norms):
//   |t~ - t_ref| <= (1) |a||db| + |da||b| + |da||db|                 a16.b16 - a.b, Cauchy-Schwarz (as task_eps)
//                 + (2) K_pad 2^-23 |a16||b16|                       FP32 accumulation of K_pad products in the tensor
//                                                                    core: order and rounding are not documented, so a
//                                                                    bound linear in K_pad with a full FP32 ulp (2^-23,
//                                                                    truncation allowed) per product of the sum
//                                                                    sum |a16_k b16_k| <= |a16||b16|
//                 + (3) d 2^-25 |b|^2 + 2^-23 (|a16||b16| + |b|^2)  prep's FP32 sum of |b|^2 (halved), the epilogue add
//                 + (4) (d + 2) 2^-25 (|a| + |b|)^2                  the reference's own rounding of d^2: d separately
//                                                                    rounded squares and d - 1 additions of terms whose
//                                                                    sum is d^2 <= (|a| + |b|)^2, halved for t
// inflated by 1 % for the FP32 evaluation of the bound.  Term (4) grows with d: at d = 3000 it is ~1.8e-4 for unit
// descriptors where task_eps's fixed 3e-5 covers d = 48 only.  tests/test_gpu_wide.py checks |t~ - t_ref| <= eps on
// every visited pair of dumped units and reports the largest ratio.
#pragma once
#include "fm_fast.cuh"

namespace fm {

constexpr int kWdCols = 256;                   // columns per step: one TMEM accumulator buffer
constexpr int kWdColBytes = kWdCols * 128;     // one k-block of a step: two 16 KB column tiles
constexpr int kWdStages = 4;                   // 4 x (16 + 32) KB = 192 KB of operand ring
constexpr int kWdSlots = 4;                    // units the scheduler warp may run ahead
constexpr int kWdEpiWarps = 8;
constexpr int kWdThreads = (3 + kWdEpiWarps) * 32;
constexpr int kWdRows = 128;                   // rows per unit

__host__ __device__ __forceinline__ float wide_task_eps(const ImageMeta& ma, const ImageMeta& mb, uint32_t d) {
  const float n2 = fmaxf(ma.max_norm2, mb.max_norm2);
  const float na = sqrtf(ma.max_norm2), nb = sqrtf(mb.max_norm2);
  const float da = sqrtf(ma.max_delta2), db = sqrtf(mb.max_delta2);
  const float ab16 = (na + da) * (nb + db);
  const float df = (float)d;
  const float e_op = na * db + da * nb + da * db;                   // (1)
  const float e_mma = (float)wide_kpad(d) * 0x1p-23f * ab16;        // (2)
  const float e_norm = df * 0x1p-25f * n2 + 0x1p-23f * (ab16 + n2);  // (3)
  const float e_ref = (df + 2.f) * 0x1p-25f * (na + nb) * (na + nb);  // (4)
  return 1.01f * (e_op + e_mma + e_norm + e_ref);
}

// certified_reject (fm_score.cuh) for the wide path: the row's |a|^2 is prep's FP32 sum of d squares, within
// d 2^-24 |a|^2 of the exact value, so the part of the margin that covers its evaluation grows with d as well.
__device__ __forceinline__ bool wide_certified_reject(float na, float a1, float a2, float eps, float thr, float ratio, uint32_t d) {
  const float margin = 2.f * eps + (1e-5f + (float)d * 0x1p-23f) * (na + 4.f);
  const float d1_lo = na - 2.f * a1 - margin;
  const float d2_hi = na - 2.f * a2 + margin;
  bool rejected = d1_lo > thr * thr * 1.00001f;
  if (a2 > -INFINITY && d2_hi > 0.f && ratio < 1.0e4f) rejected = rejected || d1_lo > ratio * ratio * d2_hi * 1.0001f;
  return rejected;
}

struct WdUnit {
  const uint8_t* rowop;  // the unit's row tile of k-block 0 (k-block kb is kb * 16 KB further)
  const uint8_t* colop;  // the column image's operand
  const float* cnorm;    // the column image's norm2_sorted
  uint32_t n_rows, row_off, s0;
  uint32_t step0, n_steps;  // column steps [step0, step0 + n_steps) of kWdCols columns
  uint32_t cmin, cmax;      // union of the unit's bands (empty: cmax <= cmin)
  uint32_t kblocks;
  uint32_t skip;            // task takes the exact kernel: nothing to write
};

struct alignas(1024) WideSmem {
  uint8_t a[kWdStages][kOpTileBytes];
  uint8_t b[kWdStages][kWdColBytes];
  uint2 band[kWdSlots][kWdRows];
  float nrm[kWdEpiWarps][128];   // per epilogue warp: -|b|^2/2 of its 128 columns of the current step
  Cand part[kTopK][kWdRows];     // unit end: the list of warp (q, 1) for warp (q, 0), [slot][row]
  WdUnit unit[kWdSlots];
  uint64_t bar_full[kWdStages], bar_empty[kWdStages];
  uint64_t bar_accfull[2], bar_accempty[2];
  uint64_t bar_ufull[kWdSlots], bar_uempty[kWdSlots];
  uint32_t tmem_base;
};
constexpr size_t kWdSmemBytes = sizeof(WideSmem) + 1024;

// Insert (v, col) into the descending list (t, c) of kTopK entries, dropping the smallest.  Static indices only: the
// list stays in registers.
__device__ __forceinline__ void wd_insert(float (&t)[kTopK], uint32_t (&c)[kTopK], float v, uint32_t col) {
#pragma unroll
  for (int k = 0; k < kTopK; k++) {
    const bool sw = v > t[k];
    const float tv = t[k];
    const uint32_t tc = c[k];
    t[k] = sw ? v : tv;
    c[k] = sw ? col : tc;
    v = sw ? tv : v;
    col = sw ? tc : col;
  }
}

// 32 columns of one row: score = accumulator + nrm, gated to [lo, lo + width).  kDump: also stores the scores of the
// columns the MMA computed (dmask) to drow.
template <bool kDump>
__device__ __forceinline__ void wd_cols(const uint32_t (&r)[32], const float* nrm, uint32_t col0, uint32_t lo, uint32_t width,
                                        float (&t)[kTopK], uint32_t (&c)[kTopK], float* drow, uint32_t dlo, uint32_t dhi) {
#pragma unroll
  for (int e = 0; e < 32; e++) {
    const uint32_t col = col0 + e;
    const float v = __uint_as_float(r[e]) + nrm[e];
    if constexpr (kDump) {
      if (drow != nullptr && col >= dlo && col < dhi) drow[col] = v;
    }
    if (col - lo < width && v > t[kTopK - 1]) wd_insert(t, c, v, col);
  }
}

// blk_off: 128-row blocks per task (prefix, n_tasks + 1 entries); units [unit_base, units) are the blocks to score
// (unit_base != 0 only for the single-unit debug launch).  cands: [batch rows][kTopK].  scored_cols += 128 x N per MMA
// chain.  kDump (test hook fm_debug_wide_unit): dump[row_in_unit * dump_ld + col] = t~ of every column the MMAs
// computed, *dump_eps = the task's eps.
template <bool kDump>
__global__ void __launch_bounds__(kWdThreads, 1)
wide_score_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks, const uint32_t* __restrict__ blk_off,
                  uint32_t n_tasks, uint32_t unit_base, uint32_t units, const uint2* __restrict__ bands, Cand* __restrict__ cands,
                  unsigned long long* __restrict__ scored_cols, float* __restrict__ dump, uint32_t dump_ld,
                  float* __restrict__ dump_eps) {
  extern __shared__ uint8_t smem_raw[];
  WideSmem& sm = *reinterpret_cast<WideSmem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 2 && lane == 0) {
    for (int i = 0; i < kWdStages; i++) { ptx::mbar_init(&sm.bar_full[i], 1); ptx::mbar_init(&sm.bar_empty[i], 1); }
    for (int i = 0; i < 2; i++) { ptx::mbar_init(&sm.bar_accfull[i], 1); ptx::mbar_init(&sm.bar_accempty[i], kWdEpiWarps); }
    for (int i = 0; i < kWdSlots; i++) {
      ptx::mbar_init(&sm.bar_ufull[i], 32);                // every lane of the scheduler warp
      ptx::mbar_init(&sm.bar_uempty[i], 2 + kWdEpiWarps);  // TMA thread, MMA thread, one arrival per epilogue warp
    }
    ptx::fence_mbar_init();
  }
  if (warp == 0) ptx::tmem_alloc<512>(&sm.tmem_base);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  const uint32_t first = unit_base + blockIdx.x;

  if (warp == 0) {
    // ---- scheduler --------------------------------------------------------------------------------------------
    uint32_t k = 0;
    for (uint32_t unit = first; unit < units; unit += gridDim.x, k++) {
      const uint32_t slot = k % kWdSlots;
      if (k >= (uint32_t)kWdSlots) ptx::mbar_wait(&sm.bar_uempty[slot], (k / kWdSlots - 1) & 1);
      const uint32_t t = find_segment_near(blk_off, n_tasks, unit, units);
      const Task task = tasks[t];
      const ImageDev A = images[task.col_img];
      const ImageDev B = images[task.row_img];
      const uint32_t s0 = (unit - blk_off[t]) * kWdRows;
      const bool skip = (task.flags & kTaskExact) != 0;
      uint32_t cmin = 0xFFFFFFFFu, cmax = 0u;
#pragma unroll
      for (int j = 0; j < kWdRows / 32; j++) {
        const uint32_t r = j * 32 + lane, s = s0 + r;
        uint2 bd = make_uint2(0u, 0u);
        if (!skip && s < B.n) bd = bands[task.row_off + s];
        if (bd.y > bd.x) { cmin = min(cmin, bd.x); cmax = max(cmax, bd.y); }
        sm.band[slot][r] = bd;
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        cmin = min(cmin, __shfl_xor_sync(0xffffffffu, cmin, o));
        cmax = max(cmax, __shfl_xor_sync(0xffffffffu, cmax, o));
      }
      if (lane == 0) {
        const uint32_t kblocks = wide_kpad(A.d) / 64u;
        WdUnit u;
        u.rowop = reinterpret_cast<const uint8_t*>(B.wideop) + (size_t)(s0 / kWdRows) * kblocks * kOpTileBytes;
        u.colop = reinterpret_cast<const uint8_t*>(A.wideop);
        u.cnorm = A.norm2_sorted;
        u.n_rows = B.n;
        u.row_off = task.row_off;
        u.s0 = s0;
        u.cmin = cmin;
        u.cmax = cmax;
        u.step0 = cmax > cmin ? cmin / kWdCols : 0u;
        u.n_steps = cmax > cmin ? (cmax + kWdCols - 1) / kWdCols - u.step0 : 0u;
        u.kblocks = kblocks;
        u.skip = skip ? 1u : 0u;
        sm.unit[slot] = u;
        if constexpr (kDump) *dump_eps = skip ? 0.f : wide_task_eps(*A.meta, *B.meta, A.d);
      }
      ptx::mbar_arrive(&sm.bar_ufull[slot]);
    }
  } else if (warp == 1) {
    // ---- TMA ----------------------------------------------------------------------------------------------------
    if (lane == 0) {
      uint32_t k = 0, q = 0;
      for (uint32_t unit = first; unit < units; unit += gridDim.x, k++) {
        const uint32_t slot = k % kWdSlots;
        ptx::mbar_wait(&sm.bar_ufull[slot], (k / kWdSlots) & 1);
        const WdUnit& us = sm.unit[slot];
        const uint8_t* rowop = us.rowop;
        const uint8_t* colop = us.colop;
        const uint32_t step0 = us.step0, n_steps = us.n_steps, kblocks = us.kblocks;
        ptx::mbar_arrive(&sm.bar_uempty[slot]);
        for (uint32_t i = 0; i < n_steps; i++) {
          // the step's two column tiles (n_pad is a multiple of 256: in bounds)
          const uint8_t* c0 = colop + (size_t)(2 * (step0 + i)) * kblocks * kOpTileBytes;
          const uint8_t* c1 = c0 + (size_t)kblocks * kOpTileBytes;
          for (uint32_t kb = 0; kb < kblocks; kb++, q++) {
            const uint32_t stg = q % kWdStages, use = q / kWdStages;
            if (use > 0) ptx::mbar_wait(&sm.bar_empty[stg], (use - 1) & 1);
            ptx::mbar_expect_tx(&sm.bar_full[stg], kOpTileBytes + kWdColBytes);
            ptx::bulk_g2s(sm.a[stg], rowop + (size_t)kb * kOpTileBytes, kOpTileBytes, &sm.bar_full[stg]);
            ptx::bulk_g2s(sm.b[stg], c0 + (size_t)kb * kOpTileBytes, kOpTileBytes, &sm.bar_full[stg]);
            ptx::bulk_g2s(sm.b[stg] + kOpTileBytes, c1 + (size_t)kb * kOpTileBytes, kOpTileBytes, &sm.bar_full[stg]);
          }
        }
      }
    }
  } else if (warp == 2) {
    // ---- MMA ----------------------------------------------------------------------------------------------------
    if (lane == 0) {
      uint32_t k = 0, q = 0, g = 0;
      unsigned long long issued = 0;
      for (uint32_t unit = first; unit < units; unit += gridDim.x, k++) {
        const uint32_t slot = k % kWdSlots;
        ptx::mbar_wait(&sm.bar_ufull[slot], (k / kWdSlots) & 1);
        const WdUnit& us = sm.unit[slot];
        const uint32_t step0 = us.step0, n_steps = us.n_steps, kblocks = us.kblocks, cmin = us.cmin, cmax = us.cmax;
        ptx::mbar_arrive(&sm.bar_uempty[slot]);
        for (uint32_t i = 0; i < n_steps; i++, g++) {
          const uint32_t buf = g & 1, c0 = (step0 + i) * kWdCols;
          if (g >= 2) ptx::mbar_wait(&sm.bar_accempty[buf], ((g >> 1) - 1) & 1);
          ptx::tc_fence_after();
          // only the step's columns inside the band union, in whole 16-column pieces (a B operand starting 16 j rows
          // into the step starts on a 1024 B swizzle atom); the buffer's other columns keep stale values, outside
          // every band of the unit
          const uint32_t lo = max(cmin, c0), hi = min(cmax, c0 + kWdCols);
          const uint32_t off = (lo - c0) & ~15u, n = ((hi - c0 + 15) & ~15u) - off;
          const uint32_t idesc = ptx::umma_idesc_f16_f32(128, (int)n);
          for (uint32_t kb = 0; kb < kblocks; kb++, q++) {
            const uint32_t stg = q % kWdStages;
            ptx::mbar_wait(&sm.bar_full[stg], (q / kWdStages) & 1);
            ptx::tc_fence_after();
            const uint64_t adesc = ptx::umma_desc_sw128(ptx::smem_u32(sm.a[stg]));
            const uint64_t bdesc = ptx::umma_desc_sw128(ptx::smem_u32(sm.b[stg]) + off * 128);
#pragma unroll
            for (uint32_t kk = 0; kk < 4; kk++)  // +32 B per K step inside the 128 B swizzle row
              ptx::mma_f16_ss(tmem + buf * kWdCols + off, adesc + 2 * kk, bdesc + 2 * kk, idesc, (kb | kk) != 0);
            ptx::mma_commit(&sm.bar_empty[stg]);
          }
          ptx::mma_commit(&sm.bar_accfull[buf]);
          issued += 128ull * n;
        }
      }
      if (scored_cols != nullptr) atomicAdd(scored_cols, issued);
    }
  } else {
    // ---- epilogue -----------------------------------------------------------------------------------------------
    // Warp (q, c): TMEM lane quadrant q = warp % 4 (the lanes the warp may access), rows 32 q + lane of the unit, and
    // columns [128 c, 128 c + 128) of every step.
    const uint32_t c = (warp - 3) >> 2, q = warp & 3, ew = warp - 3;
    const uint32_t r = q * 32 + lane;
    uint32_t taddr = tmem + ((q * 32) << 16) + c * 128;
    asm volatile("" : "+r"(taddr));
    float* nrm = sm.nrm[ew];
    uint32_t g = 0, k = 0;
    for (uint32_t unit = first; unit < units; unit += gridDim.x, k++) {
      const uint32_t slot = k % kWdSlots;
      ptx::mbar_wait(&sm.bar_ufull[slot], (k / kWdSlots) & 1);
      // (the slot is released at unit end)
      const WdUnit& us = sm.unit[slot];
      const uint32_t step0 = us.step0, n_steps = us.n_steps;
      const float* cnorm = us.cnorm;
      const uint2 bd = sm.band[slot][r];
      const uint32_t lo = bd.x, width = bd.y > bd.x ? bd.y - bd.x : 0u;
      uint32_t wmin = width ? bd.x : 0xFFFFFFFFu, wmax = width ? bd.y : 0u;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        wmin = min(wmin, __shfl_xor_sync(0xffffffffu, wmin, o));
        wmax = max(wmax, __shfl_xor_sync(0xffffffffu, wmax, o));
      }
      const uint32_t s = us.s0 + r;
      float* drow = nullptr;
      if constexpr (kDump) drow = s < us.n_rows ? dump + (size_t)r * dump_ld : nullptr;
      float tl[kTopK];
      uint32_t cl[kTopK];
#pragma unroll
      for (int e = 0; e < kTopK; e++) { tl[e] = -INFINITY; cl[e] = 0u; }
      for (uint32_t i = 0; i < n_steps; i++, g++) {
        const uint32_t buf = g & 1, cs = (step0 + i) * kWdCols, c0 = cs + c * 128;
        const bool need = kDump || (c0 < wmax && c0 + 128 > wmin);  // warp-uniform
        ptx::mbar_wait(&sm.bar_accfull[buf], (g >> 1) & 1);
        ptx::tc_fence_after();
        // The 128 columns in two halves of 64: the first is reduced while the buffer is still held, the second is
        // loaded, then the buffer goes back to the MMA warp before it is reduced.  (All 128 at once need 128 data
        // registers next to the list and spill.)
        uint32_t r0[32], r1[32];
        const uint32_t t = taddr + buf * kWdCols;
        uint32_t dlo = 0, dhi = 0;  // kDump: the columns the MMAs computed (the MMA warp's trim)
        if constexpr (kDump) {
          const uint32_t ml = max(us.cmin, cs), mh = min(us.cmax, cs + kWdCols);
          dlo = cs + ((ml - cs) & ~15u);
          dhi = cs + ((mh - cs + 15) & ~15u);
        }
        if (need) {
          __syncwarp();  // every lane is done with the previous step's norms
          const float4 nv = __ldg(reinterpret_cast<const float4*>(cnorm + c0) + lane);  // norm2_sorted holds n_pad floats
          ptx::tmem_ld32(r0, t);
          ptx::tmem_ld32(r1, t + 32);
          reinterpret_cast<float4*>(nrm)[lane] = make_float4(-0.5f * nv.x, -0.5f * nv.y, -0.5f * nv.z, -0.5f * nv.w);
          ptx::tmem_ld_wait(r0, r1);
          __syncwarp();
          wd_cols<kDump>(r0, nrm, c0, lo, width, tl, cl, drow, dlo, dhi);
          wd_cols<kDump>(r1, nrm + 32, c0 + 32, lo, width, tl, cl, drow, dlo, dhi);
          ptx::tmem_ld32(r0, t + 64);
          ptx::tmem_ld32(r1, t + 96);
          ptx::tmem_ld_wait(r0, r1);
        }
        ptx::tc_fence_before();
        __syncwarp();
        if (lane == 0) ptx::mbar_arrive(&sm.bar_accempty[buf]);
        if (need) {
          wd_cols<kDump>(r0, nrm + 64, c0 + 64, lo, width, tl, cl, drow, dlo, dhi);
          wd_cols<kDump>(r1, nrm + 96, c0 + 96, lo, width, tl, cl, drow, dlo, dhi);
        }
      }
      // unit end: warp (q, 1) passes its list to warp (q, 0), which merges and writes the row's candidates
      if (c == 1) {
#pragma unroll
        for (int e = 0; e < kTopK; e++) sm.part[e][r] = Cand{tl[e], cl[e]};
      }
      ptx::named_bar_sync(1 + q, 64);
      if (c == 0) {
#pragma unroll
        for (int e = 0; e < kTopK; e++) {
          const Cand o = sm.part[e][r];
          if (o.t > tl[kTopK - 1]) wd_insert(tl, cl, o.t, o.col);
        }
        if (!us.skip && s < us.n_rows) {
          Cand* out = cands + (size_t)(us.row_off + s) * kTopK;
#pragma unroll
          for (int e = 0; e < kTopK; e++)
            out[e] = Cand{tl[e], cl[e] | (e == 0 && width > (uint32_t)kTopK ? kCandTruncated : 0u)};
        }
      }
      ptx::named_bar_sync(1 + q, 64);  // warp (q, 1) may overwrite sm.part only after it has been read
      if (lane == 0) ptx::mbar_arrive(&sm.bar_uempty[slot]);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(sm.tmem_base);
  }
}

// The reference's norm (match.cpp:243-251) for any d: k ascending, separately rounded sub / mul / add (exact_norm48
// generalised).  Rows of a d % 4 == 0 image are 16-byte aligned and are read four values at a time.
__device__ __forceinline__ float exact_norm_any(const float* __restrict__ a, const float* __restrict__ b, uint32_t d) {
  float acc = 0.f, e;
  uint32_t k = 0;
  if ((d & 3u) == 0) {
    for (; k < d; k += 4) {
      const float4 x = __ldg(reinterpret_cast<const float4*>(a + k)), y = __ldg(reinterpret_cast<const float4*>(b + k));
      e = __fsub_rn(x.x, y.x); acc = __fadd_rn(acc, __fmul_rn(e, e));
      e = __fsub_rn(x.y, y.y); acc = __fadd_rn(acc, __fmul_rn(e, e));
      e = __fsub_rn(x.z, y.z); acc = __fadd_rn(acc, __fmul_rn(e, e));
      e = __fsub_rn(x.w, y.w); acc = __fadd_rn(acc, __fmul_rn(e, e));
    }
  }
  for (; k < d; k++) {
    e = __fsub_rn(__ldg(a + k), __ldg(b + k));
    acc = __fadd_rn(acc, __fmul_rn(e, e));
  }
  return acc;
}

// rescore_kernel's logic for the wide path: eight threads per sorted row (a CTA = one 128-row block), thread e of a
// row evaluates the exact distance of candidate e -- d sequential operations each -- and the row's (d1, match, d2) is
// the order-independent merge of the eight (top2_merge_sets, fm_rescore.cuh).
constexpr int kWdRescoreThreads = kWdRows * kTopK;

__global__ void __launch_bounds__(kWdRescoreThreads)
wide_rescore_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks,
                    const uint32_t* __restrict__ task_blk_off, uint32_t n_tasks, const Cand* __restrict__ cands, float thr,
                    float ratio, uint32_t* __restrict__ rowres, uint2* __restrict__ redo_list,
                    RescoreCounters* __restrict__ counters, float* __restrict__ rowdist, fm_row* __restrict__ rows) {
  const uint32_t t = find_segment_near(task_blk_off, n_tasks, blockIdx.x, gridDim.x);
  const Task task = tasks[t];
  if (task.flags & kTaskExact) return;  // CTA-uniform
  const ImageDev A = images[task.col_img];
  const ImageDev B = images[task.row_img];
  const uint32_t e = threadIdx.x & (kTopK - 1);
  const uint32_t s = (blockIdx.x - task_blk_off[t]) * kWdRows + threadIdx.x / kTopK;
  const bool active = s < B.n;  // uniform over a row's eight threads; every thread stays for the shuffles
  const uint32_t d = A.d;
  const float eps = wide_task_eps(*A.meta, *B.meta, d);
  const Cand* c = cands + (size_t)(task.row_off + (active ? s : 0u)) * kTopK;
  float a1 = -INFINITY, a2 = -INFINITY;
  bool overflow = false;
  if (active) {
    for (int k = 0; k < kTopK; k++) {
      const float v = c[k].t;
      if (v == INFINITY) overflow = true;
      else if (v > a1) { a2 = a1; a1 = v; }
      else if (v > a2) { a2 = v; }
    }
  }
  const float band = a2 - 2.f * eps;
  // a truncated list dropped columns scoring <= its smallest kept entry: complete iff that entry is below the band
  if (active && !overflow && c[0].t > -INFINITY && (c[0].col & kCandTruncated)) {
    float lowest = c[0].t;
    for (int k = 1; k < kTopK; k++) lowest = fminf(lowest, c[k].t);
    if (lowest >= band) overflow = true;
  }
  bool rejected = false;  // (never with a row table, as in rescore_kernel)
  if (active && !overflow && a1 > -INFINITY && !rows) rejected = wide_certified_reject(B.norm2_sorted[s], a1, a2, eps, thr, ratio, d);
  const bool eval = active && !overflow && !rejected && a1 > -INFINITY;
  const uint32_t row = active ? B.perm[s] : 0u;
  float d1 = FLT_MAX, d2 = FLT_MAX;
  uint32_t best = kNone, n_eval = 0;
  if (eval) {
    const Cand cd = c[e];
    if (cd.t > -INFINITY && cd.t >= band) {
      const uint32_t j = A.perm[cd.col & ~kCandTruncated];
      d1 = exact_norm_any(B.desc + (size_t)row * d, A.desc + (size_t)j * d, d);
      best = j;
      n_eval = 1;
    }
  }
#pragma unroll
  for (int o = 1; o < kTopK; o <<= 1) {  // within the row's eight threads
    const float od1 = __shfl_xor_sync(0xffffffffu, d1, o);
    const float od2 = __shfl_xor_sync(0xffffffffu, d2, o);
    const uint32_t om = __shfl_xor_sync(0xffffffffu, best, o);
    top2_merge_sets(od1, od2, om, d1, d2, best);
  }
  if (active && e == 0) {
    rowres[task.row_off + row] = eval && accept_rule(d1, d2, thr, ratio) ? best : kNone;
    if (eval && rowdist) rowdist[task.row_off + row] = d1;
    if (rows && !overflow) put_row(rows, task.row_off + row, d1, d2, best);
    if (overflow) redo_list[atomicAdd(&counters->redo_rows, 1ull)] = make_uint2(t, s);
  }
  // statistics: one atomic per warp
  uint32_t n_rej = (rejected && e == 0) ? 1u : 0u;
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

// exact_rows_kernel's logic for the wide path: one CTA per queued row, the row's descriptor in shared memory, threads
// striding over its gate band, each evaluating the reference's gates and exact distance on its columns.
__global__ void __launch_bounds__(kRedoThreads)
wide_exact_rows_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks, const uint2* __restrict__ bands,
                       const uint2* __restrict__ redo_list, const RescoreCounters* __restrict__ counters, float thr,
                       float ratio, uint32_t* __restrict__ rowres, float* __restrict__ rowdist, fm_row* __restrict__ rows) {
  __shared__ __align__(16) float s_row[kWideMaxD];
  __shared__ float s_d1[kRedoThreads / 32], s_d2[kRedoThreads / 32];
  __shared__ uint32_t s_m[kRedoThreads / 32];
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const unsigned long long n = counters->redo_rows;
  for (unsigned long long w = blockIdx.x; w < n; w += gridDim.x) {
    const uint2 item = redo_list[w];
    const Task task = tasks[item.x];
    const ImageDev A = images[task.col_img];
    const ImageDev B = images[task.row_img];
    const uint32_t d = A.d;
    const uint32_t row = B.perm[item.y];
    const uint2 band = bands[task.row_off + item.y];
    for (uint32_t k = threadIdx.x; k < d; k += kRedoThreads) s_row[k] = B.desc[(size_t)row * d + k];
    __syncthreads();
    const float sc = B.scale[row], lp = B.lap[row];
    float d1 = FLT_MAX, d2 = FLT_MAX;
    uint32_t match = 0;
    for (uint32_t c = band.x + threadIdx.x; c < band.y; c += kRedoThreads) {
      const uint32_t j = A.perm[c];
      if (lp != A.lap[j]) continue;                    // match.cpp:270
      if (scale_gate_fails(sc, A.scale[j])) continue;  // match.cpp:273-275
      const float* col = A.desc + (size_t)j * d;
      float acc = 0.f, e;
      uint32_t k = 0;
      if ((d & 3u) == 0) {  // 16-byte aligned rows: four values per load, same order
        for (; k < d; k += 4) {
          const float4 y = __ldg(reinterpret_cast<const float4*>(col + k));
          const float4 x = *reinterpret_cast<const float4*>(s_row + k);
          e = __fsub_rn(x.x, y.x); acc = __fadd_rn(acc, __fmul_rn(e, e));
          e = __fsub_rn(x.y, y.y); acc = __fadd_rn(acc, __fmul_rn(e, e));
          e = __fsub_rn(x.z, y.z); acc = __fadd_rn(acc, __fmul_rn(e, e));
          e = __fsub_rn(x.w, y.w); acc = __fadd_rn(acc, __fmul_rn(e, e));
        }
      }
      for (; k < d; k++) {
        e = __fsub_rn(s_row[k], __ldg(col + k));
        acc = __fadd_rn(acc, __fmul_rn(e, e));
      }
      top2_merge_one(acc, j, d1, d2, match);
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

// One batch on the wide path: bands -> wide score -> wide rescore -> wide redo -> fold.  (Never two-phase: the reject
// pass is built for K = 64.)
inline cudaError_t wide_match_batch(fm_ctx* c, const FastBatchArgs& a) {
  cudaError_t e;
  if ((e = c->d_bands.ensure((size_t)a.rows * sizeof(uint2))) != cudaSuccess) return e;
  if ((e = c->d_cands.ensure((size_t)a.rows * kTopK * sizeof(Cand))) != cudaSuccess) return e;
  if ((e = c->d_redo.ensure((size_t)a.rows * sizeof(uint2))) != cudaSuccess) return e;
  if (!c->wide_attr_set) {
    if ((e = cudaFuncSetAttribute(wide_score_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWdSmemBytes)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(wide_score_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWdSmemBytes)) != cudaSuccess) return e;
    c->wide_attr_set = true;
  }
  {
    Span sp(&c->ev_match, c->stream, kPhBands);
    bands_kernel<<<a.blocks128, 128, 0, c->stream>>>(a.images, a.tasks, a.blk_off, a.n_tasks, c->d_bands.as<uint2>());
  }
  {
    Span sp(&c->ev_match, c->stream, kPhScore);
    const uint32_t grid = std::min<uint32_t>(a.blocks128, (uint32_t)c->sm_count);  // persistent: one CTA per SM
    wide_score_kernel<false><<<grid, kWdThreads, kWdSmemBytes, c->stream>>>(
        a.images, a.tasks, a.blk_off, a.n_tasks, 0u, a.blocks128, c->d_bands.as<uint2>(), c->d_cands.as<Cand>(),
        &a.counters->scored_cols, nullptr, 0u, nullptr);
  }
  {
    Span sp(&c->ev_match, c->stream, kPhRescore);
    wide_rescore_kernel<<<a.blocks128, kWdRescoreThreads, 0, c->stream>>>(
        a.images, a.tasks, a.blk_off, a.n_tasks, c->d_cands.as<Cand>(), a.thr, a.ratio, a.rowres, c->d_redo.as<uint2>(),
        &a.counters->rescore, a.rowdist, a.table);
    // two CTAs per SM: a queued row is a long dependent chain per column, so the latency hiding comes from residency
    wide_exact_rows_kernel<<<2 * c->sm_count, kRedoThreads, 0, c->stream>>>(a.images, a.tasks, c->d_bands.as<uint2>(), c->d_redo.as<uint2>(),
                                                                        &a.counters->rescore, a.thr, a.ratio, a.rowres, a.rowdist, a.table);
    fold_redo_kernel<<<1, 1, 0, c->stream>>>(a.counters);
  }
  c->stats.kernel_launches += 5;
  c->stats.score_launches += 1;
  return cudaGetLastError();
}

}  // namespace fm
