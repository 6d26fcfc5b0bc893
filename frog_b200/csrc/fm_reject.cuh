// fm_reject.cuh -- reject pass of two-phase scoring (fm_fast.cuh): for every row of a 256-row unit, the row's best
// approximate score g1 and the second largest 16-column chunk maximum g2 over its gated-in columns, then the certified
// rejection test (certified_reject, fm_score.cuh) and the survivor list the capture pass works on.
//
// One persistent CTA per SM walks units blockIdx.x, blockIdx.x + gridDim.x, ...  Per 256-column step the unit's two
// row halves each take one tcgen05.mma M=128 x N<=256 x K=16 chain into their own 256-column TMEM buffer.
// Against the single pass's N=64 this reads the row operand once per 256 columns instead of once per 64: 12 KB of
// shared-memory operand reads per 128 cycles of MMA math instead of 6 KB per 32, which is what kept the tensor pipe
// below half its rate.  Two cuts keep the MMAs to the work the result needs:
//   * a half's chain covers only the step's columns inside that half's own band union, rounded out to 16 columns;
//   * for column images whose squared norms barely vary (normalised descriptors) the chain is 3 K-steps, not 4: the
//     norm term moves out of the MMA into the rejection test as the image's norm range (rj_ksteps).
// Any other image keeps the single pass's accumulator (M=128, FP32, K=64 in four steps), so its scores, and therefore
// its g1, g2 and rejected rows, are the single pass's.
//   warp 0      scheduler  : task lookup, the unit's 256 bands and its column-step range -> a 4-slot ring in shared
//                            memory, so unit prologues (dependent global loads) run ahead of the pipeline
//   warp 1      TMA        : the unit's two 16 KB row-operand tiles (double-buffered across units) and 32 KB column
//                            steps into a 4-stage ring
//   warp 2      MMA        : buffer h <- row half h, alternating, so one half's MMAs run while the other is drained
//   warps 3..10 epilogue   : (TMEM lane quadrant = warp % 4) x (column round c): every warp drains every buffer, in
//                            the order the MMA warp fills them, loading its 128 columns [128 c, 128 c + 128) and
//                            releasing the buffer before it reduces them, so a buffer goes back to the MMA warp one
//                            TMEM load after it was published.  Whether a round is skipped, interior (straight-line
//                            max trees) or masked is decided once per round, warp-uniformly.  Each thread keeps a
//                            partial (g1, g2) for its row in both halves; at unit end the quadrant's two warps merge
//                            them (exactly: max and min) and warp (q, c) tests the rows of half c.  (Eight warps, not
//                            sixteen: eleven warps leave 168 registers per thread for the 128-column rounds, nineteen
//                            would leave 96.)
// Scores never leave the SM.
#pragma once
#include "fm_score.cuh"

namespace fm {

// One step is 256 columns (N = 256): TMEM's 512 columns hold one accumulator buffer per row half, and each epilogue
// warp drains one 128-column round of every buffer.  (N = 128 with two stages per half measured 1.3x slower: the row
// operand is re-read from shared memory for every 128 columns.)
constexpr int kRjCols = 256;
constexpr int kRjStepBytes = kRjCols * 128;  // one step of the column operand: two stored operand tiles
constexpr int kRjStages = 4;                 // 128 KB of column-operand ring
constexpr int kRjSlots = 4;                  // units the scheduler warp may run ahead
constexpr int kRjEpiWarps = 8;
constexpr int kRjThreads = (3 + kRjEpiWarps) * 32;

struct RjUnit {
  const uint8_t* rowop;  // the unit's two row-operand tiles (row halves 0 and 1)
  const uint8_t* colop;
  uint32_t task, n_rows, row_off, s0;  // s0: sorted position of the unit's first row
  uint32_t step0, n_steps;             // column steps [step0, step0 + n_steps) of kRjCols columns
  uint2 span[2];                       // row half h's bands lie in columns [span[h].x, span[h].y) (empty: y <= x)
  uint32_t ksteps;                     // K-steps per MMA chain: 4, or 3 without the norm slots (see rj_ksteps)
  float noff1, noff2;                  // ksteps == 3: n_min / 2 and n_max / 2 of the column image; else 0
  float eps;
  uint32_t skip;                       // task takes the exact kernel: nothing to write
};

// K = 48 instead of 64 for a column image whose squared norms barely vary (SURF3D descriptors are L2-normalised).
// The fourth K-step (slots 48..63) only adds the column's -|b|^2/2 through slots 48 and 49.  Without it the MMA yields
// t' = fp16(a).fp16(b) in FP32, and the K = 64 score is t = t' - n_b/2 with n_b in [n_min, n_max] (FP32 norms, the values
// the operand carries).  The unit end then tests, instead of the row's g1 and g2 of t,
//   a1 = g1' - n_min/2  (rounded up)    >= best t       (every column's t <= t' - n_min/2 <= g1' - n_min/2)
//   a2 = g2' - n_max/2  (rounded down)  <= second t     (two columns of different chunks reach t' >= g2')
// so certified_reject keeps its meaning: rounding toward +-inf makes the FP32 subtractions one-sided, with no slack
// term.  The existing eps still bounds |t' - n_b/2 - (a.b - |b|^2/2)|: of its additive part, the hi/lo split of
// -|b|^2/2 is gone, and the FP32 accumulation inside the tensor core now sums 48 products without the norm term,
// less than the 64-term bound it was given; the operand rounding terms are the same.  What the rows lose is
// (n_max - n_min)/2 of certification margin, hence the rule: K = 48 when that is at most eps, so that normalised inputs
// reject as before (differences only at the certification edge), while any other image keeps its exact K = 64 chain.
__device__ __forceinline__ uint32_t rj_ksteps(const ImageMeta& col, float eps) {
  return 0.5f * (col.max_norm2 - min_norm2(col)) <= eps ? 3u : 4u;  // (no keypoint: min_norm2 is NaN, 4)
}

struct RjWarpRange {
  uint32_t cmin, cmax;  // columns some row of the warp accepts lie in [cmin, cmax)
  uint32_t imin, imax;  // every row of the warp accepts [imin, imax)
};

struct alignas(1024) RejectSmem {
  uint8_t a[2][2][kOpTileBytes];        // [unit buffer][row half]
  uint8_t b[kRjStages][kRjStepBytes];
  uint2 band[kRjSlots][kUnitRows];      // the unit's bands, (0, 0) for rows past the image
  float norm2[kRjSlots][kUnitRows];     // the rows' squared norms (rows with a band only)
  RjUnit unit[kRjSlots];
  uint64_t bar_afull[2], bar_aempty[2];
  uint64_t bar_bfull[kRjStages], bar_bempty[kRjStages];
  uint64_t bar_accfull[2], bar_accempty[2];  // [row half]
  uint64_t bar_ufull[kRjSlots], bar_uempty[kRjSlots];
  float2 part[2][kUnitRows];                 // [unit parity][row]: (g1, g2) of one column round, passed at unit end
  RjWarpRange wrange[kRjEpiWarps][2];        // [epilogue warp][row half], warp-uniform (kept out of registers)
  uint32_t tmem_base;
};
constexpr size_t kRjSmemBytes = sizeof(RejectSmem) + 1024;

// Maximum of the 16 columns r[O .. O + 16) of a 32-column group; kMasked: column O + e counts only if bit O + e of
// the group's mask m is set (a bit test and a select per score), otherwise as -inf.
template <bool kMasked, int O>
__device__ __forceinline__ float rj_chunk(const uint32_t (&r)[32], uint32_t m) {
  float f[16];
#pragma unroll
  for (int e = 0; e < 16; e++) {
    f[e] = __uint_as_float(r[O + e]);
    if (kMasked) f[e] = (m & (1u << (O + e))) ? f[e] : -INFINITY;
  }
  const float ga = max3(max3(f[0], f[1], f[2]), max3(f[3], f[4], f[5]), max3(f[6], f[7], f[8]));
  const float gb = max3(max3(f[9], f[10], f[11]), max3(f[12], f[13], f[14]), f[15]);
  return fmaxf(ga, gb);
}

// (a1 >= a2) and (b1 >= b2) are the two largest values of two multisets: make (a1, a2) those of their union.  Max and
// min are exact, so the result does not depend on how a row's chunk maxima are grouped.
__device__ __forceinline__ void rj_top2(float& a1, float& a2, float b1, float b2) {
  a2 = max3(a2, b2, fminf(a1, b1));
  a1 = fmaxf(a1, b1);
}

// Bits [0, n) set, n clamped to [0, 32].
__device__ __forceinline__ uint32_t rj_bits_below(int n) { return __funnelshift_lc(0xFFFFFFFFu, 0u, (uint32_t)max(n, 0)); }

// One 128-column round (r0 .. r3, 32 columns each, starting at a multiple of 128, so its eight 16-column chunks are the
// single pass's chunks): fold the chunk maxima into the row's top two (g1 >= g2).  kMasked: only columns
// [a, a + width) of the round count (a relative to the round's first column, may be negative).
template <bool kMasked>
__device__ __forceinline__ void rj_round(const uint32_t (&r0)[32], const uint32_t (&r1)[32], const uint32_t (&r2)[32],
                                         const uint32_t (&r3)[32], int a, int width, float& g1, float& g2) {
  uint32_t m[4] = {0u, 0u, 0u, 0u};  // group j's columns [a - 32 j, a + width - 32 j) as bits
  if (kMasked)
#pragma unroll
    for (int j = 0; j < 4; j++) m[j] = rj_bits_below(a + width - 32 * j) & ~rj_bits_below(a - 32 * j);
  const float c[8] = {rj_chunk<kMasked, 0>(r0, m[0]), rj_chunk<kMasked, 16>(r0, m[0]),
                      rj_chunk<kMasked, 0>(r1, m[1]), rj_chunk<kMasked, 16>(r1, m[1]),
                      rj_chunk<kMasked, 0>(r2, m[2]), rj_chunk<kMasked, 16>(r2, m[2]),
                      rj_chunk<kMasked, 0>(r3, m[3]), rj_chunk<kMasked, 16>(r3, m[3])};
  float t1[4], t2[4];
#pragma unroll
  for (int p = 0; p < 4; p++) {
    t1[p] = fmaxf(c[2 * p], c[2 * p + 1]);
    t2[p] = fminf(c[2 * p], c[2 * p + 1]);
  }
  rj_top2(t1[0], t2[0], t1[1], t2[1]);
  rj_top2(t1[2], t2[2], t1[3], t2[3]);
  rj_top2(t1[0], t2[0], t1[2], t2[2]);
  rj_top2(g1, g2, t1[0], t2[0]);
}

// units = unit_off[n_tasks] (segs = 1).  scored_cols += (row, column) scores the tensor cores computed: 128 x N per
// MMA chain issued, band-edge and 16-column round-out columns included.  Writes rowstat[row] (1 = rejected) for every row of every fast task and
// appends the sorted position of each surviving row to its task's survivor list (surv_count / surv_rows, any order).
// kDump (test hook fm_debug_reject_rows): also writes dump[row] = (a1, a2, |a|^2, eps), the arguments the row's
// certified_reject receives, for every row with a non-empty band, and NaNs for every other row of a fast task.
template <bool kDump>
__global__ void __launch_bounds__(kRjThreads, 1)
reject_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks, const uint32_t* __restrict__ unit_off,
              uint32_t n_tasks, uint32_t units, const uint2* __restrict__ bands, unsigned long long* __restrict__ scored_cols,
              float thr, float ratio, uint8_t* __restrict__ rowstat, uint32_t* __restrict__ surv_count,
              uint32_t* __restrict__ surv_rows, float4* __restrict__ dump) {
  extern __shared__ uint8_t smem_raw[];
  RejectSmem& sm = *reinterpret_cast<RejectSmem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 2 && lane == 0) {
    for (int i = 0; i < 2; i++) {
      ptx::mbar_init(&sm.bar_afull[i], 1);
      ptx::mbar_init(&sm.bar_aempty[i], 1);
    }
    for (int h = 0; h < 2; h++) {
      ptx::mbar_init(&sm.bar_accfull[h], 1);
      ptx::mbar_init(&sm.bar_accempty[h], kRjEpiWarps);  // every epilogue warp drains every buffer
    }
    for (int i = 0; i < kRjStages; i++) { ptx::mbar_init(&sm.bar_bfull[i], 1); ptx::mbar_init(&sm.bar_bempty[i], 1); }
    for (int i = 0; i < kRjSlots; i++) {
      ptx::mbar_init(&sm.bar_ufull[i], 32);                // every lane of the scheduler warp
      ptx::mbar_init(&sm.bar_uempty[i], 2 + kRjEpiWarps);  // TMA thread, MMA thread, one arrival per epilogue warp
    }
    ptx::fence_mbar_init();
  }
  if (warp == 0) ptx::tmem_alloc<512>(&sm.tmem_base);
  ptx::tc_fence_before();
  __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem = sm.tmem_base;

  if (warp == 0) {
    // ---- scheduler --------------------------------------------------------------------------------------------
    uint32_t k = 0;
    for (uint32_t unit = blockIdx.x; unit < units; unit += gridDim.x, k++) {
      const uint32_t slot = k % kRjSlots;
      if (k >= (uint32_t)kRjSlots) ptx::mbar_wait(&sm.bar_uempty[slot], (k / kRjSlots - 1) & 1);
      const uint32_t t = find_segment_near(unit_off, n_tasks, unit, units);
      const Task task = tasks[t];
      const ImageDev A = images[task.col_img];
      const ImageDev B = images[task.row_img];
      const uint32_t s0 = (unit - unit_off[t]) * kUnitRows;
      const bool skip = (task.flags & kTaskExact) != 0;
      uint32_t cmin[2] = {0xFFFFFFFFu, 0xFFFFFFFFu}, cmax[2] = {0u, 0u};  // per row half
#pragma unroll
      for (int j = 0; j < kUnitRows / 32; j++) {
        const uint32_t r = j * 32 + lane, s = s0 + r;
        const int h = j / (kUnitRows / 64);
        uint2 bd = make_uint2(0u, 0u);
        if (!skip && s < B.n) bd = bands[task.row_off + s];
        if (bd.y > bd.x) { cmin[h] = min(cmin[h], bd.x); cmax[h] = max(cmax[h], bd.y); }
        sm.band[slot][r] = bd;
        if (bd.y > bd.x) sm.norm2[slot][r] = B.norm2_sorted[s];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int h = 0; h < 2; h++) {
          cmin[h] = min(cmin[h], __shfl_xor_sync(0xffffffffu, cmin[h], o));
          cmax[h] = max(cmax[h], __shfl_xor_sync(0xffffffffu, cmax[h], o));
        }
      if (lane == 0) {
        const uint32_t umin = min(cmin[0], cmin[1]), umax = max(cmax[0], cmax[1]);
        RjUnit u;
        u.rowop = reinterpret_cast<const uint8_t*>(B.rowop) + (size_t)s0 / 128 * kOpTileBytes;
        u.colop = reinterpret_cast<const uint8_t*>(A.colop);
        u.task = t;
        u.n_rows = B.n;
        u.row_off = task.row_off;
        u.s0 = s0;
        u.step0 = umax > umin ? umin / kRjCols : 0u;
        u.n_steps = umax > umin ? (umax + kRjCols - 1) / kRjCols - u.step0 : 0u;
        u.span[0] = make_uint2(cmin[0], cmax[0]);
        u.span[1] = make_uint2(cmin[1], cmax[1]);
        u.eps = skip ? 0.f : task_eps(A.meta, B.meta);
        u.ksteps = skip ? 4u : rj_ksteps(*A.meta, u.eps);
        u.noff1 = u.ksteps == 3 ? 0.5f * min_norm2(*A.meta) : 0.f;
        u.noff2 = u.ksteps == 3 ? 0.5f * A.meta->max_norm2 : 0.f;
        u.skip = skip ? 1u : 0u;
        sm.unit[slot] = u;
      }
      ptx::mbar_arrive(&sm.bar_ufull[slot]);
    }
  } else if (warp == 1) {
    // ---- TMA ----------------------------------------------------------------------------------------------------
    if (lane == 0) {
      uint32_t k = 0, a_use = 0, bq = 0;
      for (uint32_t unit = blockIdx.x; unit < units; unit += gridDim.x, k++) {
        const uint32_t slot = k % kRjSlots;
        ptx::mbar_wait(&sm.bar_ufull[slot], (k / kRjSlots) & 1);
        const RjUnit& us = sm.unit[slot];
        const uint8_t* rowop = us.rowop;
        const uint8_t* colop = us.colop;
        const uint32_t step0 = us.step0, n_steps = us.n_steps;
        ptx::mbar_arrive(&sm.bar_uempty[slot]);
        if (n_steps == 0) continue;
        const uint32_t ab = a_use & 1;
        if (a_use >= 2) ptx::mbar_wait(&sm.bar_aempty[ab], (a_use / 2 - 1) & 1);
        a_use++;
        ptx::mbar_expect_tx(&sm.bar_afull[ab], 2 * kOpTileBytes);
        ptx::bulk_g2s(sm.a[ab][0], rowop, kOpTileBytes, &sm.bar_afull[ab]);
        ptx::bulk_g2s(sm.a[ab][1], rowop + kOpTileBytes, kOpTileBytes, &sm.bar_afull[ab]);
        for (uint32_t i = 0; i < n_steps; i++, bq++) {
          const uint32_t stg = bq % kRjStages, use = bq / kRjStages;
          if (use > 0) ptx::mbar_wait(&sm.bar_bempty[stg], (use - 1) & 1);
          const uint8_t* src = colop + (size_t)(step0 + i) * kRjStepBytes;  // n_pad is a multiple of 256: in bounds
          ptx::mbar_expect_tx(&sm.bar_bfull[stg], kRjStepBytes);
          ptx::bulk_g2s(sm.b[stg], src, kRjStepBytes / 2, &sm.bar_bfull[stg]);
          ptx::bulk_g2s(sm.b[stg] + kRjStepBytes / 2, src + kRjStepBytes / 2, kRjStepBytes / 2, &sm.bar_bfull[stg]);
        }
      }
    }
  } else if (warp == 2) {
    // ---- MMA ----------------------------------------------------------------------------------------------------
    if (lane == 0) {
      uint32_t k = 0, a_use = 0, bq = 0, g = 0;
      unsigned long long issued = 0;
      for (uint32_t unit = blockIdx.x; unit < units; unit += gridDim.x, k++) {
        const uint32_t slot = k % kRjSlots;
        ptx::mbar_wait(&sm.bar_ufull[slot], (k / kRjSlots) & 1);
        const RjUnit& us = sm.unit[slot];
        const uint32_t step0 = us.step0, n_steps = us.n_steps, ksteps = us.ksteps;
        const uint2 span[2] = {us.span[0], us.span[1]};
        ptx::mbar_arrive(&sm.bar_uempty[slot]);
        if (n_steps == 0) continue;
        const uint32_t ab = a_use & 1;
        ptx::mbar_wait(&sm.bar_afull[ab], (a_use / 2) & 1);
        a_use++;
        const uint64_t adesc[2] = {ptx::umma_desc_sw128(ptx::smem_u32(sm.a[ab][0])), ptx::umma_desc_sw128(ptx::smem_u32(sm.a[ab][1]))};
        for (uint32_t i = 0; i < n_steps; i++, bq++, g++) {
          const uint32_t stg = bq % kRjStages, c0 = (step0 + i) * kRjCols;
          ptx::mbar_wait(&sm.bar_bfull[stg], (bq / kRjStages) & 1);
#pragma unroll
          for (int h = 0; h < 2; h++) {
            if (g > 0) ptx::mbar_wait(&sm.bar_accempty[h], (g - 1) & 1);
            ptx::tc_fence_after();
            // Only the step's columns inside this half's span, in whole 16-column pieces (N = 16 .. 256; a B operand
            // starting 16 j rows into the step starts on a 1024 B swizzle atom).  The buffer's other columns keep
            // stale values: they lie outside every band of the half, so the epilogue masks or skips them.  A half
            // whose span misses the step (or that has no rows) is still handed to its epilogue warps, unscored.
            const uint32_t lo = max(span[h].x, c0), hi = min(span[h].y, c0 + kRjCols);
            if (hi > lo) {
              const uint32_t off = (lo - c0) & ~15u, n = ((hi - c0 + 15) & ~15u) - off;
              const uint32_t idesc = ptx::umma_idesc_f16_f32(128, (int)n);
              const uint64_t bdesc = ptx::umma_desc_sw128(ptx::smem_u32(sm.b[stg]) + off * 128);
#pragma unroll
              for (uint32_t kk = 0; kk < kKPad / 16; kk++)  // +32 B per K step inside the 128 B swizzle row
                if (kk < ksteps)
                  ptx::mma_f16_ss(tmem + h * kRjCols + off, adesc[h] + 2 * kk, bdesc + 2 * kk, idesc, kk > 0);
              issued += 128 * n;
            }
            ptx::mma_commit(&sm.bar_accfull[h]);
          }
          ptx::mma_commit(&sm.bar_bempty[stg]);
        }
        ptx::mma_commit(&sm.bar_aempty[ab]);
      }
      if (scored_cols != nullptr) atomicAdd(scored_cols, issued);
    }
  } else {
    // ---- epilogue -----------------------------------------------------------------------------------------------
    // Warp (q, c): TMEM lane quadrant q = warp % 4 (the lanes the warp may access) and column round c: columns
    // [128 c, 128 c + 128) of every step, in both row halves' buffers.  Per row half h, thread `lane` keeps row
    // 128 h + 32 q + lane: its band and the (g1, g2) of the chunks in the warp's rounds.  At unit end the quadrant's two
    // warps exchange their partial pairs through shared memory, and warp (q, c) tests the rows of half c.
    const uint32_t c = (warp - 3) >> 2, q = warp & 3;
    uint32_t taddr = tmem + ((q * 32) << 16) + c * 128;
    asm volatile("" : "+r"(taddr));
    uint32_t g = 0, k = 0;
    for (uint32_t unit = blockIdx.x; unit < units; unit += gridDim.x, k++) {
      const uint32_t slot = k % kRjSlots;
      ptx::mbar_wait(&sm.bar_ufull[slot], (k / kRjSlots) & 1);
      // (the slot is released at unit end, after the rejection tail has read the rest of it)
      const RjUnit& us = sm.unit[slot];
      const uint32_t step0 = us.step0, n_steps = us.n_steps;
      const uint2* band = sm.band[slot] + q * 32 + lane;  // + 128 h: this thread's row of half h
      RjWarpRange* wr = sm.wrange[warp - 3];
#pragma unroll
      for (int h = 0; h < 2; h++) {
        const uint2 bd = band[h * 128];
        const bool valid = bd.y > bd.x;
        RjWarpRange w{valid ? bd.x : 0xFFFFFFFFu, valid ? bd.y : 0u, valid ? bd.x : 0u, valid ? bd.y : 0xFFFFFFFFu};
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
          w.cmin = min(w.cmin, __shfl_xor_sync(0xffffffffu, w.cmin, o));
          w.cmax = max(w.cmax, __shfl_xor_sync(0xffffffffu, w.cmax, o));
          w.imin = max(w.imin, __shfl_xor_sync(0xffffffffu, w.imin, o));
          w.imax = min(w.imax, __shfl_xor_sync(0xffffffffu, w.imax, o));
        }
        if (lane == 0) wr[h] = w;
      }
      __syncwarp();
      float g1[2] = {-INFINITY, -INFINITY}, g2[2] = {-INFINITY, -INFINITY};
      for (uint32_t i = 0; i < n_steps; i++, g++) {
        const uint32_t c0 = (step0 + i) * kRjCols + c * 128;
#pragma unroll
        for (int h = 0; h < 2; h++) {  // in the order the MMA warp fills the buffers
          ptx::mbar_wait(&sm.bar_accfull[h], g & 1);
          ptx::tc_fence_after();
          const RjWarpRange w = wr[h];
          const bool need = c0 < w.cmax && c0 + 128 > w.cmin;        // warp-uniform
          const bool interior = c0 >= w.imin && c0 + 128 <= w.imax;  // warp-uniform: every row accepts the round
          uint32_t r0[32], r1[32], r2[32], r3[32];
          if (need) {
            const uint32_t t = taddr + h * kRjCols;
            ptx::tmem_ld32(r0, t);
            ptx::tmem_ld32(r1, t + 32);
            ptx::tmem_ld32(r2, t + 64);
            ptx::tmem_ld32(r3, t + 96);
            ptx::tmem_ld_wait(r0, r1, r2, r3);
          }
          // every column this warp needs is in registers: hand the buffer back to the MMA warp before reducing
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&sm.bar_accempty[h]);
          if (need) {
            if (interior) {
              rj_round<false>(r0, r1, r2, r3, 0, 0, g1[h], g2[h]);
            } else {
              const uint2 bd = band[h * 128];
              rj_round<true>(r0, r1, r2, r3, (int)(bd.x - c0), bd.y > bd.x ? (int)(bd.y - bd.x) : 0, g1[h], g2[h]);
            }
          }
        }
      }
      // the partner warp (q, 1 - c) has the other round of every step: pass it this warp's pairs for half 1 - c and
      // take its pairs for half c (double-buffered by unit, so a partner already at the next unit end cannot
      // overwrite a pair before it has been read)
      const uint32_t row = c * 128 + q * 32 + lane, s = us.s0 + row;  // the row this thread tests
      float2* part = sm.part[k & 1];
      part[(c ^ 1) * 128 + q * 32 + lane] = c ? make_float2(g1[0], g2[0]) : make_float2(g1[1], g2[1]);
      ptx::named_bar_sync(1 + q, 64);
      const float2 o = part[row];
      float t1 = c ? g1[1] : g1[0], t2 = c ? g2[1] : g2[0];
      rj_top2(t1, t2, o.x, o.y);
      if (!us.skip && s < us.n_rows) {
        // a row with no gated-in column has nothing to emit; otherwise the certified test (g1 = a1, g2 <= a2)
        bool rejected = true;
        const uint2 bd = sm.band[slot][row];
        // (K = 48: the bounds of rj_ksteps; K = 64: the offsets are 0 and a1, a2 are g1, g2)
        if (bd.y > bd.x && t1 > -INFINITY)
          rejected = certified_reject(sm.norm2[slot][row], __fsub_ru(t1, us.noff1), __fsub_rd(t2, us.noff2), us.eps, thr, ratio);
        if constexpr (kDump)
          dump[us.row_off + s] = bd.y > bd.x ? make_float4(__fsub_ru(t1, us.noff1), __fsub_rd(t2, us.noff2), sm.norm2[slot][row], us.eps)
                                             : make_float4(NAN, NAN, NAN, NAN);
        const uint32_t row_off = us.row_off;
        rowstat[row_off + s] = rejected ? 1 : 0;
        if (!rejected) surv_rows[row_off + atomicAdd(surv_count + us.task, 1u)] = s;  // at most n_rows survivors
      }
      __syncwarp();
      if (lane == 0) ptx::mbar_arrive(&sm.bar_uempty[slot]);
    }
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<512>(sm.tmem_base);  // (re-read: keeps the address out of the epilogue's registers)
  }
}

}  // namespace fm
