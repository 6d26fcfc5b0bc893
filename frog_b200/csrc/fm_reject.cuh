// fm_reject.cuh -- reject pass of two-phase scoring (fm_fast.cuh): for every row of a 512-row unit, the row's best
// approximate score g1 and the second largest 16-column chunk maximum g2 over its gated-in columns, then the certified
// rejection test (certified_reject, fm_score.cuh) and the survivor list the capture pass works on.
//
// One persistent CTA per SM walks units blockIdx.x, blockIdx.x + gridDim.x, ...  Per 256-column step the unit's four
// 128-row quarters each take one tcgen05.mma M=128 x N<=256 x K=16 chain into one of two 256-column TMEM buffers
// (quarter q -> buffer q % 2, in quarter order).  Against the single pass's N=64 this reads the row operand once per 256
// columns instead of once per 64: 12 KB of shared-memory operand reads per 128 cycles of MMA math instead of 6 KB per
// 32, which is what kept the tensor pipe below half its rate.  512 rows per unit, not 256, because what bounds the pass
// is delivering the column operand from L2: a 32 KB column step now feeds four chains instead of two, and the band
// union of 512 sorted rows is only a few percent wider than that of 256, so the column bytes per launch almost halve.
// Two cuts keep the MMAs to the work the result needs:
//   * a quarter's chain covers only the step's columns inside that quarter's own band union, rounded out to 16 columns;
//   * for column images whose squared norms barely vary (normalised descriptors) the chain is 3 K-steps, not 4: the
//     norm term moves out of the MMA into the rejection test as the image's norm range (rj_ksteps).
// Any other image keeps the single pass's accumulator (M=128, FP32, K=64 in four steps), so its scores, and therefore
// its g1, g2 and rejected rows, are the single pass's.
//   warp 0      scheduler  : task lookup, the unit's 512 bands, its four quarter spans and its column-step range ->
//                            a 2-slot ring in shared memory, so unit prologues (dependent global loads) run ahead of
//                            the pipeline
//   warp 1      TMA        : the unit's (up to) four 16 KB row-operand tiles (double-buffered across units) and 32 KB
//                            column steps into a 2-stage ring
//   warp 2      MMA        : buffer q % 2 <- quarter q, alternating, so one quarter's MMAs run while the previous
//                            quarter's buffer is drained; the column stage is released after the fourth fill
//   warps 3..10 epilogue   : (TMEM lane quadrant = warp % 4) x (column round c): every warp drains every fill, in
//                            the order the MMA warp makes them, loading its 128 columns [128 c, 128 c + 128) and
//                            releasing the buffer before it reduces them, so a buffer goes back to the MMA warp one
//                            TMEM load after it was published.  Whether a round is skipped, interior (straight-line
//                            max trees) or masked is decided once per round, warp-uniformly.  Each thread keeps a
//                            partial (g1, g2) for its row in every quarter; at unit end the quadrant's two warps
//                            merge them (exactly: max and min) and warp (q, c) tests the rows of quarters 2c and
//                            2c + 1.  (Eight warps, not sixteen: eleven warps leave 168 registers per thread for the
//                            128-column rounds, nineteen would leave 96.)
// Scores never leave the SM.
#pragma once
#include "fm_score.cuh"

namespace fm {

// One step is 256 columns (N = 256): TMEM's 512 columns hold two accumulator buffers, and each epilogue warp drains one
// 128-column round of every fill.  (N = 128 measured 1.3x slower: the row operand is re-read from shared memory for
// every 128 columns.)
constexpr int kRjCols = 256;
constexpr int kRjStepBytes = kRjCols * 128;  // one step of the column operand: two stored operand tiles
constexpr int kRjUnitRows = 512;             // rows per unit of this pass (the capture pass keeps kUnitRows = 256)
constexpr int kRjQuarters = kRjUnitRows / 128;
constexpr int kRjRowBufs = 2;                // row-operand buffers (4 tiles each): the next unit's tiles load under this one
constexpr int kRjStages = 2;                 // 64 KB of column-operand ring (a third stage does not fit)
constexpr int kRjSlots = 2;                  // units the scheduler warp may run ahead
constexpr int kRjEpiWarps = 8;
constexpr int kRjThreads = (3 + kRjEpiWarps) * 32;

struct RjUnit {
  const uint8_t* rowop;  // the unit's row-operand tiles (quarters 0 .. n_tiles - 1)
  const uint8_t* colop;
  uint32_t task, n_rows, row_off, s0;  // s0: sorted position of the unit's first row
  uint32_t n_tiles;                    // quarters with rows (1 .. 4): the row-operand tiles the unit loads
  uint32_t step0, n_steps;             // column steps [step0, step0 + n_steps) of kRjCols columns
  uint2 span[kRjQuarters];             // quarter q's bands lie in columns [span[q].x, span[q].y) (empty: y <= x)
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
  uint8_t a[kRjRowBufs][kRjQuarters][kOpTileBytes];  // [unit buffer][quarter]
  uint8_t b[kRjStages][kRjStepBytes];
  uint2 band[kRjSlots][kRjUnitRows];         // the unit's bands, (0, 0) for rows past the image
  float norm2[kRjSlots][kRjUnitRows];        // the rows' squared norms (rows with a band only)
  RjUnit unit[kRjSlots];
  uint64_t bar_afull[kRjRowBufs], bar_aempty[kRjRowBufs];
  uint64_t bar_bfull[kRjStages], bar_bempty[kRjStages];
  uint64_t bar_accfull[2], bar_accempty[2];  // [TMEM buffer]
  uint64_t bar_ufull[kRjSlots], bar_uempty[kRjSlots];
  float2 part[2][kRjUnitRows];               // [unit parity][row]: (g1, g2) of one column round, passed at unit end
  RjWarpRange wrange[kRjEpiWarps][kRjQuarters];  // [epilogue warp][quarter], warp-uniform (kept out of registers)
  uint32_t tmem_base;
};
constexpr size_t kRjSmemBytes = sizeof(RejectSmem) + 1024;
static_assert(kRjSmemBytes <= 227 * 1024, "reject pass: shared memory over the per-block limit");

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

// rj_unit_off[t] = first unit of task t (n_tasks + 1 entries), units of kRjUnitRows rows; units = rj_unit_off[n_tasks].
// scored_cols += (row, column) scores the tensor cores computed: 128 x N per MMA chain issued, band-edge and 16-column
// round-out columns included.  Writes rowstat[row] (1 = rejected) for every row of every fast task and appends the
// sorted position of each surviving row to its task's survivor list (surv_count / surv_rows, any order).
// kDump (test hook fm_debug_reject_rows): also writes dump[row] = (a1, a2, |a|^2, eps), the arguments the row's
// certified_reject receives, for every row with a non-empty band, and NaNs for every other row of a fast task.
template <bool kDump>
__global__ void __launch_bounds__(kRjThreads, 1)
reject_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks, const uint32_t* __restrict__ rj_unit_off,
              uint32_t n_tasks, uint32_t units, const uint2* __restrict__ bands, unsigned long long* __restrict__ scored_cols,
              float thr, float ratio, uint8_t* __restrict__ rowstat, uint32_t* __restrict__ surv_count,
              uint32_t* __restrict__ surv_rows, float4* __restrict__ dump) {
  extern __shared__ uint8_t smem_raw[];
  RejectSmem& sm = *reinterpret_cast<RejectSmem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 2 && lane == 0) {
    for (int i = 0; i < kRjRowBufs; i++) {
      ptx::mbar_init(&sm.bar_afull[i], 1);
      ptx::mbar_init(&sm.bar_aempty[i], 1);
    }
    for (int h = 0; h < 2; h++) {
      ptx::mbar_init(&sm.bar_accfull[h], 1);
      ptx::mbar_init(&sm.bar_accempty[h], kRjEpiWarps);  // every epilogue warp drains every fill
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
      const uint32_t t = find_segment_near(rj_unit_off, n_tasks, unit, units);
      const Task task = tasks[t];
      const ImageDev A = images[task.col_img];
      const ImageDev B = images[task.row_img];
      const uint32_t s0 = (unit - rj_unit_off[t]) * kRjUnitRows;
      const bool skip = (task.flags & kTaskExact) != 0;
      uint32_t cmin[kRjQuarters], cmax[kRjQuarters];  // per quarter
#pragma unroll
      for (int h = 0; h < kRjQuarters; h++) { cmin[h] = 0xFFFFFFFFu; cmax[h] = 0u; }
#pragma unroll
      for (int j = 0; j < kRjUnitRows / 32; j++) {
        const uint32_t r = j * 32 + lane, s = s0 + r;
        const int h = j / (128 / 32);
        uint2 bd = make_uint2(0u, 0u);
        if (!skip && s < B.n) bd = bands[task.row_off + s];
        if (bd.y > bd.x) { cmin[h] = min(cmin[h], bd.x); cmax[h] = max(cmax[h], bd.y); }
        sm.band[slot][r] = bd;
        if (bd.y > bd.x) sm.norm2[slot][r] = B.norm2_sorted[s];
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1)
#pragma unroll
        for (int h = 0; h < kRjQuarters; h++) {
          cmin[h] = min(cmin[h], __shfl_xor_sync(0xffffffffu, cmin[h], o));
          cmax[h] = max(cmax[h], __shfl_xor_sync(0xffffffffu, cmax[h], o));
        }
      if (lane == 0) {
        uint32_t umin = cmin[0], umax = cmax[0];
#pragma unroll
        for (int h = 1; h < kRjQuarters; h++) { umin = min(umin, cmin[h]); umax = max(umax, cmax[h]); }
        RjUnit u;
        u.rowop = reinterpret_cast<const uint8_t*>(B.rowop) + (size_t)s0 / 128 * kOpTileBytes;
        u.colop = reinterpret_cast<const uint8_t*>(A.colop);
        u.task = t;
        u.n_rows = B.n;
        u.row_off = task.row_off;
        u.s0 = s0;
        u.n_tiles = min((uint32_t)kRjQuarters, (B.n - min(B.n, s0) + 127) / 128);  // tiles past the image's rows are not read
        u.step0 = umax > umin ? umin / kRjCols : 0u;
        u.n_steps = umax > umin ? (umax + kRjCols - 1) / kRjCols - u.step0 : 0u;
#pragma unroll
        for (int h = 0; h < kRjQuarters; h++) u.span[h] = make_uint2(cmin[h], cmax[h]);
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
        const uint32_t step0 = us.step0, n_steps = us.n_steps, n_tiles = us.n_tiles;
        ptx::mbar_arrive(&sm.bar_uempty[slot]);
        if (n_steps == 0) continue;
        const uint32_t ab = a_use % kRjRowBufs;
        if (a_use >= (uint32_t)kRjRowBufs) ptx::mbar_wait(&sm.bar_aempty[ab], (a_use / kRjRowBufs - 1) & 1);
        a_use++;
        // only the tiles of quarters with rows: a quarter without rows has an empty span and issues no MMA
        ptx::mbar_expect_tx(&sm.bar_afull[ab], n_tiles * kOpTileBytes);
        for (uint32_t h = 0; h < n_tiles; h++)
          ptx::bulk_g2s(sm.a[ab][h], rowop + (size_t)h * kOpTileBytes, kOpTileBytes, &sm.bar_afull[ab]);
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
        uint2 span[kRjQuarters];
#pragma unroll
        for (int h = 0; h < kRjQuarters; h++) span[h] = us.span[h];
        ptx::mbar_arrive(&sm.bar_uempty[slot]);
        if (n_steps == 0) continue;
        const uint32_t ab = a_use % kRjRowBufs;
        ptx::mbar_wait(&sm.bar_afull[ab], (a_use / kRjRowBufs) & 1);
        a_use++;
        uint64_t adesc[kRjQuarters];
#pragma unroll
        for (int h = 0; h < kRjQuarters; h++) adesc[h] = ptx::umma_desc_sw128(ptx::smem_u32(sm.a[ab][h]));
        for (uint32_t i = 0; i < n_steps; i++, bq++, g++) {
          const uint32_t stg = bq % kRjStages, c0 = (step0 + i) * kRjCols;
          ptx::mbar_wait(&sm.bar_bfull[stg], (bq / kRjStages) & 1);
#pragma unroll
          for (int h = 0; h < kRjQuarters; h++) {
            // quarter h fills buffer h % 2; f counts that buffer's fills (two per step)
            const uint32_t buf = h & 1, f = 2 * g + h / 2;
            if (f > 0) ptx::mbar_wait(&sm.bar_accempty[buf], (f - 1) & 1);
            ptx::tc_fence_after();
            // Only the step's columns inside this quarter's span, in whole 16-column pieces (N = 16 .. 256; a B
            // operand starting 16 j rows into the step starts on a 1024 B swizzle atom).  The buffer's other columns
            // keep stale values: they lie outside every band of the quarter, so the epilogue masks or skips them.  A
            // quarter whose span misses the step (or that has no rows) is still handed to its epilogue warps, unscored.
            const uint32_t lo = max(span[h].x, c0), hi = min(span[h].y, c0 + kRjCols);
            if (hi > lo) {
              const uint32_t off = (lo - c0) & ~15u, n = ((hi - c0 + 15) & ~15u) - off;
              const uint32_t idesc = ptx::umma_idesc_f16_f32(128, (int)n);
              const uint64_t bdesc = ptx::umma_desc_sw128(ptx::smem_u32(sm.b[stg]) + off * 128);
#pragma unroll
              for (uint32_t kk = 0; kk < kKPad / 16; kk++)  // +32 B per K step inside the 128 B swizzle row
                if (kk < ksteps)
                  ptx::mma_f16_ss(tmem + buf * kRjCols + off, adesc[h] + 2 * kk, bdesc + 2 * kk, idesc, kk > 0);
              issued += 128 * n;
            }
            ptx::mma_commit(&sm.bar_accfull[buf]);
          }
          ptx::mma_commit(&sm.bar_bempty[stg]);  // after the fourth fill
        }
        ptx::mma_commit(&sm.bar_aempty[ab]);
      }
      if (scored_cols != nullptr) atomicAdd(scored_cols, issued);
    }
  } else {
    // ---- epilogue -----------------------------------------------------------------------------------------------
    // Warp (q, c): TMEM lane quadrant q = warp % 4 (the lanes the warp may access) and column round c: columns
    // [128 c, 128 c + 128) of every step, in every quarter's fill.  Per quarter h, thread `lane` keeps row
    // 128 h + 32 q + lane: its band and the (g1, g2) of the chunks in the warp's rounds.  At unit end the quadrant's two
    // warps exchange their partial pairs through shared memory, and warp (q, c) tests the rows of quarters 2c, 2c + 1.
    const uint32_t c = (warp - 3) >> 2, q = warp & 3;
    uint32_t taddr = tmem + ((q * 32) << 16) + c * 128;
    asm volatile("" : "+r"(taddr));
    // (unit blockIdx.x + k gridDim.x: the index is recomputed rather than carried, one register fewer across the step
    // loop, which needs every register it can get)
    for (uint32_t k = 0; blockIdx.x + k * gridDim.x < units; k++) {
      const uint32_t slot = k % kRjSlots;
      ptx::mbar_wait(&sm.bar_ufull[slot], (k / kRjSlots) & 1);
      // (the slot is released at unit end, after the rejection tail has read the rest of it)
      const RjUnit& us = sm.unit[slot];
      const uint32_t c_end = (us.step0 + us.n_steps) * kRjCols;
      const uint2* band = sm.band[slot] + q * 32 + lane;  // + 128 h: this thread's row of quarter h
      RjWarpRange* wr = sm.wrange[warp - 3];
#pragma unroll
      for (int h = 0; h < kRjQuarters; h++) {
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
      float g1[kRjQuarters], g2[kRjQuarters];
#pragma unroll
      for (int h = 0; h < kRjQuarters; h++) { g1[h] = -INFINITY; g2[h] = -INFINITY; }
      for (uint32_t c0 = us.step0 * kRjCols + c * 128; c0 < c_end; c0 += kRjCols) {
#pragma unroll
        for (int h = 0; h < kRjQuarters; h++) {  // in the order the MMA warp fills the buffers
          // each buffer takes two fills per step, so fill 2 g + h / 2 of buffer h % 2 completes phase parity h / 2
          const uint32_t buf = h & 1;
          ptx::mbar_wait(&sm.bar_accfull[buf], h / 2);
          ptx::tc_fence_after();
          const RjWarpRange w = wr[h];
          const bool need = c0 < w.cmax && c0 + 128 > w.cmin;        // warp-uniform
          const bool interior = c0 >= w.imin && c0 + 128 <= w.imax;  // warp-uniform: every row accepts the round
          uint32_t r0[32], r1[32], r2[32], r3[32];
          if (need) {
            const uint32_t t = taddr + buf * kRjCols;
            ptx::tmem_ld32(r0, t);
            ptx::tmem_ld32(r1, t + 32);
            ptx::tmem_ld32(r2, t + 64);
            ptx::tmem_ld32(r3, t + 96);
            ptx::tmem_ld_wait(r0, r1, r2, r3);
          }
          // every column this warp needs is in registers: hand the buffer back to the MMA warp before reducing
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive(&sm.bar_accempty[buf]);
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
      // the partner warp (q, 1 - c) has the other round of every step: pass it this warp's pairs for quarters
      // 2 (1 - c) and 2 (1 - c) + 1 and take its pairs for quarters 2c and 2c + 1 (double-buffered by unit, so a partner
      // already at the next unit end cannot overwrite a pair before it has been read)
      float2* part = sm.part[k & 1];
#pragma unroll
      for (int j = 0; j < 2; j++)
        part[(2 * (c ^ 1) + j) * 128 + q * 32 + lane] = c ? make_float2(g1[j], g2[j]) : make_float2(g1[2 + j], g2[2 + j]);
      ptx::named_bar_sync(1 + q, 64);
#pragma unroll
      for (int j = 0; j < 2; j++) {
        const uint32_t row = (2 * c + j) * 128 + q * 32 + lane, s = us.s0 + row;  // the row this thread tests
        const float2 o = part[row];
        float t1 = c ? g1[2 + j] : g1[j], t2 = c ? g2[2 + j] : g2[j];
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
