// fm_score.cuh -- the tensor-core scoring kernel (replaces norm() + the inner loop of
// ComputeMatches, match.cpp:243-251 and :267-317) and the band kernel that feeds it.
//
// One CTA scores a "unit": 256 consecutive (laplacian, scale)-sorted rows of image `second`
// against one contiguous range of 64-column tiles of image `first`.  Two CTAs share an SM
// (256 of the 512 TMEM columns and ~110 KB of shared memory each), so 16 epilogue warps hide each
// other's latencies and one CTA's prologue / tail overlaps the other's steady state.
//   warp 0      TMEM allocator, then TMA producer: cp.async.bulk 8 KB pre-swizzled FP16 tiles ->
//                             smem ring (mbarrier tx)
//   warp 1      MMA issuer  : tcgen05.mma kind::f16, M=128 N=64 K=16, 4 K-steps x 2 row halves per
//                             tile, FP32 accumulators double-buffered in TMEM (2 x 2 x 64 columns)
//   warps 2..9  epilogue    : tcgen05.ld (TMEM lane == row, so a row's scan over columns is
//                             thread-local), gate mask on band-edge tiles only, 3-input max tree
//                             per 16 columns, capture of the few columns above a running
//                             threshold into a per-row shared-memory list
// Scores never touch HBM: per row only <= 8 (t, column) candidates leave the SM.
// t = a.b - |b|^2/2 comes straight out of the MMA (K slots 48,49, see fm_prep.cuh), so
// larger t <=> smaller squared distance.
#pragma once
#include <cstddef>

#include "fm_common.cuh"
#include "fm_exact.cuh"
#include "fm_ptx.cuh"

namespace fm {

constexpr int kOpTileBytes = 16384;  // operand tile as stored: 128 keypoints x 64 halves, SWIZZLE_128B
constexpr int kTileCols = 64;        // columns per MMA tile: one half of a stored operand tile
constexpr int kTileBytes = kTileCols * 128;
constexpr int kUnitRows = 256;
constexpr int kStages = 4;
constexpr int kTopK = 8;        // candidate slots written per (row, column segment)
constexpr int kCapSlots = 22;  // capture list entries per row in shared memory
constexpr int kAccCols = 2 * 2 * kTileCols;  // TMEM columns: 2 stages x 2 row halves
constexpr int kEpiWarps = 8;
constexpr uint32_t kPreTiles = 8;  // look-ahead tiles per unit (score_kernel); FM_PRE overrides it for experiments
constexpr int kScoreThreads = (2 + kEpiWarps) * 32;  // warp 0: TMA + TMEM allocator, warp 1: MMA, warps 2..9: epilogue

struct Cand {
  float t;       // approximate score, -inf for an empty slot
  uint32_t col;  // sorted column position in image `first` (bit 31 of slot 0: list truncated)
};
constexpr uint32_t kCandTruncated = 0x80000000u;

struct alignas(1024) ScoreSmem {
  uint8_t a[2][kOpTileBytes];
  uint8_t b[kStages][kTileBytes];
  uint64_t bar_a;
  uint64_t bar_bfull[kStages];
  uint64_t bar_bempty[kStages];
  uint64_t bar_accfull[2][2];   // [stage][row half]: MMA -> the half's four epilogue warps
  uint64_t bar_accempty[2][2];  // [stage][row half]: those warps -> MMA (each row half has its own accumulators)
  uint32_t tmem_base;
  uint32_t cmin, cmax;
  uint32_t srow[kUnitRows];       // capture pass on survivors: sorted position of each unit row (0xFFFFFFFF: none)
  uint2 cap[kCapSlots][kUnitRows];  // [slot][row]: lanes of a warp hit distinct banks whatever their slot
};
constexpr size_t kScoreSmemBytes = sizeof(ScoreSmem) + 1024;

// ------------------------------------------------------------------------------------------------
// Band kernel: for every sorted row of image `second`, the interval [lo, hi) of sorted columns of
// image `first` that pass BOTH reference gates.  Within one laplacian class columns are sorted
// by scale and float division is monotone, so
//   lo = first column with !(s_row / s_col > 1.3f)      (match.cpp:273)
//   hi = first column with  (s_col / s_row > 1.3f)      (match.cpp:274)
// found by binary search with the reference's own float predicate.
__global__ void __launch_bounds__(128)
bands_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks,
             const uint32_t* __restrict__ task_blk_off, uint32_t n_tasks, uint2* __restrict__ bands) {
  const uint32_t t = find_segment_near(task_blk_off, n_tasks, blockIdx.x, gridDim.x);
  const Task task = tasks[t];
  if (task.flags & kTaskExact) return;
  const ImageDev A = images[task.col_img];
  const ImageDev B = images[task.row_img];
  const uint32_t s = (blockIdx.x - task_blk_off[t]) * 128 + threadIdx.x;
  if (s >= B.n) return;
  const ImageMeta* mb = B.meta;
  const ImageMeta* ma = A.meta;
  // class of this row in B, then the class with the same laplacian value in A
  uint32_t cb = 0;
  while (cb + 1 < mb->n_classes && mb->class_begin[cb + 1] <= s) cb++;
  const float lap = mb->class_lap[cb];
  uint32_t beg = 0, end = 0;  // the class with the same laplacian value in A (empty if there is none)
  for (uint32_t ca = 0; ca < ma->n_classes; ca++)
    if (ma->class_lap[ca] == lap) { beg = ma->class_begin[ca]; end = ma->class_begin[ca + 1]; break; }
  const float sr = B.scale_sorted[s];
  const float* __restrict__ sc = A.scale_sorted;
  // The reference's predicate is fdiv_rn(x, y) > 1.3f (match.cpp:273-274).  The IEEE division is a dozen instructions,
  // and 26 of them per row made this kernel instruction-bound; away from the boundary one multiplication decides:
  // x > 1.3001f y  =>  x / y > 1.30009  =>  the rounded quotient exceeds 1.3f;  x < 1.2999f y  =>  it does not.  (Scales
  // are finite and positive here: other images are flagged and take the exact kernel.)  Only quotients within 1e-4 of
  // 1.3 pay for the division.
  auto ratio_gt = [](float x, float y) {
    if (x > 1.3001f * y) return true;
    if (x < 1.2999f * y) return false;
    return __fdiv_rn(x, y) > 1.3f;
  };
  uint32_t l = beg, h = end;
  while (l < h) {  // first col with !(sr / sc > 1.3f)
    const uint32_t m = (l + h) >> 1;
    if (ratio_gt(sr, sc[m])) l = m + 1; else h = m;
  }
  uint32_t lo = l, hi;
  h = end;
  while (l < h) {  // first col >= lo with (sc / sr > 1.3f)
    const uint32_t m = (l + h) >> 1;
    if (ratio_gt(sc[m], sr)) h = m; else l = m + 1;
  }
  hi = l;
  if (hi < lo) hi = lo;
  bands[task.row_off + s] = make_uint2(lo, hi);
}

// ------------------------------------------------------------------------------------------------
// Two-phase scoring, between the passes: cut every task's survivor list (written by the reject pass) into units of
// 256 rows.  unit_off[t] = first survivor unit of task t (n_tasks + 1 entries), clamped to `cap_units` -- the grid the
// capture pass is launched with.  Survivors that do not fit (only when far more rows survive than two-phase scoring is
// meant for) are marked rejected for the rescoring kernel and queued for the exact row kernel instead.
struct RescoreCounters;
__global__ void __launch_bounds__(1024)
surv_plan_kernel(const uint32_t* __restrict__ surv_count, uint32_t n_tasks, uint32_t* __restrict__ unit_off,
                 uint32_t cap_units, const Task* __restrict__ tasks, const uint32_t* __restrict__ surv_rows,
                 uint8_t* __restrict__ rowstat, uint2* __restrict__ redo_list, unsigned long long* __restrict__ redo_rows) {
  __shared__ unsigned long long s_part[1024];
  const uint32_t per = (n_tasks + 1023u) / 1024u;
  const uint32_t t0 = min(n_tasks, threadIdx.x * per), t1 = min(n_tasks, t0 + per);
  unsigned long long sum = 0;
  for (uint32_t t = t0; t < t1; t++) sum += (surv_count[t] + kUnitRows - 1) / kUnitRows;
  s_part[threadIdx.x] = sum;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {  // inclusive scan of the 1024 partial sums
    const unsigned long long v = threadIdx.x >= (uint32_t)o ? s_part[threadIdx.x - o] : 0ull;
    __syncthreads();
    s_part[threadIdx.x] += v;
    __syncthreads();
  }
  unsigned long long run = s_part[threadIdx.x] - sum;
  for (uint32_t t = t0; t < t1; t++) {
    const uint32_t cnt = surv_count[t];
    const unsigned long long units = (cnt + kUnitRows - 1) / kUnitRows;
    unit_off[t] = (uint32_t)min(run, (unsigned long long)cap_units);
    if (run + units > cap_units) {
      const unsigned long long fit = run < cap_units ? (cap_units - run) * kUnitRows : 0ull;  // survivors that still get a unit
      const Task task = tasks[t];
      for (unsigned long long k = fit; k < cnt; k++) {
        const uint32_t s = surv_rows[task.row_off + k];
        rowstat[task.row_off + s] = 1;
        redo_list[atomicAdd(redo_rows, 1ull)] = make_uint2(t, s);
      }
    }
    run += units;
  }
  if (threadIdx.x == 1023) unit_off[n_tasks] = (uint32_t)min(s_part[1023], (unsigned long long)cap_units);
}

// ------------------------------------------------------------------------------------------------

__device__ __forceinline__ float max3(float a, float b, float c) { return fmaxf(fmaxf(a, b), c); }

// Certified bound on |t~ - t| (FP16-operand score vs exact a.b - |b|^2/2) for every pair of a task.
// With a16 = a + da, b16 = b + db the rounded operands (da, db = the ACTUAL rounding residuals,
// whose largest norms the prep kernel measured):
//   a16.b16 - a.b = a.db + da.b + da.db   =>   |.| <= |a||db| + |da||b| + |da||db|   (Cauchy-Schwarz)
// which is ~3x tighter than the format bound 2^-10 |a||b|.  The additive term covers the hi/lo
// split of -|b|^2/2 (2^-22 relative), FP32 accumulation inside the tensor core (<= 64 x 2^-23
// of the summed magnitudes), the FP32 evaluation of the norms (1% inflation below) and the
// reference's own FP32 rounding of d^2 (<= 48 x 2^-24 d^2).
__device__ __forceinline__ float task_eps(const ImageMeta* ma, const ImageMeta* mb) {
  const float na = sqrtf(ma->max_norm2), nb = sqrtf(mb->max_norm2);
  const float da = sqrtf(ma->max_delta2), db = sqrtf(mb->max_delta2);
  return 1.01f * (na * db + da * nb + da * db) + 3e-5f * fmaxf(1.f, fmaxf(ma->max_norm2, mb->max_norm2));
}

// Certified early rejection (used by the reject pass here and by rescore_kernel).  With na = |a|^2 of the row, a
// column's squared distance is na - 2t, and the reference's FP32 value of it lies within `margin` of na - 2t~ (2 eps
// for the score, the rest for the FP32 evaluation of na and of the distance).  For a1 = the row's best approximate
// score and a2 <= its second best:   d1_ref >= d1_lo = na - 2 a1 - margin,   d2_ref <= d2_hi = na - 2 a2 + margin.
//   * d1_lo > thr^2 (1 + 1e-5)            =>  sqrtf(d1) < thr is false                               (match.cpp:321)
//   * d1_lo > ratio^2 d2_hi (1 + 1e-4)    =>  sqrtf(d1 / d2) < ratio is false, and d2 != FLT_MAX because a second
//                                              gated-in column exists (a2 > -inf)                     (match.cpp:320)
// Either way the row emits nothing.  (ratio >= 1 can never trigger the second test: a1 >= a2.)
__device__ __forceinline__ bool certified_reject(float na, float a1, float a2, float eps, float thr, float ratio) {
  const float margin = 2.f * eps + 1e-5f * (na + 4.f);
  const float d1_lo = na - 2.f * a1 - margin;
  const float d2_hi = na - 2.f * a2 + margin;
  bool rejected = d1_lo > thr * thr * 1.00001f;
  if (a2 > -INFINITY && d2_hi > 0.f && ratio < 1.0e4f) rejected = rejected || d1_lo > ratio * ratio * d2_hi * 1.0001f;
  return rejected;
}

// Per-row scan state (registers of the row's epilogue thread).
//   g1 >= g2 : the two largest 16-column chunk maxima seen so far.  They belong to two distinct
//              columns, so g2 <= (row's second-best score) at any time, and
//   thr = g2 - 2 eps  is a capture threshold that never exceeds the final (2nd best - 2 eps):
//              every column that can be -- or tie with -- the exact nearest or second-nearest
//              neighbour scores above it (proof in fm_rescore.cuh).
// Keeping thr needs 4 branch-free ALU ops per 16 columns; only columns above thr (about
// 2 ln N per row) are appended to the row's shared-memory list.
struct RowScan {
  float g1, g2, thr;
  uint32_t cap;   // shared-space address of sm.cap[0][row]; slot k lives kCapStride bytes further per k
  uint32_t capw;  // address of the next free slot: cap + (live entries) * kCapStride
  uint32_t ovf;   // list could not hold every column above thr: row must be redone exactly
};
constexpr uint32_t kCapStride = kUnitRows * sizeof(uint2);

__device__ __forceinline__ void cap_store(uint32_t addr, float v, uint32_t col) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(addr), "r"(__float_as_uint(v)), "r"(col) : "memory");
}
__device__ __forceinline__ uint2 cap_load(uint32_t addr) {
  uint2 e;
  asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];" : "=r"(e.x), "=r"(e.y) : "r"(addr) : "memory");
  return e;
}

// Drop captured entries that the (risen) threshold has made irrelevant; returns the new count.
__device__ __noinline__ uint32_t cap_compress(uint32_t cap, uint32_t cnt, float thr) {
  uint32_t k = 0;
  for (uint32_t i = 0; i < cnt; i++) {
    const uint2 e = cap_load(cap + i * kCapStride);
    if (__uint_as_float(e.x) > thr) {
      cap_store(cap + k * kCapStride, __uint_as_float(e.x), e.y);
      k++;
    }
  }
  return k;
}

// Move the kTopK largest of cnt (> kTopK) entries to the front (selection sort in shared memory;
// only rows whose column segment is too short to establish a threshold get here).
__device__ __noinline__ void cap_select_top(uint32_t cap, uint32_t cnt) {
  for (uint32_t k = 0; k < (uint32_t)kTopK; k++) {
    uint32_t best = k;
    uint2 eb = cap_load(cap + k * kCapStride);
    const uint2 ek = eb;
    for (uint32_t i = k + 1; i < cnt; i++) {
      const uint2 e = cap_load(cap + i * kCapStride);
      if (__uint_as_float(e.x) > __uint_as_float(eb.x)) { eb = e; best = i; }
    }
    if (best != k) {
      cap_store(cap + best * kCapStride, __uint_as_float(ek.x), ek.y);
      cap_store(cap + k * kCapStride, __uint_as_float(eb.x), eb.y);
    }
  }
}

// Predicated append (no branch): if v > thr, store (v, col) at capw (unless the list is full:
// capw >= cap_end) and advance capw.  A pointer past cap_end afterwards means "overflowed".
__device__ __forceinline__ void cap_append_if_above(uint32_t& capw, uint32_t cap_end, float v, float thr, uint32_t col) {
  asm volatile(
      "{\n\t.reg .pred q, s;\n\t"
      "setp.gt.f32 q, %1, %2;\n\t"
      "setp.lt.and.u32 s, %0, %6, q;\n\t"
      "@s st.shared.v2.b32 [%0], {%3, %4};\n\t"
      "@q add.u32 %0, %0, %5;\n\t}"
      : "+r"(capw)
      : "f"(v), "f"(thr), "r"(__float_as_uint(v)), "r"(col), "n"(kCapStride), "r"(cap_end)
      : "memory");
}

// Make room in a row's capture list: drop the entries the risen threshold has retired.  Returns
// the new write address; bit 0 set = more than half of the list is still live, i.e. the row must
// be redone by the exact kernel (the list restarts empty).
__device__ __noinline__ uint32_t cap_make_room(uint32_t cap, uint32_t capw, float thr) {
  const uint32_t cnt = cap_compress(cap, min((capw - cap) / kCapStride, (uint32_t)kCapSlots), thr);
  if (cnt > (uint32_t)(kCapSlots / 2)) return cap | 1u;
  return cap + cnt * kCapStride;
}

// Max tree of 16 consecutive columns of one row: five 3-column nodes + the 16th column, two
// group maxima (columns 0..8 and 9..15) and the chunk maximum.
struct ChunkMax {
  float m0, m1, m2, m3, m4, ga, gb, m;
};

// kMasked: columns outside [lo, lo + width) are gated out (band-edge tiles only).
template <bool kMasked>
__device__ __forceinline__ ChunkMax chunk_max(const uint32_t (&r)[16], uint32_t col0, uint32_t lo, uint32_t width,
                                              float (&f)[16]) {
#pragma unroll
  for (int e = 0; e < 16; e++) {
    f[e] = __uint_as_float(r[e]);
    if (kMasked) f[e] = ((col0 + e) - lo < width) ? f[e] : -INFINITY;
  }
  ChunkMax c;
  c.m0 = max3(f[0], f[1], f[2]);
  c.m1 = max3(f[3], f[4], f[5]);
  c.m2 = max3(f[6], f[7], f[8]);
  c.m3 = max3(f[9], f[10], f[11]);
  c.m4 = max3(f[12], f[13], f[14]);
  c.ga = max3(c.m0, c.m1, c.m2);
  c.gb = max3(c.m3, c.m4, f[15]);
  c.m = fmaxf(c.ga, c.gb);
  return c;
}

// Second largest of {h} U nodes of c, folded into (h, sec): h = running maximum.
__device__ __forceinline__ void fold_second(const ChunkMax& c, float f15, float& h, float& sec) {
  sec = fmaxf(sec, fminf(h, c.m0)); h = fmaxf(h, c.m0);
  sec = fmaxf(sec, fminf(h, c.m1)); h = fmaxf(h, c.m1);
  sec = fmaxf(sec, fminf(h, c.m2)); h = fmaxf(h, c.m2);
  sec = fmaxf(sec, fminf(h, c.m3)); h = fmaxf(h, c.m3);
  sec = fmaxf(sec, fminf(h, c.m4)); h = fmaxf(h, c.m4);
  sec = fmaxf(sec, fminf(h, f15));  h = fmaxf(h, f15);
}

// 32 consecutive columns (two TMEM loads) of one row.
// Fast path (every pair, branch-free): two 3-input max trees, the two largest chunk maxima seen so
// far, the capture threshold, one compare, one warp vote.  The slow path is entered by the WARP
// when any of its 32 rows has a column above its threshold.  It walks the max tree top-down with
// warp votes -- four 8-column groups, then the 3-column nodes of a group some row hit -- so every
// branch is warp-uniform, and the per-row captures are predicated stores: lanes never diverge
// and a typical entry (one row, one column) costs ~45 instructions.
//
// upd / cap (warp-uniform): the first tiles of a unit are visited twice (see score_kernel) -- a look-ahead visit
// that only tracks the two largest chunk maxima (upd, !cap) and a capture visit against the threshold the
// look-ahead established (!upd, cap: the chunk maxima must not be folded in a second time, g2 has to stay the
// score of a column distinct from g1's).  Every other tile is visited once with both set.
template <bool kMasked, int kProbe, int kVar>
__device__ __forceinline__ void score_pair(const uint32_t (&ra)[16], const uint32_t (&rb)[16], uint32_t col0, uint32_t lo,
                                           uint32_t width, RowScan& st, float two_eps, bool upd, bool cap) {
  constexpr uint32_t kAll = 0xffffffffu;
  // An entry may append up to kEntryRoom columns per row without further checks; beyond that the
  // predicated store is suppressed and the row is marked for the exact kernel.
  constexpr uint32_t kEntryRoom = 8;
  constexpr uint32_t kFullAt = (uint32_t)(kCapSlots - kEntryRoom) * kCapStride;
  float fa[16], fb[16];
  const ChunkMax a = chunk_max<kMasked>(ra, col0, lo, width, fa);
  const ChunkMax b = chunk_max<kMasked>(rb, col0 + 16, lo, width, fb);
  const float hi = fmaxf(a.m, b.m), lw = fminf(a.m, b.m);
  // top two of {g1, g2, hi, lw} (g1 >= g2, hi >= lw)
  const float hi_u = upd ? hi : -INFINITY, lw_u = upd ? lw : -INFINITY;
  const float g2n = max3(st.g2, lw_u, fminf(st.g1, hi_u));
  st.g1 = fmaxf(st.g1, hi_u);
  st.g2 = g2n;
  if (kProbe != 1) st.thr = st.g2 - two_eps;
  float th = st.thr;
  const bool hit = cap && hi > th;
  if (__any_sync(kAll, hit)) {
    // Two rare situations share one vote: a row without a threshold yet, a row whose list is nearly full.
    if (__any_sync(kAll, hit && (st.g2 == -INFINITY || st.capw - st.cap > kFullAt))) {
      if (kProbe != 1 && __any_sync(kAll, hit && st.g2 == -INFINITY)) {
        // First scored columns of a row: seed the threshold with the second largest of the twelve
        // node maxima (disjoint column sets, so it cannot exceed the row's second-best score)
        // instead of capturing every column against thr = -inf.
        float h = -INFINITY, sec = -INFINITY;
        fold_second(a, fa[15], h, sec);
        fold_second(b, fb[15], h, sec);
        const bool seed = st.g2 == -INFINITY;
        st.g2 = seed ? sec : st.g2;
        st.thr = th = seed ? sec - two_eps : th;
      }
      // room for kEntryRoom appends, once per entry
      if (hi > th && st.capw - st.cap > kFullAt) {
        const uint32_t w = cap_make_room(st.cap, st.capw, th);
        st.ovf |= w & 1u;
        st.capw = w & ~1u;
      }
    }
    const uint32_t cap_end = st.cap + (uint32_t)kCapSlots * kCapStride;
    const bool va = __any_sync(kAll, a.ga > th), vb = __any_sync(kAll, a.gb > th);
    const bool vc = __any_sync(kAll, b.ga > th), vd = __any_sync(kAll, b.gb > th);
#define FM_TRY(f, base, e) cap_append_if_above(st.capw, cap_end, f[e], th, col0 + (base) + (e))
#define FM_NODE(v, f, base, e0, e1, e2) \
    if (v) { FM_TRY(f, base, e0); FM_TRY(f, base, e1); FM_TRY(f, base, e2); }
    // the node votes of a group are taken together, before any of its branches: one vote latency per group
    if (va) {
      const bool n0 = __any_sync(kAll, a.m0 > th), n1 = __any_sync(kAll, a.m1 > th), n2 = __any_sync(kAll, a.m2 > th);
      FM_NODE(n0, fa, 0, 0, 1, 2)
      FM_NODE(n1, fa, 0, 3, 4, 5)
      FM_NODE(n2, fa, 0, 6, 7, 8)
    }
    if (vb) {
      const bool n0 = __any_sync(kAll, a.m3 > th), n1 = __any_sync(kAll, a.m4 > th);
      FM_NODE(n0, fa, 0, 9, 10, 11)
      FM_NODE(n1, fa, 0, 12, 13, 14)
      FM_TRY(fa, 0, 15);
    }
    if (vc) {
      const bool n0 = __any_sync(kAll, b.m0 > th), n1 = __any_sync(kAll, b.m1 > th), n2 = __any_sync(kAll, b.m2 > th);
      FM_NODE(n0, fb, 16, 0, 1, 2)
      FM_NODE(n1, fb, 16, 3, 4, 5)
      FM_NODE(n2, fb, 16, 6, 7, 8)
    }
    if (vd) {
      const bool n0 = __any_sync(kAll, b.m3 > th), n1 = __any_sync(kAll, b.m4 > th);
      FM_NODE(n0, fb, 16, 9, 10, 11)
      FM_NODE(n1, fb, 16, 12, 13, 14)
      FM_TRY(fb, 16, 15);
    }
#undef FM_NODE
#undef FM_TRY
    // a row that wanted more than the list holds: its write pointer ran past the end
    st.ovf |= st.capw > cap_end ? 1u : 0u;
  }
}

// One 64-column accumulator tile of one row: two pairs of TMEM loads.
template <bool kMasked, bool kDump, int kProbe, int kVar>
__device__ __forceinline__ void score_tile(uint32_t taddr, uint32_t cb, uint32_t lo, uint32_t width, RowScan& st,
                                           float two_eps, uint32_t bar_release, float* dump_row, bool upd, bool cap) {
  uint32_t ra[16], rb[16];
  // Rolled on purpose: one copy of the capture code stays resident in the instruction cache.
#pragma unroll 1
  for (int c = 0; c < kTileCols / 16; c += 2) {
    ptx::tmem_ld16(ra, taddr + c * 16);
    ptx::tmem_ld16(rb, taddr + (c + 1) * 16);
    ptx::tmem_ld_wait(ra);
    ptx::tmem_ld_wait(rb);
    if (c + 2 >= kTileCols / 16) {
      // every column of this accumulator is now in registers: hand it back to the MMA warp
      ptx::tc_fence_before();
      __syncwarp();
      if ((threadIdx.x & 31) == 0) ptx::mbar_arrive_u32(bar_release);
    }
    if (kDump) {
#pragma unroll
      for (int e = 0; e < 16; e++) {
        dump_row[cb + c * 16 + e] = __uint_as_float(ra[e]);
        dump_row[cb + (c + 1) * 16 + e] = __uint_as_float(rb[e]);
      }
    }
    score_pair<kMasked, kProbe, kVar>(ra, rb, cb + c * 16, lo, width, st, two_eps, upd, cap);
  }
}

// unit_off: exclusive prefix of units per task (n_tasks + 1 entries).  A task with n rows has
// ceil(n / 256) * segs units; unit = row_block * segs + seg.
// cands: [batch rows][segs][kTopK]: the columns above the row's final threshold (-inf padded).
//        If more than kTopK qualify, the kTopK best are kept and bit 31 of slot 0's column is set
//        ("truncated": every dropped column scores <= the smallest kept one).  Slot 0 =
//        (+inf, kNone) marks a list that overflowed during the scan.
// dump (kDump only): [256][dump_ld] raw t of the unit.
// kProbe (performance attribution only, results are garbage): 1 = capture threshold pinned at +inf,
// i.e. the max-tree fast path alone; 2 = epilogue skips the TMEM loads too (TMA + MMA pipeline alone).
// kVar = mode of the TWO-PHASE path (fm_fast.cuh decides when to use it; 0 = the ordinary single pass).  Its first
// pass, the reject pass, is reject_kernel (fm_reject.cuh): it writes rowstat and the survivor lists.
//   2  capture pass on the survivors: surv_plan_kernel cuts every task's survivor list into units of 256 rows and
//      `unit_off` is the prefix of THOSE units; a unit's row operand tiles are gathered row by row from the image's
//      operand tiles (generic-proxy stores into the swizzled shared-memory image, then a proxy fence), everything
//      else -- bands, MMAs, capture epilogue, candidate lists written at the rows' own positions -- is the ordinary pass.
// With -d2 < 1 on images that have little in common nearly every row is rejected (random descriptors at -d2 0.8:
// 99.9 %): the capture pass then works on ~20 rows per 20 000-row task.
// Experiments tried and
// dropped in round 2, all measured on C2 (profiles/r2_summary.md): nanosleep back-off in the two single-thread warps
// (no change: their polling does not take issue slots the epilogue needs), testing against the previous step's
// threshold to shorten the compare -> vote chain (-1 %), and loading the second half of a tile under the processing
// of the first (needs ~130 registers per epilogue thread; 104 is the most setmaxnreg can hand out at two CTAs per SM).
template <bool kDump, int kProbe = 0, int kVar = 0>
__global__ void __launch_bounds__(kScoreThreads, 2)
score_kernel(const ImageDev* __restrict__ images, const Task* __restrict__ tasks,
             const uint32_t* __restrict__ unit_off, uint32_t n_tasks, uint32_t segs,
             const uint2* __restrict__ bands, Cand* __restrict__ cands, unsigned long long* __restrict__ scored_cols,
             float* __restrict__ dump, uint32_t dump_ld, uint32_t unit_base, uint32_t pre_tiles,
             float thr, float ratio, uint8_t* __restrict__ rowstat, uint32_t* __restrict__ surv_count,
             uint32_t* __restrict__ surv_rows) {
  extern __shared__ uint8_t smem_raw[];
  ScoreSmem& sm = *reinterpret_cast<ScoreSmem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);

  const uint32_t unit = blockIdx.x + unit_base;  // unit_base != 0 only for single-unit debug launches
  if (kVar == 2 && unit >= unit_off[n_tasks]) return;  // the grid is an upper bound on the survivor units
  const uint32_t t = find_segment_near(unit_off, n_tasks, unit, (kDump || kVar == 2) ? unit_off[n_tasks] : gridDim.x);
  const Task task = tasks[t];
  if (task.flags & kTaskExact) return;
  const ImageDev A = images[task.col_img];
  const ImageDev B = images[task.row_img];
  const uint32_t local = unit - unit_off[t];
  const uint32_t rb = local / segs, seg = local - rb * segs;

  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const bool is_epi = warp >= 2;
  // epilogue thread -> row: TMEM sub-partition = warp % 4 (hardware rule), accumulator half = (warp - 2) / 4
  const uint32_t half = is_epi ? (warp - 2) >> 2 : 0;
  const uint32_t row_in_unit = half * 128 + (warp & 3) * 32 + lane;
  uint32_t s = rb * kUnitRows + row_in_unit;
  if (kVar == 2) {
    // survivor unit: row k of the task's survivor list (any order), or no row at all
    const uint32_t k = rb * kUnitRows + row_in_unit;
    s = (is_epi && k < min(surv_count[t], B.n)) ? surv_rows[task.row_off + k] : 0xFFFFFFFFu;
    if (is_epi) sm.srow[row_in_unit] = s;
  }
  uint32_t lo = 0, hi = 0;
  if (is_epi && s < B.n) {
    uint2 bd = bands[task.row_off + s];
    lo = bd.x;
    hi = bd.y;
  }
  // warp-level and CTA-level column ranges
  uint32_t w_cmin = (hi > lo) ? lo : 0xFFFFFFFFu, w_cmax = (hi > lo) ? hi : 0u;
  uint32_t w_imin = lo, w_imax = hi;  // interior: columns every row of the warp accepts
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    w_cmin = min(w_cmin, __shfl_xor_sync(0xffffffffu, w_cmin, o));
    w_cmax = max(w_cmax, __shfl_xor_sync(0xffffffffu, w_cmax, o));
    w_imin = max(w_imin, __shfl_xor_sync(0xffffffffu, w_imin, o));
    w_imax = min(w_imax, __shfl_xor_sync(0xffffffffu, w_imax, o));
  }
  if (threadIdx.x == 0) { sm.cmin = 0xFFFFFFFFu; sm.cmax = 0u; }
  __syncthreads();
  if (is_epi && lane == 0 && w_cmax > w_cmin) { atomicMin(&sm.cmin, w_cmin); atomicMax(&sm.cmax, w_cmax); }
  __syncthreads();
  const uint32_t cmin = sm.cmin, cmax = sm.cmax;
  uint32_t tile0 = 0, n_tiles = 0;
  if (cmax > cmin) {
    const uint32_t tb = cmin / kTileCols, te = (cmax + kTileCols - 1) / kTileCols;
    const uint32_t nt = te - tb;
    tile0 = tb + (uint32_t)(((uint64_t)nt * seg) / segs);
    n_tiles = tb + (uint32_t)(((uint64_t)nt * (seg + 1)) / segs) - tile0;
  }
  // Look-ahead: the first n_pre tiles are scored twice.  A streaming top-2 scan captures ~2 ln(columns) columns per
  // row, most of them early, while the running threshold is still far below its final value -- and a capture by
  // ONE row costs its whole warp the slow path.  Visiting the first tiles once without capturing establishes
  // the threshold of a 64 * n_pre column prefix before the first column is captured: a few tiles of extra
  // MMA work (the tensor pipe has slack) for about a third fewer slow-path entries and no list overflow handling.
  const uint32_t n_pre = min(pre_tiles, n_tiles / 4);  // (the single-unit debug launch passes pre_tiles = 0)
  const uint32_t n_sched = n_tiles + n_pre;

  RowScan st;
  st.g1 = st.g2 = -INFINITY;
  st.thr = kProbe == 1 ? INFINITY : -INFINITY;
  st.ovf = 0;
  st.cap = ptx::smem_u32(&sm.cap[0][is_epi ? row_in_unit : 0]);
  asm volatile("" : "+r"(st.cap));  // opaque: keep the list base in a register, do not rebuild it from the thread id
  st.capw = st.cap;

  if (n_tiles > 0) {  // CTA-uniform
    if (warp == 1 && lane == 0) {
      ptx::mbar_init(&sm.bar_a, 1);
      for (int i = 0; i < kStages; i++) { ptx::mbar_init(&sm.bar_bfull[i], 1); ptx::mbar_init(&sm.bar_bempty[i], 1); }
      for (int i = 0; i < 2; i++)
        for (int h = 0; h < 2; h++) { ptx::mbar_init(&sm.bar_accfull[i][h], 1); ptx::mbar_init(&sm.bar_accempty[i][h], kEpiWarps / 2); }
      ptx::fence_mbar_init();
    }
    if (warp == 0) ptx::tmem_alloc<kAccCols>(&sm.tmem_base);
    if (kVar == 2) {
      // Gather the unit's two row-operand tiles: 16-byte chunk q of unit row r comes from chunk q of sorted row
      // srow[r] in the image's pre-swizzled tiles and lands where SWIZZLE_128B wants it; rows without a survivor are
      // zero.  (sm.srow was written before the two barriers of the column-range exchange above.)
      const uint8_t* rowop_img = reinterpret_cast<const uint8_t*>(B.rowop);
      for (uint32_t idx = threadIdx.x; idx < (uint32_t)kUnitRows * 8u; idx += kScoreThreads) {
        const uint32_t r = idx >> 3, q = idx & 7u;
        const uint32_t sr = sm.srow[r];
        uint4 v = make_uint4(0u, 0u, 0u, 0u);
        if (sr != 0xFFFFFFFFu) v = __ldg(reinterpret_cast<const uint4*>(rowop_img + (size_t)(sr >> 7) * kOpTileBytes + sw128_offset(sr & 127u, q)));
        *reinterpret_cast<uint4*>(sm.a[r >> 7] + sw128_offset(r & 127u, q)) = v;
      }
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to tcgen05.mma
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem = sm.tmem_base;

    if (warp == 0) {
      if (lane == 0) {
        // ---- TMA producer ------------------------------------------------------------------
        if (kVar != 2) {
          const uint8_t* rowop = reinterpret_cast<const uint8_t*>(B.rowop) + (size_t)rb * 2 * kOpTileBytes;
          ptx::mbar_expect_tx(&sm.bar_a, 2 * kOpTileBytes);
          ptx::bulk_g2s(sm.a[0], rowop, kOpTileBytes, &sm.bar_a);
          ptx::bulk_g2s(sm.a[1], rowop + kOpTileBytes, kOpTileBytes, &sm.bar_a);
        }
        const uint8_t* colop = reinterpret_cast<const uint8_t*>(A.colop);
        for (uint32_t i = 0; i < n_sched; i++) {
          const uint32_t stg = i % kStages, use = i / kStages;
          const uint32_t tile = tile0 + (i < n_pre ? i : i - n_pre);
          if (use > 0) ptx::mbar_wait(&sm.bar_bempty[stg], (use - 1) & 1);
          ptx::mbar_expect_tx(&sm.bar_bfull[stg], kTileBytes);
          ptx::bulk_g2s(sm.b[stg], colop + (size_t)tile * kTileBytes, kTileBytes, &sm.bar_bfull[stg]);
        }
      }
    } else if (warp == 1) {
      if (lane == 0) {
        // ---- MMA issuer ----------------------------------------------------------------------
        constexpr uint32_t idesc = ptx::umma_idesc_f16_f32(128, kTileCols);
        const uint64_t adesc0 = ptx::umma_desc_sw128(ptx::smem_u32(sm.a[0]));
        const uint64_t adesc1 = ptx::umma_desc_sw128(ptx::smem_u32(sm.a[1]));
        if (kVar != 2) ptx::mbar_wait(&sm.bar_a, 0);  // (survivor units: the gathered tiles are in place since the barrier above)
        for (uint32_t i = 0; i < n_sched; i++) {
          const uint32_t stg = i % kStages, acc = i & 1, use = i >> 1;
          if (use > 0) ptx::mbar_wait(&sm.bar_accempty[acc][0], (use - 1) & 1);
          ptx::mbar_wait(&sm.bar_bfull[stg], (i / kStages) & 1);
          ptx::tc_fence_after();
          const uint64_t bdesc = ptx::umma_desc_sw128(ptx::smem_u32(sm.b[stg]));
#pragma unroll
          for (int k = 0; k < kKPad / 16; k++)  // +32 B per K step inside the 128 B swizzle row
            ptx::mma_f16_ss(tmem + acc * (2 * kTileCols), adesc0 + 2 * k, bdesc + 2 * k, idesc, k > 0);
          ptx::mma_commit(&sm.bar_accfull[acc][0]);
          if (use > 0) {
            ptx::mbar_wait(&sm.bar_accempty[acc][1], (use - 1) & 1);
            ptx::tc_fence_after();
          }
#pragma unroll
          for (int k = 0; k < kKPad / 16; k++)
            ptx::mma_f16_ss(tmem + acc * (2 * kTileCols) + kTileCols, adesc1 + 2 * k, bdesc + 2 * k, idesc, k > 0);
          ptx::mma_commit(&sm.bar_bempty[stg]);
          ptx::mma_commit(&sm.bar_accfull[acc][1]);
        }
      }
    } else if (is_epi) {
      // ---- epilogue ------------------------------------------------------------------------------
      const uint32_t width = hi - lo;
      const float two_eps = 2.f * task_eps(A.meta, B.meta);
      float* dump_row = kDump ? dump + (size_t)row_in_unit * dump_ld : nullptr;
      unsigned long long scored = 0;
      // this thread's TMEM window: lane = its row, first column of its row half.  Kept opaque so
      // the compiler holds it in a register instead of rebuilding it from the thread id per chunk.
      uint32_t tmem_lane = tmem + (((warp & 3) * 32) << 16) + half * kTileCols;
      asm volatile("" : "+r"(tmem_lane));
      // shared-space address of this row half's accfull[0] barrier; accfull[1] is 16 B further,
      // the matching accempty barriers 32 B further (layout of ScoreSmem)
      uint32_t bar_full = ptx::smem_u32(&sm.bar_accfull[0][half]);
      asm volatile("" : "+r"(bar_full));
      static_assert(offsetof(ScoreSmem, bar_accempty) - offsetof(ScoreSmem, bar_accfull) == 32, "barrier layout");
      for (uint32_t i = 0; i < n_sched; i++) {
        const uint32_t acc = i & 1;
        const uint32_t cb = (tile0 + (i < n_pre ? i : i - n_pre)) * kTileCols;
        const bool cap = i >= n_pre, upd = i < n_pre || i >= 2 * n_pre;  // look-ahead visit, capture visit, both
        ptx::mbar_wait_u32(bar_full + acc * 16, (i >> 1) & 1);
        ptx::tc_fence_after();
        const uint32_t taddr = tmem_lane + acc * (2 * kTileCols);
        const bool needed = kProbe != 2 && (kDump || (cb < w_cmax && cb + kTileCols > w_cmin));  // warp-uniform
        if (!needed) {
          ptx::tc_fence_before();
          __syncwarp();
          if (lane == 0) ptx::mbar_arrive_u32(bar_full + 32 + acc * 16);
        } else if (!kDump && cb >= w_imin && cb + kTileCols <= w_imax) {
          score_tile<false, kDump, kProbe, kVar>(taddr, cb, lo, width, st, two_eps, bar_full + 32 + acc * 16, dump_row, upd, cap);
          scored += kTileCols;
        } else {
          score_tile<true, kDump, kProbe, kVar>(taddr, cb, lo, width, st, two_eps, bar_full + 32 + acc * 16, dump_row, upd, cap);
          scored += kTileCols;
        }
      }
      if (scored_cols != nullptr) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) scored += __shfl_xor_sync(0xffffffffu, scored, o);
        if (lane == 0) atomicAdd(scored_cols, scored);
      }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 0) {
      ptx::tc_fence_after();
      ptx::tmem_dealloc<kAccCols>(tmem);
    }
  }

  if (is_epi && s < B.n) {
    // Final list: the entries above the final threshold.
    uint32_t cnt = st.ovf ? 0u : cap_compress(st.cap, min((st.capw - st.cap) / kCapStride, (uint32_t)kCapSlots), st.thr);
    uint32_t trunc = 0;
    if (cnt > (uint32_t)kTopK) {
      cap_select_top(st.cap, cnt);
      cnt = kTopK;
      trunc = kCandTruncated;
    }
    Cand* out = cands + ((size_t)(task.row_off + s) * segs + seg) * kTopK;
#pragma unroll
    for (int k = 0; k < kTopK; k++) {
      Cand cd{-INFINITY, 0u};
      if (st.ovf) {
        if (k == 0) cd = Cand{INFINITY, kNone};
      } else if ((uint32_t)k < cnt) {
        const uint2 e = cap_load(st.cap + k * kCapStride);
        cd = Cand{__uint_as_float(e.x), e.y | (k == 0 ? trunc : 0u)};
      }
      out[k] = cd;
    }
  }
}

}  // namespace fm
