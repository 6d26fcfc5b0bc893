// fm_compact.cuh -- stable stream compaction of accepted matches (replaces push_back, match.cpp:323-327).
//
// Input : rowres[row] = matched column id or kNone, rows laid out task after task.
// Output: per task a dense list of (first, second) uint32 pairs ordered by row -- exactly the
//         order ComputeMatches appends them in -- written at the running output offset so that
//         consecutive tasks (and the two directions of a -sym pair) are contiguous.
//
// HBM-bound by nature: 4 B read per row, 8 B written per match (+ 4 B per match with distances).
// The rows of a batch are cut into chunks of <= 4096 rows of one task, described by a host-built 16-byte record each
// (no per-chunk searches or dependent loads on the device).  Three launches without any inter-CTA wait:
//   count    one CTA per chunk: fully coalesced 4-byte loads (sixteen in flight per thread), warp ballots, the chunk's
//            total -- and, when the chunk holds few matches (<= 64: the usual case when most rows are rejected), the
//            compacted pairs themselves, parked in a small per-chunk staging slot;
//   scan     one CTA: exclusive prefix of the chunk totals, per-pair counts, the running total;
//   scatter  one CTA per chunk: a parked chunk only moves its few pairs to their final place (the rows are not read
//            again); a dense chunk re-reads its rows (still L2-resident), ranks them, stages the pairs in shared
//            memory in output order and writes them with 16-byte stores.
// Batches of at most kOnePassChunks chunks take the single-launch kernel at the end of this file instead.
#pragma once
#include "fm_common.cuh"

namespace fm {

constexpr int kCompactThreads = 256;
constexpr int kCompactPer = 16;                                 // rows per thread
constexpr int kCompactChunk = kCompactThreads * kCompactPer;    // rows per chunk
constexpr int kCompactSlices = kCompactPer * (kCompactThreads / 32);  // (iteration, warp) slices of 32 rows

// One chunk: rows [row_abs, row_abs + n) of the batch's rowres array = rows row_local.. of their task.
struct ChunkDesc {
  uint32_t row_abs;
  uint32_t n_swap;     // [30:0] rows in the chunk, [31] the task is a -sym reverse pass: emit (row, match)
  uint32_t row_local;  // index, inside its task, of the chunk's first row
  uint32_t pair;       // caller's pair index the task belongs to
};

// Status word of a chunk: [63:34] launch epoch, [33:32] state, [31:0] value.
constexpr unsigned long long kChunkAggregate = 1ull;  // value = the chunk's own total
constexpr unsigned long long kChunkPrefix = 2ull;     // value = inclusive prefix up to and including the chunk
__device__ __forceinline__ unsigned long long chunk_word(uint32_t epoch, unsigned long long state, uint32_t value) {
  return ((unsigned long long)epoch << 34) | (state << 32) | value;
}

constexpr uint32_t kOnePassChunks = 1536;  // batches up to this many chunks: one launch (compact_onepass_kernel)
constexpr uint32_t kStageCap = 64;  // matches a chunk may park in its staging slot during the count pass

struct CompactArgs {
  const ChunkDesc* chunks;
  uint32_t n_chunks;
  const uint32_t* rowres;
  const float* rowdist;           // kDist only: squared distance of the row's match
  uint32_t* chunk_count;          // n_chunks
  unsigned long long* chunk_out;  // n_chunks: index of the chunk's first output pair
  uint2* stage;                   // n_chunks x kStageCap parked pairs
  uint32_t* pair_count;           // per caller pair: += matches
  unsigned long long* running_total;  // matches written before this batch; += this batch's
  uint2* out_pairs;
  float* out_dist;                // kDist only
  unsigned long long* status;     // one-pass kernel: n_chunks look-back words (epoch-tagged; cleared when the epoch wraps)
  uint32_t epoch;                 // one-pass kernel: 30 bits, different from the previous launches that used `status`
};

// Loads, ranks and slice offsets of one chunk (shared by the count and the scatter pass).  Returns the chunk total;
// afterwards s_slice holds the exclusive prefix of the (iteration, warp) slices and rank[i] the rank inside a slice.
__device__ __forceinline__ uint32_t chunk_rank(const ChunkDesc& d, const uint32_t* __restrict__ rowres, uint32_t (&m)[kCompactPer],
                                               uint32_t (&rank)[kCompactPer], uint32_t* s_slice, uint32_t* s_total) {
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t n = d.n_swap & 0x7FFFFFFFu;
  const uint32_t* src = rowres + d.row_abs;
#pragma unroll
  for (int i = 0; i < kCompactPer; i++) {
    const uint32_t r = i * kCompactThreads + tid;
    m[i] = r < n ? __ldg(src + r) : kNone;
  }
#pragma unroll
  for (int i = 0; i < kCompactPer; i++) {
    const uint32_t b = __ballot_sync(0xffffffffu, m[i] != kNone);
    rank[i] = __popc(b & ((1u << lane) - 1u));
    if (lane == 0) s_slice[i * (kCompactThreads / 32) + warp] = __popc(b);
  }
  __syncthreads();
  if (warp == 0) {  // exclusive scan of the slice totals (row order = slice order)
    uint32_t carry = 0;
#pragma unroll
    for (int k = 0; k < kCompactSlices / 32; k++) {
      const uint32_t v = s_slice[32 * k + lane];
      uint32_t inc = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t nb = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += nb;
      }
      s_slice[32 * k + lane] = carry + inc - v;
      carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) *s_total = carry;
  }
  __syncthreads();
  return *s_total;
}

// (Both kernels accept any grid: chunks are walked with a grid-stride loop.  The scatter pass is launched with 8 CTAs per
// SM -- dispatching one 256-thread CTA per chunk cost it ~0.4 us of block scheduling each for next to no work when the
// chunks are parked; the count pass measured faster with one CTA per chunk.)
template <bool kDist>
__global__ void __launch_bounds__(kCompactThreads)
compact_count_kernel(const CompactArgs a) {
  __shared__ uint32_t s_slice[kCompactSlices];
  __shared__ uint32_t s_total;
  const uint32_t tid = threadIdx.x, warp = tid >> 5;
  for (uint32_t chunk = blockIdx.x; chunk < a.n_chunks; chunk += gridDim.x) {
    const uint4 dv = __ldg(reinterpret_cast<const uint4*>(a.chunks) + chunk);
    const ChunkDesc d{dv.x, dv.y, dv.z, dv.w};
    uint32_t m[kCompactPer], rank[kCompactPer];
    const uint32_t total = chunk_rank(d, a.rowres, m, rank, s_slice, &s_total);
    if (tid == 0) a.chunk_count[chunk] = total;
    if (!kDist && total != 0 && total <= kStageCap) {  // CTA-uniform
      const bool swap = d.n_swap >> 31;
      uint2* st = a.stage + (size_t)chunk * kStageCap;
#pragma unroll
      for (int i = 0; i < kCompactPer; i++) {
        if (m[i] != kNone) {
          const uint32_t row = d.row_local + i * kCompactThreads + tid;
          st[s_slice[i * (kCompactThreads / 32) + warp] + rank[i]] = swap ? make_uint2(row, m[i]) : make_uint2(m[i], row);
        }
      }
    }
    __syncthreads();  // s_slice / s_total are rewritten by the next chunk
  }
}

// One CTA: exclusive prefix of the chunk totals (offsets relative to *running_total), per-pair counts, new total.
__global__ void __launch_bounds__(1024)
compact_scan_kernel(const CompactArgs a) {
  __shared__ unsigned long long s_warp[32];
  const unsigned long long base0 = *a.running_total;
  const uint32_t n = a.n_chunks, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t per = (n + 1023u) / 1024u;
  const uint32_t c0 = min(n, threadIdx.x * per), c1 = min(n, c0 + per);
  unsigned long long sum = 0;
  for (uint32_t c = c0; c < c1; c++) sum += a.chunk_count[c];
  unsigned long long inc = sum;  // inclusive scan inside the warp, then across the 32 warps
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (uint32_t)o) inc += v;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const unsigned long long w = s_warp[lane];
    unsigned long long winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long v = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= (uint32_t)o) winc += v;
    }
    s_warp[lane] = winc - w;  // exclusive prefix of the warp totals
    if (lane == 31) *a.running_total = base0 + winc;
  }
  __syncthreads();
  unsigned long long run = base0 + s_warp[warp] + inc - sum;
  for (uint32_t c = c0; c < c1; c++) {
    const uint32_t cnt = a.chunk_count[c];
    a.chunk_out[c] = run;
    run += cnt;
    if (cnt) atomicAdd(a.pair_count + a.chunks[c].pair, cnt);
  }
}

template <bool kDist>
__global__ void __launch_bounds__(kCompactThreads)
compact_scatter_kernel(const CompactArgs a) {
  __shared__ uint32_t s_slice[kCompactSlices];
  __shared__ uint32_t s_total;
  __shared__ __align__(16) uint2 s_stage[kCompactChunk + 2];
  const uint32_t tid = threadIdx.x, warp = tid >> 5;
  for (uint32_t chunk = blockIdx.x; chunk < a.n_chunks; chunk += gridDim.x) {
    const uint32_t total = a.chunk_count[chunk];
    if (total == 0) continue;  // CTA-uniform
    const unsigned long long dst0 = a.chunk_out[chunk];  // index of this chunk's first output pair
    if (!kDist && total <= kStageCap) {  // parked by the count pass: the rows are not read again
      if (tid < total) a.out_pairs[dst0 + tid] = a.stage[(size_t)chunk * kStageCap + tid];
      continue;
    }
    const uint4 dv = __ldg(reinterpret_cast<const uint4*>(a.chunks) + chunk);
    const ChunkDesc d{dv.x, dv.y, dv.z, dv.w};
    uint32_t m[kCompactPer], rank[kCompactPer];
    chunk_rank(d, a.rowres, m, rank, s_slice, &s_total);
    // ---- stage in output order ----
    const uint32_t shift = (uint32_t)(dst0 & 1ull);  // staged one slot late when the destination is not 16-byte aligned
    const bool swap = d.n_swap >> 31;
#pragma unroll
    for (int i = 0; i < kCompactPer; i++) {
      if (m[i] != kNone) {
        const uint32_t row = d.row_local + i * kCompactThreads + tid;
        const uint32_t pos = s_slice[i * (kCompactThreads / 32) + warp] + rank[i];
        s_stage[pos + shift] = swap ? make_uint2(row, m[i]) : make_uint2(m[i], row);
      }
    }
    __syncthreads();
    // ---- 16-byte stores: [dst0 - shift, ...) is 16-byte aligned; the slot before the first and the one after the
    // last pair are not this chunk's
    uint2* dst = a.out_pairs + (dst0 - shift);
    const uint32_t n_slots = total + shift;
    const uint4* st4 = reinterpret_cast<const uint4*>(s_stage);
    for (uint32_t q = tid; q < (n_slots + 1) / 2; q += kCompactThreads) {
      const uint32_t s0 = 2 * q;
      const bool lo_ok = s0 >= shift, hi_ok = s0 + 1 < n_slots;
      if (lo_ok && hi_ok) __stcs(reinterpret_cast<uint4*>(dst) + q, st4[q]);
      else if (lo_ok) dst[s0] = s_stage[s0];
      else if (hi_ok) dst[s0 + 1] = s_stage[s0 + 1];
    }
    if (kDist) {  // the distances take the same route through the (now free) staging area
      __syncthreads();
      float* s_dist = reinterpret_cast<float*>(s_stage);
#pragma unroll
      for (int i = 0; i < kCompactPer; i++) {
        if (m[i] != kNone)
          s_dist[s_slice[i * (kCompactThreads / 32) + warp] + rank[i]] = a.rowdist[d.row_abs + i * kCompactThreads + tid];
      }
      __syncthreads();
      float* dd = a.out_dist + dst0;
      for (uint32_t q = tid; q < total; q += kCompactThreads) dd[q] = s_dist[q];
    }
    __syncthreads();  // the staging area and s_slice are rewritten by the next chunk
  }
}

// ---- version 2 of the three passes (fm_debug_set_option("compact_v", 1) selects the ones above for comparison) ----
// What the per-launch profile of the passes above showed on 24 M-row batches (100 MB of rows): count 32 us at 40 % of
// DRAM throughput, scan 11 us in a single CTA, scatter 14 us of dependent loads.  The count pass keeps rows in flight
// only while a CTA waits for its own loads -- descriptor, then rows, then two barriers and a serial warp scan during
// which nothing is in flight.  Here the CTAs are persistent and software-pipelined: the rows (and the descriptor after
// next) of the FOLLOWING chunk are requested before the current chunk is ranked, so every resident CTA always has
// 16 KB on its way; ranks are recomputed in the rare parking branch instead of being held in registers, which keeps
// three CTAs per SM.  Per-pair counts are accumulated here (one atomic per non-empty chunk, spread over the grid)
// instead of by the single scan CTA, and the scatter pass moves parked chunks with one WARP per chunk.
struct ChunkRows {
  uint32_t m[kCompactPer];
};

__device__ __forceinline__ void chunk_load(const uint32_t* __restrict__ rowres, const ChunkDesc& d, ChunkRows& r) {
  const uint32_t n = d.n_swap & 0x7FFFFFFFu;
  const uint32_t* src = rowres + d.row_abs;
#pragma unroll
  for (int i = 0; i < kCompactPer; i++) {
    const uint32_t q = i * kCompactThreads + threadIdx.x;
    r.m[i] = q < n ? __ldg(src + q) : kNone;  // default caching: dense chunks are read again by the scatter pass, from L2
  }
}

template <bool kDist>
__global__ void __launch_bounds__(kCompactThreads, 3)
compact_count2_kernel(const CompactArgs a) {
  __shared__ uint32_t s_slice[kCompactSlices];
  __shared__ uint32_t s_total;
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  uint32_t chunk = blockIdx.x;
  if (chunk >= a.n_chunks) return;
  const uint4* descs = reinterpret_cast<const uint4*>(a.chunks);
  uint4 dv = __ldg(descs + chunk);
  ChunkRows cur, nxt;
  chunk_load(a.rowres, ChunkDesc{dv.x, dv.y, dv.z, dv.w}, cur);
  uint4 dnext = chunk + gridDim.x < a.n_chunks ? __ldg(descs + chunk + gridDim.x) : dv;
  for (;;) {
    const uint32_t next = chunk + gridDim.x;
    const bool has_next = next < a.n_chunks;  // CTA-uniform
    uint4 dnext2 = dnext;
    if (has_next) {
      chunk_load(a.rowres, ChunkDesc{dnext.x, dnext.y, dnext.z, dnext.w}, nxt);  // in flight while `cur` is ranked
      if (next + gridDim.x < a.n_chunks) dnext2 = __ldg(descs + next + gridDim.x);
    }
    const ChunkDesc d{dv.x, dv.y, dv.z, dv.w};
    // slice totals, their exclusive prefix, the chunk total
#pragma unroll
    for (int i = 0; i < kCompactPer; i++) {
      const uint32_t b = __ballot_sync(0xffffffffu, cur.m[i] != kNone);
      if (lane == 0) s_slice[i * (kCompactThreads / 32) + warp] = __popc(b);
    }
    __syncthreads();
    if (warp == 0) {
      uint32_t carry = 0;
#pragma unroll
      for (int k = 0; k < kCompactSlices / 32; k++) {
        const uint32_t v = s_slice[32 * k + lane];
        uint32_t inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const uint32_t nb = __shfl_up_sync(0xffffffffu, inc, o);
          if (lane >= (uint32_t)o) inc += nb;
        }
        s_slice[32 * k + lane] = carry + inc - v;
        carry += __shfl_sync(0xffffffffu, inc, 31);
      }
      if (lane == 0) {
        s_total = carry;
        a.chunk_count[chunk] = carry;
        if (carry) atomicAdd(a.pair_count + d.pair, carry);
      }
    }
    __syncthreads();
    const uint32_t total = s_total;
    if (!kDist && total != 0 && total <= kStageCap) {  // CTA-uniform: park the few pairs, the rows are not read again
      const bool swap = d.n_swap >> 31;
      uint2* st = a.stage + (size_t)chunk * kStageCap;
#pragma unroll
      for (int i = 0; i < kCompactPer; i++) {
        const uint32_t b = __ballot_sync(0xffffffffu, cur.m[i] != kNone);
        if (cur.m[i] != kNone) {
          const uint32_t row = d.row_local + i * kCompactThreads + tid;
          const uint32_t pos = s_slice[i * (kCompactThreads / 32) + warp] + __popc(b & ((1u << lane) - 1u));
          st[pos] = swap ? make_uint2(row, cur.m[i]) : make_uint2(cur.m[i], row);
        }
      }
    }
    if (!has_next) break;
    __syncthreads();  // s_slice / s_total are rewritten by the next chunk
    cur = nxt;
    dv = dnext;
    dnext = dnext2;
    chunk = next;
  }
}

// Count pass, version 3: the per-launch profile of version 2 (29 us per 100 MB: 43 % of DRAM throughput with the next
// chunk's rows always in flight) says the ranking work bounds the pass, not the loads -- two barriers, a serial
// 128-slice scan by one warp while seven wait, and a second round of ballots for the parked pairs.  Here every WARP owns
// 512 CONSECUTIVE rows of the chunk (16 coalesced 128-byte loads), so the rank of a match inside its warp needs nothing
// but that warp's own ballots, and the chunk needs one barrier: eight warp totals through shared memory.
template <bool kDist>
__global__ void __launch_bounds__(kCompactThreads, 3)
compact_count3_kernel(const CompactArgs a) {
  __shared__ uint32_t s_warp[2][kCompactThreads / 32];  // warp totals, double-buffered: one barrier per chunk
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  constexpr uint32_t kWarpRows = 32 * kCompactPer;  // 512
  uint32_t chunk = blockIdx.x;
  if (chunk >= a.n_chunks) return;
  const uint4* descs = reinterpret_cast<const uint4*>(a.chunks);
  auto load = [&](const uint4& dq, ChunkRows& r) {
    const uint32_t n = dq.y & 0x7FFFFFFFu;
    const uint32_t* src = a.rowres + dq.x + warp * kWarpRows;
#pragma unroll
    for (int i = 0; i < kCompactPer; i++) {
      const uint32_t q = warp * kWarpRows + i * 32 + lane;  // row inside the chunk
      r.m[i] = q < n ? __ldg(src + i * 32 + lane) : kNone;
    }
  };
  uint4 dv = __ldg(descs + chunk);
  ChunkRows cur, nxt;
  load(dv, cur);
  uint4 dnext = chunk + gridDim.x < a.n_chunks ? __ldg(descs + chunk + gridDim.x) : dv;
  uint32_t buf = 0;
  for (;;) {
    const uint32_t next = chunk + gridDim.x;
    const bool has_next = next < a.n_chunks;  // CTA-uniform
    uint4 dnext2 = dnext;
    if (has_next) {
      load(dnext, nxt);  // in flight while `cur` is counted
      if (next + gridDim.x < a.n_chunks) dnext2 = __ldg(descs + next + gridDim.x);
    }
    uint32_t ball[kCompactPer];
    uint32_t mine = 0;
#pragma unroll
    for (int i = 0; i < kCompactPer; i++) {
      ball[i] = __ballot_sync(0xffffffffu, cur.m[i] != kNone);
      mine += __popc(ball[i]);
    }
    if (lane == 0) s_warp[buf][warp] = mine;
    __syncthreads();
    uint32_t before = 0, total = 0;
#pragma unroll
    for (int w = 0; w < kCompactThreads / 32; w++) {
      const uint32_t t = s_warp[buf][w];
      before += w < (int)warp ? t : 0u;
      total += t;
    }
    if (tid == 0) {
      a.chunk_count[chunk] = total;
      if (total) atomicAdd(a.pair_count + dv.w, total);
    }
    if (!kDist && total != 0 && total <= kStageCap && mine != 0) {  // warp-uniform: park this warp's few pairs in row order
      const bool swap = dv.y >> 31;
      uint2* st = a.stage + (size_t)chunk * kStageCap + before;
      uint32_t run = 0;
#pragma unroll
      for (int i = 0; i < kCompactPer; i++) {
        if (cur.m[i] != kNone) {
          const uint32_t row = dv.z + warp * kWarpRows + i * 32 + lane;
          st[run + __popc(ball[i] & ((1u << lane) - 1u))] = swap ? make_uint2(row, cur.m[i]) : make_uint2(cur.m[i], row);
        }
        run += __popc(ball[i]);
      }
    }
    if (!has_next) break;
    buf ^= 1u;  // the other buffer was last read before the barrier above
    cur = nxt;
    dv = dnext;
    dnext = dnext2;
    chunk = next;
  }
}

// One CTA: exclusive prefix of the chunk totals (offsets relative to *running_total) and the new total.
__global__ void __launch_bounds__(1024)
compact_scan2_kernel(const CompactArgs a) {
  __shared__ unsigned long long s_warp[32];
  const unsigned long long base0 = *a.running_total;
  const uint32_t n = a.n_chunks, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // thread t owns chunks [t * per, (t + 1) * per), per a multiple of 4 so that the counts load as uint4
  const uint32_t per = ((n + 1023u) / 1024u + 3u) & ~3u;
  const uint32_t c0 = min(n, threadIdx.x * per), c1 = min(n, c0 + per);
  constexpr uint32_t kMaxPer = 32;  // 32 K chunks = 134 M rows per batch; larger batches take the loop below
  uint32_t cnt[kMaxPer];
  unsigned long long sum = 0;
  const bool in_regs = per <= kMaxPer;
  if (in_regs) {
#pragma unroll
    for (uint32_t q = 0; q < kMaxPer; q += 4) {
      uint4 v = make_uint4(0, 0, 0, 0);
      if (q < per && c0 + q < c1) {
        if (c0 + q + 4 <= c1) v = *reinterpret_cast<const uint4*>(a.chunk_count + c0 + q);
        else {
          v.x = a.chunk_count[c0 + q];
          if (c0 + q + 1 < c1) v.y = a.chunk_count[c0 + q + 1];
          if (c0 + q + 2 < c1) v.z = a.chunk_count[c0 + q + 2];
        }
      }
      cnt[q] = v.x; cnt[q + 1] = v.y; cnt[q + 2] = v.z; cnt[q + 3] = v.w;
      sum += (unsigned long long)v.x + v.y + v.z + v.w;
    }
  } else {
    for (uint32_t c = c0; c < c1; c++) sum += a.chunk_count[c];
  }
  unsigned long long inc = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const unsigned long long v = __shfl_up_sync(0xffffffffu, inc, o);
    if (lane >= (uint32_t)o) inc += v;
  }
  if (lane == 31) s_warp[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    const unsigned long long w = s_warp[lane];
    unsigned long long winc = w;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned long long v = __shfl_up_sync(0xffffffffu, winc, o);
      if (lane >= (uint32_t)o) winc += v;
    }
    s_warp[lane] = winc - w;
    if (lane == 31) *a.running_total = base0 + winc;
  }
  __syncthreads();
  unsigned long long run = base0 + s_warp[warp] + inc - sum;
  if (in_regs) {
#pragma unroll
    for (uint32_t q = 0; q < kMaxPer; q++) {
      if (q < per && c0 + q < c1) {
        a.chunk_out[c0 + q] = run;
        run += cnt[q];
      }
    }
  } else {
    for (uint32_t c = c0; c < c1; c++) {
      a.chunk_out[c] = run;
      run += a.chunk_count[c];
    }
  }
}

// Scatter: parked chunks by one warp each (count, offset and the <= 64 staged pairs are three short dependent loads;
// a CTA per chunk spent its whole life waiting for them), then the dense chunks by whole CTAs as before.
template <bool kDist>
__global__ void __launch_bounds__(kCompactThreads)
compact_scatter2_kernel(const CompactArgs a) {
  __shared__ uint32_t s_slice[kCompactSlices];
  __shared__ uint32_t s_total;
  __shared__ __align__(16) uint2 s_stage[kCompactChunk + 2];
  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (!kDist) {
    const uint32_t n_warps = gridDim.x * (kCompactThreads / 32);
    for (uint32_t chunk = blockIdx.x * (kCompactThreads / 32) + warp; chunk < a.n_chunks; chunk += n_warps) {
      const uint32_t total = a.chunk_count[chunk];
      if (total == 0 || total > kStageCap) continue;  // warp-uniform
      const unsigned long long dst0 = a.chunk_out[chunk];
      const uint2* st = a.stage + (size_t)chunk * kStageCap;
      for (uint32_t q = lane; q < total; q += 32) a.out_pairs[dst0 + q] = st[q];
    }
  }
  for (uint32_t chunk = blockIdx.x; chunk < a.n_chunks; chunk += gridDim.x) {
    const uint32_t total = a.chunk_count[chunk];
    if (total == 0 || (!kDist && total <= kStageCap)) continue;  // CTA-uniform
    const unsigned long long dst0 = a.chunk_out[chunk];
    const uint4 dv = __ldg(reinterpret_cast<const uint4*>(a.chunks) + chunk);
    const ChunkDesc d{dv.x, dv.y, dv.z, dv.w};
    uint32_t m[kCompactPer], rank[kCompactPer];
    chunk_rank(d, a.rowres, m, rank, s_slice, &s_total);
    const uint32_t shift = (uint32_t)(dst0 & 1ull);
    const bool swap = d.n_swap >> 31;
#pragma unroll
    for (int i = 0; i < kCompactPer; i++) {
      if (m[i] != kNone) {
        const uint32_t row = d.row_local + i * kCompactThreads + tid;
        const uint32_t pos = s_slice[i * (kCompactThreads / 32) + warp] + rank[i];
        s_stage[pos + shift] = swap ? make_uint2(row, m[i]) : make_uint2(m[i], row);
      }
    }
    __syncthreads();
    uint2* dst = a.out_pairs + (dst0 - shift);
    const uint32_t n_slots = total + shift;
    const uint4* st4 = reinterpret_cast<const uint4*>(s_stage);
    for (uint32_t q = tid; q < (n_slots + 1) / 2; q += kCompactThreads) {
      const uint32_t s0 = 2 * q;
      const bool lo_ok = s0 >= shift, hi_ok = s0 + 1 < n_slots;
      if (lo_ok && hi_ok) __stcs(reinterpret_cast<uint4*>(dst) + q, st4[q]);
      else if (lo_ok) dst[s0] = s_stage[s0];
      else if (hi_ok) dst[s0 + 1] = s_stage[s0 + 1];
    }
    if (kDist) {
      __syncthreads();
      float* s_dist = reinterpret_cast<float*>(s_stage);
#pragma unroll
      for (int i = 0; i < kCompactPer; i++) {
        if (m[i] != kNone)
          s_dist[s_slice[i * (kCompactThreads / 32) + warp] + rank[i]] = a.rowdist[d.row_abs + i * kCompactThreads + tid];
      }
      __syncthreads();
      float* dd = a.out_dist + dst0;
      for (uint32_t q = tid; q < total; q += kCompactThreads) dd[q] = s_dist[q];
    }
    __syncthreads();
  }
}

// ---- small batches: ONE launch -------------------------------------------------------------------------
// Up to a wave or two of chunks the three launches above are launch latency and nothing else (C2: 19 us against 11).
// Here a chunk obtains the exclusive prefix of the chunk totals by decoupled look-back over one 64-bit status word per
// chunk (launch epoch | state | value: no clearing between launches, only when the 30-bit epoch counter wraps back to
// 1; 1024 predecessors inspected per round).  CTAs of
// a 1-D grid are dispatched in index order, so a chunk's predecessors are always running or done (the assumption every
// single-pass scan makes).  For large batches the look-back chain is what bounds this design (95-140 us per 24 M rows
// in every variant measured), hence the three-launch form there.
constexpr int kCompactLook = 4;  // status words inspected per thread and look-back round

// kLookAll (test study, fm_debug_compact): every chunk but chunk 0 publishes only its aggregate, so chunk k sums all k
// predecessors in ceil(k / 1024) look-back rounds -- the multi-round path that production batches rarely reach.
template <bool kDist, bool kLookAll = false>
__global__ void __launch_bounds__(kCompactThreads)
compact_onepass_kernel(const CompactArgs a) {
  __shared__ uint32_t s_slice[kCompactSlices];  // slice totals, then their exclusive prefix
  __shared__ uint32_t s_total, s_first, s_unready, s_sum;
  __shared__ __align__(16) uint2 s_stage[kCompactChunk + 2];

  const uint32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const uint32_t chunk = blockIdx.x;
  volatile unsigned long long* status = a.status;
  // written again only by the CTA of the LAST chunk, after every other chunk has published -- i.e. after every CTA has
  // passed this load
  const unsigned long long base0 = *reinterpret_cast<volatile unsigned long long*>(a.running_total);
  const uint4 dv = __ldg(reinterpret_cast<const uint4*>(a.chunks) + chunk);
  const ChunkDesc d{dv.x, dv.y, dv.z, dv.w};
  const uint32_t n = d.n_swap & 0x7FFFFFFFu;
  const uint32_t* src = a.rowres + d.row_abs;

  // ---- coalesced loads: iteration i covers rows i*128 .. +127 of the chunk, a warp 32 consecutive rows ----
  uint32_t m[kCompactPer], rank[kCompactPer];
#pragma unroll
  for (int i = 0; i < kCompactPer; i++) {
    const uint32_t r = i * kCompactThreads + tid;
    m[i] = r < n ? __ldcs(src + r) : kNone;
  }
  if (tid == 0) { s_first = 0xFFFFFFFFu; s_unready = 0xFFFFFFFFu; s_sum = 0u; }
#pragma unroll
  for (int i = 0; i < kCompactPer; i++) {
    const uint32_t b = __ballot_sync(0xffffffffu, m[i] != kNone);
    rank[i] = __popc(b & ((1u << lane) - 1u));
    if (lane == 0) s_slice[i * (kCompactThreads / 32) + warp] = __popc(b);
  }
  __syncthreads();

  // ---- warp 0: exclusive scan of the 64 slice totals (row order = slice order), publish the chunk total ----
  if (warp == 0) {
    uint32_t carry = 0;
#pragma unroll
    for (int k = 0; k < kCompactSlices / 32; k++) {
      const uint32_t v = s_slice[32 * k + lane];
      uint32_t inc = v;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const uint32_t nb = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (uint32_t)o) inc += nb;
      }
      s_slice[32 * k + lane] = carry + inc - v;
      carry += __shfl_sync(0xffffffffu, inc, 31);
    }
    if (lane == 0) {
      s_total = carry;
      // successors can add this chunk's total while it is still looking back itself
      // (the 64-bit word is all a successor reads from this chunk: no fence is needed around the store)
      status[chunk] = chunk_word(a.epoch, chunk == 0 ? kChunkPrefix : kChunkAggregate, carry);
    }
  }
  __syncthreads();
  const uint32_t total = s_total;

  // ---- decoupled look-back: thread t inspects the predecessors at distance t + 128 r, r = 0..3, per round ----
  uint32_t excl = 0;
  {
    int64_t look = (int64_t)chunk - 1;
    while (look >= 0) {  // CTA-uniform
      unsigned long long w[kCompactLook];
      uint32_t unready = 0xFFFFFFFFu, mine = 0xFFFFFFFFu;  // smallest distance not published yet / holding a prefix
#pragma unroll
      for (int r = kCompactLook - 1; r >= 0; r--) {
        const int64_t idx = look - (int64_t)(tid + r * kCompactThreads);
        w[r] = idx >= 0 ? status[idx] : chunk_word(a.epoch, kChunkAggregate, 0u);
        const bool ok = (uint32_t)(w[r] >> 34) == a.epoch && ((w[r] >> 32) & 3ull) != 0ull;
        if (!ok) unready = tid + r * kCompactThreads;
        else if (((w[r] >> 32) & 3ull) == kChunkPrefix) mine = tid + r * kCompactThreads;
      }
      if (unready != 0xFFFFFFFFu) atomicMin(&s_unready, unready);
      if (mine != 0xFFFFFFFFu) atomicMin(&s_first, mine);
      __syncthreads();
      const uint32_t first = s_first;
      // only the predecessors NEARER than the first inclusive prefix matter: poll again if one of them has not published
      if (s_unready < first) {  // CTA-uniform
        __syncthreads();
        if (tid == 0) { s_unready = 0xFFFFFFFFu; s_first = 0xFFFFFFFFu; }
        __syncthreads();
        continue;
      }
      uint32_t val = 0;
#pragma unroll
      for (int r = 0; r < kCompactLook; r++)
        if (tid + r * kCompactThreads <= first) val += (uint32_t)w[r];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) val += __shfl_xor_sync(0xffffffffu, val, o);
      if (lane == 0 && val) atomicAdd(&s_sum, val);
      __syncthreads();
      if (first != 0xFFFFFFFFu) break;
      look -= kCompactLook * kCompactThreads;  // (s_unready is 0xFFFFFFFF here: every word of the window was published)
    }
    excl = s_sum;
    if (tid == 0) {
      if (!kLookAll && chunk != 0) status[chunk] = chunk_word(a.epoch, kChunkPrefix, excl + total);
      if (total) atomicAdd(a.pair_count + d.pair, total);
      if (chunk == a.n_chunks - 1) *a.running_total = base0 + excl + total;
    }
  }
  if (total == 0) return;  // CTA-uniform

  // ---- stage in output order ----
  const unsigned long long dst0 = base0 + excl;    // index of this chunk's first output pair
  const uint32_t shift = (uint32_t)(dst0 & 1ull);  // staged one slot late when the destination is not 16-byte aligned
  const bool swap = d.n_swap >> 31;
#pragma unroll
  for (int i = 0; i < kCompactPer; i++) {
    if (m[i] != kNone) {
      const uint32_t row = d.row_local + i * kCompactThreads + tid;
      const uint32_t pos = s_slice[i * (kCompactThreads / 32) + warp] + rank[i];
      s_stage[pos + shift] = swap ? make_uint2(row, m[i]) : make_uint2(m[i], row);
    }
  }
  __syncthreads();
  // ---- 16-byte stores: [dst0 - shift, ...) is 16-byte aligned; the slot before the first and the one after the last
  // pair are not this chunk's
  uint2* dst = a.out_pairs + (dst0 - shift);
  const uint32_t n_slots = total + shift;
  const uint4* st4 = reinterpret_cast<const uint4*>(s_stage);
  for (uint32_t q = tid; q < (n_slots + 1) / 2; q += kCompactThreads) {
    const uint32_t s0 = 2 * q;
    const bool lo_ok = s0 >= shift, hi_ok = s0 + 1 < n_slots;
    if (lo_ok && hi_ok) __stcs(reinterpret_cast<uint4*>(dst) + q, st4[q]);
    else if (lo_ok) dst[s0] = s_stage[s0];
    else if (hi_ok) dst[s0 + 1] = s_stage[s0 + 1];
  }
  if (kDist) {  // the distances take the same route through the (now free) staging area
    __syncthreads();
    float* s_dist = reinterpret_cast<float*>(s_stage);
#pragma unroll
    for (int i = 0; i < kCompactPer; i++) {
      if (m[i] != kNone)
        s_dist[s_slice[i * (kCompactThreads / 32) + warp] + rank[i]] = a.rowdist[d.row_abs + i * kCompactThreads + tid];
    }
    __syncthreads();
    float* dd = a.out_dist + dst0;
    for (uint32_t q = tid; q < total; q += kCompactThreads) dd[q] = s_dist[q];
  }
}


}  // namespace fm
