// fm_group.cuh -- the gather of fm_group_match: every member's compacted lists into one buffer on the lead GPU, in the
// caller's pair order.
//
// A member matched its shard (local pairs k = 0 .. n-1, global positions idx[k], ascending) into its own compacted
// lists.  Its stream then runs group_counts_kernel (per-pair counts stored into the lead's counts at idx[k]: peer
// stores) and links_scan_kernel on its own counts (local offsets).  The lead scans the gathered counts into
// submission-order offsets, and each member runs group_push_kernel: its lists, and distances, are stored straight into
// the lead's buffers at those offsets.  Every store of a non-lead member crosses NVLink, so the body of a list goes out
// as 16-byte stores; only an unaligned first or last element is stored alone.
#pragma once
#include "fm_common.cuh"

namespace fm {

constexpr int kGatherThreads = 256;
constexpr int kGatherWarps = kGatherThreads / 32;
// lists up to this many matches are pushed by one warp; longer ones by the whole CTA
constexpr uint32_t kGatherWarpMax = 1024;

__global__ void __launch_bounds__(256)
group_counts_kernel(const uint32_t* __restrict__ counts, const uint32_t* __restrict__ idx, uint32_t n,
                    uint32_t* __restrict__ lead_counts) {
  for (uint32_t k = blockIdx.x * blockDim.x + threadIdx.x; k < n; k += gridDim.x * blockDim.x) lead_counts[idx[k]] = counts[k];
}

// Copy `n` matches src[0, n) to dst[0, n) with lane `lane` of `lanes` threads: dst is 8-byte aligned; the 16-byte
// aligned body of dst is written with uint4 stores (src read as uint4 when it shares dst's alignment, else as two uint2).
__device__ __forceinline__ void push_pairs(const uint2* __restrict__ src, uint2* __restrict__ dst, unsigned long long n,
                                           uint32_t lane, uint32_t lanes) {
  if (n == 0) return;
  const unsigned long long head = (reinterpret_cast<uintptr_t>(dst) & 15u) ? 1ull : 0ull;
  if (head && lane == 0) dst[0] = src[0];
  const unsigned long long body = (n - head) >> 1;  // 16-byte stores
  uint4* d4 = reinterpret_cast<uint4*>(dst + head);
  const uint2* s = src + head;
  if ((reinterpret_cast<uintptr_t>(s) & 15u) == 0) {
    const uint4* s4 = reinterpret_cast<const uint4*>(s);
    for (unsigned long long i = lane; i < body; i += lanes) d4[i] = __ldg(s4 + i);
  } else {
    for (unsigned long long i = lane; i < body; i += lanes) {
      const uint2 a = __ldg(s + 2 * i), b = __ldg(s + 2 * i + 1);
      d4[i] = make_uint4(a.x, a.y, b.x, b.y);
    }
  }
  const unsigned long long tail = head + 2 * body;
  if (tail < n && lane == 0) dst[tail] = src[tail];
}

// The same for distances: 4-byte aligned dst, float4 stores for its 16-byte aligned body.
__device__ __forceinline__ void push_dist(const float* __restrict__ src, float* __restrict__ dst, unsigned long long n,
                                          uint32_t lane, uint32_t lanes) {
  if (n == 0) return;
  const unsigned long long mis = (reinterpret_cast<uintptr_t>(dst) >> 2) & 3u;
  const unsigned long long head = min(n, mis ? 4ull - mis : 0ull);
  if (lane < head) dst[lane] = src[lane];
  const unsigned long long body = (n - head) >> 2;
  float4* d4 = reinterpret_cast<float4*>(dst + head);
  const float* s = src + head;
  if ((reinterpret_cast<uintptr_t>(s) & 15u) == 0) {
    const float4* s4 = reinterpret_cast<const float4*>(s);
    for (unsigned long long i = lane; i < body; i += lanes) d4[i] = __ldg(s4 + i);
  } else {
    for (unsigned long long i = lane; i < body; i += lanes)
      d4[i] = make_float4(__ldg(s + 4 * i), __ldg(s + 4 * i + 1), __ldg(s + 4 * i + 2), __ldg(s + 4 * i + 3));
  }
  const unsigned long long tail = head + 4 * body;
  if (lane < n - tail) dst[tail + lane] = src[tail + lane];
}

// One CTA per kGatherWarps local pairs: warp w pushes pair kGatherWarps * blockIdx.x + w if its list is short, and the
// CTA then pushes the long lists of its pairs one after another with all its threads.
//   loff       : local exclusive offsets (n + 1), into src_pairs / src_dist
//   idx        : global position of each local pair;  lead_off : the lead's submission-order offsets (read over NVLink)
template <bool kDist>
__global__ void __launch_bounds__(kGatherThreads)
group_push_kernel(const uint2* __restrict__ src_pairs, const float* __restrict__ src_dist,
                  const unsigned long long* __restrict__ loff, const uint32_t* __restrict__ idx, uint32_t n,
                  const unsigned long long* __restrict__ lead_off, uint2* __restrict__ dst_pairs, float* __restrict__ dst_dist) {
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31u;
  const uint32_t k0 = blockIdx.x * kGatherWarps;
  {
    const uint32_t k = k0 + warp;
    if (k < n) {
      const unsigned long long s = loff[k], cnt = loff[k + 1] - s;
      if (cnt <= kGatherWarpMax) {
        const unsigned long long d = lead_off[idx[k]];
        push_pairs(src_pairs + s, dst_pairs + d, cnt, lane, 32);
        if (kDist) push_dist(src_dist + s, dst_dist + d, cnt, lane, 32);
      }
    }
  }
  for (uint32_t k = k0; k < min(n, k0 + kGatherWarps); k++) {
    const unsigned long long s = loff[k], cnt = loff[k + 1] - s;
    if (cnt <= kGatherWarpMax) continue;
    const unsigned long long d = lead_off[idx[k]];
    push_pairs(src_pairs + s, dst_pairs + d, cnt, threadIdx.x, kGatherThreads);
    if (kDist) push_dist(src_dist + s, dst_dist + d, cnt, threadIdx.x, kGatherThreads);
  }
}

}  // namespace fm
