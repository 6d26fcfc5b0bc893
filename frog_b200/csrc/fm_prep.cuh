// fm_prep.cuh -- per-image preparation, run once at upload (replaces the AoS Point vector the
// reference's readers build, match.cpp:39-48).
//
// Produces, all device-resident:
//   * keypoints ordered by (laplacian value, scale): `perm`, `scale_sorted`, class table.  In that
//     order both reference gates (match.cpp:270, :273-275) select, for any row, one contiguous
//     column interval -- so whole operand tiles outside the band are never scored.
//   * FP16 operand images `rowop` / `colop`, already in the 128-row x 128-byte SWIZZLE_128B K-major
//     tile layout tcgen05.mma reads, so one 16 KB cp.async.bulk lands a ready tile in shared memory.
//     K is padded 48 -> 64: slots 48,49 carry (1, 1) on the row side and the hi/lo FP16 halves of
//     -|b|^2/2 on the column side, so the MMA itself yields  t = a.b - |b|^2/2  = (|a|^2 - d^2)/2.
//   * for d != 48 (d <= kWideMaxD) instead ONE operand image `wideop` of K_pad = wide_kpad(d) slots, fp16(desc) and
//     zeros, in k-blocks of the same tiles (fm_wide.cuh adds the norm term in its epilogue).
//   * per-image flags + max squared norm (certification inputs for the FP32 rescoring) and min squared
//     norm (the reject pass drops the norm slots for column images whose norms barely vary, fm_reject.cuh).
#pragma once
#include <cub/device/device_radix_sort.cuh>

#include "fm_common.cuh"
#include "fm_prep_types.h"

namespace fm {

constexpr float kMaxNorm2 = 16.0f;  // FP16 operands certified for |desc|^2 <= 16

__device__ __forceinline__ uint32_t float_sortable(float f) {
  uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float float_unsortable(uint32_t k) {
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7fffffffu) : ~k);
}

// Preparation is batched: every image uploaded since the last fm_match is prepared by ONE set of
// launches (keys, one radix sort over all their keypoints, class tables, operand packing), not one
// set per image -- at 20k keypoints an image's sort passes are pure launch latency.
// Largest s with segs[s].<field> <= b.
__device__ __forceinline__ uint32_t prep_find(const PrepSeg* __restrict__ segs, uint32_t n_segs, uint32_t b, bool pack) {
  uint32_t lo = 0, hi = n_segs;
  while (hi - lo > 1) {
    const uint32_t mid = (lo + hi) >> 1;
    if ((pack ? segs[mid].blk_pack : segs[mid].blk_keys) <= b) lo = mid; else hi = mid;
  }
  return lo;
}

__global__ void prep_reset_kernel(const PrepSeg* __restrict__ segs, ImageMeta* __restrict__ metas) {
  ImageMeta* m = metas + segs[blockIdx.x].img;
  uint32_t* w = reinterpret_cast<uint32_t*>(m);
  for (uint32_t i = threadIdx.x; i < sizeof(ImageMeta) / 4; i += blockDim.x) w[i] = 0u;
}

// Grouping code of a laplacian value: the top 16 bits of its float pattern.  Keypoints only have
// to be GROUPED by laplacian value (the class tables are matched by value, not by order), so 16
// bits in the sort key are enough as long as they separate the values present; prep_finish checks
// that they do and otherwise routes the image to the exact kernel.
__device__ __forceinline__ uint32_t lap_code(float l) { return __float_as_uint(l) >> 16; }

// One thread per keypoint: validity flags, squared norm, 64-bit sort key
// (batch segment | laplacian code | scale bits).
__global__ void __launch_bounds__(256)
prep_keys_kernel(const ImageDev* __restrict__ images, const PrepSeg* __restrict__ segs, uint32_t n_segs,
                 ImageMeta* __restrict__ metas, unsigned long long* __restrict__ keys, uint32_t* __restrict__ idx,
                 float* __restrict__ norm2) {
  const uint32_t sg = prep_find(segs, n_segs, blockIdx.x, false);
  const PrepSeg seg = segs[sg];
  const ImageDev im = images[seg.img];
  ImageMeta* meta = metas + seg.img;
  const uint32_t i = (blockIdx.x - seg.blk_keys) * blockDim.x + threadIdx.x;
  const uint32_t d = im.d;
  uint32_t flags = 0;
  float n2 = 0.f, dl2 = 0.f;
  if (i < seg.n) {
    const float* p = im.desc + (size_t)i * d;
    for (uint32_t k = 0; k < d; k++) {
      float v = __ldg(p + k);
      if (!isfinite(v)) flags |= kImgNotFinite;
      n2 = fmaf(v, v, n2);
      const float r = __half2float(__float2half_rn(v)) - v;  // exact: the operand's FP16 rounding residual
      dl2 = fmaf(r, r, dl2);
    }
    float s = im.scale[i], l = im.lap[i];
    if (!isfinite(s) || !isfinite(l)) flags |= kImgNotFinite;
    if (!(s > 0.f)) flags |= kImgBadScale;
    if (!(n2 <= kMaxNorm2)) flags |= kImgBigNorm;
    if (l == 0.f) l = 0.f;  // -0.0 == +0.0 for the reference's float compare: one class
    keys[seg.off + i] = ((unsigned long long)sg << 48) | ((unsigned long long)lap_code(l) << 32) | __float_as_uint(s);
    idx[seg.off + i] = i;
    norm2[seg.off + i] = n2;
  }
  // warp-aggregate then one atomic per warp
  float m = isfinite(n2) ? n2 : 0.f;
  float md = isfinite(dl2) ? dl2 : 0.f;
  // the min: complemented patterns, 0 (contributes nothing to the atomicMax) past the image and for non-finite norms
  uint32_t mn_inv = (i < seg.n && isfinite(n2)) ? ~__float_as_uint(n2) : 0u;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    md = fmaxf(md, __shfl_xor_sync(0xffffffffu, md, o));
    mn_inv = max(mn_inv, __shfl_xor_sync(0xffffffffu, mn_inv, o));
    flags |= __shfl_xor_sync(0xffffffffu, flags, o);
  }
  if ((threadIdx.x & 31) == 0) {
    if (flags) atomicOr(&meta->flags, flags);
    atomicMax(reinterpret_cast<unsigned int*>(&meta->max_norm2), __float_as_uint(m));   // non-negative floats
    atomicMax(reinterpret_cast<unsigned int*>(&meta->max_delta2), __float_as_uint(md));  // order like uints
    if (mn_inv) atomicMax(&meta->min_norm2_inv, mn_inv);
  }
}

// One CTA per image: un-zip its slice of the sorted (key, idx) pairs into perm / scale_sorted and
// build the laplacian class table.
__global__ void __launch_bounds__(1024)
prep_finish_kernel(const ImageDev* __restrict__ images, const PrepSeg* __restrict__ segs, ImageMeta* __restrict__ metas,
                   const unsigned long long* __restrict__ keys_sorted, const uint32_t* __restrict__ idx_sorted,
                   const float* __restrict__ norm2_all) {
  __shared__ uint32_t s_pos[kMaxClasses + 1];
  __shared__ uint32_t s_cnt, s_collide;
  const PrepSeg seg = segs[blockIdx.x];
  const ImageDev im = images[seg.img];
  ImageMeta* meta = metas + seg.img;
  uint32_t* perm = const_cast<uint32_t*>(im.perm);
  float* scale_sorted = const_cast<float*>(im.scale_sorted);
  float* norm2_sorted = const_cast<float*>(im.norm2_sorted);
  const float* norm2 = norm2_all + seg.off;
  const unsigned long long* ks = keys_sorted + seg.off;
  const uint32_t* is = idx_sorted + seg.off;
  const uint32_t n = seg.n;
  if (threadIdx.x == 0) { s_cnt = 0; s_collide = 0; }
  __syncthreads();
  for (uint32_t s = threadIdx.x; s < n; s += blockDim.x) {
    const unsigned long long k = ks[s];
    const uint32_t o = is[s];
    perm[s] = o;
    scale_sorted[s] = __uint_as_float((uint32_t)k);
    norm2_sorted[s] = norm2[o];
    if (s == 0 || (uint32_t)(ks[s - 1] >> 32) != (uint32_t)(k >> 32)) {
      uint32_t slot = atomicAdd(&s_cnt, 1u);
      if (slot <= kMaxClasses) s_pos[slot] = s;
    } else {
      // same 16-bit code as the left neighbour: the values themselves must agree too
      float l0 = im.lap[is[s - 1]], l1 = im.lap[o];
      if (l0 == 0.f) l0 = 0.f;
      if (l1 == 0.f) l1 = 0.f;
      if (__float_as_uint(l0) != __float_as_uint(l1)) s_collide = 1;
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t cnt = s_cnt;
    uint32_t flags = 0;
    if (im.d > (uint32_t)kWideMaxD) flags |= kImgBadDim;
    if (cnt > kMaxClasses || s_collide) { flags |= kImgManyClasses; cnt = min(cnt, (uint32_t)kMaxClasses); }
    for (uint32_t a = 1; a < cnt; a++) {  // insertion sort of <= 8 boundaries
      uint32_t v = s_pos[a];
      int b = (int)a - 1;
      while (b >= 0 && s_pos[b] > v) { s_pos[b + 1] = s_pos[b]; b--; }
      s_pos[b + 1] = v;
    }
    meta->n_classes = cnt;
    for (uint32_t a = 0; a < cnt; a++) {
      meta->class_begin[a] = s_pos[a];
      float l = im.lap[is[s_pos[a]]];
      if (l == 0.f) l = 0.f;
      meta->class_lap[a] = l;
    }
    for (uint32_t a = cnt; a <= kMaxClasses; a++) meta->class_begin[a] = n;
    if (flags) atomicOr(&meta->flags, flags);
  }
}

// One thread per (sorted keypoint, 16-byte chunk): FP16 operand tiles for both roles.
__global__ void __launch_bounds__(256)
prep_pack_kernel(const ImageDev* __restrict__ images, const PrepSeg* __restrict__ segs, uint32_t n_segs,
                 const float* __restrict__ norm2_all) {
  const uint32_t sg = prep_find(segs, n_segs, blockIdx.x, true);
  const PrepSeg seg = segs[sg];
  const ImageDev im = images[seg.img];
  if (im.d != (uint32_t)kD || im.rowop == nullptr) return;
  const float* __restrict__ desc = im.desc;
  const float* __restrict__ norm2 = norm2_all + seg.off;
  const uint32_t* __restrict__ perm = im.perm;
  uint8_t* rowop = reinterpret_cast<uint8_t*>(const_cast<__half*>(im.rowop));
  uint8_t* colop = reinterpret_cast<uint8_t*>(const_cast<__half*>(im.colop));
  const uint32_t n = seg.n, n_pad = im.n_pad;
  const uint32_t g = (blockIdx.x - seg.blk_pack) * blockDim.x + threadIdx.x;
  const uint32_t s = g >> 3, q = g & 7u;
  if (s >= n_pad) return;
  __align__(16) __half h[8];
#pragma unroll
  for (int k = 0; k < 8; k++) h[k] = __float2half_rn(0.f);
  __align__(16) __half hc[8];
#pragma unroll
  for (int k = 0; k < 8; k++) hc[k] = h[k];
  if (s < n) {
    const uint32_t o = perm[s];
    if (q < 6) {
      const float4* p = reinterpret_cast<const float4*>(desc + (size_t)o * kD + q * 8);
      float4 v0 = __ldg(p), v1 = __ldg(p + 1);
      h[0] = __float2half_rn(v0.x); h[1] = __float2half_rn(v0.y); h[2] = __float2half_rn(v0.z); h[3] = __float2half_rn(v0.w);
      h[4] = __float2half_rn(v1.x); h[5] = __float2half_rn(v1.y); h[6] = __float2half_rn(v1.z); h[7] = __float2half_rn(v1.w);
#pragma unroll
      for (int k = 0; k < 8; k++) hc[k] = h[k];
    } else if (q == 6) {
      h[0] = __float2half_rn(1.f);
      h[1] = __float2half_rn(1.f);
      float x = -0.5f * norm2[o];
      __half hi = __float2half_rn(x);
      hc[0] = hi;
      hc[1] = __float2half_rn(x - __half2float(hi));
    }
  }
  const size_t off = (size_t)(s >> 7) * 16384u + sw128_offset(s & 127u, q);
  *reinterpret_cast<uint4*>(rowop + off) = *reinterpret_cast<const uint4*>(h);
  *reinterpret_cast<uint4*>(colop + off) = *reinterpret_cast<const uint4*>(hc);
}

// Wide path (d != 48, fm_wide.cuh): one thread per (sorted keypoint, 16-byte chunk of its K_pad halves), the image's
// single FP16 operand.  Tile (s / 128, k-block kb) is 16 KB at ((s / 128) * kblocks + kb) * 16 KB, so the row tile or
// one column tile of a k-block is one contiguous cp.async.bulk.  A descriptor row is d floats: unless d is a multiple of
// 4 its rows are not 16-byte aligned, so the eight values are read with scalar loads (consecutive threads read
// consecutive chunks of one row: the loads still coalesce).
__global__ void __launch_bounds__(256)
prep_wide_pack_kernel(const ImageDev* __restrict__ images, const PrepSeg* __restrict__ segs, uint32_t n_segs) {
  const uint32_t sg = prep_find(segs, n_segs, blockIdx.x, true);
  const PrepSeg seg = segs[sg];
  const ImageDev im = images[seg.img];
  if (im.wideop == nullptr) return;
  const uint32_t d = im.d, chunks = wide_kpad(d) / 8u;
  const uint32_t g = (blockIdx.x - seg.blk_pack) * blockDim.x + threadIdx.x;
  const uint32_t s = g / chunks, c = g - s * chunks;
  if (s >= im.n_pad) return;
  __align__(16) __half h[8];
#pragma unroll
  for (int k = 0; k < 8; k++) h[k] = __float2half_rn(0.f);
  if (s < seg.n) {
    const float* __restrict__ p = im.desc + (size_t)im.perm[s] * d;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      const uint32_t kk = c * 8u + k;
      if (kk < d) h[k] = __float2half_rn(__ldg(p + kk));
    }
  }
  uint8_t* op = reinterpret_cast<uint8_t*>(const_cast<__half*>(im.wideop));
  const size_t off = ((size_t)(s >> 7) * (chunks / 8u) + (c >> 3)) * 16384u + sw128_offset(s & 127u, c & 7u);
  *reinterpret_cast<uint4*>(op + off) = *reinterpret_cast<const uint4*>(h);
}

}  // namespace fm
