// Device side of libfrogsurf.so: the SURF3D producer's stages as CUDA kernels for sm_100a.
//
// Every kernel here is integer / gather work over the 64-bit integral volume, bound by L2 and HBM
// traffic, not by arithmetic.  None of it is GEMM-shaped, so there is no tensor-core code in this
// file: the rules that matter are coalesced x-fastest access, enough loads in flight per thread and
// grids that fill the 148 SMs.
//
// Exactness: the reference computes in float / double on x86-64 without FMA contraction.  Every
// floating-point operation below that takes part in a result is written as an explicit IEEE
// round-to-nearest intrinsic (__fmul_rn, __dadd_rn, ...) in the reference's evaluation order, so the
// compiler can neither fuse nor reassociate it, whatever -fmad says.  Integer box sums are exact in
// any order (unsigned 64-bit, wrapping like the reference's).
#pragma once

#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>
#include <string.h>

#include "../../include/frogsurf.h"

namespace fs {

typedef unsigned long long u64;

// ---------------------------------------------------------------------------------------------
// cast + shift (vtk3DSURF.cxx:158-176): vtkImageCast to int with ClampOverflow, then
// vtkImageShiftScale with shift = -range[0], both through double and static_cast<int>.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int clamp_to_int(double v) {
  if (v > 2147483647.0) v = 2147483647.0;
  if (v < -2147483648.0) v = -2147483648.0;
  return __double2int_rz(v);
}

template <typename T>
__device__ __forceinline__ int cast_shift(T v, double shift) {
  const int c = clamp_to_int((double)v);
  return clamp_to_int(__dmul_rn(__dadd_rn((double)c, shift), 1.0));
}

// per-block minimum of the volume, as double (exact for every supported voxel type); +inf for a block without voxels
template <typename T>
__global__ void volume_min_kernel(const T* __restrict__ in, size_t n, double* __restrict__ block_min) {
  double m = CUDART_INF;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    const double v = (double)in[i];
    m = v < m ? v : m;
  }
  for (int o = 16; o; o >>= 1) {
    const double t = __shfl_xor_sync(0xffffffffu, m, o);
    m = t < m ? t : m;
  }
  __shared__ double wm[32];
  if ((threadIdx.x & 31) == 0) wm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    for (unsigned w = 1; w < (blockDim.x >> 5); w++) m = wm[w] < m ? wm[w] : m;
    block_min[blockIdx.x] = m;
  }
}

// ---------------------------------------------------------------------------------------------
// Integral volume (integral.cxx:11-121).  The reference runs three in-place passes (x, y, z); sums
// of unsigned 64-bit integers are exact in any order, so this does x and y in one pass per z slice
// and z in a second, fully coalesced pass.  HBM traffic: voxel read + 8 B write, then 8 B read +
// 16 B write (the second copy is the parity-split layout the response kernel gathers from)
// = 36 B / voxel for 4-byte voxels, against 4 + 6 x 8 = 52 B for three separate passes.
//
// x/y pass: one CTA per z slice works through the slice in tiles of `rows` rows.  Phase 1: each warp
// scans one row of the tile along x (32 voxels per step, shuffle scan, carry in lane 31) into shared
// memory; phase 2: each thread owns columns, adds the tile's rows onto its running column sum (the
// 2-D integral of the row above) and stores them, coalesced.  Two barriers per tile.
// ---------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(512) integral_xy_kernel(const T* __restrict__ in, int32_t* __restrict__ cast_out,
                                                           u64* __restrict__ out, int nx, int ny, int rows, double shift) {
  extern __shared__ u64 fs_sm[];
  u64* col = fs_sm;        // nx running column sums
  u64* tile = fs_sm + nx;  // rows x nx row prefixes
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
  const size_t slice = (size_t)nx * ny, base = (size_t)blockIdx.x * slice;
  for (int x = tid; x < nx; x += blockDim.x) col[x] = 0;
  for (int y0 = 0; y0 < ny; y0 += rows) {
    const int nr = min(rows, ny - y0);
    for (int r = warp; r < nr; r += nwarps) {
      const size_t row = base + (size_t)(y0 + r) * nx;
      u64 carry = 0;
      for (int x0 = 0; x0 < nx; x0 += 32) {
        const int x = x0 + lane;
        u64 v = 0;
        if (x < nx) {
          const int c = cast_shift(in[row + x], shift);
          if (cast_out) cast_out[row + x] = c;
          v = (u64)(long long)c;  // int -> unsigned long long as the reference's assignment does (integral.cxx:113)
        }
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const u64 t = __shfl_up_sync(0xffffffffu, v, o);
          if (lane >= o) v += t;
        }
        v += carry;
        if (x < nx) tile[(size_t)r * nx + x] = v;
        carry = __shfl_sync(0xffffffffu, v, 31);
      }
    }
    __syncthreads();
    for (int x = tid; x < nx; x += blockDim.x) {
      u64 c = col[x];
      for (int r = 0; r < nr; r++) {
        c += tile[(size_t)r * nx + x];
        out[base + (size_t)(y0 + r) * nx + x] = c;
      }
      col[x] = c;
    }
    __syncthreads();
  }
}

// z pass, in place, plus the parity-split copy: split[x & 1][z][y][x >> 1] with row pitch hx = (nx + 1) / 2.  The
// response layers sample the volume at even x only (steps 2 .. 16), and every box corner sits at a fixed offset
// from that x, so one gather instruction of a warp touches x of ONE parity: in the split layout those 32 addresses
// are contiguous (256 B) instead of strided over 512 B.
__global__ void integral_z_kernel(u64* __restrict__ vol, u64* __restrict__ split, int nx, int ny, int nz) {
  const size_t slice = (size_t)nx * ny;
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= slice) return;
  const int x = (int)(i % nx), y = (int)(i / nx);
  const int hx = (nx + 1) / 2;
  const size_t sslice = (size_t)hx * ny;
  u64* sp = split + (size_t)(x & 1) * sslice * nz + (size_t)y * hx + (x >> 1);
  u64 acc = vol[i];
  sp[0] = acc;
  int z = 1;
  for (; z + 4 <= nz; z += 4) {
    u64* p = vol + (size_t)z * slice + i;
    u64* q = sp + (size_t)z * sslice;
    const u64 a = p[0], b = p[slice], c = p[2 * slice], d = p[3 * slice];
    acc += a; p[0] = acc; q[0] = acc;
    acc += b; p[slice] = acc; q[sslice] = acc;
    acc += c; p[2 * slice] = acc; q[2 * sslice] = acc;
    acc += d; p[3 * slice] = acc; q[3 * sslice] = acc;
  }
  for (; z < nz; z++) {
    u64* p = vol + (size_t)z * slice + i;
    acc += *p;
    *p = acc;
    sp[(size_t)z * sslice] = acc;
  }
}

// ---------------------------------------------------------------------------------------------
// Box sums over the integral volume (integral.h:66-115, BoxIntegralOptim: no clamping).
// ---------------------------------------------------------------------------------------------
struct Integral {
  const u64* p;
  long long sy, sz;  // increments along y and z (x increment 1)
  int nx, ny, nz;
};

// parity-split copy (see integral_z_kernel): (x odd ? p1 : p0) + (x >> 1) + y * sy + z * sz, element offsets in 32 bits
// (volumes up to 2^32 voxels)
struct IntegralSplit {
  const u64 *p0, *p1;  // even-x and odd-x halves
  uint32_t sy, sz;
};

// Box sum (BoxIntegralOptim) for the voxel whose element offset in the split layout is `base` (its x is even: the
// layers sample at steps 2 .. 16), the box given RELATIVE to the voxel.  Everything but `base` is the same for all
// threads, so the corner offsets live in uniform registers and each gather costs one 32-bit add and one widening
// multiply-add for its address instead of 64-bit arithmetic per corner.
__device__ __forceinline__ u64 box_sum(const IntegralSplit& I, uint32_t base, int dx, int dy, int dz, int sx, int sy, int sz) {
  const int x1 = dx - 1, x2 = dx + sx - 1;
  const uint32_t y1 = (uint32_t)(dy - 1) * I.sy, y2 = (uint32_t)(dy + sy - 1) * I.sy;
  const uint32_t z1 = (uint32_t)(dz - 1) * I.sz, z2 = (uint32_t)(dz + sz - 1) * I.sz;
  const u64* a = (x1 & 1) ? I.p1 : I.p0;
  const u64* b = (x2 & 1) ? I.p1 : I.p0;
  const uint32_t oa = base + (uint32_t)(x1 >> 1), ob = base + (uint32_t)(x2 >> 1);  // modulo 2^32: the sums are offsets >= 0
  return __ldg(b + (uint32_t)(ob + y2 + z2)) - __ldg(b + (uint32_t)(ob + y2 + z1)) - __ldg(b + (uint32_t)(ob + y1 + z2)) -
         __ldg(a + (uint32_t)(oa + y2 + z2)) + __ldg(a + (uint32_t)(oa + y1 + z2)) + __ldg(a + (uint32_t)(oa + y2 + z1)) +
         __ldg(b + (uint32_t)(ob + y1 + z1)) - __ldg(a + (uint32_t)(oa + y1 + z1));
}

__device__ __forceinline__ float boxf(const IntegralSplit& I, uint32_t base, int dx, int dy, int dz, int sx, int sy, int sz) {
  return __ull2float_rn(box_sum(I, base, dx, dy, dz, sx, sy, sz));
}

// ---------------------------------------------------------------------------------------------
// One response layer (FastHessian::buildResponseLayer, fasthessian.cxx:343-481): box-filter
// approximations of the six second derivatives, determinant response, laplacian sign, blob flag.
// 144 eight-byte gathers per voxel, from the parity-split copy of the integral volume: neighbouring
// threads take neighbouring layer voxels along x, so for the step-2 layers (7/8 of all voxels) each
// gather instruction reads 256 contiguous bytes, and the lines it touches are reused from L1 by the
// other corners of the same rows.
// ---------------------------------------------------------------------------------------------
struct LayerDev {
  float* responses;
  float* masked;       // response where the voxel is a blob, -1 where it is not: what the extremum search compares with
  uint8_t* laplacian;
  uint8_t* isblob;
  int width, height, depth, step, filter;
  int limit;           // fasthessian.cxx:366
  float inv_volume9;   // fasthessian.cxx:355
};

__device__ __forceinline__ void response_voxel(const IntegralSplit& I, const LayerDev& L, int ax, int ay, int az) {
  const int x = ax * L.step, y = ay * L.step, z = az * L.step;
  const uint32_t base = (uint32_t)(x >> 1) + (uint32_t)y * I.sy + (uint32_t)z * I.sz;
  const int b = (L.filter - 1) / 2, l = L.filter / 3, w = L.filter;
  const int m = 2 * l - 1;

  // boxes relative to (x, y, z), fasthessian.cxx:395-419
  const float Dxx = __fsub_rn(boxf(I, base, -b, -l + 1, -l + 1, w, m, m),
                              __fmul_rn(boxf(I, base, -(l / 2), -l + 1, -l + 1, l, m, m), 3.0f));
  const float Dyy = __fsub_rn(boxf(I, base, -l + 1, -b, -l + 1, m, w, m),
                              __fmul_rn(boxf(I, base, -l + 1, -(l / 2), -l + 1, m, l, m), 3.0f));
  const float Dzz = __fsub_rn(boxf(I, base, -l + 1, -l + 1, -b, m, m, w),
                              __fmul_rn(boxf(I, base, -l + 1, -l + 1, -(l / 2), m, m, l), 3.0f));
  const float Dxy = __fsub_rn(__fsub_rn(__fadd_rn(boxf(I, base, -l, -l, -l + 1, l, l, m), boxf(I, base, 1, 1, -l + 1, l, l, m)),
                                        boxf(I, base, -l, 1, -l + 1, l, l, m)),
                              boxf(I, base, 1, -l, -l + 1, l, l, m));
  const float Dyz = __fsub_rn(__fsub_rn(__fadd_rn(boxf(I, base, -l + 1, -l, -l, m, l, l), boxf(I, base, -l + 1, 1, 1, m, l, l)),
                                        boxf(I, base, -l + 1, -l, 1, m, l, l)),
                              boxf(I, base, -l + 1, 1, -l, m, l, l));
  const float Dxz = __fsub_rn(__fsub_rn(__fadd_rn(boxf(I, base, -l, -l + 1, -l, l, m, l), boxf(I, base, 1, -l + 1, 1, l, m, l)),
                                        boxf(I, base, -l, -l + 1, 1, l, m, l)),
                              boxf(I, base, 1, -l + 1, -l, l, m, l));

  // fasthessian.cxx:428-430, in the reference's operand order and types (the 2.0 literal makes the second term,
  // and from there the running sum, double)
  const float sq = __fadd_rn(__fadd_rn(__fmul_rn(Dxy, Dxy), __fmul_rn(Dxz, Dxz)), __fmul_rn(Dyz, Dyz));
  const float Sdet2p = __fsub_rn(__fadd_rn(__fadd_rn(__fmul_rn(Dyy, Dzz), __fmul_rn(Dxx, Dyy)), __fmul_rn(Dxx, Dzz)),
                                 __fmul_rn(0.8330f, sq));
  const float Trace = __fadd_rn(__fadd_rn(Dxx, Dyy), Dzz);
  double det = (double)__fmul_rn(__fmul_rn(Dxx, Dyy), Dzz);
  det = __dadd_rn(det, __dmul_rn(__dmul_rn(__dmul_rn(__dmul_rn(2.0, (double)Dxy), (double)Dyz), (double)Dxz), (double)0.7603f));
  det = __dsub_rn(det, (double)__fmul_rn(__fmul_rn(__fmul_rn(Dxx, Dyz), Dyz), 0.8330f));
  det = __dsub_rn(det, (double)__fmul_rn(__fmul_rn(__fmul_rn(Dyy, Dxz), Dxz), 0.8330f));
  det = __dsub_rn(det, (double)__fmul_rn(__fmul_rn(__fmul_rn(Dzz, Dxy), Dxy), 0.8330f));
  const float Det = __double2float_rn(det);

  const size_t index = (size_t)ax + (size_t)ay * L.width + (size_t)az * L.width * L.height;
  const bool blob = (Sdet2p > 0.0f) && (__fmul_rn(Trace, Det) > 0.0f);
  const float response = fabsf(__fmul_rn(Det, L.inv_volume9));
  L.isblob[index] = blob;
  L.responses[index] = response;
  L.masked[index] = blob ? response : -1.0f;
  L.laplacian[index] = Trace >= 0.0f ? 1 : 0;
}

// Thread -> voxel mapping: a CTA is a 32 x TY x TZ tile of layer voxels (each warp 32 consecutive x).  Voxels that are
// neighbours in y and z read box corners on the same integral-volume rows (corner rows of one voxel are 2 * step apart
// from its neighbour's), so a tile that extends in y and z reuses the lines it pulled into L1 instead of leaving
// that reuse to whichever CTA runs next: the kernel is bound by L2 -> L1 traffic, not by HBM (ncu, profiles/).
template <int TY, int TZ, int kMinBlocks = 1>
__global__ void __launch_bounds__(32 * TY * TZ, kMinBlocks) response_layer_kernel(IntegralSplit I, LayerDev L) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int ax = L.limit + blockIdx.x * 32 + lane;
  const int ay = L.limit + blockIdx.y * TY + warp % TY;
  const int az = L.limit + blockIdx.z * TZ + warp / TY;
  if (ax >= L.width - L.limit || ay >= L.height - L.limit || az >= L.depth - L.limit) return;
  response_voxel(I, L, ax, ay, az);
}

// flat mapping (x fastest over the whole interior): kept for comparison, fs_debug_set_option("response_tile", 0)
__global__ void __launch_bounds__(256) response_layer_flat_kernel(IntegralSplit I, LayerDev L) {
  const int iw = L.width - 2 * L.limit, ih = L.height - 2 * L.limit, id = L.depth - 2 * L.limit;
  const long long n = (long long)iw * ih * id;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n) return;
  response_voxel(I, L, L.limit + (int)(t % iw), L.limit + (int)((t / iw) % ih), L.limit + (int)(t / ((long long)iw * ih)));
}

// ---------------------------------------------------------------------------------------------
// Extremum search over one (bottom, middle, top) layer triple (fasthessian.cxx:161-218, isExtremum
// :521-548) and, for each extremum, the derivative vector and Hessian the interpolation step solves
// with (deriv4D :666-696, hessian4D :938-1014).  Extrema are rare, so the record is written by the
// thread that found it; the host orders records by `key` = the reference's loop position.
// ---------------------------------------------------------------------------------------------
struct LayerView {
  const float* responses;
  const float* masked;  // see LayerDev
  const uint8_t* laplacian;
  const uint8_t* isblob;
  int width, height, depth;
};

__device__ __forceinline__ size_t lv_index(const LayerView& v, int scale, int r, int c, int d) {
  // responselayer.h:73-80: getResponse(row, column, layer, src) with scale = this->width / src->width
  return (size_t)(scale * c) + (size_t)(scale * r) * v.width + (size_t)(scale * d) * v.width * v.height;
}
__device__ __forceinline__ float lv_resp(const LayerView& v, int scale, int r, int c, int d) {
  return __ldg(v.responses + lv_index(v, scale, r, c, d));
}
__device__ __forceinline__ float lv_masked(const LayerView& v, int scale, int r, int c, int d) {
  return __ldg(v.masked + lv_index(v, scale, r, c, d));
}

struct ExtremaPass {
  LayerView b, m, t;
  int scale_m, scale_b;        // m->width / t->width, b->width / t->width
  int limit;                   // fasthessian.cxx:181-189
  long long first_sup, first_down;  // loop positions from which `param` has lost its bits (fasthessian.cxx:202-210)
  int param0;                  // FIRST_SCALE 1, LAST_SCALE 2, NONE_SCALE 0
  int pass;
  float thresh;
};

struct Candidate {
  u64 key;
  int r, c, d, laplacian;
  float response;
  float pad_;
  double dD[4];
  double H[10];  // dxx dyy dzz dss dxy dxz dxs dyz dys dzs
};

__global__ void __launch_bounds__(256) extrema_kernel(ExtremaPass P, Candidate* __restrict__ out, unsigned* __restrict__ count, unsigned cap) {
  const int nc = P.t.width - 2 * P.limit, nr = P.t.height - 2 * P.limit, nd = P.t.depth - 2 * P.limit;
  const long long n = (long long)nc * nr * nd;
  const long long tix = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tix >= n) return;
  // x (column) fastest across threads for coalescing; the reference's loops nest r, c, d
  const int c = P.limit + (int)(tix % nc), r = P.limit + (int)((tix / nc) % nr), d = P.limit + (int)(tix / ((long long)nc * nr));
  const long long pos = ((long long)(r - P.limit) * nc + (c - P.limit)) * nd + (d - P.limit);
  int param = P.param0;
  if (pos >= P.first_sup) param &= 2;
  if (pos >= P.first_down) param &= 1;

  // isExtremum (fasthessian.cxx:521-548): the candidate must be a blob at or above the threshold, and no blob voxel of
  // the 3 x 3 x 3 neighbourhoods in the three layers may reach it (`>=`).  The reference walks the 27 offsets with an
  // early return; the result does not depend on the order, so each rr plane's 27 values (9 offsets x 3 layers) are
  // loaded together -- one latency instead of up to 54 dependent ones -- from the `masked` copy, where non-blob voxels
  // hold -1 and can never reach a candidate (responses are >= 0, the threshold is >= 0).  Kept quirks: the middle layer
  // skips every offset with rr == cc == 0 (dd = +-1 included), `param` decides whether top / bottom take part.
  const float candidate = lv_masked(P.m, P.scale_m, r, c, d);  // -1 when the candidate is not a blob
  if (!(candidate >= P.thresh) || !(candidate >= 0.0f)) return;  // (NaN = outside the layer's interior: never a candidate)
  const bool use_t = param != 2, use_b = param != 1;
  for (int rr = -1; rr <= 1; ++rr) {
    float vt[9], vm[9], vb[9];
#pragma unroll
    for (int q = 0; q < 9; q++) {
      const int cc = q / 3 - 1, dd = q % 3 - 1;
      vt[q] = use_t ? lv_masked(P.t, 1, r + rr, c + cc, d + dd) : -1.0f;
      vm[q] = (rr != 0 || cc != 0) ? lv_masked(P.m, P.scale_m, r + rr, c + cc, d + dd) : -1.0f;
      vb[q] = use_b ? lv_masked(P.b, P.scale_b, r + rr, c + cc, d + dd) : -1.0f;
    }
    bool reached = false;
#pragma unroll
    for (int q = 0; q < 9; q++) reached |= (vt[q] >= candidate) | (vm[q] >= candidate) | (vb[q] >= candidate);
    if (reached) return;
  }

  const unsigned slot = atomicAdd(count, 1u);
  if (slot >= cap) return;
  Candidate k;
  k.key = ((u64)P.pass << 48) | (u64)pos;
  k.r = r; k.c = c; k.d = d;
  k.laplacian = __ldg(P.m.laplacian + lv_index(P.m, P.scale_m, r, c, d));
  k.response = candidate;
  k.pad_ = 0.0f;
#define M_(rr, cc, dd) lv_resp(P.m, P.scale_m, r + (rr), c + (cc), d + (dd))
#define T_(rr, cc, dd) lv_resp(P.t, 1, r + (rr), c + (cc), d + (dd))
#define B_(rr, cc, dd) lv_resp(P.b, P.scale_b, r + (rr), c + (cc), d + (dd))
  // float differences, then a double division (the reference divides by the double literals 2.0 / 4.0)
  k.dD[0] = __ddiv_rn((double)__fsub_rn(M_(0, 1, 0), M_(0, -1, 0)), 2.0);
  k.dD[1] = __ddiv_rn((double)__fsub_rn(M_(1, 0, 0), M_(-1, 0, 0)), 2.0);
  k.dD[2] = __ddiv_rn((double)__fsub_rn(M_(0, 0, 1), M_(0, 0, -1)), 2.0);
  k.dD[3] = __ddiv_rn((double)__fsub_rn(T_(0, 0, 0), B_(0, 0, 0)), 2.0);
  const double v = (double)M_(0, 0, 0), v2 = __dmul_rn(2.0, v);
  k.H[0] = __dsub_rn((double)__fadd_rn(M_(0, 1, 0), M_(0, -1, 0)), v2);
  k.H[1] = __dsub_rn((double)__fadd_rn(M_(1, 0, 0), M_(-1, 0, 0)), v2);
  k.H[2] = __dsub_rn((double)__fadd_rn(M_(0, 0, 1), M_(0, 0, -1)), v2);
  k.H[3] = __dsub_rn((double)__fadd_rn(T_(0, 0, 0), B_(0, 0, 0)), v2);
#define CROSS_(a, b2, c2, d2) __ddiv_rn((double)__fadd_rn(__fsub_rn(__fsub_rn((a), (b2)), (c2)), (d2)), 4.0)
  k.H[4] = CROSS_(M_(1, 1, 0), M_(1, -1, 0), M_(-1, 1, 0), M_(-1, -1, 0));   // dxy
  k.H[5] = CROSS_(M_(1, 0, 1), M_(1, 0, -1), M_(-1, 0, 1), M_(-1, 0, -1));   // "dxz" (the reference steps r and d here)
  k.H[6] = CROSS_(T_(0, 1, 0), T_(0, -1, 0), B_(0, 1, 0), B_(0, -1, 0));     // dxs
  k.H[7] = CROSS_(M_(0, 1, 1), M_(0, 1, -1), M_(0, -1, 1), M_(0, -1, -1));   // "dyz" (steps c and d)
  k.H[8] = CROSS_(T_(1, 0, 0), T_(-1, 0, 0), B_(1, 0, 0), B_(-1, 0, 0));     // dys
  k.H[9] = CROSS_(T_(0, 0, 1), T_(0, 0, -1), B_(0, 0, 1), B_(0, 0, -1));     // dzs
#undef CROSS_
#undef M_
#undef T_
#undef B_
  out[slot] = k;
}

// ---------------------------------------------------------------------------------------------
// Interpolation step (FastHessian::interpolateStep / interpolateExtremum, fasthessian.cxx:575-661):
// X = -pinv(H) dD with singular values below 0.001 of the largest dropped, keep the extremum when all
// four offsets are below 1.  H is symmetric, so its SVD is its eigen-decomposition up to signs: a
// cyclic Jacobi eigen-solver in double gives pinv(H) = sum over kept eigenpairs of q q^T / lambda.
// The reference calls cv::SVD from OpenCV, which is not part of the reference tree; any accurate SVD
// agrees with this to rounding (~1e-13 relative), and the tests pin the step to that tolerance.
// One statement for host (CPU tests) and device (the library is compiled with -fmad=false, so both
// sides execute the same IEEE operations).
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline void solve_offsets(const double dD[4], const double Hs[10], double X[4]) {
  double A[4][4] = {{Hs[0], Hs[4], Hs[5], Hs[6]}, {Hs[4], Hs[1], Hs[7], Hs[8]}, {Hs[5], Hs[7], Hs[2], Hs[9]}, {Hs[6], Hs[8], Hs[9], Hs[3]}};
  double Q[4][4] = {{1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}};
  for (int sweep = 0; sweep < 64; sweep++) {
    double off = 0, diag = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
      diag += A[i][i] * A[i][i];
#pragma unroll
      for (int j = i + 1; j < 4; j++) off += A[i][j] * A[i][j];
    }
    if (off <= 1e-32 * diag || off == 0) break;
#pragma unroll
    for (int p = 0; p < 3; p++)
#pragma unroll
      for (int q = p + 1; q < 4; q++) {
        if (A[p][q] == 0) continue;
        const double theta = (A[q][q] - A[p][p]) / (2 * A[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1));
        const double cs = 1 / sqrt(t * t + 1), sn = t * cs;
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const double akp = A[k][p], akq = A[k][q];
          A[k][p] = cs * akp - sn * akq;
          A[k][q] = sn * akp + cs * akq;
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const double apk = A[p][k], aqk = A[q][k];
          A[p][k] = cs * apk - sn * aqk;
          A[q][k] = sn * apk + cs * aqk;
        }
#pragma unroll
        for (int k = 0; k < 4; k++) {
          const double qkp = Q[k][p], qkq = Q[k][q];
          Q[k][p] = cs * qkp - sn * qkq;
          Q[k][q] = sn * qkp + cs * qkq;
        }
      }
  }
  double wmax = 0;
  int largest = 0;
#pragma unroll
  for (int i = 0; i < 4; i++)
    if (fabs(A[i][i]) > wmax) { wmax = fabs(A[i][i]); largest = i; }
#pragma unroll
  for (int k = 0; k < 4; k++) X[k] = 0;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    const double lam = A[i][i];
    // W_inv(0,0) = 1 / W(0) unconditionally (a zero matrix gives inf -> NaN -> rejected, as in the reference);
    // the others are dropped when W(i) / W(0) < 0.001
    if (i != largest && !(fabs(lam) / wmax >= 0.001)) continue;
    double proj = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) proj += Q[k][i] * dD[k];
    const double coef = proj / lam;
#pragma unroll
    for (int k = 0; k < 4; k++) X[k] -= Q[k][i] * coef;
  }
}

struct PassScale {
  int t_step, m_filter, b_filter;
};
struct PassScales {
  PassScale p[8];
};

struct Interpolated {
  u64 key;        // loop position of the extremum (Candidate::key)
  fs_point point;
  int accepted;
  int pad_;
};

// fasthessian.cxx:591-611: the keypoint an accepted extremum becomes
__host__ __device__ inline bool make_point(const Candidate& k, const PassScale& s, fs_point& p) {
  double X[4];
  solve_offsets(k.dD, k.H, X);
  const double xX = X[0], xY = X[1], xZ = X[2], xS = X[3];
  if (!(fabs(xX) < 1.0f && fabs(xY) < 1.0f && fabs(xZ) < 1.0f && fabs(xS) < 1.0f)) return false;
  const int filterStep = s.m_filter - s.b_filter;
  p.x = static_cast<float>((k.c + xX) * s.t_step);
  p.y = static_cast<float>((k.r + xY) * s.t_step);
  p.z = static_cast<float>((k.d + xZ) * s.t_step);
  p.scale = static_cast<float>((double)(0.1333f) * (s.m_filter + xS * filterStep));
  p.laplacian = k.laplacian;
  p.response = k.response;
  return true;
}

__global__ void __launch_bounds__(128) interpolate_kernel(const Candidate* __restrict__ cand, unsigned n, PassScales scales,
                                                           Interpolated* __restrict__ out) {
  const unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const Candidate k = cand[i];
  Interpolated r;
  r.key = k.key;
  r.pad_ = 0;
  r.point = fs_point{0, 0, 0, 0, 0, 0};
  r.accepted = make_point(k, scales.p[(unsigned)(k.key >> 48) & 7], r.point) ? 1 : 0;
  out[i] = r;
}

// ---------------------------------------------------------------------------------------------
// glibc 2.39's expf (sysdeps/ieee754/flt-32/e_expf.c -- Szabolcs Nagy's table-driven algorithm:
// x * 32/ln2 = k + r, 2^(k/32) from a 32-entry table, cubic in r, all in double, one final rounding
// to float), restated from its published description.  Surf::gaussian calls expf (surf.cxx:227),
// so bit-identical descriptors need bit-identical expf: this restatement equals this image's libm
// on every float in [-104, 88.7] (exhaustive host test, tests/test_surf_host.py) but two, which are
// patched below; the table is 2^(i/32) rounded to double with i << 47 subtracted.
// ---------------------------------------------------------------------------------------------
#define FS_EXP2_TABLE                                                                                   \
  {0x3ff0000000000000ULL, 0x3fefd9b0d3158574ULL, 0x3fefb5586cf9890fULL, 0x3fef9301d0125b51ULL,          \
   0x3fef72b83c7d517bULL, 0x3fef54873168b9aaULL, 0x3fef387a6e756238ULL, 0x3fef1e9df51fdee1ULL,          \
   0x3fef06fe0a31b715ULL, 0x3feef1a7373aa9cbULL, 0x3feedea64c123422ULL, 0x3feece086061892dULL,          \
   0x3feebfdad5362a27ULL, 0x3feeb42b569d4f82ULL, 0x3feeab07dd485429ULL, 0x3feea47eb03a5585ULL,          \
   0x3feea09e667f3bcdULL, 0x3fee9f75e8ec5f74ULL, 0x3feea11473eb0187ULL, 0x3feea589994cce13ULL,          \
   0x3feeace5422aa0dbULL, 0x3feeb737b0cdc5e5ULL, 0x3feec49182a3f090ULL, 0x3feed503b23e255dULL,          \
   0x3feee89f995ad3adULL, 0x3feeff76f2fb5e47ULL, 0x3fef199bdd85529cULL, 0x3fef3720dcef9069ULL,          \
   0x3fef5818dcfba487ULL, 0x3fef7c97337b9b5fULL, 0x3fefa4afa2a490daULL, 0x3fefd0765b6e4540ULL}
__constant__ u64 kExp2TabDev[32] = FS_EXP2_TABLE;
static const u64 kExp2TabHost[32] = FS_EXP2_TABLE;

// the same statement on both sides of the compiler so that the host tests can run it against libm without a GPU
__host__ __device__ __forceinline__ float glibc_expf(float x) {
#ifdef __CUDA_ARCH__
#define FS_DMUL(a, b) __dmul_rn((a), (b))
#define FS_DADD(a, b) __dadd_rn((a), (b))
#define FS_DSUB(a, b) __dsub_rn((a), (b))
  const u64* tab = kExp2TabDev;
#else
#define FS_DMUL(a, b) ((a) * (b))  // host build: x86-64 baseline, no FMA contraction
#define FS_DADD(a, b) ((a) + (b))
#define FS_DSUB(a, b) ((a) - (b))
  const u64* tab = kExp2TabHost;
#endif
  if (!(x >= -0x1.9fe368p6f)) return x != x ? x : 0.0f;  // underflow to +0 (and NaN in, NaN out)
  if (x > 0x1.62e42ep6f) return x + x > x ? x * 3.0e38f : x;  // overflow to +inf
  if (x == -0x1.f8cbb2p+5f) return 0x1.f45326p-92f;      // the two inputs where libm's last bit differs
  if (x == 0x1.04845ep+5f) return 0x1.f93e38p+46f;
  const double z = FS_DMUL(0x1.71547652b82fep+0 * 32.0, (double)x);
  double kd = FS_DADD(z, 0x1.8p52);
  u64 ki;
  memcpy(&ki, &kd, 8);
  kd = FS_DSUB(kd, 0x1.8p52);
  const double r = FS_DSUB(z, kd);
  const u64 sbits = tab[ki & 31] + (ki << 47);
  double s;
  memcpy(&s, &sbits, 8);
  const double p = FS_DADD(FS_DMUL(0x1.c6af84b912394p-5 / 32 / 32 / 32, r), 0x1.ebfce50fac4f3p-3 / 32 / 32);
  const double r2 = FS_DMUL(r, r);
  double y = FS_DADD(FS_DMUL(0x1.62e42ff0c52d6p-1 / 32, r), 1.0);
  y = FS_DADD(FS_DMUL(p, r2), y);
  return (float)FS_DMUL(y, s);
#undef FS_DMUL
#undef FS_DADD
#undef FS_DSUB
}

// ---------------------------------------------------------------------------------------------
// Descriptors (Surf::getDescriptor surf.cxx:63-156, getRawDescriptor :161-217).  One CTA per
// keypoint: the (2 radius)^3 Haar samples are computed in parallel (20 gathers each, see the kernel)
// and parked in shared memory as doubles; 48 threads then add up their
// sub-block's samples IN THE REFERENCE'S ORDER (u, v, w nested), because the sums are double
// accumulations whose rounding depends on it.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ int f_round(float f) { return (int)floorf(__fadd_rn(f, 0.5f)); }  // surf.h:86-89

struct Clamp {
  bool hit;
};

// Integral value at (x, y, z); where the reference would read outside the volume (undefined behaviour in
// BoxIntegralOptim) this follows BoxIntegral (integral.h:30-62): negative index -> 0, index past the end -> last.
__device__ __forceinline__ u64 integ_at(const Integral& I, int x, int y, int z, Clamp& cl) {
  if (x < 0 || y < 0 || z < 0) { cl.hit = true; return 0; }
  if (x >= I.nx) { x = I.nx - 1; cl.hit = true; }
  if (y >= I.ny) { y = I.ny - 1; cl.hit = true; }
  if (z >= I.nz) { z = I.nz - 1; cl.hit = true; }
  return __ldg(I.p + x + (long long)y * I.sy + (long long)z * I.sz);
}

// sum over [xa+1..xb] x [ya+1..yb] x [za+1..zb] (inclusive corner indices as BoxIntegralOptim forms them)
__device__ __forceinline__ long long box_corners(const Integral& I, int xa, int xb, int ya, int yb, int za, int zb, Clamp& cl) {
  return (long long)(integ_at(I, xb, yb, zb, cl) - integ_at(I, xb, yb, za, cl) - integ_at(I, xb, ya, zb, cl) -
                     integ_at(I, xa, yb, zb, cl) + integ_at(I, xa, ya, zb, cl) + integ_at(I, xa, yb, za, cl) +
                     integ_at(I, xb, ya, za, cl) - integ_at(I, xa, ya, za, cl));
}

// haarXOptim / haarYOptim / haarZOptim (surf.cxx:256-281) at (x, y, z) with s = 2 * h
__device__ __forceinline__ void haar3(const Integral& I, int x, int y, int z, int h, float& hx, float& hy, float& hz, Clamp& cl) {
  const int s = 2 * h, hh = s / 2;
  const int xl = x - hh - 1, xm = x - 1, xr = x + hh - 1, xR = x - hh + s - 1;
  const int yl = y - hh - 1, ym = y - 1, yr = y + hh - 1, yR = y - hh + s - 1;
  const int zl = z - hh - 1, zm = z - 1, zr = z + hh - 1, zR = z - hh + s - 1;
  hx = __ll2float_rn(box_corners(I, xm, xr, yl, yR, zl, zR, cl) - box_corners(I, xl, xm, yl, yR, zl, zR, cl));
  hy = __ll2float_rn(box_corners(I, xl, xR, ym, yr, zl, zR, cl) - box_corners(I, xl, xR, yl, ym, zl, zR, cl));
  hz = __ll2float_rn(box_corners(I, xl, xR, yl, yR, zm, zr, cl) - box_corners(I, xl, xR, yl, yR, zl, zm, cl));
}

// Per-axis tables of one keypoint: the sample grid is separable (sample_x depends on u only, ...), so the three
// integral-volume planes a Haar wavelet touches along an axis -- lo = s - h - 1, mid = s - 1, hi = s + h - 1 for
// sample coordinate s and half size h -- and the squared Gaussian offset are computed once per axis position.
constexpr int kMaxRadius = 16;
struct AxisTables {
  long long lo[3][2 * kMaxRadius], mid[3][2 * kMaxRadius], hi[3][2 * kMaxRadius];  // premultiplied by the axis stride
  int sample[3][2 * kMaxRadius];
  float sq[3][2 * kMaxRadius];
};

__global__ void __launch_bounds__(128) describe_kernel(Integral I, const fs_point* __restrict__ pts, unsigned n, int radius,
                                                        int type, int normalize, float* __restrict__ desc,
                                                        unsigned* __restrict__ n_clamped) {
  extern __shared__ double fs_smd[];
  const unsigned id = blockIdx.x;
  if (id >= n) return;
  const fs_point pt = pts[id];
  const int r3 = radius * radius * radius, S = 8 * r3, R2 = 2 * radius;
  double* sx = fs_smd;  // [S] per component, sub-block major, (u, v, w) inside
  double* sy = fs_smd + S;
  double* sz = fs_smd + 2 * S;
  __shared__ double acc[48];
  __shared__ AxisTables tab;
  __shared__ int outside;
  if (threadIdx.x == 0) outside = 0;
  __syncthreads();

  const double scale = (double)pt.scale;
  const float halfRadius = __double2float_rn(__ddiv_rn((double)__double2float_rn((double)radius - 1.0), 2.0));
  const int h = f_round(pt.scale);                                           // s = 2 * fRound(scale)
  const float sig = __double2float_rn(__dmul_rn((double)2.5f, scale));       // gaussian(..., 2.5f * scale)
  const float sig2 = __fmul_rn(sig, sig);
  const float norm = __fdiv_rn(1.0f, __fmul_rn(sig2, sig));                  // 1.0f / (sig*sig*sig)
  const float den = __fmul_rn(__fmul_rn(2.0f, sig), sig);                    // 2.0f*sig*sig
  const size_t dsize = type == 0 ? 48 : (size_t)3 * S;

  if (threadIdx.x < 3 * R2) {
    const int axis = threadIdx.x / R2, idx = threadIdx.x - axis * R2;
    const float coord = axis == 0 ? pt.x : axis == 1 ? pt.y : pt.z;
    const int dim = axis == 0 ? I.nx : axis == 1 ? I.ny : I.nz;
    const long long stride = axis == 0 ? 1 : axis == 1 ? I.sy : I.sz;
    const int centre = f_round(coord);
    const int u = -radius + idx;
    // sample_x = fRound(x + u*scale)
    const int smp = f_round(__double2float_rn(__dadd_rn((double)centre, __dmul_rn((double)u, scale))));
    // xs = fRound(ipt->x + (ix * scale)) with ix = (float) i + halfRadius, i the sub-block's first offset
    const int i0 = -radius + (idx / radius) * radius;
    const float ix = __fadd_rn((float)i0, halfRadius);
    const int xs = f_round(__double2float_rn(__dadd_rn((double)coord, __dmul_rn((double)ix, scale))));
    const float g = __fsub_rn((float)xs, (float)smp);
    tab.sample[axis][idx] = smp;
    tab.sq[axis][idx] = __fmul_rn(g, g);
    tab.lo[axis][idx] = (long long)(smp - h - 1) * stride;
    tab.mid[axis][idx] = (long long)(smp - 1) * stride;
    tab.hi[axis][idx] = (long long)(smp + h - 1) * stride;
    if (smp - h - 1 < 0 || smp + h - 1 >= dim) outside = 1;
  }
  __syncthreads();
  const bool inside = outside == 0;

  // Threads enumerate the samples with x fastest: the lanes of a warp then gather from a few rows of the integral
  // volume (2 radius x-neighbours per row, `scale` voxels apart) instead of from 32 different z slices, which had the
  // L1 data pipe at 97 % with one wavefront per lane per gather (ncu, profiles/).  Where a sample is STORED follows the
  // reference's order -- sub-block major, (u, v, w) nested inside -- because that is the order the sums run in.
  for (int g = threadIdx.x; g < S; g += blockDim.x) {
    const int iu = g % R2, iv = (g / R2) % R2, iw = g / (R2 * R2);
    const int bu = iu >= radius, bv = iv >= radius, bw = iw >= radius;
    const int sidx = (bu * 4 + bv * 2 + bw) * r3 + ((iu - bu * radius) * radius + (iv - bv * radius)) * radius + (iw - bw * radius);
    float hx, hy, hz;
    if (inside) {
      // 20 gathers: the 8 corners {lo, hi}^3 are shared by the three wavelets, 4 more per wavelet through its mid plane
      const u64* p = I.p;
      const long long xl = tab.lo[0][iu], xm = tab.mid[0][iu], xh = tab.hi[0][iu];
      const long long yl = tab.lo[1][iv], ym = tab.mid[1][iv], yh = tab.hi[1][iv];
      const long long zl = tab.lo[2][iw], zm = tab.mid[2][iw], zh = tab.hi[2][iw];
      const u64 clll = __ldg(p + xl + yl + zl), cllh = __ldg(p + xl + yl + zh), clhl = __ldg(p + xl + yh + zl), clhh = __ldg(p + xl + yh + zh);
      const u64 chll = __ldg(p + xh + yl + zl), chlh = __ldg(p + xh + yl + zh), chhl = __ldg(p + xh + yh + zl), chhh = __ldg(p + xh + yh + zh);
      const u64 mxll = __ldg(p + xm + yl + zl), mxlh = __ldg(p + xm + yl + zh), mxhl = __ldg(p + xm + yh + zl), mxhh = __ldg(p + xm + yh + zh);
      const u64 myll = __ldg(p + xl + ym + zl), mylh = __ldg(p + xl + ym + zh), myhl = __ldg(p + xh + ym + zl), myhh = __ldg(p + xh + ym + zh);
      const u64 mzll = __ldg(p + xl + yl + zm), mzlh = __ldg(p + xl + yh + zm), mzhl = __ldg(p + xh + yl + zm), mzhh = __ldg(p + xh + yh + zm);
      // box(upper half) - box(lower half) along the wavelet's axis = hi - 2 mid + lo, inclusion-exclusion over the other two
      const u64 ax = (chhh - 2 * mxhh + clhh) - (chhl - 2 * mxhl + clhl) - (chlh - 2 * mxlh + cllh) + (chll - 2 * mxll + clll);
      const u64 ay = (chhh - 2 * myhh + chlh) - (chhl - 2 * myhl + chll) - (clhh - 2 * mylh + cllh) + (clhl - 2 * myll + clll);
      const u64 az = (chhh - 2 * mzhh + chhl) - (chlh - 2 * mzhl + chll) - (clhh - 2 * mzlh + clhl) + (cllh - 2 * mzll + clll);
      hx = __ll2float_rn((long long)ax);
      hy = __ll2float_rn((long long)ay);
      hz = __ll2float_rn((long long)az);
    } else {
      Clamp cl{false};
      haar3(I, tab.sample[0][iu], tab.sample[1][iv], tab.sample[2][iw], h, hx, hy, hz, cl);
    }
    if (type == 0) {
      const float num = __fadd_rn(__fadd_rn(tab.sq[0][iu], tab.sq[1][iv]), tab.sq[2][iw]);
      const double gauss = (double)__fmul_rn(norm, glibc_expf(__fdiv_rn(-num, den)));
      sx[sidx] = __dmul_rn(gauss, (double)hx);
      sy[sidx] = __dmul_rn(gauss, (double)hy);
      sz[sidx] = __dmul_rn(gauss, (double)hz);
    } else {
      float* o = desc + (size_t)id * dsize + (size_t)3 * sidx;
      o[0] = hx; o[1] = hy; o[2] = hz;
    }
  }
  if (threadIdx.x == 0 && !inside) atomicAdd(n_clamped, 1u);
  if (type != 0) return;
  __syncthreads();

  if (threadIdx.x < 48) {
    const int blk = threadIdx.x / 6, comp = threadIdx.x % 6;
    const double* src = (comp % 3 == 0 ? sx : comp % 3 == 1 ? sy : sz) + blk * r3;
    double a = 0.0;  // dx = dy = ... = 0.f
    if (comp < 3) {
      for (int q = 0; q < r3; q++) a = __dadd_rn(a, src[q]);
    } else {
      for (int q = 0; q < r3; q++) a = __dadd_rn(a, fabs(src[q]));
    }
    acc[threadIdx.x] = a;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    float* o = desc + (size_t)id * 48;
    double len = 0.0;
    for (int blk = 0; blk < 8; blk++) {
      const double* a = acc + blk * 6;
      double q = __dmul_rn(a[0], a[0]);
      for (int c = 1; c < 6; c++) q = __dadd_rn(q, __dmul_rn(a[c], a[c]));
      len = __dadd_rn(len, q);
    }
    len = __dsqrt_rn(len);
    for (int c = 0; c < 48; c++) {
      float f = __double2float_rn(acc[c]);  // desc[count++] = dx : double -> float
      if (normalize && len != 0.0) f = __double2float_rn(__ddiv_rn((double)f, len));
      o[c] = f;
    }
  }
}

}  // namespace fs
