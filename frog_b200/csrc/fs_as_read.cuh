// Device side of fs_get_points_as_read: each keypoint field as bin/surf3d's .csv.gz writer formats it and the matcher's
// reader parses it back, i.e. strtof(format_fixed(v, decimals)) (surf_io.cpp, keypoint_io.cpp), without the text.
//
// format_fixed forms n = v * 10^decimals rounded half-to-even exactly in 128-bit integers; the text "n / 10^decimals"
// then parses to the correctly rounded float of that quotient, with the sign of v ("-0.000000" reads as -0.0f).  Here:
//   1. n exactly as format_fixed forms it (same integer steps, same range test);
//   2. q = fl64(n) / fl64(10^decimals): within 2^-52 (relative) of the exact quotient x.  The only float midpoint that
//      can lie between q and x is the one inside q's own float interval [T, T + ulp): a double M.  x is compared with M
//      exactly (n * 2^-e vs mantissa(M) * 10^decimals, both below 2^84): below -> T, above -> T + ulp, equal -> the
//      even one of the two, as strtof rounds.
// Values outside format_fixed's integer range (decimals > 9, |v| * 10^decimals >= 9e18, inf, nan) take its snprintf
// path on the host: the kernel lists them and the host finishes them with snprintf + strtof.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/frogsurf.h"

namespace fs {

struct AsReadFallback {
  unsigned long long index;  // position in the output (head: row * 6 + col; descriptors: n * 6 + row * d + k)
  double value;              // the double the writer would format
};

struct AsReadGeom {
  double spacing[3], origin[3];
  double sspacing;  // cube root of the spacing product, as the writer computes it (host pow)
  int decimals;     // descriptor cells: -precision, 6 when negative
};

__device__ __forceinline__ unsigned long long pow10_u64(int d) {
  unsigned long long p = 1;
  for (int i = 0; i < d; i++) p *= 10ull;
  return p;
}

// strtof(format_fixed(v, decimals)); *host = true (and 0 returned) when format_fixed would take its snprintf path.
__device__ __forceinline__ float as_read_value(double v, int decimals, bool* host) {
  const unsigned long long bits = (unsigned long long)__double_as_longlong(v);
  const unsigned long long frac = bits & ((1ull << 52) - 1);
  const int expo = (int)((bits >> 52) & 0x7FF);
  const bool neg = (bits >> 63) != 0;
  if (decimals < 0 || decimals > 9) { *host = true; return 0.f; }
  const unsigned long long p10 = pow10_u64(decimals);
  const double p10d = (double)p10;
  if (expo == 0x7FF || !(__dmul_rn(fabs(v), p10d) < 9e18)) { *host = true; return 0.f; }
  *host = false;
  // 1. n = v * 10^decimals, rounded half-to-even (format_fixed, line for line)
  const unsigned long long mant = expo ? (frac | (1ull << 52)) : frac;
  const int e2 = (expo ? expo : 1) - 1075;
  const unsigned __int128 prod = (unsigned __int128)mant * p10;  // < 2^83
  unsigned long long n;
  if (e2 >= 0) {
    n = (unsigned long long)(prod << e2);  // the range test keeps this below 2^64
  } else {
    const int k = -e2;
    if (k >= 100) {
      n = 0;
    } else {
      const unsigned __int128 q = prod >> k, rem = prod & ((((unsigned __int128)1) << k) - 1),
                              half = ((unsigned __int128)1) << (k - 1);
      n = (unsigned long long)q;
      if (rem > half || (rem == half && (n & 1ull))) n++;
    }
  }
  if (n == 0) return neg ? -0.f : 0.f;
  // 2. the float nearest to x = n / 10^decimals (x >= 1e-9 and < 2^63: always a normal float)
  const double q = __ddiv_rn(__ull2double_rn(n), p10d);
  const unsigned long long qb = (unsigned long long)__double_as_longlong(q);
  const unsigned long long tb = qb & ~0x1FFFFFFFull;  // q truncated to float precision: T, exactly a float
  const unsigned long long mb = tb | 0x10000000ull;   // M = T + ulp / 2
  const float t = __double2float_rn(__longlong_as_double((long long)tb));
  const unsigned long long mm = (mb & ((1ull << 52) - 1)) | (1ull << 52);
  const int em = (int)((mb >> 52) & 0x7FF) - 1075;
  unsigned __int128 lhs = n, rhs = (unsigned __int128)mm * p10;  // x <> M  <=>  n * 2^-em <> mm * 10^decimals
  if (em >= 0) rhs <<= em;
  else lhs <<= -em;
  const float up = __int_as_float(__float_as_int(t) + 1);
  const float r = lhs < rhs ? t : lhs > rhs ? up : ((__float_as_int(t) & 1) ? up : t);
  return neg ? -r : r;
}

// A value for the host is counted always and listed while the list has room (the host re-runs with a longer list when
// the count exceeds it).
struct AsReadList {
  AsReadFallback* entries;
  unsigned long long* count;
  unsigned long long cap;
};

__device__ __forceinline__ void as_read_store(float* out, unsigned long long at, double v, int decimals, AsReadList list) {
  bool host;
  const float r = as_read_value(v, decimals, &host);
  out[at] = r;
  if (host) {
    const unsigned long long slot = atomicAdd(list.count, 1ull);
    if (slot < list.cap) list.entries[slot] = AsReadFallback{at, v};
  }
}

// out = head (n x 6) followed by the descriptors (n x d); one thread per value, grid-stride
__global__ void __launch_bounds__(256) as_read_kernel(const fs_point* __restrict__ pts, const float* __restrict__ desc,
                                                      unsigned n, unsigned d, AsReadGeom g, float* __restrict__ out,
                                                      AsReadList list) {
  const unsigned long long head_total = (unsigned long long)n * 6, total = head_total + (unsigned long long)n * d;
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < total;
       i += (unsigned long long)gridDim.x * blockDim.x) {
    if (i >= head_total) {
      as_read_store(out, i, (double)desc[i - head_total], g.decimals, list);
      continue;
    }
    const unsigned row = (unsigned)(i / 6), col = (unsigned)(i % 6);
    const fs_point p = pts[row];
    if (col == 4) {  // "%d": an integer's text reads back as its correctly rounded float
      out[i] = __int2float_rn(p.laplacian);
      continue;
    }
    double v;
    if (col < 3) {  // origin + coordinate * spacing: two separately rounded operations, as the host writer
      const float c = col == 0 ? p.x : col == 1 ? p.y : p.z;
      const double s = col == 0 ? g.spacing[0] : col == 1 ? g.spacing[1] : g.spacing[2];
      const double o = col == 0 ? g.origin[0] : col == 1 ? g.origin[1] : g.origin[2];
      v = __dadd_rn(__dmul_rn((double)c, s), o);
    } else if (col == 3) {
      v = __dmul_rn((double)p.scale, g.sspacing);
    } else {
      v = (double)p.response;
    }
    as_read_store(out, i, v, 6, list);
  }
}

// fs_debug_as_read: the same conversion over given doubles
__global__ void __launch_bounds__(256) as_read_values_kernel(const double* __restrict__ in, unsigned long long n, int decimals,
                                                             float* __restrict__ out, AsReadList list) {
  for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < n;
       i += (unsigned long long)gridDim.x * blockDim.x)
    as_read_store(out, i, in[i], decimals, list);
}

}  // namespace fs
