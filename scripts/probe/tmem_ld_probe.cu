// tmem_ld_probe.cu -- how fast can an SM's warps read tensor memory?  (measurement tool, not product code)
//   tmem_ld_probe [-iters N]
// One CTA per SM holds all 512 TMEM columns.  Each warp reads 128 columns of its lane quadrant (warp % 4) with
// tcgen05.ld.32x32b.x32, 16 KB per warp and round, in one of two schedules:
//   batched : four loads, then tcgen05.wait::ld  (the reject pass's schedule)
//   serial  : load, wait, load, wait, ...        (one load in flight: the round trip)
// for 1, 2 and 4 warps per SM sub-partition.  Prints bytes per clock per SM (all warps of the CTA, over the slowest
// warp's cycles) and cycles per round and per load of one warp, from clock64 inside the kernel.
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

__device__ __forceinline__ void ld32(uint32_t (&r)[32], uint32_t taddr) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ uint32_t fold(const uint32_t (&r)[32]) {
  uint32_t x = 0;
#pragma unroll
  for (int i = 0; i < 32; i++) x ^= r[i];
  return x;
}

template <bool kSerial>
__global__ void __launch_bounds__(512, 1) probe(int iters, unsigned long long* cycles, uint32_t* sink) {
  __shared__ uint32_t tmem_base;
  const uint32_t warp = threadIdx.x >> 5;
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(
                     (uint32_t)__cvta_generic_to_shared(&tmem_base)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  // lane quadrant warp % 4; warps of one sub-partition read different 128-column ranges
  const uint32_t taddr = tmem_base + (((warp & 3) * 32) << 16) + ((warp >> 2) & 3) * 128;
  uint32_t r0[32], r1[32], r2[32], r3[32], x = 0;
  const long long t0 = clock64();
  for (int it = 0; it < iters; it++) {
    if (kSerial) {
      ld32(r0, taddr); wait_ld(); x ^= fold(r0);
      ld32(r1, taddr + 32); wait_ld(); x ^= fold(r1);
      ld32(r2, taddr + 64); wait_ld(); x ^= fold(r2);
      ld32(r3, taddr + 96); wait_ld(); x ^= fold(r3);
    } else {
      ld32(r0, taddr); ld32(r1, taddr + 32); ld32(r2, taddr + 64); ld32(r3, taddr + 96);
      wait_ld();
      x ^= fold(r0) ^ fold(r1) ^ fold(r2) ^ fold(r3);
    }
  }
  const long long t1 = clock64();
  if ((threadIdx.x & 31) == 0) cycles[blockIdx.x * 16 + warp] = (unsigned long long)(t1 - t0);
  sink[blockIdx.x * blockDim.x + threadIdx.x] = x;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem_base) : "memory");
}

#define CK(x)                                                                        \
  do {                                                                               \
    cudaError_t e = (x);                                                             \
    if (e != cudaSuccess) { printf("%s: %s\n", #x, cudaGetErrorString(e)); return 1; } \
  } while (0)

int main(int argc, char** argv) {
  int iters = 20000;
  for (int i = 1; i + 1 < argc; i += 2)
    if (!strcmp(argv[i], "-iters")) iters = atoi(argv[i + 1]);
  cudaDeviceProp p;
  CK(cudaGetDeviceProperties(&p, 0));
  int clk_khz = 0;
  CK(cudaDeviceGetAttribute(&clk_khz, cudaDevAttrClockRate, 0));
  const int sms = p.multiProcessorCount;
  unsigned long long* cyc;
  uint32_t* sink;
  CK(cudaMalloc(&cyc, sms * 16 * sizeof(unsigned long long)));
  CK(cudaMalloc(&sink, sms * 512 * sizeof(uint32_t)));
  printf("%s, %d SMs, max clock %d MHz, %d iterations of 128 columns per warp\n", p.name, sms, clk_khz / 1000, iters);
  printf("%-8s %-13s %12s %15s %15s %10s\n", "schedule", "warps/SMSP", "B/clk/SM", "clk/round/warp", "clk/load/warp", "ms");
  for (int serial = 0; serial < 2; serial++)
    for (int wps : {1, 2, 4}) {
      const int threads = wps * 4 * 32;
      for (int rep = 0; rep < 2; rep++) {  // first launch warms up
        cudaEvent_t e0, e1;
        CK(cudaEventCreate(&e0));
        CK(cudaEventCreate(&e1));
        CK(cudaEventRecord(e0));
        if (serial) probe<true><<<sms, threads>>>(iters, cyc, sink);
        else probe<false><<<sms, threads>>>(iters, cyc, sink);
        CK(cudaEventRecord(e1));
        CK(cudaGetLastError());
        CK(cudaEventSynchronize(e1));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        if (rep == 0) continue;
        unsigned long long h[16 * 160];
        CK(cudaMemcpy(h, cyc, sms * 16 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        double bpc = 0, per_round = 0;
        for (int b = 0; b < sms; b++) {
          unsigned long long mx = 0;
          for (int w = 0; w < wps * 4; w++) { mx = h[b * 16 + w] > mx ? h[b * 16 + w] : mx; per_round += h[b * 16 + w]; }
          bpc += (double)wps * 4 * iters * 128 * 32 * 4 / mx;
        }
        per_round /= (double)sms * wps * 4 * iters;
        printf("%-8s %-13d %12.1f %15.1f %15.1f %10.3f\n", serial ? "serial" : "batched", wps, bpc / sms, per_round,
               per_round / 4, ms);
        CK(cudaEventDestroy(e0));
        CK(cudaEventDestroy(e1));
      }
    }
  return 0;
}
