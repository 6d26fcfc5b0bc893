// fm_select.cuh -- fm_result_select: a finished call re-decided at other thresholds from its row table
// (FM_FLAG_ROW_TABLE, include/frogmatch.h).
//
// The reference's accept test (match.cpp:320-321, accept_rule) reads three values per row -- d1, d2 and the nearest
// column -- and none of them depends on -d or -d2, so the table the decision sites wrote (put_row) decides a row at any
// thresholds.  One thread per row turns a batch's records into the rowres / rowdist arrays the decision sites would
// have written at (thr, ratio); the unchanged compaction (fm_compact.cuh) then runs on the call's own chunk records.
// HBM-bound: 12 B read, 4 B (+ 4 B with distances) written per row.
#pragma once
#include "fm_common.cuh"
#include "fm_exact.cuh"

namespace fm {

constexpr int kSelectThreads = 256;

__global__ void __launch_bounds__(kSelectThreads)
select_kernel(const fm_row* __restrict__ rows, uint32_t n_rows, float thr, float ratio, uint32_t* __restrict__ rowres,
              float* __restrict__ rowdist) {
  for (uint32_t i = blockIdx.x * kSelectThreads + threadIdx.x; i < n_rows; i += gridDim.x * kSelectThreads) {
    const float d1 = __ldg(&rows[i].d1), d2 = __ldg(&rows[i].d2);
    const uint32_t nearest = __ldg(&rows[i].nearest);
    // (nearest == kNone means d1 == FLT_MAX, which accept_rule never accepts below dist = 1.8e19)
    rowres[i] = nearest != kNone && accept_rule(d1, d2, thr, ratio) ? nearest : kNone;
    if (rowdist) rowdist[i] = d1;
  }
}

}  // namespace fm
