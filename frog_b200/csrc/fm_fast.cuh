// fm_fast.cuh -- host-side driver of the tensor-core path: per-image preparation at upload and
// the bands -> score -> rescore -> redo kernel sequence for one batch of tasks.
#pragma once

#include "fm_host.h"
#include "fm_prep.cuh"
#include "fm_reject.cuh"
#include "fm_rescore.cuh"
#include "fm_score.cuh"

namespace fm {

// Device-side counters shared by a fm_match call (one 128-byte block, zeroed per call).
struct DeviceCounters {
  unsigned long long running_total;  // matches compacted so far (fm_compact.cuh)
  unsigned long long scored_cols;    // row x column scores evaluated by score_kernel
  RescoreCounters rescore;           // candidates, redo_rows (redo_rows is reset per batch)
  unsigned long long redo_total;     // redo rows accumulated over batches
  unsigned long long pad[10];
};
static_assert(sizeof(DeviceCounters) == 128, "DeviceCounters layout");

__global__ void fold_redo_kernel(DeviceCounters* c) {
  c->redo_total += c->rescore.redo_rows;
  c->rescore.redo_rows = 0;
}

inline cudaError_t ensure_metas(fm_ctx* c, uint32_t n_images) {
  if (n_images <= c->metas_cap) return cudaSuccess;
  uint32_t cap = std::max<uint32_t>(1024, c->metas_cap * 2);
  while (cap < n_images) cap *= 2;
  DevBuf nb;
  cudaError_t e = nb.ensure((size_t)cap * sizeof(ImageMeta));
  if (e != cudaSuccess) return e;
  if (c->metas_cap) {
    e = cudaMemcpyAsync(nb.p, c->d_metas.p, (size_t)c->metas_cap * sizeof(ImageMeta), cudaMemcpyDeviceToDevice, c->stream);
    if (e != cudaSuccess) return e;
    e = cudaStreamSynchronize(c->stream);
    if (e != cudaSuccess) return e;
  }
  c->d_metas.release();
  c->d_metas = nb;
  c->metas_cap = cap;
  for (size_t i = 0; i < c->h_images.size(); i++) c->h_images[i].meta = c->d_metas.as<ImageMeta>() + i;
  c->images_dirty = true;
  return cudaSuccess;
}

// Build the sorted / FP16 tensors of every image uploaded since the last call (c->dirty), in one
// batch: desc/scale/lap were already copied to the images' slabs, perm/scale_sorted/rowop/colop
// point into them (fm_upload_image laid the slabs out) and the ImageDev table on the device is
// current.
inline cudaError_t fast_prepare_dirty(fm_ctx* c) {
  if (c->dirty.empty()) return cudaSuccess;
  std::sort(c->dirty.begin(), c->dirty.end());
  c->dirty.erase(std::unique(c->dirty.begin(), c->dirty.end()), c->dirty.end());
  std::vector<PrepSeg> segs;
  uint32_t off = 0, blk_keys = 0, blk_pack = 0;
  bool wide = false;  // the images carry the wide operand (d != 48): prep_wide_pack_kernel instead of prep_pack_kernel
  for (uint32_t img : c->dirty) {
    if (img >= c->images.size() || !c->images[img].valid) continue;
    const uint32_t n = c->images[img].n;
    const ImageDev& v = c->h_images[img];
    PrepSeg sg{};
    sg.img = img; sg.n = n; sg.off = off; sg.blk_keys = blk_keys; sg.blk_pack = blk_pack;
    segs.push_back(sg);
    off += n;
    blk_keys += (n + 255) / 256;
    if (v.wideop) wide = true;
    // 16-byte chunks per sorted keypoint: 8 of the K = 64 operands, wide_kpad(d) / 8 of the wide operand
    const uint64_t chunks = (uint64_t)v.n_pad * (v.wideop ? wide_kpad(v.d) / 8u : 8u);
    blk_pack += (uint32_t)((chunks + 255) / 256);
  }
  c->dirty.clear();
  if (segs.empty()) return cudaSuccess;
  if (segs.size() > 65535) return cudaErrorInvalidValue;  // 16 bits of the sort key name the batch segment
  const uint32_t n_segs = (uint32_t)segs.size(), n_tot = std::max(off, 1u);
  cudaError_t e;
  if ((e = c->s_segs.ensure(segs.size() * sizeof(PrepSeg))) != cudaSuccess) return e;
  if ((e = c->s_keys.ensure((size_t)n_tot * 8)) != cudaSuccess) return e;
  if ((e = c->s_keys_sorted.ensure((size_t)n_tot * 8)) != cudaSuccess) return e;
  if ((e = c->s_idx.ensure((size_t)n_tot * 4)) != cudaSuccess) return e;
  if ((e = c->s_idx_sorted.ensure((size_t)n_tot * 4)) != cudaSuccess) return e;
  if ((e = c->s_norm2.ensure((size_t)n_tot * 4)) != cudaSuccess) return e;
  // the segment table is read by kernels after this function returns: stage it in memory that outlives the call
  c->h_segs = segs;
  if ((e = cudaMemcpyAsync(c->s_segs.p, c->h_segs.data(), segs.size() * sizeof(PrepSeg), cudaMemcpyHostToDevice, c->stream)) != cudaSuccess) return e;
  // (pageable source: cudaMemcpyAsync returns once c->h_segs has been staged, so no synchronisation is needed)
  const PrepSeg* d_segs = c->s_segs.as<PrepSeg>();
  const ImageDev* d_images = c->d_images.as<ImageDev>();
  ImageMeta* d_metas = c->d_metas.as<ImageMeta>();
  unsigned long long* keys = c->s_keys.as<unsigned long long>();
  unsigned long long* keys_sorted = c->s_keys_sorted.as<unsigned long long>();
  prep_reset_kernel<<<n_segs, 64, 0, c->stream>>>(d_segs, d_metas);
  if (blk_keys)
    prep_keys_kernel<<<blk_keys, 256, 0, c->stream>>>(d_images, d_segs, n_segs, d_metas, keys, c->s_idx.as<uint32_t>(),
                                                     c->s_norm2.as<float>());
  if (off) {
    int end_bit = 48;
    while (end_bit < 64 && (1u << (end_bit - 48)) < n_segs) end_bit++;
    size_t tmp_bytes = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, keys, keys_sorted, c->s_idx.as<uint32_t>(), c->s_idx_sorted.as<uint32_t>(),
                                    (int)off, 0, end_bit, c->stream);
    if ((e = c->s_sort.ensure(tmp_bytes)) != cudaSuccess) return e;
    e = cub::DeviceRadixSort::SortPairs(c->s_sort.p, tmp_bytes, keys, keys_sorted, c->s_idx.as<uint32_t>(),
                                        c->s_idx_sorted.as<uint32_t>(), (int)off, 0, end_bit, c->stream);
    if (e != cudaSuccess) return e;
  }
  prep_finish_kernel<<<n_segs, 1024, 0, c->stream>>>(d_images, d_segs, d_metas, keys_sorted, c->s_idx_sorted.as<uint32_t>(),
                                                     c->s_norm2.as<float>());
  if (blk_pack && wide) prep_wide_pack_kernel<<<blk_pack, 256, 0, c->stream>>>(d_images, d_segs, n_segs);
  else if (blk_pack) prep_pack_kernel<<<blk_pack, 256, 0, c->stream>>>(d_images, d_segs, n_segs, c->s_norm2.as<float>());
  return cudaGetLastError();
}

// Experiment switches (fm_debug_set_option, frogmatch_debug.h).  Process-wide, explicit calls only: no environment
// variable changes what the production kernel does.
struct DebugOptions {
  int probe = 0;       // 1 | 2: timing-attribution builds of score_kernel (results are garbage)
  int variant = 0;     // experiment builds of score_kernel (results are exact)
  int pre_tiles = -1;  // look-ahead depth override; -1 = kPreTiles
  int surv_cap = -1;   // two-phase scoring: survivor-unit capacity override (tests of the overflow route); -1 = built-in
  int two_phase = -1;  // two-phase scoring: -1 = the library decides (fm_api.cu), 0 = never, 1 = whenever it is applicable
  int compact_v = 3;   // large-batch compaction (fm_compact.cuh): 3 = warp-autonomous pipelined count, 2 = pipelined count with the
                       // block-wide ranking, 1 = the first version (one CTA per chunk, scan with the per-pair counts)
  int reject_dump = 0;  // two-phase scoring: 1 = keep every task's reject-pass output on the host (fm_debug_reject_rows)
  int group_repeat = 0;  // 1 = fm_group_create takes a device more than once (one context per entry): the group path on one GPU
};
inline DebugOptions g_debug;

struct FastBatchArgs {
  const ImageDev* images;
  const Task* tasks;        // device, this batch
  const Task* h_tasks;      // host copy of `tasks` (row_off set)
  uint32_t task0;           // index of the batch's first task in the call
  uint32_t n_tasks;
  uint32_t rows;            // rows in the batch
  const uint32_t* blk_off;  // device: 128-row blocks per task (prefix)
  uint32_t blocks128;
  const uint32_t* unit_off;  // device: score units per task (prefix), already multiplied by segs
  uint32_t units;
  const uint32_t* rj_unit_off;  // device: reject-pass units per task (prefix, kRjUnitRows rows each)
  uint32_t rj_units;
  uint32_t segs;
  float thr, ratio;
  uint32_t* rowres;
  float* rowdist;  // null unless FM_FLAG_DISTANCES
  fm_row* table;   // null unless FM_FLAG_ROW_TABLE: the batch's records (then two_phase is false)
  bool two_phase;  // reject pass + capture pass instead of the single pass (see score_kernel)
  DeviceCounters* counters;
};

// g_debug.reject_dump: copy what the reject pass left for each task of the batch -- its dump, rowstat, bands and
// survivor list -- to c->reject_rows, before anything later in the batch changes rowstat.
inline cudaError_t stash_reject_rows(fm_ctx* c, const FastBatchArgs& a, const float4* dump, const uint8_t* rowstat,
                                     const uint32_t* surv_count, const uint32_t* surv_rows) {
  std::vector<float4> h_dump(a.rows);
  std::vector<uint8_t> h_stat(a.rows);
  std::vector<uint2> h_bands(a.rows);
  std::vector<uint32_t> h_count(a.n_tasks), h_surv(a.rows);
  cudaError_t e;
  if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return e;
  if ((e = cudaMemcpy(h_dump.data(), dump, (size_t)a.rows * sizeof(float4), cudaMemcpyDeviceToHost)) != cudaSuccess) return e;
  if ((e = cudaMemcpy(h_stat.data(), rowstat, a.rows, cudaMemcpyDeviceToHost)) != cudaSuccess) return e;
  if ((e = cudaMemcpy(h_bands.data(), c->d_bands.p, (size_t)a.rows * sizeof(uint2), cudaMemcpyDeviceToHost)) != cudaSuccess) return e;
  if ((e = cudaMemcpy(h_count.data(), surv_count, (size_t)a.n_tasks * sizeof(uint32_t), cudaMemcpyDeviceToHost)) != cudaSuccess) return e;
  if ((e = cudaMemcpy(h_surv.data(), surv_rows, (size_t)a.rows * sizeof(uint32_t), cudaMemcpyDeviceToHost)) != cudaSuccess) return e;
  for (uint32_t t = 0; t < a.n_tasks; t++) {
    const Task& task = a.h_tasks[t];
    if (task.flags & kTaskExact) continue;
    const uint32_t n = c->images[task.row_img].n, r0 = task.row_off;
    auto& st = c->reject_rows[a.task0 + t];
    st.valid = true;
    st.args.assign(h_dump.begin() + r0, h_dump.begin() + r0 + n);
    st.rowstat.assign(h_stat.begin() + r0, h_stat.begin() + r0 + n);
    st.bands.assign(h_bands.begin() + r0, h_bands.begin() + r0 + n);
    st.survivors.assign(h_surv.begin() + r0, h_surv.begin() + r0 + std::min(h_count[t], n));
    std::sort(st.survivors.begin(), st.survivors.end());  // the kernel appends in any order
  }
  return cudaSuccess;
}

inline cudaError_t fast_match_batch(fm_ctx* c, const FastBatchArgs& a) {
  cudaError_t e;
  if ((e = c->d_bands.ensure((size_t)a.rows * sizeof(uint2))) != cudaSuccess) return e;
  if ((e = c->d_cands.ensure((size_t)a.rows * a.segs * kTopK * sizeof(Cand))) != cudaSuccess) return e;
  if ((e = c->d_redo.ensure((size_t)a.rows * sizeof(uint2))) != cudaSuccess) return e;
  // two-phase scoring: survivor units the capture pass is launched with (an upper bound; a hundred times what the
  // >= 99 %-rejection regime needs, and never more than there could be)
  const uint32_t cap_units = g_debug.surv_cap > 0 ? (uint32_t)g_debug.surv_cap
                                                  : std::min<uint32_t>(a.units + a.n_tasks, std::max<uint32_t>(1024u, 4u * a.n_tasks));
  if (a.two_phase) {
    if ((e = c->d_rowstat.ensure((size_t)a.rows)) != cudaSuccess) return e;
    if ((e = c->d_surv.ensure(((size_t)a.rows + 2 * (size_t)a.n_tasks + 2) * sizeof(uint32_t))) != cudaSuccess) return e;
  }
  if (!c->score_attr_set) {
    // two CTAs per SM: ask for the full shared-memory carveout
    auto prep = [](auto kern) -> cudaError_t {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kScoreSmemBytes);
      if (e != cudaSuccess) return e;
      return cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
    };
    if ((e = prep(score_kernel<false, 0, 0>)) != cudaSuccess) return e;
    if ((e = prep(score_kernel<false, 0, 2>)) != cudaSuccess) return e;
    if ((e = prep(score_kernel<false, 1, 0>)) != cudaSuccess) return e;
    if ((e = prep(score_kernel<false, 2, 0>)) != cudaSuccess) return e;
    if ((e = prep(score_kernel<true, 0, 0>)) != cudaSuccess) return e;
    // the reject pass: one CTA per SM
    if ((e = cudaFuncSetAttribute(reject_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRjSmemBytes)) != cudaSuccess) return e;
    if ((e = cudaFuncSetAttribute(reject_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kRjSmemBytes)) != cudaSuccess) return e;
    c->score_attr_set = true;
  }
  bool two_phase_ran = false;
  {
    Span sp(&c->ev_match, c->stream, kPhBands);
    bands_kernel<<<a.blocks128, 128, 0, c->stream>>>(a.images, a.tasks, a.blk_off, a.n_tasks, c->d_bands.as<uint2>());
  }
  {
    Span sp(&c->ev_match, c->stream, kPhScore);
    // fm_debug_set_option("probe" | "variant" | "pre_tiles") selects experiment builds of the kernel (frogmatch_debug.h);
    // the defaults are the production kernel
    const int probe = g_debug.probe, var = g_debug.variant;
    const uint32_t pre_tiles = g_debug.pre_tiles >= 0 ? (uint32_t)g_debug.pre_tiles : kPreTiles;
    auto kern = probe == 1 ? score_kernel<false, 1, 0> : probe == 2 ? score_kernel<false, 2, 0> : score_kernel<false, 0, 0>;
    (void)var;
    uint8_t* rowstat = a.two_phase ? c->d_rowstat.as<uint8_t>() : nullptr;
    if (a.two_phase && probe == 0) {
      // d_surv: survivor counts per task | survivor-unit prefix per task (+1) | survivor lists, laid out like the rows
      uint32_t* surv_count = c->d_surv.as<uint32_t>();
      uint32_t* surv_off = surv_count + a.n_tasks;
      uint32_t* surv_rows = surv_off + a.n_tasks + 1;
      if ((e = cudaMemsetAsync(surv_count, 0, (size_t)a.n_tasks * sizeof(uint32_t), c->stream)) != cudaSuccess) return e;
      // persistent: one CTA per SM walks the units
      const uint32_t grid = std::min<uint32_t>(a.rj_units, (uint32_t)c->sm_count);
      if (g_debug.reject_dump) {
        DevBuf dump;
        if ((e = dump.ensure((size_t)a.rows * sizeof(float4))) != cudaSuccess) return e;
        if ((e = cudaMemsetAsync(dump.p, 0xFF, (size_t)a.rows * sizeof(float4), c->stream)) != cudaSuccess) return e;
        reject_kernel<true><<<grid, kRjThreads, kRjSmemBytes, c->stream>>>(
            a.images, a.tasks, a.rj_unit_off, a.n_tasks, a.rj_units, c->d_bands.as<uint2>(), &a.counters->scored_cols, a.thr,
            a.ratio, rowstat, surv_count, surv_rows, dump.as<float4>());
        if ((e = cudaGetLastError()) == cudaSuccess) e = stash_reject_rows(c, a, dump.as<float4>(), rowstat, surv_count, surv_rows);
        dump.release();
        if (e != cudaSuccess) return e;
      } else {
        reject_kernel<false><<<grid, kRjThreads, kRjSmemBytes, c->stream>>>(
            a.images, a.tasks, a.rj_unit_off, a.n_tasks, a.rj_units, c->d_bands.as<uint2>(), &a.counters->scored_cols, a.thr,
            a.ratio, rowstat, surv_count, surv_rows, nullptr);
      }
      surv_plan_kernel<<<1, 1024, 0, c->stream>>>(surv_count, a.n_tasks, surv_off, cap_units, a.tasks, surv_rows, rowstat,
                                                  c->d_redo.as<uint2>(), &a.counters->rescore.redo_rows);
      score_kernel<false, 0, 2><<<cap_units, kScoreThreads, kScoreSmemBytes, c->stream>>>(
          a.images, a.tasks, surv_off, a.n_tasks, 1u, c->d_bands.as<uint2>(), c->d_cands.as<Cand>(),
          &a.counters->scored_cols, nullptr, 0, 0, pre_tiles, a.thr, a.ratio, rowstat, surv_count, surv_rows);
      c->stats.kernel_launches += 2;
      c->stats.two_phase_batches += 1;
    } else {
      rowstat = nullptr;
      kern<<<a.units, kScoreThreads, kScoreSmemBytes, c->stream>>>(
          a.images, a.tasks, a.unit_off, a.n_tasks, a.segs, c->d_bands.as<uint2>(), c->d_cands.as<Cand>(),
          &a.counters->scored_cols, nullptr, 0, 0, pre_tiles, a.thr, a.ratio, nullptr, nullptr, nullptr);
    }
    two_phase_ran = rowstat != nullptr;
  }
  {
    Span sp(&c->ev_match, c->stream, kPhRescore);
    // two-phase: rows the reject pass threw out are not touched by the rescoring kernel at all
    if (two_phase_ran && (e = cudaMemsetAsync(a.rowres, 0xFF, (size_t)a.rows * sizeof(uint32_t), c->stream)) != cudaSuccess) return e;
    rescore_kernel<<<a.blocks128, 128, 0, c->stream>>>(a.images, a.tasks, a.blk_off, a.n_tasks, a.segs,
                                                       c->d_cands.as<Cand>(), a.thr, a.ratio, a.rowres,
                                                       c->d_redo.as<uint2>(), &a.counters->rescore, a.rowdist,
                                                       two_phase_ran ? c->d_rowstat.as<uint8_t>() : nullptr, a.table);
    exact_rows_kernel<<<c->sm_count, kRedoThreads, 0, c->stream>>>(a.images, a.tasks, c->d_bands.as<uint2>(), c->d_redo.as<uint2>(),
                                                             &a.counters->rescore, a.thr, a.ratio, a.rowres, a.rowdist, a.table);
    fold_redo_kernel<<<1, 1, 0, c->stream>>>(a.counters);
  }
  c->stats.kernel_launches += 5;
  c->stats.score_launches += 1;
  return cudaGetLastError();
}

}  // namespace fm
