// fm_host.h -- host-side state of libfrogmatch shared by fm_api.cu and the fast-path driver.
#pragma once
#include <algorithm>
#include <string>
#include <vector>

#include "../../include/frogmatch.h"
#include "fm_common.cuh"
#include "fm_prep_types.h"

namespace fm {

struct DevBuf {
  void* p = nullptr;
  size_t cap = 0;
  cudaError_t ensure(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
    size_t want = std::max(bytes, (size_t)256);
    cudaError_t e = cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) cudaFree(p);
    p = nullptr;
    cap = 0;
  }
  template <class T> T* as() const { return reinterpret_cast<T*>(p); }
};

enum Phase { kPhScore = 0, kPhRescore, kPhExact, kPhCompact, kPhPrep, kPhBands, kPhTotal, kNumPhases };

struct EventPair {
  cudaEvent_t a, b;
  int phase;
};

struct EventPool {
  std::vector<cudaEvent_t> pool;
  size_t next = 0;
  std::vector<EventPair> spans;
  cudaEvent_t get() {
    if (next == pool.size()) {
      cudaEvent_t e;
      cudaEventCreate(&e);
      pool.push_back(e);
    }
    return pool[next++];
  }
  void reset() { next = 0; spans.clear(); }
  void destroy() {
    for (auto e : pool) cudaEventDestroy(e);
    pool.clear();
    reset();
  }
};

// RAII CUDA-event bracket around a phase on the context stream.
struct Span {
  EventPool* pool;
  cudaStream_t stream;
  EventPair ep;
  Span(EventPool* p, cudaStream_t s, int phase) : pool(p), stream(s) {
    ep.a = pool->get();
    ep.b = pool->get();
    ep.phase = phase;
    cudaEventRecord(ep.a, stream);
  }
  ~Span() {
    cudaEventRecord(ep.b, stream);
    pool->spans.push_back(ep);
  }
};

// Bump allocator for the per-image device tensors: cudaMalloc costs ~0.1-1 ms a call, a 200-image
// group needs 1400 tensors.  Chunks are kept across fm_clear_images() and reused.
struct Arena {
  static constexpr size_t kChunk = (size_t)256 << 20;
  std::vector<DevBuf> chunks;
  size_t cur = 0, off = 0;
  cudaError_t alloc(size_t bytes, void** out) {
    bytes = (bytes + 1023) & ~(size_t)1023;  // operand tiles want 1 KB alignment
    while (cur < chunks.size() && off + bytes > chunks[cur].cap) { cur++; off = 0; }
    if (cur == chunks.size()) {
      chunks.emplace_back();
      cudaError_t e = chunks.back().ensure(std::max(bytes, kChunk));
      if (e != cudaSuccess) { chunks.pop_back(); return e; }
      off = 0;
    }
    *out = static_cast<char*>(chunks[cur].p) + off;
    off += bytes;
    return cudaSuccess;
  }
  void reset() { cur = 0; off = 0; }
  void release() {
    for (auto& c : chunks) c.release();
    chunks.clear();
    reset();
  }
};

// Device tensors of one image (see ImageDev in fm_common.cuh); all of them live in one arena slab.
struct Image {
  bool valid = false;
  uint32_t n = 0, d = 0;
  void* slab = nullptr;
  size_t slab_bytes = 0;
};

}  // namespace fm

struct fm_ctx {
  int device = 0;
  cudaStream_t stream = nullptr, own_stream = nullptr;
  int sm_count = 0;
  std::vector<fm::Image> images;
  std::vector<fm::ImageDev> h_images;
  std::vector<fm::ImageMeta> h_metas;
  fm::DevBuf d_images, d_metas;
  fm::Arena arena;                                            // per-image tensors
  fm::DevBuf s_keys, s_keys_sorted, s_idx, s_idx_sorted, s_norm2, s_sort, s_segs;  // batched-prep scratch (stream-ordered)
  std::vector<uint32_t> dirty;          // images uploaded since the last preparation
  std::vector<fm::PrepSeg> h_segs;
  uint32_t metas_cap = 0;
  bool images_dirty = true;
  uint32_t dim = 0;
  // per-call scratch
  fm::DevBuf d_meta_blob, d_rowres, d_rowdist, d_chunk_count, d_chunk_out, d_chunk_stage, d_chunk_status, d_totals;
  // tags the look-back status words of a one-pass compaction launch (fm_compact.cuh); d_chunk_status is cleared when
  // the buffer is allocated and each time this counter wraps back to 1 (compact_launch in fm_api.cu)
  uint32_t compact_epoch = 0;
  fm::DevBuf d_bands, d_cands, d_redo, d_taskinfo;
  fm::DevBuf d_rowstat, d_surv;  // two-phase scoring: per-row rejection flags; survivor counts / unit prefix / lists
  // fm_debug_set_option("reject_dump", 1): per task of the most recent fm_match, what its reject pass computed
  // (fm_debug_reject_rows); `valid` is false for a task that did not go through the reject pass
  struct RejectRows {
    bool valid = false;
    std::vector<float4> args;        // per sorted row: certified_reject's (a1, a2, |a|^2, eps), NaNs for a row without a band
    std::vector<uint8_t> rowstat;    // 1 = rejected
    std::vector<uint2> bands;        // gate band [x, y) of sorted columns
    std::vector<uint32_t> survivors;  // sorted positions of the surviving rows, ascending
  };
  std::vector<RejectRows> reject_rows;
  // Fraction of tensor-path rows the certified rejection test threw out in the most recent finished call with
  // -d2 < 1 (-1: unknown).  At >= kTwoPhaseMin the next such call scores in two phases from its first batch on.
  double reject_hint = -1.0;
  fm::DevBuf d_all, d_all_tasks;  // -all mode: per-row count / final / carry / offset, per-task totals and bases
  // free lists handed to results (several results may be in flight: FM_FLAG_ASYNC)
  std::vector<fm::DevBuf> out_free, counts_free, dist_free;
  std::vector<std::pair<void*, size_t>> pin_free;  // pinned blocks: DeviceCounters + per-pair counts
  std::vector<fm::EventPool> ev_free;
  fm_result* last = nullptr;  // most recent result of fm_match (cleared when it is freed)
  void* cache_pinned = nullptr;
  size_t cache_pinned_cap = 0;
  unsigned long long* h_pinned = nullptr;  // 8 x u64 scratch for small D2H reads
  fm::EventPool ev_match, ev_prep;
  float ms_prep_acc = 0.f;  // CUDA-event time of the preparation batches since the last fm_clear_images
  fm_stats stats{};
  bool score_attr_set = false;
  bool wide_attr_set = false;  // shared-memory attribute of wide_score_kernel (fm_wide.cuh) set
  std::string err;
};
