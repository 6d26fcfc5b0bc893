// fm_api.cu -- C ABI of libfrogmatch.so (include/frogmatch.h): context, keypoint upload,
// task batching and kernel orchestration.  sm_100a only; there is no CPU fallback.
#include <cstdio>
#include <cstring>
#include <new>

#include "../../include/frogmatch.h"
#include "../../include/frogmatch_debug.h"
#include "fm_all.cuh"
#include "fm_compact.cuh"
#include "fm_exact.cuh"
#include "fm_fast.cuh"
#include "fm_generic.cuh"
#include "fm_group.cuh"
#include "fm_host.h"
#include "fm_links.cuh"
#include "fm_select.cuh"
#include "fm_shard.h"
#include "fm_wide.cuh"

using namespace fm;

// One batch of a row-table call, as fm_result_select needs it: its rows' place in the table and its chunk records.
struct SelectBatch {
  uint64_t row0;  // first table row of the batch
  uint32_t rows, chunk0, chunks;  // chunk0: first record in fm_result::sel_chunks
};

// One member's share of a group result (fm_group_match): the member's own result of its shard, whose device buffers go
// back to the member's free lists once the gather is queued (its pinned block and events stay until the group result is
// complete), and the member-side scratch of the gather.
struct GroupPart {
  fm_result* sub = nullptr;
  uint32_t member = 0;            // the member's index in the group
  std::vector<uint32_t> idx;      // submission indices of the member's pairs, in its call's order
  DevBuf scratch;                 // member device: local offsets (n + 1 u64) | global positions (n u32)
  void* pin = nullptr;            // member's pinned staging of the global positions
  size_t pin_cap = 0;
};

struct fm_result {
  fm_ctx* ctx = nullptr;
  size_t n_pairs = 0;
  uint64_t total = 0;
  uint32_t flags = 0;
  float ratio = 1.f;
  bool d48 = false;  // a d = 48 call: only these feed the two-phase hint (reject_hint)
  std::vector<uint32_t> counts;
  std::vector<uint64_t> offsets;
  DevBuf d_out, d_counts, d_dist;
  uint32_t* h_pairs = nullptr;  // pinned
  size_t h_cap = 0;
  float* h_dist = nullptr;  // pinned, FM_FLAG_DISTANCES only
  bool fetched = false;
  // completion: the call's DeviceCounters and per-pair counts land in a pinned block, `done` fires behind them
  void* h_block = nullptr;
  size_t h_block_cap = 0;
  cudaEvent_t done = nullptr;
  bool waited = false;
  EventPool ev;     // this call's phase brackets (and `done`)
  fm_stats stats{};  // launch-side counters; device counters and event times are filled in by finalize()
  uint64_t slots = 0;  // matches d_out is sized for: the call's outer-loop rows (-all: its exact total)
  // group results (fm_group_match): one part per member that had pairs; the lead's submission-order offsets
  std::vector<GroupPart> parts;
  DevBuf d_goff;
  fm_group* group = nullptr;  // the group of a group result (fm_result_select gathers through it)
  // FM_FLAG_ROW_TABLE: the table, and the host records fm_result_select compacts with (a group result holds no table of
  // its own: each part's result holds its share's)
  bool table = false;
  DevBuf d_table;                         // one fm_row per outer-loop row, task after task
  std::vector<uint64_t> row_off;          // n_pairs + 1: pair p's first row, submission order over the whole call
  std::vector<SelectBatch> sel_batches;   // the call's batches
  std::vector<ChunkDesc> sel_chunks;      // their compaction chunk records, batch after batch
  std::vector<uint32_t> pair_part, pair_local;  // group result: pair p's part and its index in that part's call
};

struct fm_links {
  fm_ctx* ctx = nullptr;
  uint64_t total = 0;        // half-links
  uint32_t n_points = 0;     // points of all images of the context
  std::vector<uint64_t> point_base;  // per image index: global id of its point 0 (n_images + 1 entries)
  DevBuf d_off, d_links;
  unsigned long long* h_off = nullptr;  // pinned, after fm_links_fetch
  uint32_t* h_links = nullptr;
  float ms_build = 0.f;
};

namespace {

thread_local std::string g_create_error;

int fail(fm_ctx* c, int code, const std::string& msg) {
  if (c) c->err = msg; else g_create_error = msg;
  return code;
}

int cuda_fail(fm_ctx* c, cudaError_t e, const char* what) {
  return fail(c, e == cudaErrorMemoryAllocation ? FM_ERR_NOMEM : FM_ERR_CUDA, std::string(what) + ": " + cudaGetErrorString(e));
}

#define FM_CUDA(ctx, expr)                                     \
  do {                                                         \
    cudaError_t e__ = (expr);                                  \
    if (e__ != cudaSuccess) return cuda_fail((ctx), e__, #expr); \
  } while (0)

// Upload the ImageDev table, prepare the images uploaded since the last call (one batch of
// kernels) and read the per-image metas (flags, class tables) back.  prep_queue queues the table and the kernels;
// prep_finish reads the metas back (a pageable copy: it waits for the stream).  A group queues every member's
// preparation before it waits for any, so that its members prepare at the same time.
int prep_queue(fm_ctx* c) {
  if (!c->images_dirty) return FM_OK;
  const size_t n = c->h_images.size();
  FM_CUDA(c, cudaSetDevice(c->device));
  FM_CUDA(c, c->d_images.ensure(std::max<size_t>(1, n) * sizeof(ImageDev)));
  c->h_metas.assign(n, ImageMeta{});
  if (n) {
    FM_CUDA(c, cudaMemcpyAsync(c->d_images.p, c->h_images.data(), n * sizeof(ImageDev), cudaMemcpyHostToDevice, c->stream));
    Span sp(&c->ev_prep, c->stream, kPhPrep);
    cudaError_t e = fast_prepare_dirty(c);
    if (e != cudaSuccess) return cuda_fail(c, e, "image preparation");
  }
  return FM_OK;
}

int prep_finish(fm_ctx* c) {
  if (!c->images_dirty) return FM_OK;
  const size_t n = c->h_images.size();
  FM_CUDA(c, cudaSetDevice(c->device));
  if (n) {
    FM_CUDA(c, cudaMemcpyAsync(c->h_metas.data(), c->d_metas.p, n * sizeof(ImageMeta), cudaMemcpyDeviceToHost, c->stream));
    FM_CUDA(c, cudaStreamSynchronize(c->stream));
    // the bracket above has completed: fold it into the running sum and recycle its events (a long-lived context that
    // re-uploads images without ever clearing must not accumulate events)
    for (auto& sp : c->ev_prep.spans) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) c->ms_prep_acc += ms;
    }
    c->ev_prep.reset();
  }
  c->images_dirty = false;
  return FM_OK;
}

int sync_images(fm_ctx* c) {
  int rc = prep_queue(c);
  return rc != FM_OK ? rc : prep_finish(c);
}

// Small free lists so that several results can be in flight (FM_FLAG_ASYNC) without a cudaMalloc /
// cudaFree (a device-wide synchronisation) per call.
DevBuf take_buf(std::vector<DevBuf>& list, size_t bytes) {
  int best = -1;
  for (size_t i = 0; i < list.size(); i++)
    if (list[i].cap >= bytes && (best < 0 || list[i].cap < list[best].cap)) best = (int)i;
  if (best < 0 && !list.empty()) {  // none fits: grow the largest
    best = 0;
    for (size_t i = 1; i < list.size(); i++)
      if (list[i].cap > list[best].cap) best = (int)i;
  }
  DevBuf b;
  if (best >= 0) {
    b = list[best];
    list.erase(list.begin() + best);
  }
  return b;
}

void give_buf(std::vector<DevBuf>& list, DevBuf& b) {
  if (!b.p) return;
  if (list.size() < 4) list.push_back(b);
  else cudaFree(b.p);
  b = DevBuf{};
}

// give_buf for a buffer that queued work still reads: it goes back only when the list has room, and otherwise stays
// with its result until fm_result_free (a cudaFree now would wait for the whole device).
void give_buf_queued(std::vector<DevBuf>& list, DevBuf& b) {
  if (b.p && list.size() < 4) give_buf(list, b);
}

cudaError_t take_pinned(fm_ctx* c, size_t bytes, void** out, size_t* cap) {
  for (size_t i = 0; i < c->pin_free.size(); i++)
    if (c->pin_free[i].second >= bytes) {
      *out = c->pin_free[i].first;
      *cap = c->pin_free[i].second;
      c->pin_free.erase(c->pin_free.begin() + i);
      return cudaSuccess;
    }
  const size_t want = std::max<size_t>(bytes + bytes / 4, 4096);
  cudaError_t e = cudaMallocHost(out, want);
  if (e == cudaSuccess) *cap = want;
  return e;
}

void give_pinned(fm_ctx* c, void* p, size_t cap) {
  if (!p) return;
  if (c->pin_free.size() < 8) c->pin_free.emplace_back(p, cap);
  else cudaFreeHost(p);
}

// Complete a result: wait for its `done` event, then read the totals, per-pair counts and phase
// times the device left in the pinned block / the call's events.
int finalize(fm_result* r) {
  if (r->waited) return FM_OK;
  fm_ctx* c = r->ctx;
  FM_CUDA(c, cudaSetDevice(c->device));
  FM_CUDA(c, cudaEventSynchronize(r->done));
  const DeviceCounters* hc = static_cast<const DeviceCounters*>(r->h_block);
  const uint32_t* hcounts = reinterpret_cast<const uint32_t*>(static_cast<const char*>(r->h_block) + sizeof(DeviceCounters));
  r->total = hc->running_total;
  r->counts.assign(hcounts, hcounts + r->n_pairs);
  r->offsets.assign(r->n_pairs + 1, 0);
  for (size_t p = 0; p < r->n_pairs; p++) r->offsets[p + 1] = r->offsets[p] + r->counts[p];
  r->stats.scored_pairs = hc->scored_cols;
  r->stats.candidates = hc->rescore.candidates;
  r->stats.rows_rejected_early = hc->rescore.rejected_early;
  if (r->ratio < 1.f && r->d48 && r->stats.rows > r->stats.rows_exact)
    c->reject_hint = (double)hc->rescore.rejected_early / (double)(r->stats.rows - r->stats.rows_exact);
  r->stats.rows_exact += hc->redo_total;
  float acc[kNumPhases] = {0};
  for (auto& s : r->ev.spans) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, s.a, s.b) == cudaSuccess) acc[s.phase] += ms;
  }
  r->stats.ms_total = acc[kPhTotal];
  r->stats.ms_score = acc[kPhScore];
  r->stats.ms_rescore = acc[kPhRescore] + acc[kPhBands];
  r->stats.ms_exact = acc[kPhExact];
  r->stats.ms_compact = acc[kPhCompact];
  if (!r->parts.empty()) {
    // a group result: counters summed over the members' calls, each phase time the longest member's
    fm_stats s{};
    for (auto& gp : r->parts) {
      fm_result* q = gp.sub;
      if (finalize(q) != FM_OK) return fail(c, FM_ERR_CUDA, "fm_group_match: device " + std::to_string(q->ctx->device) + ": " + q->ctx->err);
      const fm_stats& t = q->stats;
      s.descriptor_pairs += t.descriptor_pairs;
      s.scored_pairs += t.scored_pairs;
      s.rows += t.rows;
      s.rows_exact += t.rows_exact;
      s.candidates += t.candidates;
      s.kernel_launches += t.kernel_launches;
      s.score_launches += t.score_launches;
      s.rows_rejected_early += t.rows_rejected_early;
      s.two_phase_batches += t.two_phase_batches;
      s.ms_total = std::max(s.ms_total, t.ms_total);
      s.ms_score = std::max(s.ms_score, t.ms_score);
      s.ms_rescore = std::max(s.ms_rescore, t.ms_rescore);
      s.ms_exact = std::max(s.ms_exact, t.ms_exact);
      s.ms_compact = std::max(s.ms_compact, t.ms_compact);
    }
    r->stats = s;
  }
  r->waited = true;
  const float ms_prep = c->stats.ms_prep;
  c->stats = r->stats;
  c->stats.ms_prep = ms_prep;
  if (r->offsets[r->n_pairs] != r->total)
    return fail(c, FM_ERR_CUDA, "fm_match: internal error, per-pair counts do not sum to the compacted total");
  return FM_OK;
}

// The common end of a call on one context: totals and per-pair counts to the result's pinned block, `done` behind them,
// and the call's counters and event brackets handed to the result.
cudaError_t queue_tail(fm_ctx* c, fm_result* r) {
  cudaError_t e = cudaMemcpyAsync(r->h_block, c->d_totals.p, sizeof(DeviceCounters), cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess && r->n_pairs)
    e = cudaMemcpyAsync(static_cast<char*>(r->h_block) + sizeof(DeviceCounters), r->d_counts.p, r->n_pairs * sizeof(uint32_t),
                        cudaMemcpyDeviceToHost, c->stream);
  if (e != cudaSuccess) return e;
  r->done = c->ev_match.get();
  if ((e = cudaEventRecord(r->done, c->stream)) != cudaSuccess) return e;
  r->stats = c->stats;
  r->ev = std::move(c->ev_match);
  c->ev_match = EventPool{};
  return cudaSuccess;
}

struct Batch {
  uint32_t t0, t1, rows, blocks, chunks, units;
  uint32_t rj_units;  // reject-pass units (kRjUnitRows rows each, fast tasks only)
  size_t cursor;      // first entry of this batch in the concatenated prefix arrays
  bool any_exact, any_fast;
};

// The look-back status words of the one-pass compaction kernel: fresh memory may hold anything, so it is cleared once
// here; afterwards the launch epoch tells stale words from current ones (and compact_launch clears the words again
// whenever the epoch counter wraps).
cudaError_t ensure_chunk_status(fm_ctx* c) {
  if (c->d_chunk_status.p) return cudaSuccess;
  cudaError_t e = c->d_chunk_status.ensure((size_t)kOnePassChunks * sizeof(unsigned long long));
  if (e != cudaSuccess) return e;
  return cudaMemsetAsync(c->d_chunk_status.p, 0, c->d_chunk_status.cap, c->stream);
}

// Compaction of one batch (fm_compact.cuh) on the context stream: `ca` carries the batch's chunks, rows and outputs;
// the context's scratch (d_chunk_count / d_chunk_out / d_chunk_stage, sized for ca.n_chunks, and d_chunk_status) and
// its epoch counter are filled in here.  `path` is an FM_COMPACT_* value (include/frogmatch_debug.h): fm_match passes
// FM_COMPACT_AUTO, fm_debug_compact whatever the test asks for.  Returns the number of kernel launches.
uint32_t compact_launch(fm_ctx* c, CompactArgs ca, bool want_dist, int path) {
  ca.chunk_count = c->d_chunk_count.as<uint32_t>();
  ca.chunk_out = c->d_chunk_out.as<unsigned long long>();
  ca.stage = c->d_chunk_stage.as<uint2>();
  if (path == FM_COMPACT_AUTO) path = ca.n_chunks <= kOnePassChunks ? FM_COMPACT_ONE : FM_COMPACT_THREE;
  if (path == FM_COMPACT_ONE || path == FM_COMPACT_LOOKALL) {
    ca.status = c->d_chunk_status.as<unsigned long long>();
    const uint32_t prev = c->compact_epoch;
    c->compact_epoch = (c->compact_epoch % 0x3FFFFFFEu) + 1u;  // 1 .. 2^30 - 2: never the cleared value 0
    // Back at epoch 1 after a wrap: words an earlier epoch-1 launch left past the chunks later launches rewrote would
    // pass for current ones.  (A failure here is left to the caller's cudaGetLastError.)
    if (c->compact_epoch == 1u && prev != 0u) cudaMemsetAsync(c->d_chunk_status.p, 0, c->d_chunk_status.cap, c->stream);
    ca.epoch = c->compact_epoch;
    if (path == FM_COMPACT_LOOKALL) {
      if (want_dist) compact_onepass_kernel<true, true><<<ca.n_chunks, kCompactThreads, 0, c->stream>>>(ca);
      else compact_onepass_kernel<false, true><<<ca.n_chunks, kCompactThreads, 0, c->stream>>>(ca);
    } else {
      if (want_dist) compact_onepass_kernel<true><<<ca.n_chunks, kCompactThreads, 0, c->stream>>>(ca);
      else compact_onepass_kernel<false><<<ca.n_chunks, kCompactThreads, 0, c->stream>>>(ca);
    }
    return 1;
  }
  const uint32_t grid = std::min<uint32_t>(ca.n_chunks, (uint32_t)c->sm_count * 8u);  // grid-stride over the chunks
  if (g_debug.compact_v >= 2) {
    // persistent, software-pipelined count pass: three CTAs per SM, each with the next chunk's rows in flight
    const uint32_t grid_count = std::min<uint32_t>(ca.n_chunks, (uint32_t)c->sm_count * 3u);
    if (want_dist) {
      if (g_debug.compact_v >= 3) compact_count3_kernel<true><<<grid_count, kCompactThreads, 0, c->stream>>>(ca);
      else compact_count2_kernel<true><<<grid_count, kCompactThreads, 0, c->stream>>>(ca);
      compact_scan2_kernel<<<1, 1024, 0, c->stream>>>(ca);
      compact_scatter2_kernel<true><<<grid, kCompactThreads, 0, c->stream>>>(ca);
    } else {
      if (g_debug.compact_v >= 3) compact_count3_kernel<false><<<grid_count, kCompactThreads, 0, c->stream>>>(ca);
      else compact_count2_kernel<false><<<grid_count, kCompactThreads, 0, c->stream>>>(ca);
      compact_scan2_kernel<<<1, 1024, 0, c->stream>>>(ca);
      compact_scatter2_kernel<false><<<grid, kCompactThreads, 0, c->stream>>>(ca);
    }
  } else if (want_dist) {
    compact_count_kernel<true><<<ca.n_chunks, kCompactThreads, 0, c->stream>>>(ca);  // (one CTA per chunk measured faster here)
    compact_scan_kernel<<<1, 1024, 0, c->stream>>>(ca);
    compact_scatter_kernel<true><<<grid, kCompactThreads, 0, c->stream>>>(ca);
  } else {
    compact_count_kernel<false><<<ca.n_chunks, kCompactThreads, 0, c->stream>>>(ca);
    compact_scan_kernel<<<1, 1024, 0, c->stream>>>(ca);
    compact_scatter_kernel<false><<<grid, kCompactThreads, 0, c->stream>>>(ca);
  }
  return 3;
}

}  // namespace

extern "C" {

const char* fm_version(void) { return "frogmatch 0.1 (sm_100a: tcgen05 + TMA bulk copy)"; }

int fm_device_count(int* n) {
  if (!n) return FM_ERR_INVALID;
  *n = 0;
  int k = 0;
  cudaError_t e = cudaGetDeviceCount(&k);
  if (e != cudaSuccess) return cuda_fail(nullptr, e, "fm_device_count");
  *n = k;
  return FM_OK;
}

int fm_create(int device, fm_ctx** out) {
  if (!out) return fail(nullptr, FM_ERR_INVALID, "fm_create: out is NULL");
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return fail(nullptr, FM_ERR_CUDA, std::string("fm_create: no CUDA device (") + cudaGetErrorString(e) +
                                          "); libfrogmatch has no CPU fallback");
  if (device < 0 || device >= n_dev) return fail(nullptr, FM_ERR_INVALID, "fm_create: device index out of range");
  cudaDeviceProp prop{};
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess)
    return cuda_fail(nullptr, e, "fm_create");
  if (prop.major != 10)
    return fail(nullptr, FM_ERR_UNSUPPORTED, "fm_create: device is sm_" + std::to_string(prop.major) +
                                                 std::to_string(prop.minor) + ", this library is built for sm_100a only");
  fm_ctx* c = new (std::nothrow) fm_ctx();
  if (!c) return fail(nullptr, FM_ERR_NOMEM, "fm_create: out of host memory");
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking)) != cudaSuccess ||
      (e = cudaMallocHost(reinterpret_cast<void**>(&c->h_pinned), 256)) != cudaSuccess) {
    if (c->own_stream) cudaStreamDestroy(c->own_stream);
    delete c;
    return cuda_fail(nullptr, e, "fm_create");
  }
  c->stream = c->own_stream;
  *out = c;
  return FM_OK;
}

void fm_destroy(fm_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  cudaStreamSynchronize(c->stream);
  c->arena.release();
  DevBuf* bufs[] = {&c->s_keys, &c->s_keys_sorted, &c->s_idx, &c->s_idx_sorted, &c->s_norm2, &c->s_sort, &c->s_segs, &c->d_images, &c->d_metas, &c->d_meta_blob, &c->d_rowres, &c->d_rowdist, &c->d_chunk_count, &c->d_chunk_out, &c->d_chunk_stage, &c->d_chunk_status,
                    &c->d_totals, &c->d_bands, &c->d_cands, &c->d_redo, &c->d_taskinfo, &c->d_rowstat, &c->d_surv, &c->d_all, &c->d_all_tasks};
  for (auto* b : bufs) b->release();
  for (auto& b : c->out_free) b.release();
  for (auto& b : c->counts_free) b.release();
  for (auto& b : c->dist_free) b.release();
  for (auto& pb : c->pin_free) cudaFreeHost(pb.first);
  if (c->cache_pinned) cudaFreeHost(c->cache_pinned);
  if (c->h_pinned) cudaFreeHost(c->h_pinned);
  c->ev_match.destroy();
  for (auto& e : c->ev_free) e.destroy();
  c->ev_prep.destroy();
  cudaStreamDestroy(c->own_stream);
  delete c;
}

const char* fm_last_error(const fm_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int fm_set_stream(fm_ctx* c, void* s) {
  if (!c) return FM_ERR_INVALID;
  FM_CUDA(c, cudaSetDevice(c->device));
  FM_CUDA(c, cudaStreamSynchronize(c->stream));
  c->stream = s ? reinterpret_cast<cudaStream_t>(s) : c->own_stream;
  return FM_OK;
}

int fm_synchronize(fm_ctx* c) {
  if (!c) return FM_ERR_INVALID;
  FM_CUDA(c, cudaSetDevice(c->device));
  FM_CUDA(c, cudaStreamSynchronize(c->stream));
  return FM_OK;
}

int fm_clear_images(fm_ctx* c) {
  if (!c) return FM_ERR_INVALID;
  for (auto& im : c->images) { im.valid = false; im.slab = nullptr; im.slab_bytes = 0; }
  c->dirty.clear();
  c->images_dirty = true;
  c->dim = 0;
  // the arena is handed out again right away: everything that still reads the old tensors must have finished
  FM_CUDA(c, cudaSetDevice(c->device));
  FM_CUDA(c, cudaStreamSynchronize(c->stream));
  c->arena.reset();
  c->ev_prep.reset();
  c->ms_prep_acc = 0.f;
  return FM_OK;
}

int fm_image_points(const fm_ctx* c, uint32_t img, uint32_t* n) {
  if (!c || !n || img >= c->images.size() || !c->images[img].valid) return FM_ERR_INVALID;
  *n = c->images[img].n;
  return FM_OK;
}

int fm_upload_image(fm_ctx* c, uint32_t img, const float* desc, const float* scale, const float* lap, uint32_t n,
                    uint32_t d) {
  if (!c) return FM_ERR_INVALID;
  if ((n && (!desc || !scale || !lap)) || d == 0) return fail(c, FM_ERR_INVALID, "fm_upload_image: null input or d == 0");
  if (d > (1u << 20)) return fail(c, FM_ERR_UNSUPPORTED, "fm_upload_image: descriptor length above 2^20 is not supported");
  if (img >= 65536u) return fail(c, FM_ERR_INVALID, "fm_upload_image: image index above 65535 (pairs.bin ids are u16, match.cpp:735)");
  if (c->dim != 0 && c->dim != d) return fail(c, FM_ERR_INVALID, "fm_upload_image: all images of a context must share d");
  FM_CUDA(c, cudaSetDevice(c->device));
  c->dim = d;
  if (img >= c->images.size()) c->images.resize(img + 1);
  if (img >= c->h_images.size()) c->h_images.resize(img + 1, ImageDev{});
  Image& im = c->images[img];
  // One slab per image: desc | scale | lap | perm | scale_sorted | norm2_sorted | rowop | colop | wideop (1 KB aligned pieces).
  auto pad = [](size_t x) { return (x + 1023) & ~(size_t)1023; };
  const uint32_t n_pad = (n + 255u) & ~255u;  // rows are consumed 256 at a time, columns 64
  const size_t b_desc = pad((size_t)n * d * sizeof(float)), b_vec = pad((size_t)std::max(n, 1u) * sizeof(float));
  const size_t b_op = d == (uint32_t)kD ? pad((size_t)n_pad * kKPad * sizeof(__half)) : 0;
  // d != 48: one operand image of wide_kpad(d) halves per keypoint (fm_wide.cuh); longer descriptors have none
  const bool wide = d != (uint32_t)kD && d <= (uint32_t)kWideMaxD;
  const size_t b_wide = wide ? pad((size_t)n_pad * wide_kpad(d) * sizeof(__half)) : 0;
  const size_t need = b_desc + 5 * b_vec + 2 * b_op + b_wide + 1024;
  if (!im.slab || im.slab_bytes < need) {  // a re-upload that fits reuses the image's slab
    void* p = nullptr;
    FM_CUDA(c, c->arena.alloc(need, &p));
    im.slab = p;
    im.slab_bytes = need;
  }
  char* base = static_cast<char*>(im.slab);
  float* d_desc = reinterpret_cast<float*>(base);
  float* d_scale = reinterpret_cast<float*>(base + b_desc);
  float* d_lap = reinterpret_cast<float*>(base + b_desc + b_vec);
  if (n) {
    FM_CUDA(c, cudaMemcpyAsync(d_desc, desc, (size_t)n * d * sizeof(float), cudaMemcpyDefault, c->stream));
    FM_CUDA(c, cudaMemcpyAsync(d_scale, scale, (size_t)n * sizeof(float), cudaMemcpyDefault, c->stream));
    FM_CUDA(c, cudaMemcpyAsync(d_lap, lap, (size_t)n * sizeof(float), cudaMemcpyDefault, c->stream));
  }
  im.valid = true;
  im.n = n;
  im.d = d;
  ImageDev& v = c->h_images[img];
  v = ImageDev{};
  v.desc = d_desc;
  v.scale = d_scale;
  v.lap = d_lap;
  v.n = n;
  v.d = d;
  v.n_pad = n_pad;
  v.perm = reinterpret_cast<uint32_t*>(base + b_desc + 2 * b_vec);
  v.scale_sorted = reinterpret_cast<float*>(base + b_desc + 3 * b_vec);
  v.norm2_sorted = reinterpret_cast<float*>(base + b_desc + 4 * b_vec);
  v.rowop = b_op ? reinterpret_cast<__half*>(base + b_desc + 5 * b_vec) : nullptr;
  v.colop = b_op ? reinterpret_cast<__half*>(base + b_desc + 5 * b_vec + b_op) : nullptr;
  v.wideop = wide ? reinterpret_cast<__half*>(base + b_desc + 5 * b_vec + 2 * b_op) : nullptr;
  {
    cudaError_t e = ensure_metas(c, (uint32_t)c->h_images.size());
    if (e != cudaSuccess) return cuda_fail(c, e, "fm_upload_image");
    v.meta = c->d_metas.as<ImageMeta>() + img;
  }
  c->dirty.push_back(img);  // sorted / FP16 tensors are built in one batch at the next fm_match
  c->images_dirty = true;
  return FM_OK;
}

int fm_match(fm_ctx* c, const uint32_t* pair_first, const uint32_t* pair_second, size_t n_pairs, float dist,
             float dist2second, uint32_t flags, fm_result** out) {
  if (!c || !out) return FM_ERR_INVALID;
  *out = nullptr;
  if (n_pairs && (!pair_first || !pair_second)) return fail(c, FM_ERR_INVALID, "fm_match: null pair arrays");
  // match.cpp:320-321: a row with no surviving column has d1 == FLT_MAX and is emitted (with a
  // stale column id) only if sqrt(FLT_MAX) = 1.8e19 < dist.  No caller passes such a threshold
  // (FROG.py uses 1e10); refuse it rather than imitate an index leak.
  if (!(dist < 1.8e19f)) return fail(c, FM_ERR_UNSUPPORTED, "fm_match: distance threshold must be below 1.8e19");
  if ((flags & FM_FLAG_ROW_TABLE) && (flags & FM_FLAG_MATCH_ALL))
    return fail(c, FM_ERR_INVALID, "fm_match: FM_FLAG_ROW_TABLE does not combine with FM_FLAG_MATCH_ALL");
  FM_CUDA(c, cudaSetDevice(c->device));
  for (size_t p = 0; p < n_pairs; p++) {
    uint32_t a = pair_first[p], b = pair_second[p];
    if (a >= c->images.size() || b >= c->images.size() || !c->images[a].valid || !c->images[b].valid)
      return fail(c, FM_ERR_INVALID, "fm_match: pair " + std::to_string(p) + " names an image that was not uploaded");
  }
  int rc = sync_images(c);
  if (rc != FM_OK) return rc;
  const bool sym = flags & FM_FLAG_SYM;
  const bool match_all = flags & FM_FLAG_MATCH_ALL;
  const bool force_exact = (flags & FM_FLAG_FORCE_EXACT) != 0;
  const bool table = (flags & FM_FLAG_ROW_TABLE) != 0;
  // d != 48: the wide tensor-core path (fm_wide.cuh); images it cannot take (kImgBadDim and the other flags) are exact
  const bool wide = c->dim != (uint32_t)kD;

  // ---- tasks --------------------------------------------------------------------------------
  std::vector<Task> tasks;
  std::vector<uint32_t> pair_of_task;
  tasks.reserve(n_pairs * (sym ? 2 : 1));
  uint64_t total_rows = 0, desc_pairs = 0;
  auto add_task = [&](uint32_t col, uint32_t row, uint32_t tflags, size_t p) {
    if (force_exact || c->h_metas[col].flags || c->h_metas[row].flags) tflags |= kTaskExact;
    tasks.push_back(Task{col, row, 0, tflags});
    pair_of_task.push_back((uint32_t)p);
    total_rows += c->images[row].n;
    desc_pairs += (uint64_t)c->images[col].n * c->images[row].n;
  };
  for (size_t p = 0; p < n_pairs; p++) {
    add_task(pair_first[p], pair_second[p], 0, p);
    if (sym) add_task(pair_second[p], pair_first[p], kTaskSwap, p);
  }
  const uint32_t n_tasks = (uint32_t)tasks.size();
  c->reject_rows.clear();
  if (g_debug.reject_dump) c->reject_rows.resize(n_tasks);

  // ---- batches + prefix arrays (blocks of 128 rows, compaction chunks, score units, reject-pass units) ------------
  uint64_t base_units = 0;
  for (auto& t : tasks)
    if (!(t.flags & kTaskExact)) base_units += (c->images[t.row_img].n + kUnitRows - 1) / kUnitRows;
  uint32_t segs = 1;
  if (!wide && base_units > 0 && base_units < (uint64_t)2 * c->sm_count)  // (the wide path scores whole rows: segs = 1)
    segs = (uint32_t)std::min<uint64_t>(8, ((uint64_t)2 * c->sm_count + base_units - 1) / base_units);
  if (match_all && total_rows > 0xFFFFFFF0ull) return fail(c, FM_ERR_UNSUPPORTED, "fm_match: -all supports at most 2^32 outer-loop rows per call");
  const uint32_t kMaxBatchRows = match_all ? 0xFFFFFFF0u : (24u << 20);  // -all: one batch (its scan spans all rows)
  std::vector<Batch> batches;
  std::vector<uint32_t> blk_off, unit_off, rj_unit_off;
  std::vector<ChunkDesc> chunk_desc;  // compaction chunks of every batch, batch after batch (fm_compact.cuh)
  std::vector<size_t> chunk_cursor;   // first chunk of each batch in chunk_desc
  for (uint32_t t = 0; t < n_tasks;) {
    chunk_cursor.push_back(chunk_desc.size());
    Batch b{t, t, 0, 0, 0, 0, 0, blk_off.size(), false, false};
    while (b.t1 < n_tasks) {
      const uint32_t nr = c->images[tasks[b.t1].row_img].n;
      if (b.t1 > b.t0 && (uint64_t)b.rows + nr > kMaxBatchRows) break;
      tasks[b.t1].row_off = b.rows;
      blk_off.push_back(b.blocks);
      unit_off.push_back(b.units);
      rj_unit_off.push_back(b.rj_units);
      for (uint32_t r0 = 0; r0 < nr; r0 += kCompactChunk)
        chunk_desc.push_back(ChunkDesc{b.rows + r0, std::min<uint32_t>(kCompactChunk, nr - r0) | ((tasks[b.t1].flags & kTaskSwap) ? 0x80000000u : 0u),
                                       r0, pair_of_task[b.t1]});
      b.rows += nr;
      b.blocks += (nr + 127) / 128;
      b.chunks += (nr + kCompactChunk - 1) / kCompactChunk;
      if (tasks[b.t1].flags & kTaskExact) b.any_exact = true;
      else {
        b.any_fast = true;
        b.units += ((nr + kUnitRows - 1) / kUnitRows) * segs;
        b.rj_units += (nr + kRjUnitRows - 1) / kRjUnitRows;  // (two-phase scoring runs at segs = 1 only)
      }
      b.t1++;
    }
    blk_off.push_back(b.blocks);
    unit_off.push_back(b.units);
    rj_unit_off.push_back(b.rj_units);
    batches.push_back(b);
    t = b.t1;
  }

  fm_result* r = new (std::nothrow) fm_result();
  if (!r) return fail(c, FM_ERR_NOMEM, "fm_match: out of host memory");
  r->ctx = c;
  r->n_pairs = n_pairs;
  r->flags = flags;
  r->ratio = dist2second;
  r->d48 = !wide && !table;  // (a table call rejects nothing early: it says nothing about the two-phase choice)
  r->slots = total_rows;
  if (table) {
    // first, so that a table that does not fit leaves nothing behind
    cudaError_t e = r->d_table.ensure(std::max<uint64_t>(total_rows, 1) * sizeof(fm_row));
    if (e != cudaSuccess) {
      cudaGetLastError();  // (an allocation failure is not sticky: clear it for the context's next call)
      delete r;
      return cuda_fail(c, e, ("fm_match: row table of " + std::to_string(total_rows) + " rows").c_str());
    }
    r->table = true;
    r->row_off.assign(n_pairs + 1, 0);
    for (size_t p = 0; p < n_pairs; p++)
      r->row_off[p + 1] = r->row_off[p] + c->images[pair_second[p]].n + (sym ? c->images[pair_first[p]].n : 0u);
    for (size_t bi = 0, row0 = 0; bi < batches.size(); row0 += batches[bi].rows, bi++)
      r->sel_batches.push_back(SelectBatch{row0, batches[bi].rows, (uint32_t)chunk_cursor[bi], batches[bi].chunks});
    r->sel_chunks = chunk_desc;
  }
  r->d_out = take_buf(c->out_free, std::max<uint64_t>(total_rows, 1) * sizeof(uint2));
  r->d_counts = take_buf(c->counts_free, std::max<size_t>(n_pairs, 1) * sizeof(uint32_t));
  const bool want_dist = (flags & FM_FLAG_DISTANCES) && !match_all;
  if (want_dist) r->d_dist = take_buf(c->dist_free, std::max<uint64_t>(total_rows, 1) * sizeof(float));
#define FM_CUDA_R(expr)                       \
  do {                                        \
    cudaError_t e__ = (expr);                 \
    if (e__ != cudaSuccess) {                 \
      int code__ = cuda_fail(c, e__, #expr);  \
      fm_result_free(r);                      \
      return code__;                          \
    }                                         \
  } while (0)

  if (c->ev_match.pool.empty() && !c->ev_free.empty()) {
    c->ev_match = std::move(c->ev_free.back());
    c->ev_free.pop_back();
  }
  c->ev_match.reset();
  fm_stats prev = c->stats;
  c->stats = fm_stats{};
  c->stats.ms_prep = prev.ms_prep;
  c->stats.descriptor_pairs = desc_pairs;
  c->stats.rows = total_rows;

  // metadata blob: tasks | chunk descriptors | blk_off | unit_off | rj_unit_off   (16-byte records first: alignment)
  const size_t np = blk_off.size();
  const size_t off_chunk = sizeof(Task) * n_tasks;
  const size_t off_blk = off_chunk + sizeof(ChunkDesc) * chunk_desc.size();
  const size_t off_unit = off_blk + sizeof(uint32_t) * np;
  const size_t off_rj = off_unit + sizeof(uint32_t) * np;
  const size_t blob_bytes = off_rj + sizeof(uint32_t) * np;
  // The blob is staged in the result's pinned block (behind the counters and per-pair counts the device
  // writes back) so that the copy is asynchronous whatever its size: a pageable source would make
  // cudaMemcpyAsync wait for the stream, i.e. for the previous FM_FLAG_ASYNC call.
  const size_t off_blob = (sizeof(DeviceCounters) + std::max<size_t>(n_pairs, 1) * sizeof(uint32_t) + 15) & ~(size_t)15;
  FM_CUDA_R(take_pinned(c, off_blob + std::max<size_t>(blob_bytes, 16), &r->h_block, &r->h_block_cap));
  unsigned char* blob = static_cast<unsigned char*>(r->h_block) + off_blob;
  if (n_tasks) memcpy(blob, tasks.data(), sizeof(Task) * n_tasks);
  if (!chunk_desc.empty()) memcpy(blob + off_chunk, chunk_desc.data(), sizeof(ChunkDesc) * chunk_desc.size());
  if (np) {
    memcpy(blob + off_blk, blk_off.data(), sizeof(uint32_t) * np);
    memcpy(blob + off_unit, unit_off.data(), sizeof(uint32_t) * np);
    memcpy(blob + off_rj, rj_unit_off.data(), sizeof(uint32_t) * np);
  }
  FM_CUDA_R(c->d_meta_blob.ensure(std::max<size_t>(blob_bytes, 16)));
  FM_CUDA_R(cudaMemcpyAsync(c->d_meta_blob.p, blob, std::max<size_t>(blob_bytes, 16), cudaMemcpyHostToDevice, c->stream));
  const unsigned char* blob_d = c->d_meta_blob.as<unsigned char>();
  const Task* d_tasks = reinterpret_cast<const Task*>(blob_d);
  const ChunkDesc* d_chunk = reinterpret_cast<const ChunkDesc*>(blob_d + off_chunk);
  const uint32_t* d_blk = reinterpret_cast<const uint32_t*>(blob_d + off_blk);
  const uint32_t* d_unit = reinterpret_cast<const uint32_t*>(blob_d + off_unit);
  const uint32_t* d_rj_unit = reinterpret_cast<const uint32_t*>(blob_d + off_rj);

  uint32_t max_rows = 1, max_chunks = 1;
  for (auto& b : batches) { max_rows = std::max(max_rows, b.rows); max_chunks = std::max(max_chunks, b.chunks); }
  FM_CUDA_R(c->d_rowres.ensure((size_t)max_rows * sizeof(uint32_t)));
  if (want_dist) {
    FM_CUDA_R(c->d_rowdist.ensure((size_t)max_rows * sizeof(float)));
    FM_CUDA_R(r->d_dist.ensure(std::max<uint64_t>(total_rows, 1) * sizeof(float)));
  }
  FM_CUDA_R(c->d_chunk_count.ensure((size_t)max_chunks * sizeof(uint32_t)));
  FM_CUDA_R(c->d_chunk_out.ensure((size_t)max_chunks * sizeof(unsigned long long)));
  FM_CUDA_R(c->d_chunk_stage.ensure((size_t)max_chunks * kStageCap * sizeof(uint2)));
  FM_CUDA_R(ensure_chunk_status(c));
  FM_CUDA_R(c->d_totals.ensure(sizeof(DeviceCounters)));
  FM_CUDA_R(r->d_out.ensure(std::max<uint64_t>(total_rows, 1) * sizeof(uint2)));
  FM_CUDA_R(r->d_counts.ensure(std::max<size_t>(n_pairs, 1) * sizeof(uint32_t)));
  FM_CUDA_R(cudaMemsetAsync(r->d_counts.p, 0, std::max<size_t>(n_pairs, 1) * sizeof(uint32_t), c->stream));
  FM_CUDA_R(cudaMemsetAsync(c->d_totals.p, 0, sizeof(DeviceCounters), c->stream));

  const ImageDev* d_images = c->d_images.as<ImageDev>();
  uint32_t* d_rowres = c->d_rowres.as<uint32_t>();
  float* d_rowdist = want_dist ? c->d_rowdist.as<float>() : nullptr;
  DeviceCounters* d_counters = c->d_totals.as<DeviceCounters>();
  if (match_all) {
    // ---- -all: count pass, per-task scan, emit pass (fm_all.cuh); list sizes are data-dependent ----
    Span total_span(&c->ev_match, c->stream, kPhTotal);
    std::vector<unsigned long long> task_total(std::max<uint32_t>(n_tasks, 1), 0), task_base(std::max<uint32_t>(n_tasks, 1), 0);
    std::vector<uint32_t> pair_counts(std::max<size_t>(n_pairs, 1), 0);
    unsigned long long grand = 0;
    if (!batches.empty() && batches[0].rows > 0) {
      const Batch& b = batches[0];
      const size_t rows = b.rows;
      FM_CUDA_R(c->d_all.ensure(rows * (3 * sizeof(uint32_t) + sizeof(unsigned long long)) + 16));
      FM_CUDA_R(c->d_all_tasks.ensure((size_t)n_tasks * 2 * sizeof(unsigned long long)));
      unsigned long long* row_off = c->d_all.as<unsigned long long>();
      uint32_t* row_count = reinterpret_cast<uint32_t*>(row_off + rows);
      uint32_t* row_final = row_count + rows;
      uint32_t* row_carry = row_final + rows;
      unsigned long long* d_task_total = c->d_all_tasks.as<unsigned long long>();
      unsigned long long* d_task_base = d_task_total + n_tasks;
      const bool d48 = c->dim == (uint32_t)kD;
      const size_t smem = exact_smem_bytes(kD);
      {
        Span sp(&c->ev_match, c->stream, kPhExact);
        if (d48)
          match_all_kernel<kD, false><<<b.blocks, kExactRows, smem, c->stream>>>(d_images, d_tasks, d_blk, n_tasks, dist, row_count,
                                                                                 row_final, nullptr, nullptr, nullptr, nullptr);
        else
          exact_generic_kernel<1><<<b.blocks, kExactRows, 0, c->stream>>>(d_images, d_tasks, d_blk, n_tasks, dist, 1.f, 0u, nullptr, row_count,
                                                                          row_final, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr);
        all_scan_kernel<<<(n_tasks + 63) / 64, 64, 0, c->stream>>>(d_images, d_tasks, n_tasks, row_count, row_final, row_carry, row_off,
                                                                    d_task_total);
      }
      FM_CUDA_R(cudaMemcpyAsync(task_total.data(), d_task_total, (size_t)n_tasks * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
      FM_CUDA_R(cudaStreamSynchronize(c->stream));
      for (uint32_t t = 0; t < n_tasks; t++) {
        task_base[t] = grand;
        grand += task_total[t];
        const unsigned long long pc = (unsigned long long)pair_counts[pair_of_task[t]] + task_total[t];
        if (pc > 0xFFFFFFFFull) { fm_result_free(r); return fail(c, FM_ERR_UNSUPPORTED, "fm_match: an -all list exceeds 2^32 pairs (pairs.bin block sizes are u32, match.cpp:734)"); }
        pair_counts[pair_of_task[t]] = (uint32_t)pc;
      }
      FM_CUDA_R(r->d_out.ensure(std::max<unsigned long long>(grand, 1) * sizeof(uint2)));
      r->slots = grand;
      FM_CUDA_R(cudaMemcpyAsync(d_task_base, task_base.data(), (size_t)n_tasks * sizeof(unsigned long long), cudaMemcpyHostToDevice, c->stream));
      {
        Span sp(&c->ev_match, c->stream, kPhExact);
        if (d48)
          match_all_kernel<kD, true><<<b.blocks, kExactRows, smem, c->stream>>>(d_images, d_tasks, d_blk, n_tasks, dist, nullptr, nullptr,
                                                                                row_carry, row_off, d_task_base, r->d_out.as<uint2>());
        else
          exact_generic_kernel<2><<<b.blocks, kExactRows, 0, c->stream>>>(d_images, d_tasks, d_blk, n_tasks, dist, 1.f, 0u, nullptr, nullptr,
                                                                          nullptr, row_carry, row_off, d_task_base, r->d_out.as<uint2>(), nullptr, nullptr);
      }
      FM_CUDA_R(cudaStreamSynchronize(c->stream));  // task_base (pageable) must outlive the copy
      c->stats.kernel_launches += 3;
      c->stats.rows_exact += total_rows;
    }
    // hand the totals to the common tail: DeviceCounters.running_total and the per-pair counts
    DeviceCounters hc{};
    hc.running_total = grand;
    FM_CUDA_R(cudaMemcpyAsync(c->d_totals.p, &hc, sizeof hc, cudaMemcpyHostToDevice, c->stream));
    if (n_pairs)
      FM_CUDA_R(cudaMemcpyAsync(r->d_counts.p, pair_counts.data(), n_pairs * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    FM_CUDA_R(cudaStreamSynchronize(c->stream));
  } else {
    Span total_span(&c->ev_match, c->stream, kPhTotal);
    // Two-phase scoring (score_kernel kVar 1 / 2) pays only when nearly every row fails the reference's ratio test --
    // images with little in common at -d2 < 1 -- and costs ~60 % extra otherwise.  So it is used when the previous
    // call of this kind on this context rejected >= 99 % of its rows, or, inside a synchronous multi-batch call, once
    // the first batch (single pass) has shown that much.
    constexpr double kTwoPhaseMin = 0.99;
    // (reject pass: K = 64 only; a row table needs every row's exact distances)
    const bool two_phase_possible = dist2second < 1.f && segs == 1 && !force_exact && !wide && !table;
    bool two_phase = two_phase_possible && c->reject_hint >= kTwoPhaseMin;
    bool probed = false;
    if (g_debug.two_phase >= 0) {  // test hook: force the choice
      two_phase = two_phase_possible && g_debug.two_phase != 0;
      probed = true;
    }
    uint64_t row0 = 0;  // the batch's first row in the call
    for (size_t bi = 0; bi < batches.size(); row0 += batches[bi].rows, bi++) {
      const Batch& b = batches[bi];
      const uint32_t nt = b.t1 - b.t0;
      const uint32_t* blk = d_blk + b.cursor;
      const uint32_t* unt = d_unit + b.cursor;
      if (b.rows == 0) continue;
      fm_row* tab = table ? r->d_table.as<fm_row>() + row0 : nullptr;
      if (b.any_fast) {
        FastBatchArgs fa{};
        fa.images = d_images;
        fa.tasks = d_tasks + b.t0;
        fa.h_tasks = tasks.data() + b.t0;
        fa.task0 = b.t0;
        fa.n_tasks = nt;
        fa.rows = b.rows;
        fa.blk_off = blk;
        fa.blocks128 = b.blocks;
        fa.unit_off = unt;
        fa.units = b.units;
        fa.rj_unit_off = d_rj_unit + b.cursor;
        fa.rj_units = b.rj_units;
        fa.segs = segs;
        fa.thr = dist;
        fa.ratio = dist2second;
        fa.rowres = d_rowres;
        fa.rowdist = d_rowdist;
        fa.table = tab;
        fa.two_phase = two_phase;
        fa.counters = d_counters;
        cudaError_t e = wide ? wide_match_batch(c, fa) : fast_match_batch(c, fa);
        if (e != cudaSuccess) {
          int code = cuda_fail(c, e, "fm_match: tensor-core path");
          fm_result_free(r);
          return code;
        }
      }
      if (b.any_exact) {
        Span sp(&c->ev_match, c->stream, kPhExact);
        if (c->dim == (uint32_t)kD)
          exact_match_kernel<kD><<<b.blocks, kExactRows, exact_smem_bytes(kD), c->stream>>>(
              d_images, d_tasks + b.t0, blk, nt, dist, dist2second, kTaskExact, d_rowres, d_rowdist, tab);
        else
          exact_generic_kernel<0><<<b.blocks, kExactRows, 0, c->stream>>>(d_images, d_tasks + b.t0, blk, nt, dist, dist2second, kTaskExact,
                                                                          d_rowres, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, d_rowdist, tab);
        c->stats.kernel_launches++;
        for (uint32_t t = b.t0; t < b.t1; t++)
          if (tasks[t].flags & kTaskExact) c->stats.rows_exact += c->images[tasks[t].row_img].n;
      }
      {
        Span sp(&c->ev_match, c->stream, kPhCompact);
        CompactArgs ca{};
        ca.chunks = d_chunk + chunk_cursor[bi];
        ca.n_chunks = b.chunks;
        ca.rowres = d_rowres;
        ca.rowdist = d_rowdist;
        ca.pair_count = r->d_counts.as<uint32_t>();
        ca.running_total = &d_counters->running_total;
        ca.out_pairs = r->d_out.as<uint2>();
        ca.out_dist = want_dist ? r->d_dist.as<float>() : nullptr;
        c->stats.kernel_launches += compact_launch(c, ca, want_dist, FM_COMPACT_AUTO);
      }
      if (two_phase_possible && !two_phase && !probed && b.any_fast && !b.any_exact && bi + 1 < batches.size() &&
          !(flags & FM_FLAG_ASYNC)) {
        // a synchronous call with more batches to come: look at what the first one rejected
        probed = true;
        DeviceCounters* hc = reinterpret_cast<DeviceCounters*>(r->h_block);
        FM_CUDA_R(cudaMemcpyAsync(hc, c->d_totals.p, sizeof(DeviceCounters), cudaMemcpyDeviceToHost, c->stream));
        FM_CUDA_R(cudaStreamSynchronize(c->stream));
        two_phase = (double)hc->rescore.rejected_early >= kTwoPhaseMin * (double)b.rows;
      }
    }
  }
  FM_CUDA_R(cudaGetLastError());
  FM_CUDA_R(queue_tail(c, r));
  c->last = r;
  if (!(flags & FM_FLAG_ASYNC)) {
    rc = fm_result_wait(r);
    if (rc != FM_OK) { fm_result_free(r); return rc; }
  }
  *out = r;
  return FM_OK;
#undef FM_CUDA_R
}

int fm_result_wait(fm_result* r) {
  if (!r) return FM_ERR_INVALID;
  int rc = finalize(r);
  if (rc != FM_OK) return rc;
  if (!(r->flags & FM_FLAG_DEVICE_ONLY)) return fm_result_fetch(r);
  return FM_OK;
}

int fm_result_fetch(fm_result* r) {
  if (!r) return FM_ERR_INVALID;
  if (r->fetched) return FM_OK;
  fm_ctx* c = r->ctx;
  int rc = finalize(r);
  if (rc != FM_OK) return rc;
  FM_CUDA(c, cudaSetDevice(c->device));
  const size_t bytes = std::max<uint64_t>(r->total, 1) * sizeof(uint2);
  if (c->cache_pinned && c->cache_pinned_cap >= bytes) {
    r->h_pairs = static_cast<uint32_t*>(c->cache_pinned);
    r->h_cap = c->cache_pinned_cap;
    c->cache_pinned = nullptr;
    c->cache_pinned_cap = 0;
  } else {
    const size_t want = bytes + bytes / 4 + 4096;
    FM_CUDA(c, cudaMallocHost(reinterpret_cast<void**>(&r->h_pairs), want));
    r->h_cap = want;
  }
  if (r->d_dist.p && !r->h_dist) FM_CUDA(c, cudaMallocHost(reinterpret_cast<void**>(&r->h_dist), std::max<uint64_t>(r->total, 1) * sizeof(float)));
  if (r->total) {
    FM_CUDA(c, cudaMemcpyAsync(r->h_pairs, r->d_out.p, r->total * sizeof(uint2), cudaMemcpyDeviceToHost, c->stream));
    if (r->h_dist) FM_CUDA(c, cudaMemcpyAsync(r->h_dist, r->d_dist.p, r->total * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    FM_CUDA(c, cudaStreamSynchronize(c->stream));
  }
  r->fetched = true;
  return FM_OK;
}

size_t fm_result_num_pairs(const fm_result* r) { return r ? r->n_pairs : 0; }
uint64_t fm_result_total(const fm_result* r) { return (r && r->waited) ? r->total : 0; }
uint32_t fm_result_count(const fm_result* r, size_t p) { return (r && r->waited && p < r->n_pairs) ? r->counts[p] : 0; }
const uint32_t* fm_result_pairs(const fm_result* r, size_t p) {
  if (!r || p >= r->n_pairs || !r->fetched) return nullptr;
  return r->h_pairs + 2 * r->offsets[p];
}
const float* fm_result_distances(const fm_result* r, size_t p) {
  if (!r || p >= r->n_pairs || !r->fetched || !r->h_dist) return nullptr;
  return r->h_dist + r->offsets[p];
}
const uint32_t* fm_result_device_counts(const fm_result* r) { return r ? r->d_counts.as<uint32_t>() : nullptr; }
const uint32_t* fm_result_device_pairs(const fm_result* r) { return r ? r->d_out.as<uint32_t>() : nullptr; }

void fm_result_free(fm_result* r) {
  if (!r) return;
  fm_ctx* c = r->ctx;
  cudaSetDevice(c->device);
  if (r->done && !r->waited) cudaEventSynchronize(r->done);  // the pinned block is still a copy target
  if (c->last == r) c->last = nullptr;
  if (r->d_table.p) {  // fm_result_select calls may still read the table
    cudaStreamSynchronize(c->stream);
    r->d_table.release();
  }
  // hand the buffers and events back to the context so the next call does not reallocate
  give_buf(c->out_free, r->d_out);
  give_buf(c->counts_free, r->d_counts);
  give_buf(c->dist_free, r->d_dist);
  if (r->h_dist) cudaFreeHost(r->h_dist);
  give_pinned(c, r->h_block, r->h_block_cap);
  if (!r->ev.pool.empty()) {
    if (c->ev_free.size() < 8) c->ev_free.push_back(std::move(r->ev));
    else r->ev.destroy();
  }
  if (r->h_pairs) {
    if (r->h_cap > c->cache_pinned_cap) {
      if (c->cache_pinned) cudaFreeHost(c->cache_pinned);
      c->cache_pinned = r->h_pairs;
      c->cache_pinned_cap = r->h_cap;
    } else {
      cudaFreeHost(r->h_pairs);
    }
  }
  give_buf(c->counts_free, r->d_goff);
  for (auto& gp : r->parts) {  // (the lead's `done` follows every member's gather: nothing below is still in use)
    fm_ctx* m = gp.sub->ctx;
    fm_result_free(gp.sub);
    cudaSetDevice(m->device);
    give_buf(m->counts_free, gp.scratch);
    give_pinned(m, gp.pin, gp.pin_cap);
  }
  delete r;
}

int fm_get_stats(fm_ctx* c, fm_stats* out) {
  if (!c || !out) return FM_ERR_INVALID;
  FM_CUDA(c, cudaSetDevice(c->device));
  FM_CUDA(c, cudaStreamSynchronize(c->stream));
  if (c->last && !c->last->waited) {
    int rc = finalize(c->last);
    if (rc != FM_OK) return rc;
  }
  c->stats.ms_prep = c->ms_prep_acc;
  *out = c->stats;
  return FM_OK;
}

int fm_result_stats(fm_result* r, fm_stats* out) {
  if (!r || !out) return FM_ERR_INVALID;
  int rc = finalize(r);
  if (rc != FM_OK) return rc;
  *out = r->stats;
  return FM_OK;
}

// ---- consumer hand-off: link build (fm_links.cuh) -------------------------------------------------

int fm_links_build(fm_result* r, const uint32_t* pair_first, const uint32_t* pair_second, const uint32_t* block_order,
                   fm_links** out) {
  if (!r || !out) return FM_ERR_INVALID;
  *out = nullptr;
  fm_ctx* c = r->ctx;
  if (!r->waited) return fail(c, FM_ERR_INVALID, "fm_links_build: the result is not complete (fm_result_wait first)");
  if (r->flags & FM_FLAG_MATCH_ALL) return fail(c, FM_ERR_UNSUPPORTED, "fm_links_build: -all results are not supported");
  if (r->n_pairs && (!pair_first || !pair_second)) return fail(c, FM_ERR_INVALID, "fm_links_build: null pair arrays");
  FM_CUDA(c, cudaSetDevice(c->device));
  fm_links* l = new (std::nothrow) fm_links();
  if (!l) return fail(c, FM_ERR_NOMEM, "fm_links_build: out of host memory");
  l->ctx = c;
  const size_t n_img = c->images.size();
  l->point_base.assign(n_img + 1, 0);
  for (size_t i = 0; i < n_img; i++) l->point_base[i + 1] = l->point_base[i] + (c->images[i].valid ? c->images[i].n : 0);
  if (l->point_base[n_img] > 0xFFFFFFF0ull) { delete l; return fail(c, FM_ERR_UNSUPPORTED, "fm_links_build: more than 2^32 points"); }
  l->n_points = (uint32_t)l->point_base[n_img];
  // blocks in file order
  std::vector<LinkBlock> blocks(r->n_pairs);
  std::vector<unsigned long long> entry_off(r->n_pairs + 1, 0);
  for (size_t k = 0; k < r->n_pairs; k++) {
    const size_t p = block_order ? block_order[k] : k;
    if (p >= r->n_pairs || pair_first[p] >= n_img || pair_second[p] >= n_img) { delete l; return fail(c, FM_ERR_INVALID, "fm_links_build: bad block order or pair"); }
    LinkBlock& b = blocks[k];
    b.src = r->offsets[p];
    b.q0 = entry_off[k];
    b.count = r->counts[p];
    b.image1 = pair_first[p];
    b.image2 = pair_second[p];
    b.base1 = (uint32_t)l->point_base[b.image1];
    b.base2 = (uint32_t)l->point_base[b.image2];
    b.pad_ = 0;
    entry_off[k + 1] = entry_off[k] + b.count;
  }
  const unsigned long long n_entries = entry_off[r->n_pairs];
  l->total = 2ull * n_entries;
  auto bail = [&](cudaError_t e, const char* what) { int code = cuda_fail(c, e, what); fm_links_free(l); return code; };
  DevBuf d_blocks, d_eoff, d_deg, d_cursor, d_tmp;
  struct Scratch { DevBuf* b[5]; ~Scratch() { for (auto* x : b) x->release(); } } scratch{{&d_blocks, &d_eoff, &d_deg, &d_cursor, &d_tmp}};
  cudaError_t e;
  const size_t np1 = (size_t)l->n_points + 1;
  if ((e = d_blocks.ensure(std::max<size_t>(1, blocks.size()) * sizeof(LinkBlock))) != cudaSuccess) return bail(e, "fm_links_build");
  if ((e = d_eoff.ensure(entry_off.size() * sizeof(unsigned long long))) != cudaSuccess) return bail(e, "fm_links_build");
  if ((e = d_deg.ensure(np1 * sizeof(uint32_t))) != cudaSuccess) return bail(e, "fm_links_build");
  if ((e = d_cursor.ensure(np1 * sizeof(uint32_t))) != cudaSuccess) return bail(e, "fm_links_build");
  if ((e = d_tmp.ensure(std::max<uint64_t>(l->total, 1) * sizeof(HalfLink))) != cudaSuccess) return bail(e, "fm_links_build");
  if ((e = l->d_off.ensure(np1 * sizeof(unsigned long long))) != cudaSuccess) return bail(e, "fm_links_build");
  if ((e = l->d_links.ensure(std::max<uint64_t>(l->total, 1) * sizeof(uint2))) != cudaSuccess) return bail(e, "fm_links_build");
  cudaEvent_t ev0, ev1;
  cudaEventCreate(&ev0);
  cudaEventCreate(&ev1);
  if (!blocks.empty() && (e = cudaMemcpyAsync(d_blocks.p, blocks.data(), blocks.size() * sizeof(LinkBlock), cudaMemcpyHostToDevice, c->stream)) != cudaSuccess) return bail(e, "fm_links_build");
  if ((e = cudaMemcpyAsync(d_eoff.p, entry_off.data(), entry_off.size() * sizeof(unsigned long long), cudaMemcpyHostToDevice, c->stream)) != cudaSuccess) return bail(e, "fm_links_build");
  cudaMemsetAsync(d_deg.p, 0, np1 * sizeof(uint32_t), c->stream);
  cudaMemsetAsync(d_cursor.p, 0, np1 * sizeof(uint32_t), c->stream);
  cudaEventRecord(ev0, c->stream);
  const unsigned grid = (unsigned)((n_entries + 255) / 256);
  const uint2* pairs = r->d_out.as<uint2>();
  if (n_entries)
    links_scatter_kernel<false><<<grid, 256, 0, c->stream>>>(d_blocks.as<LinkBlock>(), d_eoff.as<unsigned long long>(), (uint32_t)r->n_pairs, n_entries,
                                                            pairs, d_deg.as<uint32_t>(), nullptr, nullptr, nullptr);
  links_scan_kernel<<<1, 1024, 0, c->stream>>>(d_deg.as<uint32_t>(), l->n_points, l->d_off.as<unsigned long long>());
  if (n_entries)
    links_scatter_kernel<true><<<grid, 256, 0, c->stream>>>(d_blocks.as<LinkBlock>(), d_eoff.as<unsigned long long>(), (uint32_t)r->n_pairs, n_entries,
                                                           pairs, nullptr, l->d_off.as<unsigned long long>(), d_cursor.as<uint32_t>(), d_tmp.as<HalfLink>());
  if (l->n_points)
    links_sort_kernel<<<(l->n_points + 127) / 128, 128, 0, c->stream>>>(l->d_off.as<unsigned long long>(), l->n_points, d_tmp.as<HalfLink>(),
                                                                        l->d_links.as<uint2>());
  cudaEventRecord(ev1, c->stream);
  if ((e = cudaGetLastError()) != cudaSuccess) return bail(e, "fm_links_build: launch");
  if ((e = cudaStreamSynchronize(c->stream)) != cudaSuccess) return bail(e, "fm_links_build");  // the scratch buffers and host tables die here
  cudaEventElapsedTime(&l->ms_build, ev0, ev1);
  cudaEventDestroy(ev0);
  cudaEventDestroy(ev1);
  *out = l;
  return FM_OK;
}

uint64_t fm_links_total(const fm_links* l) { return l ? l->total : 0; }

int fm_links_fetch(fm_links* l) {
  if (!l) return FM_ERR_INVALID;
  if (l->h_off) return FM_OK;
  fm_ctx* c = l->ctx;
  FM_CUDA(c, cudaSetDevice(c->device));
  const size_t np1 = (size_t)l->n_points + 1;
  FM_CUDA(c, cudaMallocHost(reinterpret_cast<void**>(&l->h_off), np1 * sizeof(unsigned long long)));
  FM_CUDA(c, cudaMallocHost(reinterpret_cast<void**>(&l->h_links), std::max<uint64_t>(l->total, 1) * sizeof(uint2)));
  FM_CUDA(c, cudaMemcpyAsync(l->h_off, l->d_off.p, np1 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
  if (l->total) FM_CUDA(c, cudaMemcpyAsync(l->h_links, l->d_links.p, l->total * sizeof(uint2), cudaMemcpyDeviceToHost, c->stream));
  FM_CUDA(c, cudaStreamSynchronize(c->stream));
  return FM_OK;
}

const uint64_t* fm_links_offsets(const fm_links* l, uint32_t img, uint32_t* n_points) {
  if (!l || !l->h_off || (size_t)img + 1 >= l->point_base.size()) return nullptr;
  if (n_points) *n_points = (uint32_t)(l->point_base[img + 1] - l->point_base[img]);
  return reinterpret_cast<const uint64_t*>(l->h_off) + l->point_base[img];
}
const uint32_t* fm_links_data(const fm_links* l) { return (l && l->h_off) ? l->h_links : nullptr; }
const uint64_t* fm_links_device_offsets(const fm_links* l) { return l ? reinterpret_cast<const uint64_t*>(l->d_off.p) : nullptr; }
const uint32_t* fm_links_device_data(const fm_links* l) { return l ? l->d_links.as<uint32_t>() : nullptr; }
float fm_links_build_ms(const fm_links* l) { return l ? l->ms_build : 0.f; }

void fm_links_free(fm_links* l) {
  if (!l) return;
  cudaSetDevice(l->ctx->device);
  l->d_off.release();
  l->d_links.release();
  if (l->h_off) cudaFreeHost(l->h_off);
  if (l->h_links) cudaFreeHost(l->h_links);
  delete l;
}

// ---- device groups (fm_group_*): several contexts that act as one -------------------------------------------------

}  // extern "C"

struct fm_group {
  std::vector<fm_ctx*> m;         // one context per device; m[0] is the lead
  std::vector<cudaEvent_t> ev;    // per member, on its device: the member's stream up to the latest hand-off
  cudaEvent_t ev_lead = nullptr;  // the lead's scan of the gathered counts
  std::vector<std::vector<char>> peer;  // peer[k][j]: member k reads member j's memory directly (same GPU, or peer access)
};

namespace {

thread_local std::string g_group_create_error;

int group_fail(fm_group* g, int code, const std::string& msg) {
  if (g) g->m[0]->err = msg; else g_group_create_error = msg;
  return code;
}

// An error of member k's own call, reported on the group with the device named.
int member_fail(fm_group* g, size_t k, int code) {
  return group_fail(g, code, "device " + std::to_string(g->m[k]->device) + ": " + g->m[k]->err);
}

// Steps 2-5 of a group call, behind the members' calls r->parts (each a device-only FM_FLAG_ASYNC result of member
// parts[i].member over the pairs parts[i].idx; the caller recorded g->ev_lead on the lead stream before queueing them):
// gather their counts and lists into r's buffers on the lead, in submission order, all in stream order, and record
// r->done behind it.  On error the caller frees r (after synchronising the members).
int group_gather(fm_group* g, fm_result* r) {
  fm_ctx* lead = g->m[0];
  const size_t G = g->m.size(), n_pairs = r->n_pairs;
  const bool want_dist = (r->flags & FM_FLAG_DISTANCES) && !(r->flags & FM_FLAG_MATCH_ALL);
#define FM_CUDA_G(expr)                                  \
  do {                                                   \
    cudaError_t e__ = (expr);                            \
    if (e__ != cudaSuccess) return cuda_fail(lead, e__, #expr); \
  } while (0)
  FM_CUDA_G(cudaSetDevice(lead->device));
  r->d_out = take_buf(lead->out_free, std::max<uint64_t>(r->slots, 1) * sizeof(uint2));
  r->d_counts = take_buf(lead->counts_free, std::max<size_t>(n_pairs, 1) * sizeof(uint32_t));
  r->d_goff = take_buf(lead->counts_free, (n_pairs + 1) * sizeof(unsigned long long));
  if (want_dist) r->d_dist = take_buf(lead->dist_free, std::max<uint64_t>(r->slots, 1) * sizeof(float));
  FM_CUDA_G(r->d_out.ensure(std::max<uint64_t>(r->slots, 1) * sizeof(uint2)));
  FM_CUDA_G(r->d_counts.ensure(std::max<size_t>(n_pairs, 1) * sizeof(uint32_t)));
  FM_CUDA_G(r->d_goff.ensure((n_pairs + 1) * sizeof(unsigned long long)));
  if (want_dist) FM_CUDA_G(r->d_dist.ensure(std::max<uint64_t>(r->slots, 1) * sizeof(float)));
  FM_CUDA_G(take_pinned(lead, sizeof(DeviceCounters) + std::max<size_t>(n_pairs, 1) * sizeof(uint32_t), &r->h_block, &r->h_block_cap));
  memset(r->h_block, 0, sizeof(DeviceCounters));

  // 2. each member's counts to their submission positions on the lead; its local offsets
  for (GroupPart& gp : r->parts) {
    const size_t k = gp.member;
    fm_ctx* c = g->m[k];
    const uint32_t nk = (uint32_t)gp.idx.size();
    FM_CUDA_G(cudaSetDevice(c->device));
    FM_CUDA_G(take_pinned(c, (size_t)nk * sizeof(uint32_t), &gp.pin, &gp.pin_cap));
    uint32_t* h_idx = static_cast<uint32_t*>(gp.pin);
    for (uint32_t i = 0; i < nk; i++) h_idx[i] = gp.idx[i];
    const size_t loff_bytes = ((size_t)nk + 1) * sizeof(unsigned long long);
    gp.scratch = take_buf(c->counts_free, loff_bytes + (size_t)nk * sizeof(uint32_t));
    FM_CUDA_G(gp.scratch.ensure(loff_bytes + (size_t)nk * sizeof(uint32_t)));
    unsigned long long* loff = gp.scratch.as<unsigned long long>();
    uint32_t* d_idx = reinterpret_cast<uint32_t*>(loff + nk + 1);
    FM_CUDA_G(cudaMemcpyAsync(d_idx, h_idx, (size_t)nk * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
    if (k) FM_CUDA_G(cudaStreamWaitEvent(c->stream, g->ev_lead, 0));
    const uint32_t* counts = gp.sub->d_counts.as<uint32_t>();
    group_counts_kernel<<<(nk + 255) / 256, 256, 0, c->stream>>>(counts, d_idx, nk, r->d_counts.as<uint32_t>());
    links_scan_kernel<<<1, 1024, 0, c->stream>>>(counts, nk, loff);
    FM_CUDA_G(cudaGetLastError());
    FM_CUDA_G(cudaEventRecord(g->ev[k], c->stream));
  }
  // 3. the lead scans the gathered counts into submission-order offsets
  FM_CUDA_G(cudaSetDevice(lead->device));
  for (const GroupPart& gp : r->parts)
    if (gp.member) FM_CUDA_G(cudaStreamWaitEvent(lead->stream, g->ev[gp.member], 0));
  links_scan_kernel<<<1, 1024, 0, lead->stream>>>(r->d_counts.as<uint32_t>(), (uint32_t)n_pairs, r->d_goff.as<unsigned long long>());
  FM_CUDA_G(cudaGetLastError());
  FM_CUDA_G(cudaEventRecord(g->ev_lead, lead->stream));
  // 4. each member pushes its lists into the lead's buffer; its own buffers go back to its free lists when they have
  // room (stream order keeps them until the push has read them), else at fm_result_free
  for (GroupPart& gp : r->parts) {
    const size_t k = gp.member;
    fm_ctx* c = g->m[k];
    fm_result* q = gp.sub;
    const uint32_t nk = (uint32_t)gp.idx.size();
    FM_CUDA_G(cudaSetDevice(c->device));
    if (k) FM_CUDA_G(cudaStreamWaitEvent(c->stream, g->ev_lead, 0));
    const unsigned long long* loff = gp.scratch.as<unsigned long long>();
    const uint32_t* d_idx = reinterpret_cast<const uint32_t*>(loff + nk + 1);
    const unsigned grid = (nk + kGatherWarps - 1) / kGatherWarps;
    if (want_dist)
      group_push_kernel<true><<<grid, kGatherThreads, 0, c->stream>>>(q->d_out.as<uint2>(), q->d_dist.as<float>(), loff, d_idx, nk,
                                                                      r->d_goff.as<unsigned long long>(), r->d_out.as<uint2>(), r->d_dist.as<float>());
    else
      group_push_kernel<false><<<grid, kGatherThreads, 0, c->stream>>>(q->d_out.as<uint2>(), nullptr, loff, d_idx, nk,
                                                                       r->d_goff.as<unsigned long long>(), r->d_out.as<uint2>(), nullptr);
    FM_CUDA_G(cudaGetLastError());
    FM_CUDA_G(cudaEventRecord(g->ev[k], c->stream));
    give_buf_queued(c->out_free, q->d_out);
    give_buf_queued(c->counts_free, q->d_counts);
    give_buf_queued(c->dist_free, q->d_dist);
  }
  // 5. the lead waits for every push; total and counts to the result's pinned block, as fm_match leaves them
  FM_CUDA_G(cudaSetDevice(lead->device));
  for (const GroupPart& gp : r->parts)
    if (gp.member) FM_CUDA_G(cudaStreamWaitEvent(lead->stream, g->ev[gp.member], 0));
  FM_CUDA_G(cudaMemcpyAsync(static_cast<char*>(r->h_block) + offsetof(DeviceCounters, running_total), r->d_goff.as<unsigned long long>() + n_pairs,
                            sizeof(unsigned long long), cudaMemcpyDeviceToHost, lead->stream));
  if (n_pairs)
    FM_CUDA_G(cudaMemcpyAsync(static_cast<char*>(r->h_block) + sizeof(DeviceCounters), r->d_counts.p, n_pairs * sizeof(uint32_t),
                              cudaMemcpyDeviceToHost, lead->stream));
  r->done = r->ev.get();
  FM_CUDA_G(cudaEventRecord(r->done, lead->stream));
#undef FM_CUDA_G
  return FM_OK;
}


}  // namespace

extern "C" {

int fm_group_create(const int* devices, int n, fm_group** out) {
  if (!out) return group_fail(nullptr, FM_ERR_INVALID, "fm_group_create: out is NULL");
  *out = nullptr;
  int n_dev = 0;
  cudaError_t e = cudaGetDeviceCount(&n_dev);
  if (e != cudaSuccess || n_dev == 0)
    return group_fail(nullptr, FM_ERR_CUDA, std::string("fm_group_create: no CUDA device (") + cudaGetErrorString(e) +
                                                "); libfrogmatch has no CPU fallback");
  if (!devices || n <= 0) return group_fail(nullptr, FM_ERR_INVALID, "fm_group_create: no devices given");
  for (int k = 0; k < n; k++) {
    if (devices[k] < 0 || devices[k] >= n_dev)
      return group_fail(nullptr, FM_ERR_INVALID, "fm_group_create: device " + std::to_string(devices[k]) + " is out of range (" +
                                                     std::to_string(n_dev) + " visible)");
    for (int j = 0; j < k && !g_debug.group_repeat; j++)
      if (devices[j] == devices[k])
        return group_fail(nullptr, FM_ERR_INVALID, "fm_group_create: device " + std::to_string(devices[k]) + " is given twice");
  }
  for (int k = 1; k < n; k++) {
    if (devices[k] == devices[0]) continue;  // (fm_debug_set_option "group_repeat")
    int can = 0;
    if ((e = cudaDeviceCanAccessPeer(&can, devices[k], devices[0])) != cudaSuccess)
      return group_fail(nullptr, FM_ERR_CUDA, std::string("fm_group_create: cudaDeviceCanAccessPeer: ") + cudaGetErrorString(e));
    if (!can)
      return group_fail(nullptr, FM_ERR_UNSUPPORTED, "fm_group_create: device " + std::to_string(devices[k]) +
                                                         " cannot access the lead device " + std::to_string(devices[0]) + " as a peer");
  }
  fm_group* g = new (std::nothrow) fm_group();
  if (!g) return group_fail(nullptr, FM_ERR_NOMEM, "fm_group_create: out of host memory");
  auto undo = [&](int code, const std::string& msg) {
    fm_group_destroy(g);
    return group_fail(nullptr, code, msg);
  };
  for (int k = 0; k < n; k++) {
    fm_ctx* c = nullptr;
    int rc = fm_create(devices[k], &c);
    if (rc != FM_OK) return undo(rc, std::string(fm_last_error(nullptr)));
    g->m.push_back(c);
    cudaEvent_t ev = nullptr;
    if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess)
      return undo(FM_ERR_CUDA, std::string("fm_group_create: ") + cudaGetErrorString(e));
    g->ev.push_back(ev);
  }
  // Peer access (process state, left enabled at destroy) for every ordered pair of members that supports it: members
  // store into the lead's memory (the gather; required, checked above), and uploads copy between members.
  g->peer.assign(n, std::vector<char>(n, 0));
  for (int k = 0; k < n; k++)
    for (int j = 0; j < n; j++) {
      if (devices[k] == devices[j]) { g->peer[k][j] = 1; continue; }  // (the same GPU: fm_debug_set_option "group_repeat")
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, devices[k], devices[j]) != cudaSuccess || !can) { cudaGetLastError(); continue; }
      cudaSetDevice(devices[k]);
      e = cudaDeviceEnablePeerAccess(devices[j], 0);
      if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
      else if (e != cudaSuccess) {
        cudaGetLastError();
        if (j == 0)
          return undo(FM_ERR_UNSUPPORTED, "fm_group_create: device " + std::to_string(devices[k]) + " cannot map the lead device " +
                                              std::to_string(devices[0]) + ": " + cudaGetErrorString(e));
        continue;
      }
      g->peer[k][j] = 1;
    }
  cudaSetDevice(devices[0]);
  if ((e = cudaEventCreateWithFlags(&g->ev_lead, cudaEventDisableTiming)) != cudaSuccess)
    return undo(FM_ERR_CUDA, std::string("fm_group_create: ") + cudaGetErrorString(e));
  *out = g;
  return FM_OK;
}

void fm_group_destroy(fm_group* g) {
  if (!g) return;
  for (size_t k = 0; k < g->m.size(); k++) {
    cudaSetDevice(g->m[k]->device);
    cudaStreamSynchronize(g->m[k]->stream);
    if (k < g->ev.size()) cudaEventDestroy(g->ev[k]);
  }
  if (g->ev_lead) {
    cudaSetDevice(g->m[0]->device);
    cudaEventDestroy(g->ev_lead);
  }
  for (auto* c : g->m) fm_destroy(c);
  delete g;
}

const char* fm_group_last_error(const fm_group* g) { return g ? g->m[0]->err.c_str() : g_group_create_error.c_str(); }

int fm_group_synchronize(fm_group* g) {
  if (!g) return FM_ERR_INVALID;
  for (size_t k = 0; k < g->m.size(); k++)
    if (int rc = fm_synchronize(g->m[k])) return member_fail(g, k, rc);
  return FM_OK;
}

int fm_group_clear_images(fm_group* g) {
  if (!g) return FM_ERR_INVALID;
  for (size_t k = 0; k < g->m.size(); k++)
    if (int rc = fm_clear_images(g->m[k])) return member_fail(g, k, rc);
  return FM_OK;
}

int fm_group_upload_image(fm_group* g, uint32_t img, const float* desc, const float* scale, const float* lap, uint32_t n,
                          uint32_t d) {
  if (!g) return FM_ERR_INVALID;
  const size_t G = g->m.size();
  if (G == 1) return fm_upload_image(g->m[0], img, desc, scale, lap, n, d);
  // The owner copies the caller's image: a host image goes to member img % n, a device image to the member on its GPU.
  // The lead, then every other member, copies a member's device copy it can read as a peer: the owner's, otherwise the
  // lead's (every member reads the lead's memory).  So each image crosses PCIe at most once.  The lead owns the image
  // when it cannot read the owner's memory (or the image lies on a GPU outside the group).
  cudaPointerAttributes attr{};
  const bool on_device = n && desc && cudaPointerGetAttributes(&attr, desc) == cudaSuccess && attr.type == cudaMemoryTypeDevice;
  cudaGetLastError();
  size_t o = img % G;
  if (on_device) {
    o = 0;
    for (size_t k = 0; k < G; k++)
      if (g->m[k]->device == attr.device) { o = k; break; }
  }
  if (!g->peer[0][o]) o = 0;
  fm_ctx* owner = g->m[o];
  if (int rc = fm_upload_image(owner, img, desc, scale, lap, n, d)) return o ? member_fail(g, o, rc) : rc;
  FM_CUDA(g->m[0], cudaSetDevice(owner->device));
  FM_CUDA(g->m[0], cudaEventRecord(g->ev[o], owner->stream));
  std::vector<size_t> order;  // the lead first: members that cannot read the owner copy the lead's copy
  if (o != 0) order.push_back(0);
  for (size_t k = 1; k < G; k++)
    if (k != o) order.push_back(k);
  for (size_t k : order) {
    const size_t src = g->peer[k][o] ? o : 0;
    const ImageDev& v = g->m[src]->h_images[img];
    fm_ctx* c = g->m[k];
    FM_CUDA(g->m[0], cudaSetDevice(c->device));
    FM_CUDA(g->m[0], cudaStreamWaitEvent(c->stream, g->ev[src], 0));
    if (int rc = fm_upload_image(c, img, v.desc, v.scale, v.lap, n, d)) return k ? member_fail(g, k, rc) : rc;
    FM_CUDA(g->m[0], cudaEventRecord(g->ev[k], c->stream));
  }
  // the sources' copies must outlive the members' reads of them (a later upload may reuse their slabs)
  for (size_t s : {o, (size_t)0}) {
    FM_CUDA(g->m[0], cudaSetDevice(g->m[s]->device));
    for (size_t k : order)
      if (k != s) FM_CUDA(g->m[0], cudaStreamWaitEvent(g->m[s]->stream, g->ev[k], 0));
  }
  return FM_OK;
}

int fm_group_match(fm_group* g, const uint32_t* pair_first, const uint32_t* pair_second, size_t n_pairs, float dist,
                   float dist2second, uint32_t flags, fm_result** out) {
  if (!g || !out) return FM_ERR_INVALID;
  *out = nullptr;
  const size_t G = g->m.size();
  fm_ctx* lead = g->m[0];
  if (G == 1) return fm_match(lead, pair_first, pair_second, n_pairs, dist, dist2second, flags, out);
  if (n_pairs && (!pair_first || !pair_second)) return fail(lead, FM_ERR_INVALID, "fm_match: null pair arrays");
  if (!(dist < 1.8e19f)) return fail(lead, FM_ERR_UNSUPPORTED, "fm_match: distance threshold must be below 1.8e19");
  if ((flags & FM_FLAG_ROW_TABLE) && (flags & FM_FLAG_MATCH_ALL))
    return fail(lead, FM_ERR_INVALID, "fm_match: FM_FLAG_ROW_TABLE does not combine with FM_FLAG_MATCH_ALL");
  for (size_t p = 0; p < n_pairs; p++) {  // (every member holds every image: the lead's table speaks for all)
    uint32_t a = pair_first[p], b = pair_second[p];
    if (a >= lead->images.size() || b >= lead->images.size() || !lead->images[a].valid || !lead->images[b].valid)
      return fail(lead, FM_ERR_INVALID, "fm_match: pair " + std::to_string(p) + " names an image that was not uploaded");
  }
  if (flags & FM_FLAG_MATCH_ALL) {  // the limit of one context's call, for the whole call rather than each shard
    uint64_t rows = 0;
    for (size_t p = 0; p < n_pairs; p++)
      rows += lead->images[pair_second[p]].n + ((flags & FM_FLAG_SYM) ? lead->images[pair_first[p]].n : 0u);
    if (rows > 0xFFFFFFF0ull) return fail(lead, FM_ERR_UNSUPPORTED, "fm_match: -all supports at most 2^32 outer-loop rows per call");
  }
  // Prepare new images on every member at once: fm_match would otherwise wait for each member's preparation in turn.
  for (size_t k = 0; k < G; k++)
    if (int rc = prep_queue(g->m[k])) return member_fail(g, k, rc);
  for (size_t k = 0; k < G; k++)
    if (int rc = prep_finish(g->m[k])) return member_fail(g, k, rc);

  std::vector<double> weight(n_pairs);
  for (size_t p = 0; p < n_pairs; p++) weight[p] = (double)lead->images[pair_first[p]].n * (double)lead->images[pair_second[p]].n;
  const std::vector<std::vector<size_t>> shard = shard_pairs(weight, (int)G);

  fm_result* r = new (std::nothrow) fm_result();
  if (!r) return fail(lead, FM_ERR_NOMEM, "fm_group_match: out of host memory");
  r->ctx = lead;
  r->n_pairs = n_pairs;
  r->flags = flags;
  r->ratio = dist2second;
  r->group = g;
  auto bail = [&](int code) {
    for (auto* c : g->m) { cudaSetDevice(c->device); cudaStreamSynchronize(c->stream); }
    fm_result_free(r);
    return code;
  };
#define FM_CUDA_G(expr)                                  \
  do {                                                   \
    cudaError_t e__ = (expr);                            \
    if (e__ != cudaSuccess) return bail(cuda_fail(lead, e__, #expr)); \
  } while (0)

  // Members store into lead buffers taken from the lead's free lists, whose earlier users may still be queued on the
  // lead stream: members start storing only behind this event.
  FM_CUDA_G(cudaSetDevice(lead->device));
  FM_CUDA_G(cudaEventRecord(g->ev_lead, lead->stream));
  // 1. every member queues the match of its shard (FM_FLAG_MATCH_ALL calls run one after another: they size on the host)
  {
    std::vector<uint32_t> pf, ps;
    for (size_t k = 0; k < G; k++) {
      if (shard[k].empty()) continue;
      pf.clear();
      ps.clear();
      for (size_t p : shard[k]) { pf.push_back(pair_first[p]); ps.push_back(pair_second[p]); }
      fm_result* q = nullptr;
      if (int rc = fm_match(g->m[k], pf.data(), ps.data(), pf.size(), dist, dist2second, flags | FM_FLAG_ASYNC | FM_FLAG_DEVICE_ONLY, &q))
        return bail(member_fail(g, k, rc));
      r->parts.push_back(GroupPart{});
      GroupPart& gp = r->parts.back();
      gp.sub = q;
      gp.member = (uint32_t)k;
      gp.idx.assign(shard[k].begin(), shard[k].end());
      r->slots += q->slots;
    }
  }
#undef FM_CUDA_G
  if (flags & FM_FLAG_ROW_TABLE) {
    // rows in submission order over the whole call, and where each pair's rows lie (fm_result_rows_copy)
    r->table = true;
    r->row_off.assign(n_pairs + 1, 0);
    for (size_t p = 0; p < n_pairs; p++)
      r->row_off[p + 1] = r->row_off[p] + lead->images[pair_second[p]].n + ((flags & FM_FLAG_SYM) ? lead->images[pair_first[p]].n : 0u);
    r->pair_part.assign(n_pairs, 0);
    r->pair_local.assign(n_pairs, 0);
    for (size_t i = 0; i < r->parts.size(); i++)
      for (size_t j = 0; j < r->parts[i].idx.size(); j++) {
        r->pair_part[r->parts[i].idx[j]] = (uint32_t)i;
        r->pair_local[r->parts[i].idx[j]] = (uint32_t)j;
      }
  }
  if (int rc = group_gather(g, r)) return bail(rc);
  if (!(flags & FM_FLAG_ASYNC)) {
    int rc = fm_result_wait(r);
    if (rc != FM_OK) { fm_result_free(r); return rc; }
  }
  *out = r;
  return FM_OK;
}

// ---- re-deciding a call at other thresholds (FM_FLAG_ROW_TABLE, fm_select.cuh) ---------------------------------------

}  // extern "C"

namespace {

// fm_result_select on a result of one context: per batch of the source call, select_kernel turns the table's rows into
// rowres / rowdist at (dist, ratio), and compact_launch compacts them with the call's own chunk records -- the
// fm_match tail, with the scoring replaced by one read of the table.
int select_one(const fm_result* s, float dist, float ratio, uint32_t flags, fm_result** out) {
  fm_ctx* c = s->ctx;
  FM_CUDA(c, cudaSetDevice(c->device));
  const bool want_dist = (flags & FM_FLAG_DISTANCES) != 0;
  const uint64_t total_rows = s->slots;
  fm_result* r = new (std::nothrow) fm_result();
  if (!r) return fail(c, FM_ERR_NOMEM, "fm_result_select: out of host memory");
  r->ctx = c;
  r->n_pairs = s->n_pairs;
  r->flags = flags;
  r->ratio = ratio;
  r->slots = total_rows;
  r->d_out = take_buf(c->out_free, std::max<uint64_t>(total_rows, 1) * sizeof(uint2));
  r->d_counts = take_buf(c->counts_free, std::max<size_t>(r->n_pairs, 1) * sizeof(uint32_t));
  if (want_dist) r->d_dist = take_buf(c->dist_free, std::max<uint64_t>(total_rows, 1) * sizeof(float));
#define FM_CUDA_R(expr)                       \
  do {                                        \
    cudaError_t e__ = (expr);                 \
    if (e__ != cudaSuccess) {                 \
      int code__ = cuda_fail(c, e__, #expr);  \
      fm_result_free(r);                      \
      return code__;                          \
    }                                         \
  } while (0)
  if (c->ev_match.pool.empty() && !c->ev_free.empty()) {
    c->ev_match = std::move(c->ev_free.back());
    c->ev_free.pop_back();
  }
  c->ev_match.reset();
  const float ms_prep = c->stats.ms_prep;
  c->stats = fm_stats{};
  c->stats.ms_prep = ms_prep;
  c->stats.rows = total_rows;

  // the chunk records, staged in the result's pinned block behind the counters and counts (as fm_match stages its blob)
  const size_t off_blob = (sizeof(DeviceCounters) + std::max<size_t>(r->n_pairs, 1) * sizeof(uint32_t) + 15) & ~(size_t)15;
  const size_t blob_bytes = std::max<size_t>(s->sel_chunks.size() * sizeof(ChunkDesc), 16);
  FM_CUDA_R(take_pinned(c, off_blob + blob_bytes, &r->h_block, &r->h_block_cap));
  unsigned char* blob = static_cast<unsigned char*>(r->h_block) + off_blob;
  if (!s->sel_chunks.empty()) memcpy(blob, s->sel_chunks.data(), s->sel_chunks.size() * sizeof(ChunkDesc));
  FM_CUDA_R(c->d_meta_blob.ensure(blob_bytes));
  FM_CUDA_R(cudaMemcpyAsync(c->d_meta_blob.p, blob, blob_bytes, cudaMemcpyHostToDevice, c->stream));
  const ChunkDesc* d_chunk = c->d_meta_blob.as<ChunkDesc>();

  uint32_t max_rows = 1, max_chunks = 1;
  for (auto& b : s->sel_batches) { max_rows = std::max(max_rows, b.rows); max_chunks = std::max(max_chunks, b.chunks); }
  FM_CUDA_R(c->d_rowres.ensure((size_t)max_rows * sizeof(uint32_t)));
  if (want_dist) {
    FM_CUDA_R(c->d_rowdist.ensure((size_t)max_rows * sizeof(float)));
    FM_CUDA_R(r->d_dist.ensure(std::max<uint64_t>(total_rows, 1) * sizeof(float)));
  }
  FM_CUDA_R(c->d_chunk_count.ensure((size_t)max_chunks * sizeof(uint32_t)));
  FM_CUDA_R(c->d_chunk_out.ensure((size_t)max_chunks * sizeof(unsigned long long)));
  FM_CUDA_R(c->d_chunk_stage.ensure((size_t)max_chunks * kStageCap * sizeof(uint2)));
  FM_CUDA_R(ensure_chunk_status(c));
  FM_CUDA_R(c->d_totals.ensure(sizeof(DeviceCounters)));
  FM_CUDA_R(r->d_out.ensure(std::max<uint64_t>(total_rows, 1) * sizeof(uint2)));
  FM_CUDA_R(r->d_counts.ensure(std::max<size_t>(r->n_pairs, 1) * sizeof(uint32_t)));
  FM_CUDA_R(cudaMemsetAsync(r->d_counts.p, 0, std::max<size_t>(r->n_pairs, 1) * sizeof(uint32_t), c->stream));
  FM_CUDA_R(cudaMemsetAsync(c->d_totals.p, 0, sizeof(DeviceCounters), c->stream));

  uint32_t* d_rowres = c->d_rowres.as<uint32_t>();
  float* d_rowdist = want_dist ? c->d_rowdist.as<float>() : nullptr;
  DeviceCounters* d_counters = c->d_totals.as<DeviceCounters>();
  {
    Span total_span(&c->ev_match, c->stream, kPhTotal);
    for (const SelectBatch& b : s->sel_batches) {
      if (b.rows == 0) continue;
      {
        Span sp(&c->ev_match, c->stream, kPhRescore);
        const uint32_t grid = std::min<uint32_t>((b.rows + kSelectThreads - 1) / kSelectThreads, (uint32_t)c->sm_count * 16u);
        select_kernel<<<grid, kSelectThreads, 0, c->stream>>>(s->d_table.as<fm_row>() + b.row0, b.rows, dist, ratio, d_rowres,
                                                              d_rowdist);
        c->stats.kernel_launches++;
      }
      {
        Span sp(&c->ev_match, c->stream, kPhCompact);
        CompactArgs ca{};
        ca.chunks = d_chunk + b.chunk0;
        ca.n_chunks = b.chunks;
        ca.rowres = d_rowres;
        ca.rowdist = d_rowdist;
        ca.pair_count = r->d_counts.as<uint32_t>();
        ca.running_total = &d_counters->running_total;
        ca.out_pairs = r->d_out.as<uint2>();
        ca.out_dist = want_dist ? r->d_dist.as<float>() : nullptr;
        c->stats.kernel_launches += compact_launch(c, ca, want_dist, FM_COMPACT_AUTO);
      }
    }
  }
  FM_CUDA_R(cudaGetLastError());
  FM_CUDA_R(queue_tail(c, r));
#undef FM_CUDA_R
  if (!(flags & FM_FLAG_ASYNC)) {
    int rc = fm_result_wait(r);
    if (rc != FM_OK) { fm_result_free(r); return rc; }
  }
  *out = r;
  return FM_OK;
}

// fm_result_select on a group result: each member selects on its part of the call, and the lists are gathered on the
// lead exactly as fm_group_match gathers them.
int select_group(const fm_result* s, float dist, float ratio, uint32_t flags, fm_result** out) {
  fm_group* g = s->group;
  fm_ctx* lead = g->m[0];
  fm_result* r = new (std::nothrow) fm_result();
  if (!r) return fail(lead, FM_ERR_NOMEM, "fm_result_select: out of host memory");
  r->ctx = lead;
  r->n_pairs = s->n_pairs;
  r->flags = flags;
  r->ratio = ratio;
  r->group = g;
  auto bail = [&](int code) {
    for (auto* c : g->m) { cudaSetDevice(c->device); cudaStreamSynchronize(c->stream); }
    fm_result_free(r);
    return code;
  };
  // members store into lead buffers only behind this event (see fm_group_match)
  cudaError_t e = cudaSetDevice(lead->device);
  if (e == cudaSuccess) e = cudaEventRecord(g->ev_lead, lead->stream);
  if (e != cudaSuccess) return bail(cuda_fail(lead, e, "fm_result_select"));
  for (const GroupPart& sp : s->parts) {
    fm_result* q = nullptr;
    if (int rc = select_one(sp.sub, dist, ratio, (flags & FM_FLAG_DISTANCES) | FM_FLAG_ASYNC | FM_FLAG_DEVICE_ONLY, &q))
      return bail(member_fail(g, sp.member, rc));
    r->parts.push_back(GroupPart{});
    GroupPart& gp = r->parts.back();
    gp.sub = q;
    gp.member = sp.member;
    gp.idx = sp.idx;
    r->slots += q->slots;
  }
  if (int rc = group_gather(g, r)) return bail(rc);
  if (!(flags & FM_FLAG_ASYNC)) {
    int rc = fm_result_wait(r);
    if (rc != FM_OK) { fm_result_free(r); return rc; }
  }
  *out = r;
  return FM_OK;
}

}  // namespace

extern "C" {

int fm_result_select(const fm_result* r, float dist, float dist2second, uint32_t flags, fm_result** out) {
  if (!r || !out) return FM_ERR_INVALID;
  *out = nullptr;
  fm_ctx* c = r->ctx;
  if (flags & ~(FM_FLAG_DISTANCES | FM_FLAG_DEVICE_ONLY | FM_FLAG_ASYNC))
    return fail(c, FM_ERR_INVALID, "fm_result_select: flags other than FM_FLAG_DISTANCES, FM_FLAG_DEVICE_ONLY and FM_FLAG_ASYNC");
  if (!r->table) return fail(c, FM_ERR_INVALID, "fm_result_select: the result has no row table (FM_FLAG_ROW_TABLE)");
  if (dist != dist || dist2second != dist2second) return fail(c, FM_ERR_INVALID, "fm_result_select: NaN threshold");
  if (!(dist < 1.8e19f)) return fail(c, FM_ERR_UNSUPPORTED, "fm_result_select: distance threshold must be below 1.8e19");
  return r->group ? select_group(r, dist, dist2second, flags, out) : select_one(r, dist, dist2second, flags, out);
}

const fm_row* fm_result_rows_device(const fm_result* r) {
  return (r && r->table && !r->group) ? r->d_table.as<fm_row>() : nullptr;
}

uint64_t fm_result_row_offset(const fm_result* r, size_t p) {
  return (r && r->table && p <= r->n_pairs) ? r->row_off[p] : UINT64_MAX;
}

int fm_result_rows_copy(fm_result* r, size_t p, fm_row* dst) {
  if (!r) return FM_ERR_INVALID;
  if (!r->table || p >= r->n_pairs || !dst) return fail(r->ctx, FM_ERR_INVALID, "fm_result_rows_copy: no row table, bad pair or null dst");
  const fm_result* t = r->group ? r->parts[r->pair_part[p]].sub : r;  // the result holding the pair's rows
  const size_t q = r->group ? r->pair_local[p] : p;
  fm_ctx* c = t->ctx;
  const uint64_t n = t->row_off[q + 1] - t->row_off[q];
  FM_CUDA(r->ctx, cudaSetDevice(c->device));
  if (n) FM_CUDA(r->ctx, cudaMemcpyAsync(dst, t->d_table.as<fm_row>() + t->row_off[q], n * sizeof(fm_row), cudaMemcpyDeviceToHost, c->stream));
  FM_CUDA(r->ctx, cudaStreamSynchronize(c->stream));
  return FM_OK;
}

// ---- debug / test hooks (include/frogmatch_debug.h) ---------------------------------------------

int fm_debug_set_option(const char* name, int value) {
  if (!name) return FM_ERR_INVALID;
  if (!strcmp(name, "probe")) g_debug.probe = value;
  else if (!strcmp(name, "variant")) g_debug.variant = value;
  else if (!strcmp(name, "pre_tiles")) g_debug.pre_tiles = value;
  else if (!strcmp(name, "two_phase")) g_debug.two_phase = value;
  else if (!strcmp(name, "surv_cap")) g_debug.surv_cap = value;
  else if (!strcmp(name, "compact_v")) g_debug.compact_v = value;
  else if (!strcmp(name, "reject_dump")) g_debug.reject_dump = value;
  else if (!strcmp(name, "group_repeat")) g_debug.group_repeat = value;
  else return FM_ERR_INVALID;
  return FM_OK;
}

int fm_debug_image(fm_ctx* c, uint32_t img, uint32_t* flags, uint32_t* n_classes, float* class_lap,
                   uint32_t* class_begin, float* max_norm2, uint32_t* perm, float* scale_sorted,
                   uint16_t* rowop, uint16_t* colop) {
  if (!c || img >= c->images.size() || !c->images[img].valid) return FM_ERR_INVALID;
  FM_CUDA(c, cudaSetDevice(c->device));
  int rc = sync_images(c);
  if (rc != FM_OK) return rc;
  const ImageMeta& m = c->h_metas[img];
  const Image& im = c->images[img];
  const ImageDev& v = c->h_images[img];
  if (flags) *flags = m.flags;
  if (n_classes) *n_classes = m.n_classes;
  if (max_norm2) *max_norm2 = m.max_norm2;
  if (class_lap) memcpy(class_lap, m.class_lap, sizeof m.class_lap);
  if (class_begin) memcpy(class_begin, m.class_begin, sizeof m.class_begin);
  if (perm && im.n) FM_CUDA(c, cudaMemcpy(perm, v.perm, im.n * 4, cudaMemcpyDeviceToHost));
  if (scale_sorted && im.n) FM_CUDA(c, cudaMemcpy(scale_sorted, v.scale_sorted, im.n * 4, cudaMemcpyDeviceToHost));
  for (int role = 0; role < 2; role++) {
    uint16_t* dst = role ? colop : rowop;
    const __half* src = role ? v.colop : v.rowop;
    if (!dst) continue;
    if (!src) return fail(c, FM_ERR_INVALID, "fm_debug_image: image has no FP16 operands (d != 48)");
    std::vector<uint8_t> raw((size_t)v.n_pad * 128);
    FM_CUDA(c, cudaMemcpy(raw.data(), src, raw.size(), cudaMemcpyDeviceToHost));
    for (uint32_t s = 0; s < v.n_pad; s++)  // undo the SWIZZLE_128B tile layout
      for (uint32_t q = 0; q < 8; q++)
        memcpy(dst + (size_t)s * 64 + q * 8, raw.data() + (size_t)(s >> 7) * 16384 + sw128_offset(s & 127u, q), 16);
  }
  return FM_OK;
}

int fm_debug_image_norms(fm_ctx* c, uint32_t img, float* min_norm2_out, float* max_norm2, float* max_delta2) {
  if (!c || img >= c->images.size() || !c->images[img].valid) return FM_ERR_INVALID;
  FM_CUDA(c, cudaSetDevice(c->device));
  int rc = sync_images(c);
  if (rc != FM_OK) return rc;
  const ImageMeta& m = c->h_metas[img];
  if (min_norm2_out) *min_norm2_out = min_norm2(m);
  if (max_norm2) *max_norm2 = m.max_norm2;
  if (max_delta2) *max_delta2 = m.max_delta2;
  return FM_OK;
}

int fm_debug_score_unit(fm_ctx* c, uint32_t first_img, uint32_t second_img, uint32_t row_block, float* t_out,
                        uint32_t ld, uint32_t* bands_out, float* cand_t, uint32_t* cand_col) {
  if (!c || first_img >= c->images.size() || second_img >= c->images.size() || !c->images[first_img].valid ||
      !c->images[second_img].valid || c->dim != (uint32_t)kD)
    return FM_ERR_INVALID;
  FM_CUDA(c, cudaSetDevice(c->device));
  int rc = sync_images(c);
  if (rc != FM_OK) return rc;
  const uint32_t nB = c->images[second_img].n;
  const uint32_t n_pad_a = c->h_images[first_img].n_pad;
  if (row_block * kUnitRows >= nB || ld < n_pad_a) return fail(c, FM_ERR_INVALID, "fm_debug_score_unit: bad row block or ld");
  Task task{first_img, second_img, 0, 0};
  const uint32_t blocks = (nB + 127) / 128, units = (nB + kUnitRows - 1) / kUnitRows;
  uint32_t meta[4] = {0, blocks, 0, units};
  DevBuf d_task, d_meta, d_dump;
  FM_CUDA(c, d_task.ensure(sizeof task));
  FM_CUDA(c, d_meta.ensure(sizeof meta));
  FM_CUDA(c, d_dump.ensure((size_t)kUnitRows * ld * sizeof(float)));
  FM_CUDA(c, c->d_bands.ensure((size_t)nB * sizeof(uint2)));
  FM_CUDA(c, c->d_cands.ensure((size_t)nB * kTopK * sizeof(Cand)));
  FM_CUDA(c, cudaMemcpyAsync(d_task.p, &task, sizeof task, cudaMemcpyHostToDevice, c->stream));
  FM_CUDA(c, cudaMemcpyAsync(d_meta.p, meta, sizeof meta, cudaMemcpyHostToDevice, c->stream));
  FM_CUDA(c, cudaMemsetAsync(d_dump.p, 0xFF, (size_t)kUnitRows * ld * sizeof(float), c->stream));  // NaN = "not written"
  FM_CUDA(c, cudaFuncSetAttribute(score_kernel<true, 0, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kScoreSmemBytes));
  bands_kernel<<<blocks, 128, 0, c->stream>>>(c->d_images.as<ImageDev>(), d_task.as<Task>(), d_meta.as<uint32_t>(), 1,
                                              c->d_bands.as<uint2>());
  score_kernel<true, 0, 0><<<1, kScoreThreads, kScoreSmemBytes, c->stream>>>(
      c->d_images.as<ImageDev>(), d_task.as<Task>(), d_meta.as<uint32_t>() + 2, 1, 1, c->d_bands.as<uint2>(),
      c->d_cands.as<Cand>(), nullptr, d_dump.as<float>(), ld, row_block, 0, 0.f, 0.f, nullptr, nullptr, nullptr);
  FM_CUDA(c, cudaGetLastError());
  FM_CUDA(c, cudaStreamSynchronize(c->stream));
  const uint32_t r0 = row_block * kUnitRows, nr = std::min<uint32_t>(kUnitRows, nB - r0);
  if (t_out) FM_CUDA(c, cudaMemcpy(t_out, d_dump.p, (size_t)kUnitRows * ld * sizeof(float), cudaMemcpyDeviceToHost));
  if (bands_out) FM_CUDA(c, cudaMemcpy(bands_out, c->d_bands.as<uint2>() + r0, (size_t)nr * sizeof(uint2), cudaMemcpyDeviceToHost));
  if (cand_t && cand_col) {
    std::vector<Cand> h((size_t)nr * kTopK);
    FM_CUDA(c, cudaMemcpy(h.data(), c->d_cands.as<Cand>() + (size_t)r0 * kTopK, h.size() * sizeof(Cand), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < h.size(); i++) { cand_t[i] = h[i].t; cand_col[i] = h[i].col; }
  }
  d_task.release(); d_meta.release(); d_dump.release();
  return FM_OK;
}

int fm_debug_wide_unit(fm_ctx* c, uint32_t first_img, uint32_t second_img, uint32_t row_block, float* t_out, uint32_t ld,
                       uint32_t* bands_out, float* cand_t, uint32_t* cand_col, float* eps_out, uint32_t* k_pad_out) {
  if (!c || first_img >= c->images.size() || second_img >= c->images.size() || !c->images[first_img].valid ||
      !c->images[second_img].valid)
    return FM_ERR_INVALID;
  if (c->dim == (uint32_t)kD || c->dim > (uint32_t)kWideMaxD)
    return fail(c, FM_ERR_INVALID, "fm_debug_wide_unit: the wide path takes descriptor lengths d != 48, d <= 4096");
  FM_CUDA(c, cudaSetDevice(c->device));
  int rc = sync_images(c);
  if (rc != FM_OK) return rc;
  const uint32_t nB = c->images[second_img].n;
  const uint32_t n_pad_a = c->h_images[first_img].n_pad;
  if (row_block * kWdRows >= nB || ld < n_pad_a) return fail(c, FM_ERR_INVALID, "fm_debug_wide_unit: bad row block or ld");
  Task task{first_img, second_img, 0, 0};
  const uint32_t blocks = (nB + kWdRows - 1) / kWdRows;
  uint32_t meta[2] = {0, blocks};
  DevBuf d_task, d_meta, d_dump, d_eps;
  FM_CUDA(c, d_task.ensure(sizeof task));
  FM_CUDA(c, d_meta.ensure(sizeof meta));
  FM_CUDA(c, d_dump.ensure((size_t)kWdRows * ld * sizeof(float)));
  FM_CUDA(c, d_eps.ensure(sizeof(float)));
  FM_CUDA(c, c->d_bands.ensure((size_t)nB * sizeof(uint2)));
  FM_CUDA(c, c->d_cands.ensure((size_t)nB * kTopK * sizeof(Cand)));
  FM_CUDA(c, cudaMemcpyAsync(d_task.p, &task, sizeof task, cudaMemcpyHostToDevice, c->stream));
  FM_CUDA(c, cudaMemcpyAsync(d_meta.p, meta, sizeof meta, cudaMemcpyHostToDevice, c->stream));
  FM_CUDA(c, cudaMemsetAsync(d_dump.p, 0xFF, (size_t)kWdRows * ld * sizeof(float), c->stream));  // NaN = "not computed"
  FM_CUDA(c, cudaFuncSetAttribute(wide_score_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWdSmemBytes));
  bands_kernel<<<blocks, 128, 0, c->stream>>>(c->d_images.as<ImageDev>(), d_task.as<Task>(), d_meta.as<uint32_t>(), 1,
                                              c->d_bands.as<uint2>());
  wide_score_kernel<true><<<1, kWdThreads, kWdSmemBytes, c->stream>>>(
      c->d_images.as<ImageDev>(), d_task.as<Task>(), d_meta.as<uint32_t>(), 1, row_block, row_block + 1, c->d_bands.as<uint2>(),
      c->d_cands.as<Cand>(), nullptr, d_dump.as<float>(), ld, d_eps.as<float>());
  FM_CUDA(c, cudaGetLastError());
  FM_CUDA(c, cudaStreamSynchronize(c->stream));
  const uint32_t r0 = row_block * kWdRows, nr = std::min<uint32_t>(kWdRows, nB - r0);
  if (t_out) FM_CUDA(c, cudaMemcpy(t_out, d_dump.p, (size_t)kWdRows * ld * sizeof(float), cudaMemcpyDeviceToHost));
  if (bands_out) FM_CUDA(c, cudaMemcpy(bands_out, c->d_bands.as<uint2>() + r0, (size_t)nr * sizeof(uint2), cudaMemcpyDeviceToHost));
  if (cand_t && cand_col) {
    std::vector<Cand> h((size_t)nr * kTopK);
    FM_CUDA(c, cudaMemcpy(h.data(), c->d_cands.as<Cand>() + (size_t)r0 * kTopK, h.size() * sizeof(Cand), cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < h.size(); i++) { cand_t[i] = h[i].t; cand_col[i] = h[i].col; }
  }
  if (eps_out) FM_CUDA(c, cudaMemcpy(eps_out, d_eps.p, sizeof(float), cudaMemcpyDeviceToHost));
  if (k_pad_out) *k_pad_out = wide_kpad(c->dim);
  d_task.release(); d_meta.release(); d_dump.release(); d_eps.release();
  return FM_OK;
}

int fm_debug_reject_rows(fm_ctx* c, uint32_t task, uint32_t n_rows, float* args, uint8_t* rowstat, uint32_t* bands,
                         uint32_t* survivors, uint32_t* n_survivors) {
  if (!c) return FM_ERR_INVALID;
  if (task >= c->reject_rows.size() || !c->reject_rows[task].valid)
    return fail(c, FM_ERR_INVALID, "fm_debug_reject_rows: the task did not go through the reject pass of the last fm_match");
  const fm_ctx::RejectRows& st = c->reject_rows[task];
  if (n_rows != st.rowstat.size()) return fail(c, FM_ERR_INVALID, "fm_debug_reject_rows: n_rows is not the task's row count");
  if (args && n_rows) memcpy(args, st.args.data(), (size_t)n_rows * sizeof(float4));
  if (rowstat && n_rows) memcpy(rowstat, st.rowstat.data(), n_rows);
  if (bands && n_rows) memcpy(bands, st.bands.data(), (size_t)n_rows * sizeof(uint2));
  if (survivors && !st.survivors.empty()) memcpy(survivors, st.survivors.data(), st.survivors.size() * sizeof(uint32_t));
  if (n_survivors) *n_survivors = (uint32_t)st.survivors.size();
  return FM_OK;
}

int fm_debug_compact(fm_ctx* c, const uint32_t* rowres, const float* rowdist, uint32_t n_rows, const uint32_t* chunks,
                     uint32_t n_chunks, int path, uint64_t base, uint32_t* out_pairs, float* out_dist, uint64_t out_slots,
                     uint32_t* pair_counts, uint32_t n_pairs, uint64_t* total_out, uint64_t* status_out,
                     uint32_t* epoch_inout) {
  if (!c) return FM_ERR_INVALID;
  if (path < FM_COMPACT_AUTO || path > FM_COMPACT_LOOKALL || n_chunks == 0 || !chunks || !out_pairs || !pair_counts ||
      (n_rows && !rowres) || (rowdist && !out_dist))
    return fail(c, FM_ERR_INVALID, "fm_debug_compact: bad path or missing argument");
  if ((path == FM_COMPACT_ONE || path == FM_COMPACT_LOOKALL) && n_chunks > kOnePassChunks)
    return fail(c, FM_ERR_INVALID, "fm_debug_compact: one launch takes at most 1536 chunks");
  const bool want_dist = rowdist != nullptr;
  uint64_t total = 0;
  for (uint32_t k = 0; k < n_chunks; k++) {
    const ChunkDesc d{chunks[4 * k], chunks[4 * k + 1], chunks[4 * k + 2], chunks[4 * k + 3]};
    const uint32_t n = d.n_swap & 0x7FFFFFFFu;
    if (n > (uint32_t)kCompactChunk || (uint64_t)d.row_abs + n > n_rows || d.pair >= n_pairs)
      return fail(c, FM_ERR_INVALID, "fm_debug_compact: a chunk has more than 4096 rows, reaches past n_rows or names no pair");
    for (uint32_t i = 0; i < n; i++) total += rowres[d.row_abs + i] != kNone;
  }
  if (base + total > out_slots) return fail(c, FM_ERR_INVALID, "fm_debug_compact: base + matches exceeds out_slots");
  FM_CUDA(c, cudaSetDevice(c->device));
  DevBuf d_chunks, d_out, d_dist, d_counts, d_total;
  auto release = [&] { d_chunks.release(); d_out.release(); d_dist.release(); d_counts.release(); d_total.release(); };
#define FM_CUDA_H(expr)                                  \
  do {                                                   \
    cudaError_t e__ = (expr);                            \
    if (e__ != cudaSuccess) {                            \
      release();                                         \
      return cuda_fail(c, e__, #expr);                   \
    }                                                    \
  } while (0)
  FM_CUDA_H(c->d_rowres.ensure(std::max<size_t>(n_rows, 1) * sizeof(uint32_t)));
  if (want_dist) FM_CUDA_H(c->d_rowdist.ensure(std::max<size_t>(n_rows, 1) * sizeof(float)));
  FM_CUDA_H(c->d_chunk_count.ensure((size_t)n_chunks * sizeof(uint32_t)));
  FM_CUDA_H(c->d_chunk_out.ensure((size_t)n_chunks * sizeof(unsigned long long)));
  FM_CUDA_H(c->d_chunk_stage.ensure((size_t)n_chunks * kStageCap * sizeof(uint2)));
  FM_CUDA_H(ensure_chunk_status(c));
  FM_CUDA_H(d_chunks.ensure((size_t)n_chunks * sizeof(ChunkDesc)));
  FM_CUDA_H(d_out.ensure(std::max<uint64_t>(out_slots, 1) * sizeof(uint2)));
  if (want_dist) FM_CUDA_H(d_dist.ensure(std::max<uint64_t>(out_slots, 1) * sizeof(float)));
  FM_CUDA_H(d_counts.ensure(std::max<size_t>(n_pairs, 1) * sizeof(uint32_t)));
  FM_CUDA_H(d_total.ensure(sizeof(unsigned long long)));
  const unsigned long long base_ull = base;
  if (n_rows) FM_CUDA_H(cudaMemcpyAsync(c->d_rowres.p, rowres, (size_t)n_rows * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  if (want_dist && n_rows)
    FM_CUDA_H(cudaMemcpyAsync(c->d_rowdist.p, rowdist, (size_t)n_rows * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  FM_CUDA_H(cudaMemcpyAsync(d_chunks.p, chunks, (size_t)n_chunks * sizeof(ChunkDesc), cudaMemcpyHostToDevice, c->stream));
  if (out_slots) FM_CUDA_H(cudaMemcpyAsync(d_out.p, out_pairs, out_slots * sizeof(uint2), cudaMemcpyHostToDevice, c->stream));
  if (want_dist && out_slots)
    FM_CUDA_H(cudaMemcpyAsync(d_dist.p, out_dist, out_slots * sizeof(float), cudaMemcpyHostToDevice, c->stream));
  if (n_pairs) FM_CUDA_H(cudaMemcpyAsync(d_counts.p, pair_counts, (size_t)n_pairs * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
  FM_CUDA_H(cudaMemcpyAsync(d_total.p, &base_ull, sizeof base_ull, cudaMemcpyHostToDevice, c->stream));
  if (epoch_inout) c->compact_epoch = *epoch_inout;
  CompactArgs ca{};
  ca.chunks = d_chunks.as<ChunkDesc>();
  ca.n_chunks = n_chunks;
  ca.rowres = c->d_rowres.as<uint32_t>();
  ca.rowdist = want_dist ? c->d_rowdist.as<float>() : nullptr;
  ca.pair_count = d_counts.as<uint32_t>();
  ca.running_total = d_total.as<unsigned long long>();
  ca.out_pairs = d_out.as<uint2>();
  ca.out_dist = want_dist ? d_dist.as<float>() : nullptr;
  compact_launch(c, ca, want_dist, path);
  FM_CUDA_H(cudaGetLastError());
  unsigned long long total_dev = 0;
  if (out_slots) FM_CUDA_H(cudaMemcpyAsync(out_pairs, d_out.p, out_slots * sizeof(uint2), cudaMemcpyDeviceToHost, c->stream));
  if (want_dist && out_slots)
    FM_CUDA_H(cudaMemcpyAsync(out_dist, d_dist.p, out_slots * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (n_pairs) FM_CUDA_H(cudaMemcpyAsync(pair_counts, d_counts.p, (size_t)n_pairs * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
  FM_CUDA_H(cudaMemcpyAsync(&total_dev, d_total.p, sizeof total_dev, cudaMemcpyDeviceToHost, c->stream));
  if (status_out)
    FM_CUDA_H(cudaMemcpyAsync(status_out, c->d_chunk_status.p, (size_t)kOnePassChunks * sizeof(unsigned long long),
                              cudaMemcpyDeviceToHost, c->stream));
  FM_CUDA_H(cudaStreamSynchronize(c->stream));
#undef FM_CUDA_H
  release();
  if (total_out) *total_out = total_dev;
  if (epoch_inout) *epoch_inout = c->compact_epoch;
  return FM_OK;
}

}  // extern "C"
