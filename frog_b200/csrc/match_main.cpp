// match_main.cpp -- drop-in replacement for valette/FROG's `bin/match` (match/match.cpp:340-747).
//
//   match <listfile-or-directory> [-o out] [-d dist] [-d2 ratio] [-n N] [-sp thr] [-np n] [-nt threads]
//         [-zmin z] [-zmax z] [-sym] [-targ k] [-all x]   (reference keys, same meaning)
//         [-gpus G] [-exact 1] [-stats file.json] [-gather nccl|host] [-plan 1] [-mp 0|1] [-dists file]
//                                                          (new keys; unknown to the reference)
//
// Same argv quirks (every key consumes two tokens except -sym, match.cpp:365-431), same keypoint
// readers, same stdout protocol, byte-identical pairs.bin.  The pairing phase (match.cpp:638-652)
// runs on B200s through the C ABI of libfrogmatch.so; there is no CPU fallback.
//
// Process model.  CUDA start-up is per process AND per visible device (cuInit: 0.6 s with one
// device visible, 5 s with eight), so a one-shot executable that wants G GPUs runs ONE PROCESS PER
// GPU: before the first CUDA call and before any thread exists, the parent forks G - 1 workers,
// each of which sees exactly one device.  Parent and workers share one anonymous MAP_SHARED arena
// created before the fork (inherited at the same address, released by the kernel when the
// processes exit: nothing to clean up, nothing to leak):
//   * the parent parses the keypoint files (OpenMP, as match.cpp:508-570 does) and drops every
//     finished image's descriptors into the arena; every worker -- worker 0 is a thread of the
//     parent -- uploads an image to its GPU as soon as it is marked ready, so host-to-device copies
//     and CUDA start-up both hide under the parsing;
//   * when all images are in, the parent shards the image pairs (longest processing time first)
//     and publishes each worker's share; workers match, copy their compacted lists into the arena
//     and leave with _exit; the parent writes pairs.bin in the reference's block order.
// `-gather nccl` sends the lists GPU-to-GPU over NVLink to worker 0 instead (one communicator rank
// per worker) -- identical bytes, but communicator start-up costs more than it saves a one-shot run.
//
// Volume entries.  A list entry ending in ".mha" or ".mhd" is a MetaImage volume (data in the header's file or in the
// file it names; raw or compressed, either byte order, the element types fsio::read_metaimage lists): the load loop
// reads it (in parallel, like the keypoint files) and hands it to the SURF3D producer, which yields exactly the
// keypoints that `surf3d <volume> <options>` followed by the .csv.gz reader would (`-surf3d "<surf3d options>"`, one token; the
// conversion to the text's values runs on the device, fs_get_points_as_read).  This removes a process start -- and so
// a CUDA start-up, ~0.55 s -- and a text round trip per volume.  Producer calls go to ONE fs_ctx on this process's
// GPU 0, created by the first volume after the workers are forked and used by one loader thread at a time: a 400^3
// volume takes ~10.5 ms there, so one GPU produces faster than a disk delivers volumes.  libfrogsurf.so is dlopen'ed
// only when the list holds a volume, so a deployment for keypoint files needs libfrogmatch.so alone.  A resident
// server keeps its producer context from job to job.
#include <dlfcn.h>
#include <omp.h>
#include <sys/mman.h>
#include <sys/wait.h>
#include <unistd.h>

#include <algorithm>
#include <array>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <iostream>
#include <mutex>
#include <numeric>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "frogmatch.h"
#include "fm_shard.h"
#include "frogsurf.h"
#include "keypoint_io.h"
#include "surf_io.h"

#ifdef FM_WITH_NCCL
#include <cuda_runtime.h>
#include <nccl.h>
#endif

namespace fs = std::filesystem;
using std::cerr;
using std::cout;
using std::endl;
using std::string;

namespace {

constexpr int kMaxWorkers = 64;

double now_s() {
  return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ---- the shared arena ---------------------------------------------------------------------------------

enum WorkerState : uint32_t { kStarting = 0, kContextUp = 1, kCountsOut = 2, kDone = 3, kFailed = 4 };

struct WorkerSlot {
  std::atomic<uint32_t> state;
  char error[480];
  char device[64];  // this worker's CUDA_VISIBLE_DEVICES entry (forked workers)
  // plan, written by the parent before Control::plan_ready
  uint64_t pairs_off;  // uint32 first[n_pairs] | uint32 second[n_pairs]
  uint64_t n_pairs;
  // result, written by the worker before state = kCountsOut (counts, total) / kDone (lists, distances)
  uint64_t counts_off, lists_off, dists_off, total;
  fm_stats stats;
  double create_s, upload_s, match_s, gather_s, nccl_init_s;
};

struct ImageSlot {
  std::atomic<uint32_t> ready;  // 1 once n, d and the three arrays are in place
  uint32_t n, d;
  uint64_t desc_off, scale_off, lap_off;
};

struct Control {
  std::atomic<uint64_t> bump;  // next free byte of the arena
  uint64_t arena_bytes;
  std::atomic<uint32_t> abort;       // somebody failed: everybody leaves
  std::atomic<uint32_t> plan_ready;  // pair shards published
  std::atomic<uint32_t> nccl_id_ready;
  uint32_t n_images, n_workers, dim;
  float dist, ratio;
  uint32_t flags;
  uint32_t use_nccl;
  unsigned char nccl_id[128];
  WorkerSlot worker[kMaxWorkers];
  // ImageSlot image[n_images] follows
  ImageSlot* images() { return reinterpret_cast<ImageSlot*>(this + 1); }
  char* base() { return reinterpret_cast<char*>(this); }
  template <class T> T* at(uint64_t off) { return reinterpret_cast<T*>(base() + off); }
  // 0 = the arena is exhausted
  uint64_t alloc(uint64_t bytes) {
    bytes = (bytes + 255) & ~(uint64_t)255;
    const uint64_t off = bump.fetch_add(bytes);
    return off + bytes <= arena_bytes ? off : 0;
  }
};

Control* map_arena(size_t n_images, uint64_t estimate_bytes) {
  const uint64_t head = sizeof(Control) + n_images * sizeof(ImageSlot);
  // Virtual space is free (pages are committed when touched): reserve far more than any group needs; a kernel that
  // refuses (strict overcommit) gets a request sized from the input files instead.
  const uint64_t tries[2] = {(uint64_t)1 << 40, head + estimate_bytes + ((uint64_t)64 << 20)};
  for (uint64_t bytes : tries) {
    void* p = mmap(nullptr, bytes, PROT_READ | PROT_WRITE, MAP_SHARED | MAP_ANONYMOUS | MAP_NORESERVE, -1, 0);
    if (p == MAP_FAILED) continue;
    Control* c = new (p) Control();
    c->arena_bytes = bytes;
    c->bump.store((head + 4095) & ~(uint64_t)4095);
    for (size_t i = 0; i < n_images; i++) new (c->images() + i) ImageSlot();
    return c;
  }
  return nullptr;
}

void worker_fail(Control* ctl, int g, const string& msg) {
  WorkerSlot& w = ctl->worker[g];
  snprintf(w.error, sizeof w.error, "%s", msg.c_str());
  w.state.store(kFailed);
  ctl->abort.store(1);
}

template <class Pred>
bool wait_for(Control* ctl, Pred ready) {  // false = aborted
  for (unsigned spins = 0; !ready(); spins++) {
    if (ctl->abort.load()) return false;
    if (spins < 64) std::this_thread::yield();
    else usleep(100);
  }
  return true;
}

#ifdef FM_WITH_NCCL
struct NcclRank {
  ncclComm_t comm = nullptr;
  cudaStream_t stream = nullptr;
  string error;
  double init_s = 0;
  void init(Control* ctl, int g, int device) {
    const double t0 = now_s();
    ncclUniqueId id;
    static_assert(sizeof(ncclUniqueId) <= sizeof(Control::nccl_id), "unique id does not fit");
    if (g == 0) {
      ncclResult_t r = ncclGetUniqueId(&id);
      if (r != ncclSuccess) { error = string("ncclGetUniqueId: ") + ncclGetErrorString(r); return; }
      memcpy(ctl->nccl_id, &id, sizeof id);
      ctl->nccl_id_ready.store(1);
    } else {
      if (!wait_for(ctl, [&] { return ctl->nccl_id_ready.load() != 0; })) { error = "aborted"; return; }
      memcpy(&id, ctl->nccl_id, sizeof id);
    }
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking);
    if (e != cudaSuccess) { error = string("NCCL gather stream: ") + cudaGetErrorString(e); return; }
    ncclResult_t r = ncclCommInitRank(&comm, (int)ctl->n_workers, id, g);
    if (r != ncclSuccess) { error = string("ncclCommInitRank: ") + ncclGetErrorString(r); comm = nullptr; return; }
    init_s = now_s() - t0;
  }
};
#endif

// One worker = one GPU.  Runs as a thread of the parent (worker 0, and every worker with -mp 0) or as the main
// thread of a forked process that sees a single device.
// `warm`: a context a resident server already holds for this device (see serve()); else one is created here.
void worker_run(Control* ctl, int g, int device, fm_ctx* warm) {
  WorkerSlot& w = ctl->worker[g];
  double t0 = now_s();
  fm_ctx* ctx = warm;
  if (ctx) {
    if (fm_clear_images(ctx) != FM_OK) { worker_fail(ctl, g, fm_last_error(ctx)); return; }
  } else if (fm_create(device, &ctx) != FM_OK) {
    worker_fail(ctl, g, fm_last_error(nullptr));
    return;
  }
  w.create_s = now_s() - t0;
  w.state.store(kContextUp);
#ifdef FM_WITH_NCCL
  NcclRank nccl;
  std::thread nccl_thread;
  if (ctl->use_nccl) nccl_thread = std::thread([&] { nccl.init(ctl, g, device); });
  struct Join { std::thread& t; ~Join() { if (t.joinable()) t.join(); } } join_nccl{nccl_thread};
#endif

  // ---- uploads, image by image as the parent finishes parsing them ----
  double upload_busy = 0;
  std::vector<uint32_t> empty;  // images without keypoints: uploaded last, with the group's descriptor length
  for (uint32_t i = 0; i < ctl->n_images; i++) {
    ImageSlot& im = ctl->images()[i];
    if (!wait_for(ctl, [&] { return im.ready.load() != 0; })) return;
    if (im.n == 0) { empty.push_back(i); continue; }
    t0 = now_s();
    if (fm_upload_image(ctx, i, ctl->at<float>(im.desc_off), ctl->at<float>(im.scale_off), ctl->at<float>(im.lap_off), im.n, im.d) != FM_OK) {
      worker_fail(ctl, g, fm_last_error(ctx));
      return;
    }
    upload_busy += now_s() - t0;
  }
  if (!wait_for(ctl, [&] { return ctl->plan_ready.load() != 0; })) return;
  for (uint32_t i : empty) {
    // match.cpp gives an image without keypoints zero matches whatever the others' descriptor length is
    const float none = 0.f;
    if (fm_upload_image(ctx, i, &none, &none, &none, 0, ctl->dim ? ctl->dim : 48u) != FM_OK) { worker_fail(ctl, g, fm_last_error(ctx)); return; }
  }
  t0 = now_s();
  if (fm_synchronize(ctx) != FM_OK) { worker_fail(ctl, g, fm_last_error(ctx)); return; }
  w.upload_s = upload_busy + (now_s() - t0);

  // ---- this worker's image pairs ----
  t0 = now_s();
  const uint32_t* pf = ctl->at<uint32_t>(w.pairs_off);
  const uint32_t* ps = pf + w.n_pairs;
  bool via_nccl = false;
#ifdef FM_WITH_NCCL
  if (ctl->use_nccl) {
    if (nccl_thread.joinable()) nccl_thread.join();
    if (!nccl.error.empty()) { worker_fail(ctl, g, "NCCL gather unavailable: " + nccl.error); return; }
    via_nccl = true;
    w.nccl_init_s = nccl.init_s;
  }
#endif
  fm_result* res = nullptr;
  const uint32_t flags = ctl->flags | ((via_nccl && g > 0) ? FM_FLAG_DEVICE_ONLY : 0u);
  if (fm_match(ctx, pf, ps, w.n_pairs, ctl->dist, ctl->ratio, flags, &res) != FM_OK) { worker_fail(ctl, g, fm_last_error(ctx)); return; }
  fm_get_stats(ctx, &w.stats);
  w.match_s = now_s() - t0;

  // ---- hand the lists over ----
  t0 = now_s();
  w.total = fm_result_total(res);
  w.counts_off = ctl->alloc(std::max<uint64_t>(w.n_pairs, 1) * sizeof(uint32_t));
  const bool want_dist = ctl->flags & FM_FLAG_DISTANCES;
  if (!via_nccl || g == 0) {
    w.lists_off = ctl->alloc(std::max<uint64_t>(w.total, 1) * 2 * sizeof(uint32_t));
    if (want_dist) w.dists_off = ctl->alloc(std::max<uint64_t>(w.total, 1) * sizeof(float));
  }
  if (!w.counts_off || ((!via_nccl || g == 0) && (!w.lists_off || (want_dist && !w.dists_off)))) {
    worker_fail(ctl, g, "shared arena exhausted while publishing the match lists");
    return;
  }
  uint32_t* counts = ctl->at<uint32_t>(w.counts_off);
  for (uint64_t p = 0; p < w.n_pairs; p++) counts[p] = fm_result_count(res, p);
  if ((!via_nccl || g == 0) && w.total) {
    memcpy(ctl->at<uint32_t>(w.lists_off), fm_result_pairs(res, 0), w.total * 2 * sizeof(uint32_t));
    if (want_dist) memcpy(ctl->at<float>(w.dists_off), fm_result_distances(res, 0), w.total * sizeof(float));
  }
  w.state.store(kCountsOut);
#ifdef FM_WITH_NCCL
  if (via_nccl) {
    // Lists of workers 1.. travel GPU-to-GPU to worker 0 (ncclSend / ncclRecv over NVLink) and reach the host in ONE
    // device-to-host copy there, mirroring the single writer of match.cpp:660-745.  (Distances stay a host-path
    // feature: -dists with -gather nccl is refused in main.)
    auto cu = [&](cudaError_t e, const char* what) {
      if (e != cudaSuccess) { worker_fail(ctl, g, string(what) + ": " + cudaGetErrorString(e)); return false; }
      return true;
    };
    auto nc = [&](ncclResult_t r, const char* what) {
      if (r != ncclSuccess) { worker_fail(ctl, g, string(what) + ": " + ncclGetErrorString(r)); return false; }
      return true;
    };
    if (g > 0) {
      if (w.total) {
        if (!nc(ncclSend(fm_result_device_pairs(res), 2 * w.total, ncclUint32, 0, nccl.comm, nccl.stream), "ncclSend")) return;
        if (!cu(cudaStreamSynchronize(nccl.stream), "gather synchronize")) return;
      }
    } else {
      uint64_t elems = 0;
      std::vector<uint64_t> off(ctl->n_workers, 0);
      for (uint32_t k = 1; k < ctl->n_workers; k++) {
        if (!wait_for(ctl, [&] { return ctl->worker[k].state.load() >= kCountsOut; })) return;
        off[k] = elems;
        elems += 2 * ctl->worker[k].total;
      }
      if (elems) {
        uint32_t* d_stage = nullptr;
        const uint64_t stage_off = ctl->alloc(elems * sizeof(uint32_t));
        if (!stage_off) { worker_fail(ctl, g, "shared arena exhausted (NCCL gather)"); return; }
        if (!cu(cudaSetDevice(device), "cudaSetDevice")) return;
        if (!cu(cudaMalloc(reinterpret_cast<void**>(&d_stage), elems * sizeof(uint32_t)), "cudaMalloc(gather stage)")) return;
        if (!nc(ncclGroupStart(), "ncclGroupStart")) return;
        for (uint32_t k = 1; k < ctl->n_workers; k++)
          if (ctl->worker[k].total && !nc(ncclRecv(d_stage + off[k], 2 * ctl->worker[k].total, ncclUint32, (int)k, nccl.comm, nccl.stream), "ncclRecv")) return;
        if (!nc(ncclGroupEnd(), "ncclGroupEnd")) return;
        if (!cu(cudaMemcpyAsync(ctl->at<uint32_t>(stage_off), d_stage, elems * sizeof(uint32_t), cudaMemcpyDeviceToHost, nccl.stream), "gather D2H")) return;
        if (!cu(cudaStreamSynchronize(nccl.stream), "gather synchronize")) return;
        for (uint32_t k = 1; k < ctl->n_workers; k++) ctl->worker[k].lists_off = stage_off + off[k] * sizeof(uint32_t);
      }
    }
  }
#endif
  w.gather_s = now_s() - t0;
  if (warm) {  // a resident server keeps the context: hand the result's buffers back to it
    fm_result_free(res);
#ifdef FM_WITH_NCCL
    if (nccl.comm) ncclCommDestroy(nccl.comm);
    if (nccl.stream) cudaStreamDestroy(nccl.stream);
#endif
  }
  w.state.store(kDone);
  // One-shot runs do not tear the context, its device memory or the communicator down: the process is about to
  // leave, and destroying one CUDA context per GPU costs more than everything above.
}

// ---- volume entries: the SURF3D producer (libfrogsurf.so, loaded at run time) --------------------------------------

bool is_volume(const string& f) {
  return f.size() > 4 && (f.compare(f.size() - 4, 4, ".mha") == 0 || f.compare(f.size() - 4, 4, ".mhd") == 0);
}

struct SurfApi {
  void* handle = nullptr;
  // (frogsurf.h's declarations give the types; nothing here links against them)
  decltype(&fs_create) create = nullptr;
  decltype(&fs_last_error) last_error = nullptr;
  decltype(&fs_set_volume) set_volume = nullptr;
  decltype(&fs_detect) detect = nullptr;
  decltype(&fs_select) select = nullptr;
  decltype(&fs_describe) describe = nullptr;
  decltype(&fs_num_points) num_points = nullptr;
  decltype(&fs_get_points_as_read) get_points_as_read = nullptr;
  decltype(&fs_get_stats) get_stats = nullptr;

  // dlopen searches the executable's run path ($ORIGIN/../frog_b200), then the usual places
  bool load(string& err) {
    if (handle) return true;
    void* h = dlopen("libfrogsurf.so", RTLD_NOW | RTLD_LOCAL);
    if (!h) { err = dlerror(); return false; }
    bool ok = true;
    auto sym = [&](auto& fn, const char* name) {
      fn = reinterpret_cast<std::remove_reference_t<decltype(fn)>>(dlsym(h, name));
      if (!fn) { ok = false; err = string("libfrogsurf.so lacks ") + name; }
    };
    sym(create, "fs_create");
    sym(last_error, "fs_last_error");
    sym(set_volume, "fs_set_volume");
    sym(detect, "fs_detect");
    sym(select, "fs_select");
    sym(describe, "fs_describe");
    sym(num_points, "fs_num_points");
    sym(get_points_as_read, "fs_get_points_as_read");
    sym(get_stats, "fs_get_stats");
    if (!ok) { dlclose(h); return false; }
    handle = h;
    return true;
  }
};

// One producer context for all volume entries of a job: created by the first volume that needs it, used by one
// loader thread at a time (an fs_ctx is one-host-thread-at-a-time).
struct VolumeProducer {
  SurfApi* api = nullptr;
  fs_ctx** ctx = nullptr;  // a resident server's, kept across jobs, or this job's
  std::mutex mu;
  uint32_t volumes = 0;
  double busy_s = 0, gpu_ms = 0;
};

// `surf3d <path> <options>` then fmio::read_keypoints of the .csv.gz it writes, without the file
bool produce_keypoints(const string& path, const fsio::SurfOptions& o, VolumeProducer& P, fmio::KeypointSet& k, string& err) {
  fsio::Volume vol;
  if (!fsio::read_metaimage(path, vol, err, stderr)) return false;
  fsio::clamp_volume(vol, o);
  std::lock_guard<std::mutex> lock(P.mu);
  const double t0 = now_s();
  const SurfApi& F = *P.api;
  if (!*P.ctx && F.create(0, P.ctx) != FS_OK) { err = string("SURF3D producer: ") + F.last_error(nullptr); return false; }
  fs_ctx* c = *P.ctx;
  uint32_t n = 0, d = 0;
  auto die = [&](const char* what) { err = string("SURF3D producer, ") + what + ": " + F.last_error(c); return false; };
  if (F.set_volume(c, vol.data.data(), vol.voxel_type, vol.dims[0], vol.dims[1], vol.dims[2]) != FS_OK) return die("volume");
  if (F.detect(c, (float)o.threshold, &n) != FS_OK) return die("detector");
  if (F.select(c, o.numberOfPoints) != FS_OK) return die("select");
  if (F.describe(c, o.descriptorType, o.subVolumeRadius, o.normalize) != FS_OK) return die("descriptors");
  F.num_points(c, &n, &d);
  k = fmio::KeypointSet{};
  k.n = n;
  k.d = n ? d : 0;  // an empty file: no row, no length
  k.head.resize((size_t)n * 6);
  k.desc.resize((size_t)n * d);
  if (F.get_points_as_read(c, o.precision, vol.spacing, vol.origin, k.head.data(), k.desc.data()) != FS_OK) return die("read back");
  fs_stats st{};
  F.get_stats(c, &st);
  P.gpu_ms += (double)st.ms_integral + st.ms_response_map + st.ms_extrema + st.ms_describe;
  P.volumes++;
  P.busy_s += now_s() - t0;
  return true;
}

// Contexts a resident server (`match -serve-daemon`) keeps warm: one per visible device, and the producer's once a
// job has needed it.
struct WarmPool {
  std::vector<fm_ctx*> ctx;
  SurfApi surf_api;
  fs_ctx* surf = nullptr;
};

}  // namespace

// One `match` invocation.  `cout` / `cerr` are the caller's streams (a resident server relays them to its client);
// with a WarmPool the GPUs' contexts already exist and no process is forked.
int run_job(int argc, char* argv[], std::ostream& cout, std::ostream& cerr, WarmPool* warm) {
  std::chrono::time_point<std::chrono::system_clock> start, end;
  int N = 1000000;
  float sp = 0;
  int np = 1000000;
  int nt = (int)std::thread::hardware_concurrency();
  if (argc < 2) {
    cout << "Usage : match pointFiles.txt [options] " << endl;  // match.cpp:347-350
    return 1;
  }
  fs::path full_path = fs::absolute(fs::path(argv[1]));
  float dist = 0.22f;  // match.cpp:352 `float dist = 0.22`
  float dist2second = 1;
  float zmin = -1e20f, zmax = 1e20f;
  bool matchAll = false, writePoints = false, symFlag = false, forceExact = false;
  char* outputFileName = nullptr;
  float anatVal = 0.0f;
  int target = -1;
  int gpus = -1;
  const char* statsFile = nullptr;
  const char* distsFile = nullptr;  // -dists f: squared distance of every emitted match (float32, block order of pairs.bin)
  bool planOnly = false;            // -plan 1: print the GPU plan (no CUDA call is made) and exit
  bool multiProcess = false;        // -mp 1: one forked worker process per GPU instead of one thread per GPU
  bool serveMode = false;           // -serve 1: handled by main(): run inside the resident server (warm CUDA contexts)
  // How the lists of GPUs 1.. reach the writer: "host" = every GPU copies its own lists over its own PCIe link,
  // "nccl" = GPU-to-GPU over NVLink to GPU 0, then one device-to-host copy.  Bringing the communicators up costs a
  // one-shot process more than matching a 50 x 50k group, so "host" is the default here.
  const char* gatherMode = "host";
  const char* surfArgs = "";  // -surf3d "<options>": bin/surf3d's options for the volume entries

  // match.cpp:365-431: key = argv[k], value = argv[k+1]; advance by 2, by 1 for -sym.
  for (int k = 2; k < argc;) {
    const char* key = argv[k];
    const char* value = (k + 1 < argc) ? argv[k + 1] : nullptr;
    auto has = [&](const char* name) { return strcmp(key, name) == 0; };
    if (value) {
      if (has("-n")) N = atoi(value);
      if (has("-sp")) sp = (float)atof(value);
      if (has("-np")) np = atoi(value);
      if (has("-nt")) nt = atoi(value);
      if (has("-d")) dist = (float)atof(value);
      if (has("-d2")) dist2second = (float)atof(value);
      if (has("-zmin")) zmin = (float)atof(value);
      if (has("-zmax")) zmax = (float)atof(value);
      if (has("-o")) outputFileName = argv[k + 1];
      if (has("-anat")) anatVal = (float)atof(value);
      if (has("-targ")) target = atoi(value);
      if (has("-gpus")) gpus = atoi(value);
      if (has("-exact")) forceExact = atoi(value) != 0;
      if (has("-stats")) statsFile = value;
      if (has("-dists")) distsFile = value;
      if (has("-gather")) gatherMode = value;
      if (has("-plan")) planOnly = atoi(value) != 0;
      if (has("-mp")) multiProcess = atoi(value) != 0;
      if (has("-serve")) serveMode = atoi(value) != 0;
      if (has("-surf3d")) surfArgs = value;
    }
    if (has("-all")) matchAll = true;
    if (has("-p")) writePoints = true;
    if (has("-sym")) { symFlag = true; k -= 1; }
    k += 2;
  }
  if (anatVal != 0.0f) {
    cerr << "match: -anat is not supported (the reference reads uninitialised transformedCoordinates, "
            "match.cpp:548-559)" << endl;
    return 1;
  }
  if (writePoints) cerr << "match: -p (debug CSV dump) is ignored by the B200 build" << endl;
  // bin/surf3d's own option loop and refusals; the file-output keys (-o -bin -csv -csvgz -gz) and -gpu have nothing
  // to act on here
  std::vector<string> surfTokens;
  {
    std::istringstream ss(surfArgs);
    for (string t; ss >> t;) surfTokens.push_back(t);
  }
  std::vector<char*> surfArgv;
  for (string& t : surfTokens) surfArgv.push_back(&t[0]);
  fsio::SurfOptions surfOpts;
  fsio::parse_surf_options((int)surfArgv.size(), surfArgv.data(), 0, surfOpts);
  if (const char* what = fsio::unsupported_surf_option(surfOpts)) {
    cerr << fsio::unsupported_surf_message(what) << endl;
    return 7;
  }
  if (surfOpts.pointFile) {
    cerr << "match: -surf3d -p (descriptors at the points of a csv file) is not available for volume entries; terminating." << endl;
    return 7;
  }
  const bool want_nccl = strcmp(gatherMode, "nccl") == 0;
  if (distsFile && (matchAll || want_nccl)) {
    cerr << "match: -dists is not available with -all or -gather nccl" << endl;
    return 1;
  }

  std::vector<std::array<double, 3>> rigids;
  std::vector<string> filenames;
  if (fs::is_directory(full_path)) {  // match.cpp:439-452
    for (fs::directory_iterator it(full_path), e; it != e; ++it)
      if (fs::is_regular_file(it->status())) filenames.push_back(it->path().native());
  } else if (fs::is_regular_file(full_path)) {  // match.cpp:454-492
    std::ifstream file(full_path.native());
    string line;
    while (std::getline(file, line)) {
      std::stringstream lineStream(line);
      string cell;
      std::getline(lineStream, cell, ',');
      if (cell.find("/") == 0) {
        filenames.push_back(cell);
        cout << cell << endl;
      } else {
        filenames.push_back(full_path.parent_path().native() + "/" + cell + ".csv");
        cout << full_path.parent_path().native() + cell << endl;
      }
      std::array<double, 3> point = {0, 0, 0};
      try {
        std::getline(lineStream, cell, ',');
        point[0] = std::stof(cell);
        std::getline(lineStream, cell, ',');
        point[1] = std::stof(cell);
        std::getline(lineStream, cell, ',');
        point[2] = std::stof(cell);
      } catch (...) {
      }
      rigids.push_back(point);
    }
  } else {
    cerr << "Bad argument, first arg must be a valid file or a directory" << endl;  // match.cpp:496
    return 1;
  }

  // ---- GPU plan, made before the first CUDA call ---------------------------------------------------------
  // The number of GPUs follows the work.  Bringing CUDA up costs a one-shot process ~0.55 s for the first GPU and
  // ~0.65 s for EVERY further one -- serialised system-wide, whether the GPUs are driven from threads or from
  // processes (profiles/r2_ctx_probe.txt) -- while one B200 matches ~1.3e13 descriptor pairs per second.  So without
  // -gpus the plan is the G that minimises  start-up(G) + pairs / (G x rate), the pairs estimated from the keypoint
  // file sizes: one GPU up to ~2e13 pairs (a 200 x 20k group is 8e12), two up to ~5e13, ...  A resident server
  // (-serve 1) has its contexts up already and uses every GPU whenever the group has work for them.
  const size_t n_load = std::min<size_t>(filenames.size(), (size_t)std::max(N, 0));
  const size_t planned_pairs = n_load < 2 ? 0 : (target >= 0 ? n_load - 1 : n_load * (n_load - 1) / 2);
  double est_bytes = 0;  // upper estimate of the float data the arena will hold
  int G_want = gpus;
  {
    double pts = 0, pts2 = 0;  // sum n_i, sum n_i^2 -> sum_{i<j} n_i n_j
    for (size_t i = 0; i < n_load; i++) {
      std::error_code ec;
      const double bytes = (double)fs::file_size(filenames[i], ec);
      if (ec) continue;
      const string& f = filenames[i];
      if (is_volume(f)) {
        // At most one extremum per middle response layer position, layers sampled every 2 voxels or more: fewer than
        // voxels / 3 keypoints.  An uncompressed .mha takes at least one byte per voxel; a .mhd header or a compressed
        // stream can be far smaller than the voxel count its header states.
        fsio::MetaHeader h;
        string herr;
        const double voxels = std::max(bytes, fsio::read_metaimage_header(f, h, herr) ? (double)h.dims[0] * h.dims[1] * h.dims[2] : 0.0);
        const double d = surfOpts.descriptorType == 1 ? 24.0 * std::pow((double)surfOpts.subVolumeRadius, 3) : 48.0;
        const double n_vol = surfOpts.numberOfPoints > 0 ? std::min<double>(surfOpts.numberOfPoints, voxels / 3) : voxels / 3;
        est_bytes += n_vol * (d + 2) * sizeof(float);
        pts += n_vol;
        pts2 += n_vol * n_vol;
        continue;
      }
      const bool gz = f.size() > 3 && f.compare(f.size() - 3, 3, ".gz") == 0;
      const bool bin = f.size() > 4 && f.compare(f.size() - 4, 4, ".bin") == 0;
      const double n_est = bytes / (bin ? 216.0 : gz ? 220.0 : 500.0);  // 54 floats; "%f" text; the same gzipped
      est_bytes += bin ? bytes + 4096 : gz ? bytes * 24 : bytes * 2;    // text: >= 2 characters per value
      pts += n_est;
      pts2 += n_est * n_est;
    }
    if (G_want <= 0) {
      const double est_pairs = target >= 0 ? pts * pts / std::max<double>(n_load, 1) : (pts * pts - pts2) / 2;
      const double rate = 1.3e13, first_gpu_s = warm ? 0.0 : 0.55, next_gpu_s = warm ? 0.01 : 0.65;
      double best_t = 1e300;
      for (int g = 1; g <= kMaxWorkers; g++) {
        const double t = first_gpu_s + next_gpu_s * (g - 1) + est_pairs / (g * rate);
        if (t < best_t) { best_t = t; G_want = g; }
      }
    }
    est_bytes += 16.0 * pts * std::max<double>(n_load, 1);  // match lists: <= 8 B per outer-loop row per image pair
  }
  G_want = (int)std::max<size_t>(1, std::min<size_t>((size_t)std::min(G_want, kMaxWorkers), std::max<size_t>(planned_pairs, 1)));
  if (planOnly) {
    cout << "Planned GPUs : " << G_want << " (" << planned_pairs << " image pairs)" << endl;
    return 0;
  }
  (void)serveMode;
  // device ids the workers may use: the caller's CUDA_VISIBLE_DEVICES list stays authoritative
  std::vector<string> dev_ids;
  if (const char* vis_env = getenv("CUDA_VISIBLE_DEVICES")) {
    std::stringstream ss(vis_env);
    for (string tok; std::getline(ss, tok, ',');)
      if (!tok.empty()) dev_ids.push_back(tok);
  } else {
    int n_phys = 0;
    for (std::error_code ec; n_phys < kMaxWorkers && fs::exists("/dev/nvidia" + std::to_string(n_phys), ec);) n_phys++;
    for (int g = 0; g < n_phys; g++) dev_ids.push_back(std::to_string(g));
  }
  const bool have_ids = !dev_ids.empty();  // (no list and no device nodes: let CUDA report what it finds)
  const int G = warm ? std::max(1, std::min<int>(G_want, (int)warm->ctx.size()))
                     : have_ids ? std::max(1, std::min<int>(G_want, (int)dev_ids.size())) : 1;
  if (nt > 0) omp_set_num_threads(nt);
  int nb = (int)n_load;
  if (nb > 65535) { cerr << "match: more than 65535 images cannot be described by pairs.bin (u16 ids)" << endl; return 1; }

  // the producer's library, before any thread or CUDA state exists (its context comes later, see the load loop)
  SurfApi own_surf_api;
  fs_ctx* own_surf_ctx = nullptr;
  VolumeProducer producer;
  producer.api = warm ? &warm->surf_api : &own_surf_api;
  producer.ctx = warm ? &warm->surf : &own_surf_ctx;
  if (std::any_of(filenames.begin(), filenames.begin() + nb, is_volume)) {
    string err;
    if (!producer.api->load(err)) {
      cerr << "match: the list holds MetaImage volumes (.mha / .mhd), which need libfrogsurf.so: " << err << endl;
      return 1;
    }
  }

  Control* ctl = map_arena((size_t)nb, (uint64_t)est_bytes);
  if (!ctl) { cerr << "match: cannot map the shared arena" << endl; return 1; }
  ctl->n_images = (uint32_t)nb;
  ctl->n_workers = (uint32_t)G;
  ctl->dist = dist;
  ctl->ratio = dist2second;
  ctl->flags = (symFlag ? FM_FLAG_SYM : 0u) | (forceExact ? FM_FLAG_FORCE_EXACT : 0u) |
               (matchAll ? FM_FLAG_MATCH_ALL : 0u) |  // -all: match.cpp:295-300, bug-compatible (fm_all.cuh)
               (distsFile ? FM_FLAG_DISTANCES : 0u);
#ifdef FM_WITH_NCCL
  ctl->use_nccl = (want_nccl && G > 1) ? 1u : 0u;
#else
  ctl->use_nccl = 0;
  if (want_nccl) cerr << "match: built without NCCL; gathering the match lists through host memory" << endl;
#endif

  // ---- workers: forked BEFORE any thread or CUDA state exists in this process -------------------------------
  cout << std::flush;
  cerr << std::flush;
  std::vector<pid_t> children;
  const bool fork_workers = multiProcess && G > 1 && !warm;
  if (fork_workers) {
    for (int g = 1; g < G; g++) {
      snprintf(ctl->worker[g].device, sizeof ctl->worker[g].device, "%s", dev_ids[g].c_str());
      pid_t pid = fork();
      if (pid < 0) { cerr << "match: fork failed" << endl; ctl->abort.store(1); return 1; }
      if (pid == 0) {
        setenv("CUDA_VISIBLE_DEVICES", ctl->worker[g].device, 1);
        worker_run(ctl, g, 0, nullptr);
        fflush(nullptr);
        _exit(ctl->worker[g].state.load() == kDone ? 0 : 2);
      }
      children.push_back(pid);
    }
  }
  if (have_ids && !warm) {
    // this process: its own device only (forked workers), or the first G devices (threads)
    string vis;
    for (int g = 0; g < (fork_workers ? 1 : G); g++) vis += (g ? "," : "") + dev_ids[g];
    setenv("CUDA_VISIBLE_DEVICES", vis.c_str(), 1);
  }
  std::vector<std::thread> local_workers;
  for (int g = 0; g < (fork_workers ? 1 : G); g++) local_workers.emplace_back(worker_run, ctl, g, g, warm ? warm->ctx[g] : nullptr);
  // Every exit path below: tell the workers, reap them, release the arena.  (A one-shot process then leaves through
  // _exit in main, without tearing CUDA down.)
  const uint64_t arena_bytes = ctl->arena_bytes;
  auto leave = [&](int code) -> int {
    if (code != 0) ctl->abort.store(1);
    for (auto& t : local_workers)
      if (t.joinable()) t.join();
    for (pid_t pid : children) { int st = 0; waitpid(pid, &st, 0); }
    cout << std::flush;
    cerr << std::flush;
    munmap(ctl, arena_bytes);
    return code;
  };
  auto report_failures = [&]() {
    for (int g = 0; g < G; g++)
      if (ctl->worker[g].state.load() == kFailed) cerr << "match: GPU " << g << ": " << ctl->worker[g].error << endl;
  };

  cout << "Found " << filenames.size() << " files, loading : " << fmin(N, filenames.size()) << endl;
  start = std::chrono::system_clock::now();
  if (filenames.size() > (size_t)N) filenames.resize(N);
  std::vector<fmio::KeypointSet> images(nb);  // header fields (pairs.bin records); descriptors move to the arena
  int load_failed = 0;

#pragma omp parallel for schedule(dynamic)
  for (int it = 0; it < nb; ++it) {  // match.cpp:508-570, with the per-image pruning of :579-609 done right away
    string err;
    fmio::KeypointSet& k = images[it];
    if (ctl->abort.load()) continue;
    if (!(is_volume(filenames[it]) ? produce_keypoints(filenames[it], surfOpts, producer, k, err)
                                   : fmio::read_keypoints(filenames[it], k, err))) {
#pragma omp critical
      { cerr << err << " (" << filenames[it] << ")" << endl; load_failed = 1; }
      ctl->abort.store(1);
      continue;
    }
    float zT = rigids.size() ? (float)rigids[it][2] : 0;
    fmio::filter_z(k, zT, zmin, zmax);
    std::array<double, 3> rg = rigids.size() ? rigids[it] : std::array<double, 3>{0, 0, 0};
#pragma omp critical
    cout << "image " << it << " rigid : " << rg[0] << ", " << rg[1] << ", " << rg[2] << " before : " << k.n
         << " points, after : " << k.n << endl << std::flush;  // the reference prints the post-filter size twice
    fmio::prune(k, sp, np);  // an image's pruning depends on that image alone
    ImageSlot& im = ctl->images()[it];
    im.n = k.n;
    im.d = k.d;
    if (k.n) {
      im.desc_off = ctl->alloc((uint64_t)k.n * k.d * sizeof(float));
      im.scale_off = ctl->alloc((uint64_t)k.n * sizeof(float));
      im.lap_off = ctl->alloc((uint64_t)k.n * sizeof(float));
      if (!im.desc_off || !im.scale_off || !im.lap_off) {
#pragma omp critical
        { cerr << "match: shared arena exhausted while loading " << filenames[it] << endl; load_failed = 1; }
        ctl->abort.store(1);
        continue;
      }
      memcpy(ctl->at<float>(im.desc_off), k.desc.data(), (size_t)k.n * k.d * sizeof(float));
      float* scale = ctl->at<float>(im.scale_off);
      float* lap = ctl->at<float>(im.lap_off);
      for (uint32_t r = 0; r < k.n; r++) { scale[r] = k.row_head(r)[3]; lap[r] = k.row_head(r)[4]; }
      std::vector<float>().swap(k.desc);  // the writer needs the header fields only
    }
    im.ready.store(1);  // workers upload it from here on
  }
  if (load_failed) { report_failures(); return leave(1); }
  if (ctl->abort.load()) {  // a worker gave up while the files were loading (typically: no CUDA device)
    for (auto& t : local_workers)
      if (t.joinable()) t.join();
    report_failures();
    bool no_device = false;
    for (int g = 0; g < G; g++) no_device = no_device || strstr(ctl->worker[g].error, "no CUDA device");
    if (no_device) cerr << "match: no CUDA device available; this build has no CPU path" << endl;
    return leave(1);
  }
  if (nb == 0) { cerr << "match: no keypoint files" << endl; return leave(1); }

  end = std::chrono::system_clock::now();
  cout << " : " << std::chrono::duration<float>(end - start).count() << "s" << endl;
  start = end;
  cout << (images[0].n ? images[0].d : 0) << " values per descriptor" << endl;  // match.cpp:575
  cout << "Sorting and pruning..." << endl;
  for (int it = 0; it < nb; ++it) cout << ". (" << images[it].n << ")" << std::flush;  // match.cpp:579-609 (done above)
  end = std::chrono::system_clock::now();
  cout << " : " << std::chrono::duration<float>(end - start).count() << "s" << endl;
  start = end;

  uint32_t dim = 0;
  for (auto& k : images)
    if (k.n) {
      if (dim == 0) dim = k.d;
      if (k.d != dim) { cerr << "match: images disagree on the descriptor length" << endl; return leave(1); }
    }
  ctl->dim = dim;

  // match.cpp:617-628
  std::vector<std::pair<int, int>> indices;
  for (int i = 0; i < nb - 1; i++) {
    if (target >= 0) {
      if (i != target) indices.push_back(std::make_pair(i, target));
    } else {
      for (int j = i + 1; j < nb; j++) indices.push_back(std::make_pair(i, j));
    }
  }
  if (target >= nb) { cerr << "match: -targ " << target << " is not a valid image index" << endl; return leave(1); }

  cout << "Pairing... " << endl;
  std::vector<std::vector<size_t>> shard;
  {
    std::vector<double> weight(indices.size());
    for (size_t id = 0; id < indices.size(); id++)
      weight[id] = (double)images[indices[id].first].n * (double)images[indices[id].second].n;
    shard = fm::shard_pairs(weight, G);
    for (int g = 0; g < G; g++) {
      WorkerSlot& w = ctl->worker[g];
      w.n_pairs = shard[g].size();
      w.pairs_off = ctl->alloc(std::max<uint64_t>(w.n_pairs, 1) * 2 * sizeof(uint32_t));
      if (!w.pairs_off) { cerr << "match: shared arena exhausted" << endl; return leave(1); }
      uint32_t* pf = ctl->at<uint32_t>(w.pairs_off);
      for (size_t k = 0; k < shard[g].size(); k++) {
        pf[k] = (uint32_t)indices[shard[g][k]].first;
        pf[w.n_pairs + k] = (uint32_t)indices[shard[g][k]].second;
      }
    }
  }
  ctl->plan_ready.store(1);

  // ---- wait for the workers (a forked worker that dies without a word is noticed through waitpid) ----
  {
    std::vector<char> reaped(children.size(), 0);
    for (;;) {
      bool all = true;
      for (int g = 0; g < G; g++) all = all && ctl->worker[g].state.load() == kDone;
      if (all) break;
      if (ctl->abort.load()) break;
      for (size_t c = 0; c < children.size(); c++) {
        if (reaped[c]) continue;
        int st = 0;
        if (waitpid(children[c], &st, WNOHANG) == children[c]) {
          reaped[c] = 1;
          const bool ok = WIFEXITED(st) && WEXITSTATUS(st) == 0;
          if (!ok && ctl->worker[c + 1].state.load() != kFailed)
            worker_fail(ctl, (int)c + 1, WIFSIGNALED(st) ? "worker process killed by signal " + std::to_string(WTERMSIG(st))
                                                         : "worker process exited with status " + std::to_string(WEXITSTATUS(st)));
        }
      }
      usleep(200);
    }
    if (ctl->abort.load()) {
      for (auto& t : local_workers)
        if (t.joinable()) t.join();
      report_failures();
      bool no_device = false;
      for (int g = 0; g < G; g++) no_device = no_device || strstr(ctl->worker[g].error, "no CUDA device");
      if (no_device) cerr << "match: no CUDA device available; this build has no CPU path" << endl;
      return leave(1);
    }
  }

  // ---- per pair, where its list lives ----
  std::vector<fmio::PairBlock> by_pair(indices.size());
  std::vector<const float*> dist_of(indices.size(), nullptr);
  long long sum = 0;
  for (int g = 0; g < G; g++) {
    WorkerSlot& w = ctl->worker[g];
    const uint32_t* counts = ctl->at<uint32_t>(w.counts_off);
    const uint32_t* lists = w.lists_off ? ctl->at<uint32_t>(w.lists_off) : nullptr;
    const float* dists = w.dists_off ? ctl->at<float>(w.dists_off) : nullptr;
    uint64_t off = 0;
    for (size_t k = 0; k < shard[g].size(); k++) {
      const size_t id = shard[g][k];
      fmio::PairBlock b;
      b.first = indices[id].first;
      b.second = indices[id].second;
      b.count = counts[k];
      b.pairs = lists ? lists + 2 * off : nullptr;
      if (dists) dist_of[id] = dists + off;
      off += b.count;
      by_pair[id] = b;
      sum += b.count;
      cout << "." << std::flush;  // match.cpp:650
    }
  }
  end = std::chrono::system_clock::now();
  const float pairing_s = std::chrono::duration<float>(end - start).count();
  cout << " : " << pairing_s << "s" << endl;
  start = end;
  cout << "Nb Match : " << (int)sum << endl;  // `int sum`, match.cpp:615,658

  // match.cpp:660-673
  std::stringstream outfilename;
  if (outputFileName) outfilename << string(outputFileName);
  else outfilename << "out_" << full_path.stem().string() << "_" << filenames.size() << ".bin";

  // match.cpp:727-742 walks pairs[i][j] row-major over a matrix in which a later store to the same
  // cell replaces an earlier one (only possible with -targ); reproduce that order.
  std::vector<size_t> order(indices.size());
  std::iota(order.begin(), order.end(), 0);
  std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return indices[a] < indices[b]; });
  std::vector<fmio::PairBlock> blocks;
  blocks.reserve(order.size());
  for (size_t id : order) blocks.push_back(by_pair[id]);

  if (!fmio::write_pairs_bin(outfilename.str(), filenames, rigids, images, blocks)) {
    cout << "write error : " << outfilename.str() << endl;  // match.cpp:677-682
    return leave(1);
  }
  cout << "Output file : " << outfilename.str() << endl;
  if (distsFile) {
    // side output for the parity checks (pairs.bin has no distances): per block, in pairs.bin's block order, `count`
    // float32 squared distances -- what the reference's norm() returns for each emitted pair (match.cpp:293)
    FILE* f = fopen(distsFile, "wb");
    if (!f) { cerr << "match: cannot write " << distsFile << endl; return leave(1); }
    for (size_t id : order)
      if (by_pair[id].count) fwrite(dist_of[id], sizeof(float), by_pair[id].count, f);
    fclose(f);
  }

  if (statsFile) {
    fm_stats tot{};
    float ms_max = 0;
    double create_s = 0, upload_s = 0, match_s = 0, gather_s = 0, nccl_init_s = 0;
    for (int g = 0; g < G; g++) {
      const WorkerSlot& j = ctl->worker[g];
      create_s = std::max(create_s, j.create_s);
      upload_s = std::max(upload_s, j.upload_s);
      match_s = std::max(match_s, j.match_s);
      gather_s = std::max(gather_s, j.gather_s);
      nccl_init_s = std::max(nccl_init_s, j.nccl_init_s);
      tot.descriptor_pairs += j.stats.descriptor_pairs;
      tot.scored_pairs += j.stats.scored_pairs;
      tot.rows += j.stats.rows;
      tot.rows_exact += j.stats.rows_exact;
      tot.candidates += j.stats.candidates;
      tot.kernel_launches += j.stats.kernel_launches;
      ms_max = std::max(ms_max, j.stats.ms_total);
    }
    std::ofstream sf(statsFile);
    sf << "{\"gpus\": " << G << ", \"processes\": " << (fork_workers ? G : 1) << ", \"image_pairs\": " << indices.size()
       << ", \"descriptor_pairs\": " << tot.descriptor_pairs << ", \"scored_pairs\": " << tot.scored_pairs << ", \"rows\": " << tot.rows
       << ", \"rows_exact\": " << tot.rows_exact << ", \"candidates\": " << tot.candidates << ", \"kernel_launches\": " << tot.kernel_launches
       << ", \"gpu_ms_max\": " << ms_max << ", \"pairing_s\": " << pairing_s << ", \"ctx_create_s\": " << create_s
       << ", \"upload_s\": " << upload_s << ", \"match_call_s\": " << match_s << ", \"gather_s\": " << gather_s
       << ", \"matches\": " << sum
       << ", \"gather\": \"" << (ctl->use_nccl ? "nccl" : (G > 1 ? "host" : "none")) << "\""
       << ", \"nccl_init_s\": " << nccl_init_s << ", \"volumes\": " << producer.volumes << ", \"produce_s\": " << producer.busy_s
       << ", \"produce_gpu_ms\": " << producer.gpu_ms << "}" << endl;
  }
  return leave(0);
}

// ---- resident server (`-serve 1`) -----------------------------------------------------------------------------
// A one-shot process pays CUDA's start-up on every call (see the GPU plan above); callers that match many groups
// (FROG.py over a study, the desk UI) can keep ONE server per user alive instead: `match <args> -serve 1` hands the
// command line to the server over a unix socket -- starting it first if nobody listens -- and relays its stdout,
// stderr and exit code, so the call looks exactly like a one-shot run to run.sh / FROG.py.  The server holds one
// context per visible GPU, runs one job at a time through the very same run_job(), and leaves after `idle` seconds
// without work (FROGMATCH_SERVE_IDLE, default 600).  Socket: $FROGMATCH_SOCKET or /tmp/frogmatch.<uid>.sock.

#include <poll.h>
#include <sys/socket.h>
#include <sys/stat.h>
#include <sys/un.h>

namespace {

string socket_path() {
  if (const char* p = getenv("FROGMATCH_SOCKET")) return p;
  return "/tmp/frogmatch." + std::to_string((unsigned)getuid()) + ".sock";
}

bool send_all(int fd, const void* p, size_t n) {
  const char* c = static_cast<const char*>(p);
  while (n) {
    ssize_t k = send(fd, c, n, MSG_NOSIGNAL);
    if (k <= 0) return false;
    c += k;
    n -= (size_t)k;
  }
  return true;
}
bool recv_all(int fd, void* p, size_t n) {
  char* c = static_cast<char*>(p);
  while (n) {
    ssize_t k = recv(fd, c, n, 0);
    if (k <= 0) return false;
    c += k;
    n -= (size_t)k;
  }
  return true;
}
// frame: u8 kind (1 stdout, 2 stderr, 3 exit code) | u32 length | payload
bool send_frame(int fd, uint8_t kind, const void* p, uint32_t n) {
  unsigned char head[5] = {kind, (unsigned char)n, (unsigned char)(n >> 8), (unsigned char)(n >> 16), (unsigned char)(n >> 24)};
  return send_all(fd, head, 5) && (n == 0 || send_all(fd, p, n));
}

// std::ostream whose bytes travel to the client as frames of one kind
class FrameBuf : public std::streambuf {
  int fd_;
  uint8_t kind_;
  char buf_[4096];
 public:
  FrameBuf(int fd, uint8_t kind) : fd_(fd), kind_(kind) { setp(buf_, buf_ + sizeof buf_); }
  int sync() override {
    if (pptr() > pbase()) send_frame(fd_, kind_, pbase(), (uint32_t)(pptr() - pbase()));
    setp(buf_, buf_ + sizeof buf_);
    return 0;
  }
  int_type overflow(int_type ch) override {
    sync();
    if (ch != traits_type::eof()) { *pptr() = (char)ch; pbump(1); }
    return ch;
  }
};

int serve(const string& path, int idle_s) {
  // contexts for every visible device, created side by side
  int n_dev = 0;
  if (fm_device_count(&n_dev) != FM_OK || n_dev <= 0) { fprintf(stderr, "match -serve: %s\n", fm_last_error(nullptr)); return 1; }
  WarmPool pool;
  pool.ctx.assign((size_t)std::min(n_dev, kMaxWorkers), nullptr);
  {
    std::vector<std::thread> th;
    for (size_t g = 0; g < pool.ctx.size(); g++) th.emplace_back([&pool, g] { fm_create((int)g, &pool.ctx[g]); });
    for (auto& t : th) t.join();
  }
  for (auto* c : pool.ctx)
    if (!c) { fprintf(stderr, "match -serve: cannot create a context on every visible device\n"); return 1; }
  int ls = socket(AF_UNIX, SOCK_STREAM, 0);
  sockaddr_un addr{};
  addr.sun_family = AF_UNIX;
  snprintf(addr.sun_path, sizeof addr.sun_path, "%s", path.c_str());
  unlink(path.c_str());
  const mode_t old_mask = umask(0077);  // the socket belongs to this user alone
  const bool bound = ls >= 0 && bind(ls, reinterpret_cast<sockaddr*>(&addr), sizeof addr) == 0 && listen(ls, 8) == 0;
  umask(old_mask);
  if (!bound) { perror("match -serve: bind"); return 1; }
  for (;;) {
    pollfd pfd{ls, POLLIN, 0};
    const int pr = poll(&pfd, 1, idle_s * 1000);
    if (pr == 0) break;  // idle: leave
    if (pr < 0) continue;
    const int fd = accept(ls, nullptr, nullptr);
    if (fd < 0) continue;
    // request: u32 length | cwd \0 arg0 \0 arg1 \0 ...
    uint32_t len = 0;
    std::vector<char> req;
    if (recv_all(fd, &len, 4) && len > 0 && len < (1u << 24)) {
      req.resize(len);
      if (!recv_all(fd, req.data(), len)) req.clear();
    }
    if (!req.empty() && req.back() == 0) {
      std::vector<char*> args;
      for (size_t i = 0; i < req.size();) { args.push_back(req.data() + i); i += strlen(req.data() + i) + 1; }
      if (args.size() >= 3 && strcmp(args[2], "-serve-stop") == 0) {
        const uint32_t zero = 0;
        send_frame(fd, 3, &zero, 4);
        close(fd);
        break;
      }
      int code = 1;
      if (args.size() >= 2 && chdir(args[0]) == 0) {
        FrameBuf ob(fd, 1), eb(fd, 2);
        std::ostream os(&ob), es(&eb);
        code = run_job((int)args.size() - 1, args.data() + 1, os, es, &pool);
        os.flush();
        es.flush();
      }
      const uint32_t c = (uint32_t)code;
      send_frame(fd, 3, &c, 4);
    }
    close(fd);
  }
  close(ls);
  unlink(path.c_str());
  return 0;
}

int connect_to(const string& path) {
  int fd = socket(AF_UNIX, SOCK_STREAM, 0);
  if (fd < 0) return -1;
  sockaddr_un addr{};
  addr.sun_family = AF_UNIX;
  snprintf(addr.sun_path, sizeof addr.sun_path, "%s", path.c_str());
  if (connect(fd, reinterpret_cast<sockaddr*>(&addr), sizeof addr) != 0) { close(fd); return -1; }
  return fd;
}

// Client side of `-serve 1`.  Returns the job's exit code, or -1 if no server could be reached or started (the caller
// then runs the job itself).
int run_served(int argc, char* argv[]) {
  const string path = socket_path();
  int fd = connect_to(path);
  if (fd < 0) {
    // nobody listens: start the server (detached, its own session), then wait for its socket
    pid_t pid = fork();
    if (pid == 0) {
      setsid();
      if (fork() != 0) _exit(0);  // the grandchild is adopted by init: no zombie, no controlling terminal
      const string log = path + ".log";
      FILE* lf = freopen(log.c_str(), "a", stderr);
      (void)lf;
      lf = freopen("/dev/null", "w", stdout);
      lf = freopen("/dev/null", "r", stdin);
      execl("/proc/self/exe", argv[0], "-serve-daemon", path.c_str(), (char*)nullptr);
      _exit(127);
    }
    if (pid > 0) { int st = 0; waitpid(pid, &st, 0); }
    for (int i = 0; i < 1200 && fd < 0; i++) {  // CUDA start-up for every visible GPU: up to a minute
      usleep(50000);
      fd = connect_to(path);
    }
    if (fd < 0) return -1;
  }
  std::vector<char> req;
  char cwd[4096];
  if (!getcwd(cwd, sizeof cwd)) { close(fd); return -1; }
  req.insert(req.end(), cwd, cwd + strlen(cwd) + 1);
  for (int i = 0; i < argc; i++) req.insert(req.end(), argv[i], argv[i] + strlen(argv[i]) + 1);
  const uint32_t len = (uint32_t)req.size();
  if (!send_all(fd, &len, 4) || !send_all(fd, req.data(), req.size())) { close(fd); return -1; }
  std::vector<char> buf;
  for (;;) {
    unsigned char head[5];
    if (!recv_all(fd, head, 5)) { fprintf(stderr, "match: the server closed the connection\n"); close(fd); return 1; }
    const uint32_t n = head[1] | (head[2] << 8) | (head[3] << 16) | ((uint32_t)head[4] << 24);
    buf.resize(n);
    if (n && !recv_all(fd, buf.data(), n)) { close(fd); return 1; }
    if (head[0] == 1) { fwrite(buf.data(), 1, n, stdout); fflush(stdout); }
    else if (head[0] == 2) { fwrite(buf.data(), 1, n, stderr); }
    else if (head[0] == 3) {
      uint32_t code = 1;
      if (n == 4) memcpy(&code, buf.data(), 4);
      close(fd);
      return (int)code;
    }
  }
}

}  // namespace

int main(int argc, char* argv[]) {
  if (argc >= 3 && strcmp(argv[1], "-serve-daemon") == 0) {
    const char* idle = getenv("FROGMATCH_SERVE_IDLE");
    const int rc = serve(argv[2], idle ? std::max(1, atoi(idle)) : 600);
    fflush(nullptr);
    _exit(rc);
  }
  bool served = false;
  for (int k = 2; k + 1 < argc; k++)
    if (strcmp(argv[k], "-serve") == 0 && atoi(argv[k + 1]) != 0) served = true;
  if ((argc >= 2 && strcmp(argv[1], "-serve-stop") == 0)) {
    const int fd = connect_to(socket_path());
    if (fd < 0) return 0;  // nothing to stop
    close(fd);
    return run_served(argc, argv) == 0 ? 0 : 1;
  }
  if (served) {
    const int rc = run_served(argc, argv);
    if (rc >= 0) return rc;
    cerr << "match: no resident server could be reached or started; running one-shot" << endl;
  }
  const int rc = run_job(argc, argv, cout, cerr, nullptr);
  // pairs.bin and the side files are closed.  Tearing down one CUDA context per GPU (and NCCL) costs a one-shot
  // process up to seconds and frees nothing the operating system does not reclaim anyway: leave at once.
  cout << std::flush;
  cerr << std::flush;
  fflush(nullptr);
  _exit(rc);
}
