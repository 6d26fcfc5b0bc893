// libfrogsurf.so: C ABI (include/frogsurf.h) + host logic of the SURF3D producer.
// Host side = what the reference does on the host between its parallel loops: layer geometry and
// loop limits (fasthessian.cxx:142-218, 287-341), ordering of the extrema, the 4 x 4 solve of the
// interpolation step (fasthessian.cxx:575-661) and the response sort (vtk3DSURF.cxx:209-226).
#include <algorithm>
#include <cmath>
#include <cerrno>
#include <cstdarg>
#include <cstdlib>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "fs_as_read.cuh"
#include "fs_kernels.cuh"

namespace {

thread_local std::string g_create_error;
int g_response_tile = 5;  // fs_debug_set_option("response_tile", v): 0 flat, 1 32x8x1, 2 32x4x2, 3 32x2x4, 4 32x1x8, 5 32x4x4 (default), 6-9 register / CTA-size variants

struct Layer {
  fs::LayerDev dev{};
  size_t voxels = 0;
};

}  // namespace

struct fs_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[2] = {nullptr, nullptr};
  std::string err;
  int nx = 0, ny = 0, nz = 0;
  int32_t* d_cast = nullptr;
  fs::u64* d_integral = nullptr;
  fs::u64* d_split = nullptr;  // parity-split copy of the integral volume (fs_kernels.cuh, integral_z_kernel)
  size_t vol_cap = 0, split_cap = 0, cast_cap = 0;
  void* d_in = nullptr;
  size_t in_cap = 0;
  double* d_blockmin = nullptr;
  std::vector<Layer> layers;
  float* d_layer_f = nullptr;
  uint8_t* d_layer_b = nullptr;
  size_t layer_f_cap = 0, layer_b_cap = 0;
  fs::Candidate* d_cand = nullptr;
  fs::Interpolated* d_interp = nullptr;
  size_t interp_cap = 0;
  std::vector<fs::Interpolated> h_interp;
  unsigned* d_count = nullptr;  // [0] candidates, [1] clamped keypoints
  unsigned cand_cap = 0;
  std::vector<fs_point> points;
  fs_point* d_points = nullptr;
  size_t points_cap = 0;
  float* d_desc = nullptr;
  size_t desc_cap = 0;
  uint32_t desc_size = 0;
  float* d_as_read = nullptr;  // fs_get_points_as_read: head + descriptors as the .csv.gz reader returns them
  size_t as_read_cap = 0;
  fs::AsReadFallback* d_fallback = nullptr;
  size_t fallback_cap = 0;
  unsigned long long* d_fallback_count = nullptr;
  bool have_volume = false;
  bool keep_cast = false;  // fs_debug_keep_cast_volume: also store vtk3DSURF::Cast (only the parity tests read it)
  fs_stats stats{};
};

namespace {

int fail(fs_ctx* c, int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf; else g_create_error = buf;
  return code;
}

#define FS_CUDA(c, call)                                                                          \
  do {                                                                                            \
    cudaError_t e_ = (call);                                                                      \
    if (e_ != cudaSuccess) return fail((c), FS_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
  } while (0)

template <typename T>
int ensure(fs_ctx* c, T*& p, size_t& cap, size_t need) {
  if (need <= cap) return FS_OK;
  if (p) cudaFree(p);
  p = nullptr;
  cap = 0;
  if (cudaMalloc((void**)&p, need * sizeof(T)) != cudaSuccess) {
    cudaGetLastError();
    return fail(c, FS_ERR_NOMEM, "cudaMalloc of %zu bytes failed", need * sizeof(T));
  }
  cap = need;
  return FS_OK;
}

size_t voxel_size(int t) {
  switch (t) {
    case FS_U8: case FS_I8: return 1;
    case FS_I16: case FS_U16: return 2;
    case FS_I32: case FS_U32: case FS_F32: return 4;
    case FS_F64: return 8;
  }
  return 0;
}

template <typename T>
int run_integral(fs_ctx* c, const T* in, double* shift_out) {
  const size_t n = (size_t)c->nx * c->ny * c->nz;
  const int blocks = 592;
  fs::volume_min_kernel<T><<<blocks, 256, 0, c->stream>>>(in, n, c->d_blockmin);
  double mins[592];
  FS_CUDA(c, cudaMemcpyAsync(mins, c->d_blockmin, sizeof mins, cudaMemcpyDeviceToHost, c->stream));
  FS_CUDA(c, cudaStreamSynchronize(c->stream));
  double mn = mins[0];
  for (int i = 1; i < blocks; i++) mn = std::min(mn, mins[i]);
  const double shift = -mn;  // Shift->SetShift( -Range[ 0 ] ), vtk3DSURF.cxx:172
  *shift_out = shift;
  // rows per tile: 16 (one per warp) while two CTAs still fit an SM's shared memory, fewer for very wide volumes
  int rows = 16;
  while (rows > 1 && ((size_t)c->nx * (rows + 1)) * sizeof(fs::u64) > 100 * 1024) rows >>= 1;
  const size_t smem = ((size_t)c->nx * (rows + 1)) * sizeof(fs::u64);
  if (smem > 200 * 1024) return fail(c, FS_ERR_UNSUPPORTED, "nx = %d is too wide for the row scan", c->nx);
  FS_CUDA(c, cudaFuncSetAttribute(fs::integral_xy_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  fs::integral_xy_kernel<T><<<c->nz, 512, smem, c->stream>>>(in, c->keep_cast ? c->d_cast : nullptr, c->d_integral, c->nx, c->ny, rows, shift);
  const size_t slice = (size_t)c->nx * c->ny;
  fs::integral_z_kernel<<<(unsigned)((slice + 255) / 256), 256, 0, c->stream>>>(c->d_integral, c->d_split, c->nx, c->ny, c->nz);
  FS_CUDA(c, cudaGetLastError());
  return FS_OK;
}

fs::IntegralSplit split_view(const fs_ctx* c) {
  fs::IntegralSplit I;
  const long long hx = (c->nx + 1) / 2;
  I.p0 = c->d_split;
  I.p1 = c->d_split + (size_t)hx * c->ny * c->nz;
  I.sy = (uint32_t)hx;
  I.sz = (uint32_t)(hx * c->ny);
  return I;
}

fs::Integral integral_view(const fs_ctx* c) {
  fs::Integral I;
  I.p = c->d_integral;
  I.sy = c->nx;
  I.sz = (long long)c->nx * c->ny;
  I.nx = c->nx; I.ny = c->ny; I.nz = c->nz;
  return I;
}

// ---- layer geometry (FastHessian constructor :53-81, buildResponseMap :287-341) ----------------
struct LayerGeom { int w, h, d, step, filter; };

int octaves_for(int nx, int ny, int nz) {
  const int min_dim = std::min(nx, std::min(ny, nz));
  int octaves = 4;  // vtk3DSURF.cxx:193 asks for 4
  if (min_dim < 51 * 2) octaves = std::min(1, octaves);
  else if (min_dim < 99 * 2) octaves = std::min(2, octaves);
  else if (min_dim < 195 * 2) octaves = std::min(3, octaves);
  else if (min_dim < 387 * 2) octaves = std::min(4, octaves);
  return octaves;
}

std::vector<LayerGeom> layer_geometry(int nx, int ny, int nz, int octaves) {
  const int s = 2;  // init_sample
  const int w = nx / s, h = ny / s, d = nz / s;
  static const int filters[10] = {9, 15, 21, 27, 39, 51, 75, 99, 147, 195};
  std::vector<LayerGeom> g;
  for (int i = 0; i < 4 && octaves >= 1; i++) g.push_back({w, h, d, s, filters[i]});
  for (int o = 2; o <= octaves && o <= 4; o++) {
    const int f = 1 << (o - 1);
    for (int i = 0; i < 2; i++) g.push_back({w / f, h / f, d / f, s * f, filters[4 + 2 * (o - 2) + i]});
  }
  return g;
}

int layer_limit(const LayerGeom& g) {
  // fasthessian.cxx:366: ceil((float)(filter + 1)/(float)step/2)+1
  return (int)(std::ceil((float)(g.filter + 1) / (float)g.step / 2) + 1);
}

// First (r, c, d) in the reference's loop order (r outer, d inner, each from `limit`) where any of the three
// per-axis predicates holds; -1 when none does.  fasthessian.cxx:202-210 clears bits of `param` there and the
// variable is never restored inside the pass, so everything from that position on sees the cleared value.
template <class PR, class PC, class PD>
long long first_hit(int limit, int nr, int nc, int nd, PR pr, PC pc, PD pd) {
  long long inner = -1;  // first (c, d) offset with pc || pd, independent of r
  for (int c = 0; c < nc && inner < 0; c++) {
    if (pc(limit + c)) { inner = (long long)c * nd; break; }
    for (int d = 0; d < nd; d++)
      if (pd(limit + d)) { inner = (long long)c * nd + d; break; }
  }
  for (int r = 0; r < nr; r++) {
    if (pr(limit + r)) return (long long)r * nc * nd;
    if (inner >= 0) return (long long)r * nc * nd + inner;
  }
  return -1;
}

// Ascending by key, equal keys in input order: LSD radix sort over the bytes that differ between keys (loop positions
// of ~25 000 extrema: four of eight bytes), a tenth of the time std::sort takes on the (key, index) pairs.
struct KeyIndex {
  uint64_t key;
  uint32_t index;
};

void sort_by_key(std::vector<KeyIndex>& v) {
  if (v.size() < 2) return;
  uint64_t all_or = 0, all_and = ~0ull;
  for (const KeyIndex& k : v) { all_or |= k.key; all_and &= k.key; }
  const uint64_t varying = all_or ^ all_and;  // bits that are not the same in every key
  std::vector<KeyIndex> tmp(v.size());
  KeyIndex* src = v.data();
  KeyIndex* dst = tmp.data();
  for (int byte = 0; byte < 8; byte++) {
    if (!((varying >> (8 * byte)) & 0xFFu)) continue;
    size_t count[257] = {0};
    for (size_t i = 0; i < v.size(); i++) count[((src[i].key >> (8 * byte)) & 0xFFu) + 1]++;
    for (int b = 0; b < 256; b++) count[b + 1] += count[b];
    for (size_t i = 0; i < v.size(); i++) dst[count[(src[i].key >> (8 * byte)) & 0xFFu]++] = src[i];
    std::swap(src, dst);
  }
  if (src != v.data()) std::memcpy(v.data(), src, v.size() * sizeof(KeyIndex));
}

// vtk3DSURF.cxx:209-226 with compareResponses (:32): partial_sort + resize when there are more points than asked for,
// sort otherwise, nothing when number_of_points <= 0.  The reference sorts its Ipoint objects; which of two equal
// responses comes first is decided by the algorithm's comparisons and moves only, never by the payload, so running the
// SAME std::partial_sort / std::sort over 8-byte (response, index) keys and gathering afterwards gives the same order
// at a third of the memory traffic.
struct ResponseKey {
  float response;
  uint32_t index;
};
struct ByResponse {  // a functor, so the comparison is inlined into the sort loops
  bool operator()(const ResponseKey& i, const ResponseKey& j) const { return i.response > j.response; }
};

void select_points(std::vector<fs_point>& pts, int number_of_points) {
  if (number_of_points <= 0) return;
  std::vector<ResponseKey> keys(pts.size());
  for (size_t i = 0; i < pts.size(); i++) keys[i] = ResponseKey{pts[i].response, (uint32_t)i};
  if (keys.size() > (size_t)number_of_points) {
    // (a plain sort of the keys would be twice as fast, but equal responses are common -- 6 among the 23 210 extrema
    // of the bench volume -- and their order is partial_sort's alone)
    std::partial_sort(keys.begin(), keys.begin() + number_of_points, keys.end(), ByResponse());
    keys.resize(number_of_points);
  } else {
    std::sort(keys.begin(), keys.end(), ByResponse());
  }
  std::vector<fs_point> out(keys.size());
  for (size_t i = 0; i < keys.size(); i++) out[i] = pts[keys[i].index];
  pts.swap(out);
}

int upload_points(fs_ctx* c) {
  const size_t n = c->points.size();
  if (int rc = ensure(c, c->d_points, c->points_cap, std::max<size_t>(n, 1))) return rc;
  if (n) FS_CUDA(c, cudaMemcpyAsync(c->d_points, c->points.data(), n * sizeof(fs_point), cudaMemcpyHostToDevice, c->stream));
  return FS_OK;
}

// format_fixed's snprintf path (surf_io.cpp) followed by the reader's strtof
float as_read_on_host(double v, int decimals, bool* range_error) {
  char fmt[16], text[512];
  std::snprintf(fmt, sizeof fmt, "%%.%df", decimals);
  std::snprintf(text, sizeof text, fmt, v);
  errno = 0;
  const float f = std::strtof(text, nullptr);
  if (errno == ERANGE) *range_error = true;
  return f;
}

// Runs the conversion kernel `launch(list)` until its list of host values holds all of them, then copies `total`
// results to `out` (split at `split`: out[0 .. split) and out2[0 .. total - split)) and finishes the listed values.
// `decimals_of(index)` gives a listed value's decimals.
template <class Launch, class Decimals>
int as_read_finish(fs_ctx* c, size_t total, size_t split, float* out, float* out2, Launch launch, Decimals decimals_of,
                   bool* range_error) {
  unsigned long long listed = 0;
  for (;;) {
    FS_CUDA(c, cudaMemsetAsync(c->d_fallback_count, 0, sizeof(unsigned long long), c->stream));
    launch(fs::AsReadList{c->d_fallback, c->d_fallback_count, (unsigned long long)c->fallback_cap});
    FS_CUDA(c, cudaGetLastError());
    FS_CUDA(c, cudaMemcpyAsync(&listed, c->d_fallback_count, sizeof listed, cudaMemcpyDeviceToHost, c->stream));
    FS_CUDA(c, cudaStreamSynchronize(c->stream));
    if (listed <= c->fallback_cap) break;
    if (int rc = ensure(c, c->d_fallback, c->fallback_cap, (size_t)listed)) return rc;
  }
  if (split) FS_CUDA(c, cudaMemcpyAsync(out, c->d_as_read, split * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  if (total > split)
    FS_CUDA(c, cudaMemcpyAsync(out2, c->d_as_read + split, (total - split) * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
  std::vector<fs::AsReadFallback> fb((size_t)listed);
  if (listed) FS_CUDA(c, cudaMemcpyAsync(fb.data(), c->d_fallback, listed * sizeof(fs::AsReadFallback), cudaMemcpyDeviceToHost, c->stream));
  FS_CUDA(c, cudaStreamSynchronize(c->stream));
  for (const fs::AsReadFallback& e : fb) {
    const float f = as_read_on_host(e.value, decimals_of(e.index), range_error);
    if (e.index < split) out[e.index] = f;
    else out2[e.index - split] = f;
  }
  return FS_OK;
}

int as_read_buffers(fs_ctx* c, size_t total) {
  if (int rc = ensure(c, c->d_as_read, c->as_read_cap, total)) return rc;
  if (!c->d_fallback_count) FS_CUDA(c, cudaMalloc((void**)&c->d_fallback_count, sizeof(unsigned long long)));
  return ensure(c, c->d_fallback, c->fallback_cap, std::min<size_t>(total, (size_t)1 << 16));
}

unsigned as_read_blocks(size_t total) { return (unsigned)std::max<size_t>(1, std::min<size_t>((total + 255) / 256, 148 * 16)); }

float elapsed(fs_ctx* c) {
  float ms = 0;
  cudaEventSynchronize(c->ev[1]);
  cudaEventElapsedTime(&ms, c->ev[0], c->ev[1]);
  return ms;
}

}  // namespace

extern "C" {

const char* fs_version(void) { return "frogsurf-b200 0.1 (sm_100a)"; }

int fs_device_count(int* n) {
  int k = 0;
  if (cudaGetDeviceCount(&k) != cudaSuccess) { cudaGetLastError(); if (n) *n = 0; return FS_ERR_CUDA; }
  if (n) *n = k;
  return k > 0 ? FS_OK : FS_ERR_CUDA;
}

int fs_create(int device, fs_ctx** out) {
  if (!out) return fail(nullptr, FS_ERR_INVALID, "fs_create: out is null");
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) {
    cudaGetLastError();
    return fail(nullptr, FS_ERR_CUDA, "fs_create: no CUDA device (libfrogsurf has no CPU path)");
  }
  if (device < 0 || device >= n) return fail(nullptr, FS_ERR_INVALID, "fs_create: device %d of %d", device, n);
  fs_ctx* c = new fs_ctx;
  c->device = device;
  if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreate(&c->ev[0]) != cudaSuccess || cudaEventCreate(&c->ev[1]) != cudaSuccess ||
      cudaMalloc((void**)&c->d_blockmin, 592 * sizeof(double)) != cudaSuccess ||
      cudaMalloc((void**)&c->d_count, 2 * sizeof(unsigned)) != cudaSuccess) {
    fail(nullptr, FS_ERR_CUDA, "fs_create: %s", cudaGetErrorString(cudaGetLastError()));
    fs_destroy(c);  // releases whatever was created before the failing call
    return FS_ERR_CUDA;
  }
  *out = c;
  return FS_OK;
}

void fs_destroy(fs_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->stream) cudaStreamSynchronize(c->stream);
  cudaFree(c->d_cast); cudaFree(c->d_integral); cudaFree(c->d_split); cudaFree(c->d_in); cudaFree(c->d_blockmin);
  cudaFree(c->d_layer_f); cudaFree(c->d_layer_b); cudaFree(c->d_cand); cudaFree(c->d_interp); cudaFree(c->d_count);
  cudaFree(c->d_points); cudaFree(c->d_desc); cudaFree(c->d_as_read); cudaFree(c->d_fallback); cudaFree(c->d_fallback_count);
  if (c->ev[0]) cudaEventDestroy(c->ev[0]);
  if (c->ev[1]) cudaEventDestroy(c->ev[1]);
  if (c->stream) cudaStreamDestroy(c->stream);
  delete c;
}

const char* fs_last_error(const fs_ctx* c) { return c ? c->err.c_str() : g_create_error.c_str(); }

int fs_set_volume(fs_ctx* c, const void* voxels, int voxel_type, int nx, int ny, int nz) {
  if (!c) return FS_ERR_INVALID;
  const size_t vs = voxel_size(voxel_type);
  if (!voxels || !vs || nx <= 0 || ny <= 0 || nz <= 0) return fail(c, FS_ERR_INVALID, "fs_set_volume: bad argument");
  FS_CUDA(c, cudaSetDevice(c->device));
  const size_t n = (size_t)nx * ny * nz;
  c->have_volume = false;
  c->nx = nx; c->ny = ny; c->nz = nz;
  if (c->keep_cast)
    if (int rc = ensure(c, c->d_cast, c->cast_cap, n)) return rc;
  if (int rc = ensure(c, c->d_integral, c->vol_cap, n)) return rc;
  if ((size_t)((nx + 1) / 2) * ny * nz >= (1ull << 32)) return fail(c, FS_ERR_UNSUPPORTED, "fs_set_volume: more than 2^33 voxels");
  if (int rc = ensure(c, c->d_split, c->split_cap, (size_t)2 * ((nx + 1) / 2) * ny * nz)) return rc;
  cudaPointerAttributes at{};
  const bool on_device = cudaPointerGetAttributes(&at, voxels) == cudaSuccess &&
                         (at.type == cudaMemoryTypeDevice || at.type == cudaMemoryTypeManaged);
  cudaGetLastError();
  const void* src = voxels;
  if (!on_device) {
    size_t bytes_cap = c->in_cap;
    unsigned char* p = static_cast<unsigned char*>(c->d_in);
    if (int rc = ensure(c, p, bytes_cap, n * vs)) { c->d_in = p; c->in_cap = bytes_cap; return rc; }
    c->d_in = p; c->in_cap = bytes_cap;
    FS_CUDA(c, cudaMemcpyAsync(c->d_in, voxels, n * vs, cudaMemcpyHostToDevice, c->stream));
    src = c->d_in;
  }
  FS_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  double shift = 0;
  int rc = FS_OK;
  switch (voxel_type) {
    case FS_U8: rc = run_integral(c, static_cast<const uint8_t*>(src), &shift); break;
    case FS_I16: rc = run_integral(c, static_cast<const int16_t*>(src), &shift); break;
    case FS_U16: rc = run_integral(c, static_cast<const uint16_t*>(src), &shift); break;
    case FS_I32: rc = run_integral(c, static_cast<const int32_t*>(src), &shift); break;
    case FS_F32: rc = run_integral(c, static_cast<const float*>(src), &shift); break;
    case FS_I8: rc = run_integral(c, static_cast<const int8_t*>(src), &shift); break;
    case FS_U32: rc = run_integral(c, static_cast<const uint32_t*>(src), &shift); break;
    case FS_F64: rc = run_integral(c, static_cast<const double*>(src), &shift); break;
  }
  if (rc) return rc;
  FS_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  FS_CUDA(c, cudaStreamSynchronize(c->stream));
  c->stats.ms_integral = elapsed(c);
  c->layers.clear();
  c->points.clear();
  c->desc_size = 0;
  c->have_volume = true;
  return FS_OK;
}

int fs_detect(fs_ctx* c, float threshold, uint32_t* n_points) {
  if (!c) return FS_ERR_INVALID;
  if (!c->have_volume) return fail(c, FS_ERR_STATE, "fs_detect: no volume");
  FS_CUDA(c, cudaSetDevice(c->device));
  const float thresh = threshold >= 0 ? threshold : 0.0004f;  // saveParameters, fasthessian.cxx:107
  const int octaves = octaves_for(c->nx, c->ny, c->nz);
  const std::vector<LayerGeom> geom = layer_geometry(c->nx, c->ny, c->nz, octaves);
  for (const LayerGeom& g : geom)
    if (g.w <= 0 || g.h <= 0 || g.d <= 0) return fail(c, FS_ERR_INVALID, "fs_detect: volume too small for the response layers");

  // ---- response layers ----
  size_t total = 0;
  for (const LayerGeom& g : geom) total += (size_t)g.w * g.h * g.d;
  if (int rc = ensure(c, c->d_layer_f, c->layer_f_cap, 2 * total)) return rc;  // responses, then the masked copy
  if (int rc = ensure(c, c->d_layer_b, c->layer_b_cap, 2 * total)) return rc;
  FS_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  FS_CUDA(c, cudaMemsetAsync(c->d_layer_f, 0, total * sizeof(float), c->stream));
  FS_CUDA(c, cudaMemsetAsync(c->d_layer_f + total, 0xFF, total * sizeof(float), c->stream));  // NaN outside the interiors: compares false
  FS_CUDA(c, cudaMemsetAsync(c->d_layer_b, 0, 2 * total, c->stream));
  c->layers.clear();
  size_t off = 0;
  uint64_t computed = 0;
  const fs::IntegralSplit I = split_view(c);
  for (const LayerGeom& g : geom) {
    Layer L;
    L.voxels = (size_t)g.w * g.h * g.d;
    L.dev.responses = c->d_layer_f + off;
    L.dev.masked = c->d_layer_f + total + off;
    L.dev.laplacian = c->d_layer_b + off;
    L.dev.isblob = c->d_layer_b + total + off;
    L.dev.width = g.w; L.dev.height = g.h; L.dev.depth = g.d; L.dev.step = g.step; L.dev.filter = g.filter;
    L.dev.limit = layer_limit(g);
    const float w = (float)g.filter;
    L.dev.inv_volume9 = 1.f / ((w * w * w) * (w * w * w) * (w * w * w));  // fasthessian.cxx:355
    off += L.voxels;
    const long long iw = g.w - 2 * L.dev.limit, ih = g.h - 2 * L.dev.limit, id = g.d - 2 * L.dev.limit;
    if (iw > 0 && ih > 0 && id > 0) {
      const long long n = iw * ih * id;
      computed += (uint64_t)n;
      auto grid = [&](int ty, int tz) { return dim3((unsigned)((iw + 31) / 32), (unsigned)((ih + ty - 1) / ty), (unsigned)((id + tz - 1) / tz)); };
      switch (g_response_tile) {
        case 0: fs::response_layer_flat_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(I, L.dev); break;
        case 1: fs::response_layer_kernel<8, 1><<<grid(8, 1), 256, 0, c->stream>>>(I, L.dev); break;
        case 3: fs::response_layer_kernel<2, 4><<<grid(2, 4), 256, 0, c->stream>>>(I, L.dev); break;
        case 4: fs::response_layer_kernel<1, 8><<<grid(1, 8), 256, 0, c->stream>>>(I, L.dev); break;
        case 2: fs::response_layer_kernel<4, 2><<<grid(4, 2), 256, 0, c->stream>>>(I, L.dev); break;
        case 6: fs::response_layer_kernel<4, 2, 5><<<grid(4, 2), 256, 0, c->stream>>>(I, L.dev); break;  // <= 51 registers
        case 7: fs::response_layer_kernel<4, 2, 6><<<grid(4, 2), 256, 0, c->stream>>>(I, L.dev); break;  // <= 42 registers
        case 8: fs::response_layer_kernel<4, 1, 8><<<grid(4, 1), 128, 0, c->stream>>>(I, L.dev); break;  // 128-thread CTAs
        case 9: fs::response_layer_kernel<2, 1, 16><<<grid(2, 1), 64, 0, c->stream>>>(I, L.dev); break;  // 64-thread CTAs
        default: fs::response_layer_kernel<4, 4><<<grid(4, 4), 512, 0, c->stream>>>(I, L.dev); break;
      }
    }
    c->layers.push_back(L);
  }
  FS_CUDA(c, cudaGetLastError());
  FS_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  FS_CUDA(c, cudaStreamSynchronize(c->stream));
  c->stats.ms_response_map = elapsed(c);
  c->stats.n_layers = (uint32_t)c->layers.size();
  c->stats.response_voxels = computed;

  // ---- extremum search, one launch per (octave, interval) pass ----
  static const int filter_map[5][4] = {{0, 1, 2, 3}, {1, 3, 4, 5}, {3, 5, 6, 7}, {5, 7, 8, 9}, {7, 9, 10, 11}};
  struct PassHost { int b, m, t, limit; };
  std::vector<PassHost> passes;
  unsigned cap = std::max(c->cand_cap, 1u << 18);
  for (int attempt = 0; attempt < 2; attempt++) {
    if (cap > c->cand_cap) {
      size_t cc = c->cand_cap;
      if (int rc = ensure(c, c->d_cand, cc, (size_t)cap)) return rc;
      c->cand_cap = (unsigned)cc;
    }
    passes.clear();
    FS_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
    FS_CUDA(c, cudaMemsetAsync(c->d_count, 0, sizeof(unsigned), c->stream));
    int pass = 0;
    for (int o = 0; o < octaves; ++o)
      for (int i = 0; i <= 1; ++i, ++pass) {
        const int bi = filter_map[o][i], mi = filter_map[o][i + 1], ti = filter_map[o][i + 2];
        const fs::LayerDev &b = c->layers[bi].dev, &m = c->layers[mi].dev, &t = c->layers[ti].dev;
        int param;
        if (o == 0 && i == 0) param = 1;                 // FIRST_SCALE
        else if (o == (octaves - 1) && i == 1) param = 2;  // LAST_SCALE
        else param = 0;
        // fasthessian.cxx:181-189, operand types as written there
        const int limit_m = (int)std::ceil((std::ceil((float)(m.filter + 1) / (float)m.step / 2.0) + 1) * (float)m.step / (float)t.step);
        const int limit_b = (int)std::ceil((std::ceil((float)(b.filter + 1) / (float)b.step / 2.0) + 1) * (float)b.step / (float)t.step);
        const int limit_t = (int)(std::ceil((float)(t.filter + 1) / (float)t.step / 2.0) + 1);
        int limit = std::max(limit_m, limit_b);
        limit = std::max(limit, limit_t);
        limit = (int)std::max((float)limit, (float)(0.6666 * t.filter + 2.5 * m.step) / (float)m.step + 2);
        passes.push_back({bi, mi, ti, limit});
        const int nr = t.height - 2 * limit, nc = t.width - 2 * limit, nd = t.depth - 2 * limit;
        if (nr <= 0 || nc <= 0 || nd <= 0) continue;
        // fasthessian.cxx:199-200
        const int lim_sup = (int)std::max((float)std::ceil((float)((t.filter - 1) / 2 + 2) / (float)t.step),
                                          (float)(0.6666 * t.filter + 2.5 * t.step + 2) / t.step);
        const int lim_down = (int)std::max((float)std::ceil((float)((b.filter - 1) / 2 + 2) / (float)b.step),
                                           (float)(0.6666 * b.filter + 2.5 * b.step + 2) / b.step);
        const int ratio = (int)(t.width / b.width);
        fs::ExtremaPass P;
        P.first_sup = first_hit(limit, nr, nc, nd,
                                [&](int r) { return r < lim_sup || r >= t.height - lim_sup; },
                                [&](int cc2) { return cc2 < lim_sup || cc2 >= t.width - lim_sup; },
                                [&](int d) { return d < lim_sup || d >= t.depth - lim_sup; });
        P.first_down = first_hit(limit, nr, nc, nd,
                                 [&](int r) { return r * ratio < lim_down || r * ratio >= b.height - lim_down; },
                                 [&](int cc2) { return cc2 * ratio < lim_down || cc2 * ratio >= b.width - lim_down; },
                                 [&](int d) { return d * ratio < lim_down || d * ratio >= b.depth - lim_down; });
        const long long never = 1LL << 62;
        if (P.first_sup < 0) P.first_sup = never;
        if (P.first_down < 0) P.first_down = never;
        auto view = [](const fs::LayerDev& l) { return fs::LayerView{l.responses, l.masked, l.laplacian, l.isblob, l.width, l.height, l.depth}; };
        P.b = view(b); P.m = view(m); P.t = view(t);
        P.scale_m = m.width / t.width;
        P.scale_b = b.width / t.width;
        P.limit = limit;
        P.param0 = param;
        P.pass = pass;
        P.thresh = thresh;
        const long long n = (long long)nr * nc * nd;
        fs::extrema_kernel<<<(unsigned)((n + 255) / 256), 256, 0, c->stream>>>(P, c->d_cand, c->d_count, c->cand_cap);
      }
    FS_CUDA(c, cudaGetLastError());
    FS_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
    unsigned found = 0;
    FS_CUDA(c, cudaMemcpyAsync(&found, c->d_count, sizeof found, cudaMemcpyDeviceToHost, c->stream));
    FS_CUDA(c, cudaStreamSynchronize(c->stream));
    c->stats.ms_extrema = elapsed(c);
    c->stats.n_candidates = found;
    if (found <= c->cand_cap) break;
    if (attempt == 1) return fail(c, FS_ERR_NOMEM, "fs_detect: candidate buffer overflow");
    cap = found + 1024;  // rerun with room for all of them
  }

  // ---- interpolation on the device, one thread per extremum; the host only restores the reference's push_back
  // order (the loop position in `key`) among the accepted ones ----
  const unsigned nc = c->stats.n_candidates;
  c->points.clear();
  if (nc) {
    size_t icap = c->interp_cap;
    if (int rc = ensure(c, c->d_interp, icap, (size_t)nc)) return rc;
    c->interp_cap = icap;
    fs::PassScales scales{};
    for (size_t i = 0; i < passes.size() && i < 8; i++)
      scales.p[i] = fs::PassScale{c->layers[passes[i].t].dev.step, c->layers[passes[i].m].dev.filter, c->layers[passes[i].b].dev.filter};
    fs::interpolate_kernel<<<(nc + 127) / 128, 128, 0, c->stream>>>(c->d_cand, nc, scales, c->d_interp);
    FS_CUDA(c, cudaGetLastError());
    c->h_interp.resize(nc);
    FS_CUDA(c, cudaMemcpyAsync(c->h_interp.data(), c->d_interp, (size_t)nc * sizeof(fs::Interpolated), cudaMemcpyDeviceToHost, c->stream));
    FS_CUDA(c, cudaStreamSynchronize(c->stream));
    std::vector<KeyIndex> order;
    order.reserve(nc);
    for (unsigned i = 0; i < nc; i++)
      if (c->h_interp[i].accepted) order.push_back(KeyIndex{c->h_interp[i].key, i});
    sort_by_key(order);
    c->points.reserve(order.size());
    for (const KeyIndex& o : order) c->points.push_back(c->h_interp[o.index].point);
  }
  c->desc_size = 0;
  c->stats.n_points = (uint32_t)c->points.size();
  if (n_points) *n_points = (uint32_t)c->points.size();
  return FS_OK;
}

int fs_select(fs_ctx* c, int number_of_points) {
  if (!c) return FS_ERR_INVALID;
  select_points(c->points, number_of_points);
  c->desc_size = 0;
  c->stats.n_points = (uint32_t)c->points.size();
  return FS_OK;
}

int fs_set_points(fs_ctx* c, const float* xyzs, uint32_t n) {
  if (!c || (n && !xyzs)) return FS_ERR_INVALID;
  c->points.resize(n);
  for (uint32_t i = 0; i < n; i++) {
    fs_point& p = c->points[i];
    p.x = xyzs[4 * i]; p.y = xyzs[4 * i + 1]; p.z = xyzs[4 * i + 2]; p.scale = xyzs[4 * i + 3];
    p.response = 0; p.laplacian = 0;  // Ipoint(), ipoint.h:33
  }
  c->desc_size = 0;
  c->stats.n_points = n;
  return FS_OK;
}

int fs_describe(fs_ctx* c, int type, int radius, int normalize) {
  if (!c) return FS_ERR_INVALID;
  if (!c->have_volume) return fail(c, FS_ERR_STATE, "fs_describe: no volume");
  if (type != 0 && type != 1) return fail(c, FS_ERR_UNSUPPORTED, "fs_describe: descriptor type %d needs vtkImageResize", type);
  if (radius < 1 || (type == 0 && radius > 10) || radius > fs::kMaxRadius) return fail(c, FS_ERR_UNSUPPORTED, "fs_describe: radius %d", radius);
  FS_CUDA(c, cudaSetDevice(c->device));
  const size_t n = c->points.size();
  const size_t S = (size_t)8 * radius * radius * radius;
  const uint32_t dsize = type == 0 ? 48u : (uint32_t)(3 * S);
  if (int rc = upload_points(c)) return rc;
  if (int rc = ensure(c, c->d_desc, c->desc_cap, std::max<size_t>(n * dsize, 1))) return rc;
  const size_t smem = type == 0 ? 3 * S * sizeof(double) : 0;
  FS_CUDA(c, cudaFuncSetAttribute(fs::describe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
  FS_CUDA(c, cudaMemsetAsync(c->d_count + 1, 0, sizeof(unsigned), c->stream));
  FS_CUDA(c, cudaEventRecord(c->ev[0], c->stream));
  if (n)
    fs::describe_kernel<<<(unsigned)n, 128, smem, c->stream>>>(integral_view(c), c->d_points, (unsigned)n, radius, type, normalize,
                                                               c->d_desc, c->d_count + 1);
  FS_CUDA(c, cudaGetLastError());
  FS_CUDA(c, cudaEventRecord(c->ev[1], c->stream));
  unsigned clamped = 0;
  FS_CUDA(c, cudaMemcpyAsync(&clamped, c->d_count + 1, sizeof clamped, cudaMemcpyDeviceToHost, c->stream));
  FS_CUDA(c, cudaStreamSynchronize(c->stream));
  c->stats.ms_describe = elapsed(c);
  c->stats.n_clamped = clamped;
  c->desc_size = dsize;
  return FS_OK;
}

int fs_num_points(fs_ctx* c, uint32_t* n, uint32_t* descriptor_size) {
  if (!c) return FS_ERR_INVALID;
  if (n) *n = (uint32_t)c->points.size();
  if (descriptor_size) *descriptor_size = c->desc_size;
  return FS_OK;
}

int fs_get_points(fs_ctx* c, fs_point* points, float* desc) {
  if (!c) return FS_ERR_INVALID;
  const size_t n = c->points.size();
  if (points && n) std::memcpy(points, c->points.data(), n * sizeof(fs_point));
  if (desc && n) {
    if (!c->desc_size) return fail(c, FS_ERR_STATE, "fs_get_points: no descriptors yet");
    FS_CUDA(c, cudaSetDevice(c->device));
    FS_CUDA(c, cudaMemcpy(desc, c->d_desc, n * c->desc_size * sizeof(float), cudaMemcpyDeviceToHost));
  }
  return FS_OK;
}

int fs_get_points_as_read(fs_ctx* c, int precision, const double spacing[3], const double origin[3], float* head, float* desc) {
  if (!c || !spacing || !origin) return FS_ERR_INVALID;
  const size_t n = c->points.size(), d = c->desc_size;
  if (!n) return FS_OK;
  if (!d) return fail(c, FS_ERR_STATE, "fs_get_points_as_read: no descriptors yet");
  if (!head || !desc) return fail(c, FS_ERR_INVALID, "fs_get_points_as_read: null output");
  FS_CUDA(c, cudaSetDevice(c->device));
  const size_t total = n * (6 + d);
  if (int rc = as_read_buffers(c, total)) return rc;
  fs::AsReadGeom g{};
  for (int i = 0; i < 3; i++) { g.spacing[i] = spacing[i]; g.origin[i] = origin[i]; }
  g.sspacing = std::pow(spacing[0] * spacing[1] * spacing[2], 1.0 / 3.0);  // the writers' Sspacing (surf_io.cpp)
  g.decimals = precision >= 0 ? precision : 6;  // "%f" = six decimals
  bool range_error = false;
  const int rc = as_read_finish(
      c, total, n * 6, head, desc,
      [&](fs::AsReadList list) {
        fs::as_read_kernel<<<as_read_blocks(total), 256, 0, c->stream>>>(c->d_points, c->d_desc, (unsigned)n, (unsigned)d, g,
                                                                          c->d_as_read, list);
      },
      [&](unsigned long long index) { return index < n * 6 ? 6 : g.decimals; }, &range_error);
  if (rc) return rc;
  // the reader's std::stof throws there: the keypoint file could not be read back
  if (range_error) return fail(c, FS_ERR_INVALID, "fs_get_points_as_read: a value's text is out of float range");
  return FS_OK;
}

int fs_get_stats(fs_ctx* c, fs_stats* out) {
  if (!c || !out) return FS_ERR_INVALID;
  *out = c->stats;
  return FS_OK;
}

/* ---- host-side pieces exposed for the CPU tests (include/frogsurf_debug.h) ---- */
float fs_debug_expf(float x) { return fs::glibc_expf(x); }
void fs_debug_expf_many(const float* x, float* y, size_t n) {
  for (size_t i = 0; i < n; i++) y[i] = fs::glibc_expf(x[i]);
}
void fs_debug_solve_offsets(const double* dD, const double* H10, double* X) { fs::solve_offsets(dD, H10, X); }
/* layer geometry and loop limits for an nx x ny x nz volume: per layer width, height, depth, step, filter, limit */
int fs_debug_layers(int nx, int ny, int nz, int32_t* out6, int cap) {
  const std::vector<LayerGeom> g = layer_geometry(nx, ny, nz, octaves_for(nx, ny, nz));
  for (size_t i = 0; i < g.size() && (int)i < cap; i++) {
    int32_t* o = out6 + 6 * i;
    o[0] = g[i].w; o[1] = g[i].h; o[2] = g[i].d; o[3] = g[i].step; o[4] = g[i].filter; o[5] = layer_limit(g[i]);
  }
  return (int)g.size();
}
/* vtk3DSURF.cxx:209-226 on n (response, original index) pairs: writes the surviving original indices, returns their count */
uint32_t fs_debug_select(const float* response, uint32_t n, int number_of_points, uint32_t* order) {
  std::vector<fs_point> pts(n);
  for (uint32_t i = 0; i < n; i++) { pts[i] = fs_point{0, 0, 0, 0, response[i], (int32_t)i}; }
  select_points(pts, number_of_points);
  for (size_t i = 0; i < pts.size(); i++) order[i] = (uint32_t)pts[i].laplacian;
  return (uint32_t)pts.size();
}

int fs_debug_set_option(const char* name, int value) {
  if (name && std::strcmp(name, "response_tile") == 0) { g_response_tile = value; return FS_OK; }
  return FS_ERR_INVALID;
}

/* the ordering fs_detect applies to its extrema: order[] receives the input indices, ascending by key, ties in input order */
void fs_debug_sort_keys(const uint64_t* keys, uint32_t n, uint32_t* order) {
  std::vector<KeyIndex> v(n);
  for (uint32_t i = 0; i < n; i++) v[i] = KeyIndex{keys[i], i};
  sort_by_key(v);
  for (uint32_t i = 0; i < n; i++) order[i] = v[i].index;
}

void fs_debug_keep_cast_volume(fs_ctx* c, int on) { if (c) c->keep_cast = on != 0; }

int fs_debug_as_read(const double* in, size_t n, int precision, float* out) {
  if (!n) return FS_OK;
  if (!in || !out) return FS_ERR_INVALID;
  fs_ctx* c = nullptr;
  if (int rc = fs_create(0, &c)) return rc;
  double* d_in = nullptr;
  size_t in_cap = 0;
  int rc = as_read_buffers(c, n);
  if (!rc) rc = ensure(c, d_in, in_cap, n);
  if (!rc && cudaMemcpy(d_in, in, n * sizeof(double), cudaMemcpyHostToDevice) != cudaSuccess) rc = FS_ERR_CUDA;
  const int decimals = precision >= 0 ? precision : 6;
  bool range_error = false;
  if (!rc)
    rc = as_read_finish(
        c, n, n, out, nullptr,
        [&](fs::AsReadList list) {
          fs::as_read_values_kernel<<<as_read_blocks(n), 256, 0, c->stream>>>(d_in, n, decimals, c->d_as_read, list);
        },
        [&](unsigned long long) { return decimals; }, &range_error);
  cudaFree(d_in);
  fs_destroy(c);
  return rc;
}

int fs_get_cast_volume(fs_ctx* c, int32_t* out) {
  if (!c || !out) return FS_ERR_INVALID;
  if (!c->have_volume) return fail(c, FS_ERR_STATE, "no volume");
  if (!c->keep_cast || c->cast_cap < (size_t)c->nx * c->ny * c->nz)
    return fail(c, FS_ERR_STATE, "the shifted volume is only kept after fs_debug_keep_cast_volume(ctx, 1)");
  FS_CUDA(c, cudaSetDevice(c->device));
  FS_CUDA(c, cudaMemcpy(out, c->d_cast, (size_t)c->nx * c->ny * c->nz * sizeof(int32_t), cudaMemcpyDeviceToHost));
  return FS_OK;
}

int fs_get_integral(fs_ctx* c, uint64_t* out) {
  if (!c || !out) return FS_ERR_INVALID;
  if (!c->have_volume) return fail(c, FS_ERR_STATE, "no volume");
  FS_CUDA(c, cudaSetDevice(c->device));
  FS_CUDA(c, cudaMemcpy(out, c->d_integral, (size_t)c->nx * c->ny * c->nz * sizeof(uint64_t), cudaMemcpyDeviceToHost));
  return FS_OK;
}

int fs_num_layers(fs_ctx* c, uint32_t* n) {
  if (!c || !n) return FS_ERR_INVALID;
  *n = (uint32_t)c->layers.size();
  return FS_OK;
}

int fs_get_layer(fs_ctx* c, uint32_t layer, int32_t info[5], float* responses, uint8_t* laplacian, uint8_t* isblob) {
  if (!c || layer >= c->layers.size()) return FS_ERR_INVALID;
  const Layer& L = c->layers[layer];
  if (info) { info[0] = L.dev.width; info[1] = L.dev.height; info[2] = L.dev.depth; info[3] = L.dev.step; info[4] = L.dev.filter; }
  FS_CUDA(c, cudaSetDevice(c->device));
  if (responses) FS_CUDA(c, cudaMemcpy(responses, L.dev.responses, L.voxels * sizeof(float), cudaMemcpyDeviceToHost));
  if (laplacian) FS_CUDA(c, cudaMemcpy(laplacian, L.dev.laplacian, L.voxels, cudaMemcpyDeviceToHost));
  if (isblob) FS_CUDA(c, cudaMemcpy(isblob, L.dev.isblob, L.voxels, cudaMemcpyDeviceToHost));
  return FS_OK;
}

}  // extern "C"
