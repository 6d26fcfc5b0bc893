#include "surf_io.h"

#include <zlib.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>

namespace fsio {

namespace {

size_t type_size(int t) { return t == FS_U8 ? 1 : (t == FS_I16 || t == FS_U16) ? 2 : 4; }

std::string trim(const std::string& s) {
  size_t a = s.find_first_not_of(" \t\r\n"), b = s.find_last_not_of(" \t\r\n");
  return a == std::string::npos ? std::string() : s.substr(a, b - a + 1);
}

template <typename T>
void flip_axis(std::vector<unsigned char>& data, const int dims[3], int axis) {
  T* p = reinterpret_cast<T*>(data.data());
  const size_t nx = dims[0], ny = dims[1], nz = dims[2];
  const size_t n[3] = {nx, ny, nz};
  for (size_t z = 0; z < nz; z++)
    for (size_t y = 0; y < ny; y++)
      for (size_t x = 0; x < nx; x++) {
        size_t c[3] = {x, y, z};
        if (c[axis] >= n[axis] / 2) continue;
        size_t o[3] = {x, y, z};
        o[axis] = n[axis] - 1 - c[axis];
        std::swap(p[c[0] + nx * (c[1] + ny * c[2])], p[o[0] + nx * (o[1] + ny * o[2])]);
      }
}

double sspacing(const double spacing[3]) { return std::pow(spacing[0] * spacing[1] * spacing[2], 1.0 / 3.0); }

// printf("%.<decimals>f", v) without printf: the writers format a million values per image and glibc's exact
// multi-precision conversion costs ~0.45 us each.  A double is M * 2^e with M < 2^53, so v * 10^decimals is the
// integer M * 10^decimals shifted by e: formed exactly in 128 bits, rounded half-to-even on the exact remainder as
// printf does in the default rounding mode.  Anything outside the comfortable range (|v| * 10^decimals >= 9e18,
// decimals > 9, inf, nan) goes to snprintf.  Returns the number of characters written (no terminator).
inline size_t format_fixed(double v, int decimals, char* out, size_t cap) {
  static const uint64_t kPow10[10] = {1ull, 10ull, 100ull, 1000ull, 10000ull, 100000ull, 1000000ull, 10000000ull, 100000000ull, 1000000000ull};
  uint64_t bits;
  std::memcpy(&bits, &v, 8);
  const uint64_t frac = bits & ((1ull << 52) - 1);
  const int expo = (int)((bits >> 52) & 0x7FF);
  if (decimals < 0 || decimals > 9 || expo == 0x7FF || !(std::fabs(v) * (double)kPow10[decimals > 9 || decimals < 0 ? 0 : decimals] < 9e18)) {
    char fmt[16];
    std::snprintf(fmt, sizeof fmt, "%%.%df", decimals < 0 ? 6 : decimals);
    return (size_t)std::snprintf(out, cap, fmt, v);
  }
  const uint64_t mant = expo ? (frac | (1ull << 52)) : frac;
  const int e2 = (expo ? expo : 1) - 1075;
  const unsigned __int128 prod = (unsigned __int128)mant * kPow10[decimals];  // < 2^53 * 2^30
  uint64_t n;
  if (e2 >= 0) {
    n = (uint64_t)(prod << e2);  // the range check keeps this below 2^64
  } else {
    const int k = -e2;
    if (k >= 100) {
      n = 0;  // prod < 2^83: far below one half
    } else {
      const unsigned __int128 q = prod >> k, rem = prod & ((((unsigned __int128)1) << k) - 1), half = ((unsigned __int128)1) << (k - 1);
      n = (uint64_t)q;
      if (rem > half || (rem == half && (n & 1ull))) n++;
    }
  }
  const uint64_t ip = n / kPow10[decimals], fp = n % kPow10[decimals];
  char tmp[40];
  size_t len = 0;
  if (bits >> 63) tmp[len++] = '-';
  char digits[24];
  int nd = 0;
  uint64_t t = ip;
  do { digits[nd++] = (char)('0' + t % 10); t /= 10; } while (t);
  while (nd) tmp[len++] = digits[--nd];
  if (decimals) {
    tmp[len++] = '.';
    uint64_t f = fp;
    for (int i = decimals - 1; i >= 0; i--) { tmp[len + i] = (char)('0' + f % 10); f /= 10; }
    len += decimals;
  }
  if (len > cap) len = cap;
  std::memcpy(out, tmp, len);
  return len;
}

}  // namespace

bool read_metaimage(const std::string& path, Volume& out, std::string& err, FILE* warnings) {
  std::ifstream f(path, std::ios::binary);
  if (!f) { err = "cannot open " + path; return false; }
  std::map<std::string, std::string> kv;
  std::string line, datafile;
  while (std::getline(f, line)) {
    const size_t eq = line.find('=');
    if (eq == std::string::npos) continue;
    const std::string k = trim(line.substr(0, eq)), v = trim(line.substr(eq + 1));
    kv[k] = v;
    if (k == "ElementDataFile") { datafile = v; break; }
  }
  auto ints = [&](const char* k, int* o, int n) { std::istringstream s(kv[k]); for (int i = 0; i < n; i++) if (!(s >> o[i])) return false; return true; };
  auto dbls = [&](const char* k, double* o, int n) { std::istringstream s(kv[k]); for (int i = 0; i < n; i++) if (!(s >> o[i])) return false; return true; };
  int ndims = 0;
  if (!ints("NDims", &ndims, 1) || ndims != 3) { err = "MetaImage: NDims must be 3"; return false; }
  if (!ints("DimSize", out.dims, 3)) { err = "MetaImage: DimSize"; return false; }
  if (kv.count("ElementSpacing")) dbls("ElementSpacing", out.spacing, 3);
  else if (kv.count("ElementSize")) dbls("ElementSize", out.spacing, 3);
  if (kv.count("Offset")) dbls("Offset", out.origin, 3);
  else if (kv.count("Position")) dbls("Position", out.origin, 3);
  else if (kv.count("Origin")) dbls("Origin", out.origin, 3);
  if (kv.count("ElementNumberOfChannels") && kv["ElementNumberOfChannels"] != "1") { err = "MetaImage: one channel only"; return false; }
  if (kv.count("CompressedData") && (kv["CompressedData"] == "True" || kv["CompressedData"] == "true")) { err = "MetaImage: compressed data unsupported"; return false; }
  if (kv.count("BinaryDataByteOrderMSB") && (kv["BinaryDataByteOrderMSB"] == "True" || kv["BinaryDataByteOrderMSB"] == "true")) { err = "MetaImage: big-endian data unsupported"; return false; }
  const std::string et = kv["ElementType"];
  if (et == "MET_UCHAR") out.voxel_type = FS_U8;
  else if (et == "MET_SHORT") out.voxel_type = FS_I16;
  else if (et == "MET_USHORT") out.voxel_type = FS_U16;
  else if (et == "MET_INT") out.voxel_type = FS_I32;
  else if (et == "MET_FLOAT") out.voxel_type = FS_F32;
  else { err = "MetaImage: unsupported ElementType " + et; return false; }
  const size_t bytes = (size_t)out.dims[0] * out.dims[1] * out.dims[2] * type_size(out.voxel_type);
  out.data.resize(bytes);
  if (datafile == "LOCAL") {
    f.read(reinterpret_cast<char*>(out.data.data()), bytes);
    if ((size_t)f.gcount() != bytes) { err = "MetaImage: short data"; return false; }
  } else {
    std::string dir;
    const size_t slash = path.find_last_of('/');
    if (slash != std::string::npos && datafile[0] != '/') dir = path.substr(0, slash + 1);
    std::ifstream d(dir + datafile, std::ios::binary);
    if (!d) { err = "cannot open " + dir + datafile; return false; }
    d.read(reinterpret_cast<char*>(out.data.data()), bytes);
    if ((size_t)d.gcount() != bytes) { err = "MetaImage: short data file"; return false; }
  }
  // vtkRobustImageReader.h:52-60, 97-113
  for (const char* key : {"TransformMatrix", "Orientation", "Rotation"}) {
    if (!kv.count(key)) continue;
    double m[9];
    if (!dbls(key, m, 9)) continue;
    for (int i = 0; i < 3; i++) {
      if (!(m[4 * i] < 0)) continue;
      if (warnings) std::fprintf(warnings, "Warning : RobustReader flipping dimension %d\n", i);
      switch (type_size(out.voxel_type)) {
        case 1: flip_axis<uint8_t>(out.data, out.dims, i); break;
        case 2: flip_axis<uint16_t>(out.data, out.dims, i); break;
        default: flip_axis<uint32_t>(out.data, out.dims, i); break;
      }
      out.origin[i] = out.origin[i] - out.spacing[i] * (out.dims[i] - 1);
    }
  }
  return true;
}

bool write_metaimage(const std::string& path, const Volume& v, std::string& err) {
  static const char* names[] = {"MET_UCHAR", "MET_SHORT", "MET_USHORT", "MET_INT", "MET_FLOAT"};
  std::ofstream f(path, std::ios::binary);
  if (!f) { err = "cannot write " + path; return false; }
  f << "ObjectType = Image\nNDims = 3\nBinaryData = True\nBinaryDataByteOrderMSB = False\nCompressedData = False\n";
  f.precision(17);
  f << "Offset = " << v.origin[0] << " " << v.origin[1] << " " << v.origin[2] << "\n";
  f << "ElementSpacing = " << v.spacing[0] << " " << v.spacing[1] << " " << v.spacing[2] << "\n";
  f << "DimSize = " << v.dims[0] << " " << v.dims[1] << " " << v.dims[2] << "\n";
  f << "ElementType = " << names[v.voxel_type] << "\nElementDataFile = LOCAL\n";
  f.write(reinterpret_cast<const char*>(v.data.data()), v.data.size());
  return (bool)f;
}

bool write_points_csv(const std::string& path, const fs_point* pts, const float* desc, size_t n, size_t dsize,
                      const double spacing[3], const double origin[3]) {
  const double ss = sspacing(spacing);
  std::ofstream f;
  f.open(path, std::ofstream::out | std::ofstream::trunc);
  if (!f) return false;
  for (size_t i = 0; i != n; i++) {
    const fs_point& p = pts[i];
    f << p.x * spacing[0] + origin[0] << ",";
    f << p.y * spacing[1] + origin[1] << ",";
    f << p.z * spacing[2] + origin[2] << ",";
    f << p.scale * ss << ",";
    f << p.laplacian << ",";
    f << p.response << ",";
    for (size_t k = 0; k < dsize; k++) {
      f << desc[i * dsize + k];
      if (k < dsize - 1) f << ",";
    }
    f << std::endl;
  }
  f.close();
  return true;
}

bool write_points_csvgz(const std::string& path, const char* gz_opts, int precision, const fs_point* pts, const float* desc,
                        size_t n, size_t dsize, const double spacing[3], const double origin[3]) {
  const double ss = sspacing(spacing);
  std::string opts("w");
  if (gz_opts) opts += gz_opts;
  gzFile gz = gzopen(path.c_str(), opts.c_str());
  if (!gz) return false;
  // one formatted row per gzwrite instead of one gzprintf per cell: the deflate stream depends on the bytes only
  const int dec = precision >= 0 ? precision : 6;  // "%f" = six decimals
  std::vector<char> row(64 * (dsize + 8) + 512);
  for (size_t i = 0; i != n; i++) {
    const fs_point& p = pts[i];
    size_t o = 0;
    auto put = [&](double v, int decimals) {
      if (row.size() - o < 400) row.resize(row.size() * 2);
      o += format_fixed(v, decimals, row.data() + o, row.size() - o);
    };
    put(p.x * spacing[0] + origin[0], 6); row[o++] = ',';
    put(p.y * spacing[1] + origin[1], 6); row[o++] = ',';
    put(p.z * spacing[2] + origin[2], 6); row[o++] = ',';
    put(p.scale * ss, 6); row[o++] = ',';
    o += std::snprintf(row.data() + o, row.size() - o, "%d,", p.laplacian);
    put(p.response, 6); row[o++] = ',';
    for (size_t k = 0; k < dsize; k++) {
      put(desc[i * dsize + k], dec);
      if (k < dsize - 1) row[o++] = ',';
    }
    row[o++] = '\n';
    if (gzwrite(gz, row.data(), (unsigned)o) != (int)o) { gzclose(gz); return false; }
  }
  return gzclose(gz) == Z_OK;
}

bool write_points_bin(const std::string& path, const fs_point* pts, const float* desc, size_t n, size_t dsize,
                      const double spacing[3], const double origin[3]) {
  const double ss = sspacing(spacing);
  FILE* file = std::fopen(path.c_str(), "wb");
  if (!file) return false;
  std::vector<float> rec(6 + dsize);
  for (size_t i = 0; i != n; i++) {
    const fs_point& p = pts[i];
    rec[0] = p.x * spacing[0] + origin[0];
    rec[1] = p.y * spacing[1] + origin[1];
    rec[2] = p.z * spacing[2] + origin[2];
    rec[3] = p.scale * ss;
    rec[4] = p.laplacian;
    rec[5] = p.response;
    if (dsize) std::memcpy(rec.data() + 6, desc + i * dsize, dsize * sizeof(float));
    std::fwrite(rec.data(), sizeof(float), rec.size(), file);
  }
  std::fclose(file);
  return true;
}

bool read_points_file(const std::string& path, const double spacing[3], const double origin[3], const int dims[3],
                      std::vector<float>& xyzs, size_t& n_outside, std::string& err) {
  std::ifstream f(path);
  if (!f) { err = "cannot open " + path; return false; }
  const double ss = sspacing(spacing);
  double lo[3], hi[3];
  for (int i = 0; i < 3; i++) { lo[i] = origin[i]; hi[i] = origin[i] + (dims[i] - 1) * spacing[i]; }
  xyzs.clear();
  n_outside = 0;
  std::string line, cell;
  size_t line_no = 0;
  while (std::getline(f, line)) {
    line_no++;
    size_t pos = 0;
    bool exhausted = line.empty();  // an empty stream yields no first cell: the line is skipped
    if (exhausted) continue;
    float v[4];
    for (int k = 0; k < 4; k++) {
      if (!exhausted) {
        if (k > 0 && pos >= line.size()) {  // the line ended with a comma: getline erases its string, extracts nothing
          cell.clear();
          exhausted = true;
        } else {
          const size_t comma = line.find(',', pos);
          if (comma == std::string::npos) { cell = line.substr(pos); exhausted = true; }
          else { cell = line.substr(pos, comma - pos); pos = comma + 1; }
        }
      }  // else: `cell` keeps its previous content, as the reference's failed getline leaves it
      try {
        v[k] = std::stof(cell);
      } catch (...) {
        err = "stof failed at line " + std::to_string(line_no) + " of " + path;
        return false;
      }
    }
    xyzs.push_back((float)((v[0] - origin[0]) / spacing[0]));
    xyzs.push_back((float)((v[1] - origin[1]) / spacing[1]));
    xyzs.push_back((float)((v[2] - origin[2]) / spacing[2]));
    xyzs.push_back((float)(v[3] / ss));
    if (!(v[0] >= lo[0] && v[0] <= hi[0] && v[1] >= lo[1] && v[1] <= hi[1] && v[2] >= lo[2] && v[2] <= hi[2])) n_outside++;
  }
  return true;
}

void parse_surf_options(int argc, char* const argv[], int first, SurfOptions& o) {
  for (int k = first; k < argc; k += 2) {
    const char* key = argv[k];
    char* value = k + 1 < argc ? argv[k + 1] : (char*)"";
    if (std::strcmp(key, "-d") == 0) o.maxSize = std::atoi(value);
    if (std::strcmp(key, "-s") == 0) o.spacing = std::atof(value);
    if (std::strcmp(key, "-t") == 0) o.threshold = std::atof(value);
    if (std::strcmp(key, "-cmin") == 0) { o.clampMinValues = true; o.clampMinValue = std::atof(value); }
    if (std::strcmp(key, "-cmax") == 0) { o.clampMaxValues = true; o.clampMaxValue = std::atof(value); }
    if (std::strcmp(key, "-m") == 0) o.maskfilename = value;
    if (std::strcmp(key, "-o") == 0) o.outfilename = value;
    if (std::strcmp(key, "-json") == 0) o.writeJSON = std::atoi(value);
    if (std::strcmp(key, "-csv") == 0) o.writeCSV = std::atoi(value);
    if (std::strcmp(key, "-bin") == 0) o.writeBIN = std::atoi(value);
    if (std::strcmp(key, "-csvgz") == 0) o.writeCSVGZ = std::atoi(value);
    if (std::strcmp(key, "-type") == 0) o.descriptorType = std::atoi(value);
    if (std::strcmp(key, "-n") == 0) o.numberOfPoints = std::atoi(value);
    if (std::strcmp(key, "-p") == 0) o.pointFile = value;
    if (std::strcmp(key, "-r") == 0) o.subVolumeRadius = std::atoi(value);
    if (std::strcmp(key, "-normalize") == 0) o.normalize = std::atoi(value);
    if (std::strcmp(key, "-pad") == 0) o.pad = std::atoi(value);
    if (std::strcmp(key, "-gz") == 0) o.gzOpts = value;
    if (std::strcmp(key, "-precision") == 0) o.precision = std::atoi(value);
    if (std::strcmp(key, "-gpu") == 0) o.gpu = std::atoi(value);
  }
}

const char* unsupported_surf_option(const SurfOptions& o) {
  if (o.spacing != 0 || o.maxSize > 0) return "-s / -d (vtkImageResample)";
  if (o.maskfilename) return "-m (mask resampling)";
  if (o.pad) return "-pad (vtkImageMirrorPad)";
  if (o.descriptorType == 2) return "-type 2 (vtkImageResize)";
  if (o.writeJSON) return "-json 1 (picojson point dump)";
  return nullptr;
}

std::string unsupported_surf_message(const char* what) {
  return std::string("surf3d (B200): ") + what + " needs a VTK image filter that this build does not restate; terminating.";
}

namespace {
template <typename T>
void clamp_values(std::vector<unsigned char>& data, bool lo_on, float lo, bool hi_on, float hi) {
  // values below -cmin become cmin, above -cmax become cmax
  T* p = reinterpret_cast<T*>(data.data());
  const size_t n = data.size() / sizeof(T);
  for (size_t i = 0; i < n; i++) {
    if (lo_on && (double)p[i] < (double)lo) p[i] = (T)lo;
    if (hi_on && (double)p[i] > (double)hi) p[i] = (T)hi;
  }
}
}  // namespace

void clamp_volume(Volume& v, const SurfOptions& o) {
  if (!o.clampMinValues && !o.clampMaxValues) return;
  const bool lo = o.clampMinValues, hi = o.clampMaxValues;
  switch (v.voxel_type) {
    case FS_U8: clamp_values<uint8_t>(v.data, lo, o.clampMinValue, hi, o.clampMaxValue); break;
    case FS_I16: clamp_values<int16_t>(v.data, lo, o.clampMinValue, hi, o.clampMaxValue); break;
    case FS_U16: clamp_values<uint16_t>(v.data, lo, o.clampMinValue, hi, o.clampMaxValue); break;
    case FS_I32: clamp_values<int32_t>(v.data, lo, o.clampMinValue, hi, o.clampMaxValue); break;
    default: clamp_values<float>(v.data, lo, o.clampMinValue, hi, o.clampMaxValue); break;
  }
}

bool write_bounds_json(const std::string& path, const Volume& v) {
  // picojson serialises a std::map (keys sorted) and numbers as "%.f" when integral below 2^53, else "%.17g"
  auto num = [](double x) {
    char buf[256];
    double tmp;
    std::snprintf(buf, sizeof buf, std::fabs(x) < (double)(1ULL << 53) && std::modf(x, &tmp) == 0 ? "%.f" : "%.17g", x);
    return std::string(buf);
  };
  double b[6];
  for (int i = 0; i < 3; i++) {
    b[2 * i] = v.origin[i];
    b[2 * i + 1] = v.origin[i] + (v.dims[i] - 1) * v.spacing[i];
  }
  std::ofstream f;
  f.open(path, std::ofstream::out | std::ofstream::trunc);
  if (!f) return false;
  f << "{\"bounds\":{\"xmax\":" << num(b[1]) << ",\"xmin\":" << num(b[0]) << ",\"ymax\":" << num(b[3]) << ",\"ymin\":" << num(b[2])
    << ",\"zmax\":" << num(b[5]) << ",\"zmin\":" << num(b[4]) << "}}";
  f.close();
  return true;
}

}  // namespace fsio

// ---- plain-C face of the host I/O (frog_b200/libfsio.so), so the CPU test suite can compare the writers with the
// reference's without a GPU ----
extern "C" {

// fmt: 0 csv, 1 csv.gz, 2 bin.  Returns 0 on success.
int fsio_write_points(const char* path, int fmt, const char* gz_opts, int precision, const fs_point* pts, const float* desc,
                      size_t n, size_t dsize, const double* spacing, const double* origin) {
  bool ok = false;
  if (fmt == 0) ok = fsio::write_points_csv(path, pts, desc, n, dsize, spacing, origin);
  else if (fmt == 1) ok = fsio::write_points_csvgz(path, gz_opts, precision, pts, desc, n, dsize, spacing, origin);
  else if (fmt == 2) ok = fsio::write_points_bin(path, pts, desc, n, dsize, spacing, origin);
  return ok ? 0 : -1;
}

// Reads a MetaImage header + data; returns 0 and fills dims / spacing / origin / voxel_type, copying at most `cap`
// bytes of voxel data into `data` (may be null to query the size through *bytes).
int fsio_read_metaimage(const char* path, int* dims, double* spacing, double* origin, int* voxel_type, void* data, size_t cap,
                        size_t* bytes) {
  fsio::Volume v;
  std::string err;
  if (!fsio::read_metaimage(path, v, err)) return -1;
  for (int i = 0; i < 3; i++) { dims[i] = v.dims[i]; spacing[i] = v.spacing[i]; origin[i] = v.origin[i]; }
  *voxel_type = v.voxel_type;
  if (bytes) *bytes = v.data.size();
  if (data) std::memcpy(data, v.data.data(), v.data.size() < cap ? v.data.size() : cap);
  return 0;
}

// x, y, z, scale per point in voxel units; returns the number of points (at most cap are copied), -1 on error
long fsio_read_points(const char* path, const double* spacing, const double* origin, const int* dims, float* xyzs, long cap,
                      long* n_outside) {
  std::vector<float> v;
  std::string err;
  size_t outside = 0;
  if (!fsio::read_points_file(path, spacing, origin, dims, v, outside, err)) return -1;
  if (n_outside) *n_outside = (long)outside;
  const long n = (long)(v.size() / 4);
  if (xyzs) std::memcpy(xyzs, v.data(), sizeof(float) * 4 * (size_t)(n < cap ? n : cap));
  return n;
}

// test hook: formats every v[i] with `decimals` decimals and compares with snprintf("%.<decimals>f"); returns the
// number of values that differ (the first one's index in *first_bad)
long fsio_debug_format_check(const double* v, long n, int decimals, long* first_bad) {
  long bad = 0;
  char fmt[16], a[512], b[512];
  std::snprintf(fmt, sizeof fmt, "%%.%df", decimals);
  for (long i = 0; i < n; i++) {
    const size_t la = fsio::format_fixed(v[i], decimals, a, sizeof a - 1);
    a[la] = 0;
    std::snprintf(b, sizeof b, fmt, v[i]);
    if (std::strcmp(a, b) != 0) { if (!bad && first_bad) *first_bad = i; bad++; }
  }
  return bad;
}

// test hook: out[i] = strtof of in[i] as the .csv.gz writer formats it with `decimals` decimals (six when negative) --
// the values the matcher's reader returns from that text; the reference for fs_get_points_as_read
void fsio_debug_as_read(const double* in, long n, int decimals, float* out) {
  const int dec = decimals >= 0 ? decimals : 6;
#pragma omp parallel for schedule(static)
  for (long i = 0; i < n; i++) {
    char a[512];
    a[fsio::format_fixed(in[i], dec, a, sizeof a - 1)] = 0;
    out[i] = std::strtof(a, nullptr);
  }
}

int fsio_write_bounds_json(const char* path, const int* dims, const double* spacing, const double* origin) {
  fsio::Volume v;
  for (int i = 0; i < 3; i++) { v.dims[i] = dims[i]; v.spacing[i] = spacing[i]; v.origin[i] = origin[i]; }
  return fsio::write_bounds_json(path, v) ? 0 : -1;
}

}  // extern "C"
