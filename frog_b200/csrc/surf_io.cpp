#include "surf_io.h"

#include <zlib.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <map>
#include <sstream>

namespace fsio {

namespace {

double now_s() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

std::string trim(const std::string& s) {
  size_t a = s.find_first_not_of(" \t\r\n"), b = s.find_last_not_of(" \t\r\n");
  return a == std::string::npos ? std::string() : s.substr(a, b - a + 1);
}

template <typename T>
void flip_axis(unsigned char* data, const int dims[3], int axis) {
  T* p = reinterpret_cast<T*>(data);
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

size_t type_size(int t) {
  switch (t) {
    case FS_U8: case FS_I8: return 1;
    case FS_I16: case FS_U16: return 2;
    case FS_F64: return 8;
    default: return 4;
  }
}

bool read_metaimage_header(const std::string& path, MetaHeader& h, std::string& err) {
  h = MetaHeader{};
  auto fail = [&](const std::string& what) { err = "MetaImage " + path + ": " + what; return false; };
  std::ifstream f(path, std::ios::binary);
  if (!f) { err = "cannot open " + path; return false; }
  std::map<std::string, std::string> kv;
  std::string line, datafile;
  bool have_datafile = false;
  while (std::getline(f, line)) {
    const size_t eq = line.find('=');
    if (eq == std::string::npos) continue;
    const std::string k = trim(line.substr(0, eq)), v = trim(line.substr(eq + 1));
    kv[k] = v;
    if (k == "ElementDataFile") { datafile = v; have_datafile = true; break; }
  }
  if (!have_datafile) return fail("no ElementDataFile");
  auto ints = [&](const char* k, int* o, int n) { std::istringstream s(kv[k]); for (int i = 0; i < n; i++) if (!(s >> o[i])) return false; return true; };
  auto dbls = [&](const char* k, double* o, int n) { std::istringstream s(kv[k]); for (int i = 0; i < n; i++) if (!(s >> o[i])) return false; return true; };
  auto is_true = [&](const char* k) { const std::string& v = kv.count(k) ? kv[k] : std::string(); return v == "True" || v == "true" || v == "TRUE"; };
  auto key_value = [&](const char* k) { return std::string(k) + " = " + kv[k]; };
  int ndims = 0;
  if (!ints("NDims", &ndims, 1) || ndims != 3) { err = "MetaImage: NDims must be 3"; return false; }
  if (!ints("DimSize", h.dims, 3) || h.dims[0] <= 0 || h.dims[1] <= 0 || h.dims[2] <= 0) { err = "MetaImage: DimSize"; return false; }
  if (kv.count("ElementSpacing")) dbls("ElementSpacing", h.spacing, 3);
  else if (kv.count("ElementSize")) dbls("ElementSize", h.spacing, 3);
  if (kv.count("Offset")) dbls("Offset", h.origin, 3);
  else if (kv.count("Position")) dbls("Position", h.origin, 3);
  else if (kv.count("Origin")) dbls("Origin", h.origin, 3);
  if (kv.count("ElementNumberOfChannels") && kv["ElementNumberOfChannels"] != "1")
    return fail(key_value("ElementNumberOfChannels") + ": one channel only");
  if (kv.count("BinaryData") && !is_true("BinaryData")) return fail(key_value("BinaryData") + ": ASCII element data is not supported");
  const std::string et = kv["ElementType"];
  if (et == "MET_UCHAR") h.voxel_type = FS_U8;
  else if (et == "MET_CHAR") h.voxel_type = FS_I8;
  else if (et == "MET_SHORT") h.voxel_type = FS_I16;
  else if (et == "MET_USHORT") h.voxel_type = FS_U16;
  else if (et == "MET_INT") h.voxel_type = FS_I32;
  else if (et == "MET_UINT") h.voxel_type = FS_U32;
  else if (et == "MET_FLOAT") h.voxel_type = FS_F32;
  else if (et == "MET_DOUBLE") h.voxel_type = FS_F64;
  else if (et == "MET_LONG" || et == "MET_ULONG")  // sizeof(long) of the program that wrote the file
    return fail(key_value("ElementType") + ": its width depends on the platform that wrote the file");
  else if (et == "MET_LONG_LONG" || et == "MET_ULONG_LONG")
    return fail(key_value("ElementType") + ": 64-bit integers above 2^53 have no exact double value");
  else return fail("unsupported " + key_value("ElementType"));
  if (datafile == "LIST" || datafile.find('%') != std::string::npos)
    return fail(key_value("ElementDataFile") + ": lists and file patterns of data files are not supported");
  h.big_endian = is_true("BinaryDataByteOrderMSB") || is_true("ElementByteOrderMSB");
  h.compressed = is_true("CompressedData");
  if (h.compressed && kv.count("CompressedDataSize")) {
    std::istringstream s(kv["CompressedDataSize"]);
    if (!(s >> h.compressed_size) || h.compressed_size < 0) return fail("bad " + key_value("CompressedDataSize"));
  }
  if (datafile == "LOCAL") {
    h.data_file = path;
    h.data_offset = (long long)f.tellg();
    if (h.data_offset < 0) {  // the header ends the file: the data read reports it short
      f.clear();
      f.seekg(0, std::ios::end);
      h.data_offset = (long long)f.tellg();
    }
  } else {
    std::string dir;
    const size_t slash = path.find_last_of('/');
    if (slash != std::string::npos && datafile[0] != '/') dir = path.substr(0, slash + 1);
    h.data_file = dir + datafile;
    if (kv.count("HeaderSize")) {
      std::istringstream s(kv["HeaderSize"]);
      if (!(s >> h.data_offset) || h.data_offset < -1) return fail("bad " + key_value("HeaderSize"));
      if (h.data_offset == -1 && h.compressed) return fail(key_value("HeaderSize") + " with compressed data: the data's start is unknown");
    }
  }
  // vtkRobustImageReader.h:52-60, 97-113
  for (const char* key : {"TransformMatrix", "Orientation", "Rotation"}) {
    if (!kv.count(key)) continue;
    double m[9];
    if (!dbls(key, m, 9)) continue;
    for (int i = 0; i < 3; i++) h.flips[i] += m[4 * i] < 0;
  }
  return true;
}

namespace {

// Inflates one zlib or gzip stream (header detected by zlib) of at most `avail` bytes (< 0: to the end of the file)
// from `in` straight into dst[0, bytes): the stream must end exactly there.
bool inflate_into(std::ifstream& in, long long avail, unsigned char* dst, size_t bytes, const std::string& file,
                  std::string& err, ReadTimes* t) {
  auto fail = [&](const std::string& what) { err = "MetaImage " + file + ": " + what; return false; };
  z_stream zs{};
  if (inflateInit2(&zs, 15 + 32) != Z_OK) return fail("inflateInit2 failed");
  std::vector<unsigned char> buf(1 << 20);
  unsigned char spare;  // receives output beyond the expected size, to tell a longer stream from a complete one
  size_t done = 0;
  bool eof = false, ok = false;
  for (;;) {
    if (zs.avail_in == 0 && !eof) {
      const double t0 = now_s();
      const size_t want = avail < 0 ? buf.size() : (size_t)std::min<long long>(avail, (long long)buf.size());
      in.read(reinterpret_cast<char*>(buf.data()), (std::streamsize)want);
      const size_t got = (size_t)in.gcount();
      if (avail >= 0) avail -= (long long)got;
      eof = got < want || avail == 0;
      zs.next_in = buf.data();
      zs.avail_in = (uInt)got;
      if (t) t->read_s += now_s() - t0;
    }
    const double t0 = now_s();
    const bool full = done == bytes;
    zs.next_out = full ? &spare : dst + done;
    zs.avail_out = full ? 1u : (uInt)std::min<size_t>(bytes - done, 1u << 30);
    const uInt out0 = zs.avail_out;
    const int rc = inflate(&zs, Z_NO_FLUSH);
    const size_t produced = out0 - zs.avail_out;
    if (t) t->inflate_s += now_s() - t0;
    if (full && produced) { err = "decompresses to more than " + std::to_string(bytes) + " bytes (DimSize x element size)"; break; }
    done += produced;
    if (rc == Z_STREAM_END) {
      if (done == bytes) ok = true;
      else err = "compressed stream ends after " + std::to_string(done) + " of " + std::to_string(bytes) + " bytes";
      break;
    }
    if (rc == Z_BUF_ERROR && zs.avail_in == 0 && eof) {
      err = "compressed stream is truncated after " + std::to_string(done) + " of " + std::to_string(bytes) + " bytes";
      break;
    }
    if (rc != Z_OK && rc != Z_BUF_ERROR) { err = std::string("corrupt compressed stream: ") + (zs.msg ? zs.msg : "inflate failed"); break; }
  }
  inflateEnd(&zs);
  return ok || fail(err);
}

template <typename T>
void swap_elements(unsigned char* p, size_t bytes) {
  for (size_t i = 0; i + sizeof(T) <= bytes; i += sizeof(T)) std::reverse(p + i, p + i + sizeof(T));
}

}  // namespace

bool read_metaimage_data(const MetaHeader& h, unsigned char* dst, std::string& err, FILE* warnings, ReadTimes* t) {
  auto fail = [&](const std::string& what) { err = "MetaImage " + h.data_file + ": " + what; return false; };
  const size_t bytes = h.bytes();
  double t0 = now_s();
  std::ifstream d(h.data_file, std::ios::binary);
  if (!d) { err = "cannot open " + h.data_file; return false; }
  d.seekg(0, std::ios::end);
  const long long file_size = (long long)d.tellg();
  long long start = h.data_offset;
  if (start < 0) start = file_size - (long long)bytes;  // HeaderSize = -1: the data ends the file
  if (start < 0 || start > file_size) return fail("short data: " + std::to_string(file_size) + " bytes, " + std::to_string(bytes) + " needed");
  d.seekg(start);
  if (h.compressed) {
    if (h.compressed_size > file_size - start)
      return fail("CompressedDataSize = " + std::to_string(h.compressed_size) + " exceeds the " + std::to_string(file_size - start) +
                  " bytes after the header");
    if (t) t->read_s += now_s() - t0;
    if (!inflate_into(d, h.compressed_size, dst, bytes, h.data_file, err, t)) return false;
  } else {
    d.read(reinterpret_cast<char*>(dst), (std::streamsize)bytes);
    if ((size_t)d.gcount() != bytes) return fail("short data: " + std::to_string(d.gcount()) + " of " + std::to_string(bytes) + " bytes");
    if (t) t->read_s += now_s() - t0;
  }
  t0 = now_s();
  const size_t es = type_size(h.voxel_type);
  if (h.big_endian) {
    switch (es) {
      case 2: swap_elements<uint16_t>(dst, bytes); break;
      case 4: swap_elements<uint32_t>(dst, bytes); break;
      case 8: swap_elements<uint64_t>(dst, bytes); break;
    }
  }
  for (int i = 0; i < 3; i++) {
    for (int k = 0; k < h.flips[i]; k++) {  // once per key with a negative diagonal, as vtkRobustImageReader.h:97-113
      if (warnings) std::fprintf(warnings, "Warning : RobustReader flipping dimension %d\n", i);
      switch (es) {
        case 1: flip_axis<uint8_t>(dst, h.dims, i); break;
        case 2: flip_axis<uint16_t>(dst, h.dims, i); break;
        case 4: flip_axis<uint32_t>(dst, h.dims, i); break;
        default: flip_axis<uint64_t>(dst, h.dims, i); break;
      }
    }
  }
  if (t) t->swap_s += now_s() - t0;
  return true;
}

bool read_metaimage(const std::string& path, Volume& out, std::string& err, FILE* warnings) {
  MetaHeader h;
  if (!read_metaimage_header(path, h, err)) return false;
  out.data.resize(h.bytes());
  if (!read_metaimage_data(h, out.data.data(), err, warnings)) return false;
  for (int i = 0; i < 3; i++) { out.dims[i] = h.dims[i]; out.spacing[i] = h.spacing[i]; out.origin[i] = h.flipped_origin(i); }
  out.voxel_type = h.voxel_type;
  return true;
}

bool write_metaimage(const std::string& path, const Volume& v, std::string& err) {
  static const char* names[] = {"MET_UCHAR", "MET_SHORT", "MET_USHORT", "MET_INT", "MET_FLOAT", "MET_CHAR", "MET_UINT", "MET_DOUBLE"};
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
    case FS_I8: clamp_values<int8_t>(v.data, lo, o.clampMinValue, hi, o.clampMaxValue); break;
    case FS_U32: clamp_values<uint32_t>(v.data, lo, o.clampMinValue, hi, o.clampMaxValue); break;
    case FS_F64: clamp_values<double>(v.data, lo, o.clampMinValue, hi, o.clampMaxValue); break;
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

namespace {
thread_local std::string g_fsio_error;
}

// Text of this thread's most recent fsio_read_metaimage failure.
const char* fsio_last_error(void) { return g_fsio_error.c_str(); }

// Reads a MetaImage header and fills dims / spacing / origin / voxel_type / *bytes; with `data` non-null it also reads
// the voxels into data[0, *bytes) (cap must hold them) and, when `seconds` is non-null, stores the time spent on the
// header, reading, inflating and byte swaps / flips there (four values).  Returns 0, or -1 with fsio_last_error().
int fsio_read_metaimage(const char* path, int* dims, double* spacing, double* origin, int* voxel_type, void* data, size_t cap,
                        size_t* bytes, double* seconds) {
  const double t0 = fsio::now_s();
  fsio::MetaHeader h;
  std::string& err = g_fsio_error;
  if (!fsio::read_metaimage_header(path, h, err)) return -1;
  for (int i = 0; i < 3; i++) { dims[i] = h.dims[i]; spacing[i] = h.spacing[i]; origin[i] = h.flipped_origin(i); }
  *voxel_type = h.voxel_type;
  if (bytes) *bytes = h.bytes();
  if (!data) return 0;
  if (cap < h.bytes()) { err = "fsio_read_metaimage: " + std::to_string(cap) + " bytes given, " + std::to_string(h.bytes()) + " needed"; return -1; }
  fsio::ReadTimes t;
  const double t1 = fsio::now_s();
  if (!fsio::read_metaimage_data(h, static_cast<unsigned char*>(data), err, stdout, &t)) return -1;
  if (seconds) { seconds[0] = t1 - t0; seconds[1] = t.read_s; seconds[2] = t.inflate_s; seconds[3] = t.swap_s; }
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
