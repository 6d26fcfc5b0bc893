// Host I/O of bin/surf3d: a MetaImage (.mhd / .mha) volume reader and the reference's keypoint writers.
#pragma once

#include <cstdint>
#include <cstdio>
#include <string>
#include <vector>

#include "frogsurf.h"

namespace fsio {

struct Volume {
  int dims[3] = {0, 0, 0};
  double spacing[3] = {1, 1, 1};
  double origin[3] = {0, 0, 0};
  int voxel_type = FS_I16;  // fs_voxel_type
  std::vector<unsigned char> data;
};

size_t type_size(int voxel_type);  // bytes per element of an fs_voxel_type

// A MetaImage header (.mha / .mhd): what read_metaimage_data needs to fill a buffer of bytes() bytes.
struct MetaHeader {
  int dims[3] = {0, 0, 0};
  double spacing[3] = {1, 1, 1};
  double origin[3] = {0, 0, 0};  // as written; flipped_origin() is the volume's
  int voxel_type = FS_I16;
  std::string data_file;          // the header's own path for ElementDataFile = LOCAL
  long long data_offset = 0;      // where the data starts in data_file; -1: it ends the file (HeaderSize = -1)
  bool compressed = false;        // CompressedData: one zlib or gzip stream
  long long compressed_size = -1; // CompressedDataSize; -1: the stream runs to the end of the file
  bool big_endian = false;        // BinaryDataByteOrderMSB or ElementByteOrderMSB
  int flips[3] = {0, 0, 0};       // keys whose direction cosine of this axis is negative
  size_t bytes() const { return (size_t)dims[0] * dims[1] * dims[2] * type_size(voxel_type); }
  double flipped_origin(int i) const {
    double o = origin[i];
    for (int k = 0; k < flips[i]; k++) o = o - spacing[i] * (dims[i] - 1);
    return o;
  }
};

// Seconds spent by read_metaimage_data: reading the file, inflating, byte swaps and axis flips.
struct ReadTimes {
  double read_s = 0, inflate_s = 0, swap_s = 0;
};

// MetaImage with one component and binary element data, in the same file (ElementDataFile = LOCAL) or in the named
// file next to the header (after HeaderSize bytes; HeaderSize = -1: the data ends the file).  Element types
// MET_UCHAR / MET_CHAR / MET_SHORT / MET_USHORT / MET_INT / MET_UINT / MET_FLOAT / MET_DOUBLE.  CompressedData = True:
// one deflate stream with a zlib or gzip wrapper, CompressedDataSize bytes long or running to the end of the file,
// inflated in chunks into the voxel buffer; it must yield exactly DimSize x element size bytes.  Big-endian data
// (BinaryDataByteOrderMSB / ElementByteOrderMSB) is swapped to native order, then axis flips for negative
// TransformMatrix diagonals (vtkRobustImageReader.h:52-60, 97-113) are applied.  Refused, with the key named:
// MET_LONG / MET_ULONG (their width is the writer's platform's), 64-bit integers (not exact through double), LIST and
// pattern data files, ASCII data, more than one channel.
// (`warnings`: where the reader's axis-flip notices go; bin/surf3d prints them on stdout like the reference.)
bool read_metaimage(const std::string& path, Volume& out, std::string& err, FILE* warnings = stdout);
// The same in two steps: the header alone, then the data into dst[0, h.bytes()) (nothing partial is reported as read:
// on failure dst's contents are undefined).
bool read_metaimage_header(const std::string& path, MetaHeader& h, std::string& err);
bool read_metaimage_data(const MetaHeader& h, unsigned char* dst, std::string& err, FILE* warnings = stdout,
                         ReadTimes* times = nullptr);
bool write_metaimage(const std::string& path, const Volume& v, std::string& err);

// vtk3DSURF::WritePointsCSV / WritePointsCSVGZ / WritePointsBinary (vtk3DSURF.cxx:405-525): voxel-unit keypoints are
// written as origin + coordinate * spacing, scale * cbrt(spacing product), laplacian, response, descriptor.
bool write_points_csv(const std::string& path, const fs_point* pts, const float* desc, size_t n, size_t dsize,
                      const double spacing[3], const double origin[3]);
bool write_points_csvgz(const std::string& path, const char* gz_opts, int precision, const fs_point* pts, const float* desc,
                        size_t n, size_t dsize, const double spacing[3], const double origin[3]);
bool write_points_bin(const std::string& path, const fs_point* pts, const float* desc, size_t n, size_t dsize,
                      const double spacing[3], const double origin[3]);
// vtk3DSURF::ReadIPoints (vtk3DSURF.cxx:34-77, surf3d -p): one keypoint per line, "x,y,z,scale" in world units; returns
// x, y, z, scale per point in VOXEL units (as fs_set_points takes them).  A cell that is missing at the end of a line
// repeats the previous cell (the reference's getline leaves its string untouched), an empty line is skipped, a cell
// that is not a number is an error (std::stof throws in the reference).  n_outside counts the points the reference
// reports as "outside image" (they are kept).
bool read_points_file(const std::string& path, const double spacing[3], const double origin[3], const int dims[3],
                      std::vector<float>& xyzs, size_t& n_outside, std::string& err);

// bin/surf3d's options (surf3d.cxx:16-157), shared with bin/match's -surf3d key so that the two cannot drift apart.
struct SurfOptions {
  double spacing = 0, threshold = 0;
  int maxSize = 0, writeJSON = 0, writeBIN = 0, writeCSV = 0, writeCSVGZ = 1, descriptorType = 0, numberOfPoints = -1;
  int pad = 0, subVolumeRadius = 5, precision = -1, gpu = 0;
  const char *maskfilename = nullptr, *pointFile = nullptr, *gzOpts = nullptr;
  bool clampMinValues = false, clampMaxValues = false, normalize = true;
  float clampMinValue = 0, clampMaxValue = 0;
  std::string outfilename = "points";
};
// The reference's option loop over argv[first ..): every key consumes two tokens, unknown keys are ignored.  The
// strings stay argv's.
void parse_surf_options(int argc, char* const argv[], int first, SurfOptions& o);
// Options that need a VTK image filter this build does not restate (-s / -d, -m, -pad, -type 2) or picojson
// (-json 1): the one to name in the refusal, nullptr when there is none.
const char* unsupported_surf_option(const SurfOptions& o);
// the refusal both executables print for it before leaving with exit code 7
std::string unsupported_surf_message(const char* what);
// -cmin / -cmax: vtkImageThreshold with ReplaceOut (surf3d.cxx:232-255) on the volume as read
void clamp_volume(Volume& v, const SurfOptions& o);

// surf3d.cxx:269-285: {"bounds":{"xmax":..,"xmin":..,...}} in picojson's number format
bool write_bounds_json(const std::string& path, const Volume& v);

}  // namespace fsio
