// bin/surf3d -- the SURF3D producer's executable over libfrogsurf.so (SURVEY.md 8f-4).
// Same command line as the reference's surf3d (vtkOpenSURF3D/surf3d.cxx:16-157): the option loop advances two
// tokens per key and ignores keys it does not know.  Options that need VTK's own image filters (-s / -d
// resampling, -m mask, -pad, -type 2) or picojson (-json 1) are rejected loudly instead of being approximated; the input is a
// MetaImage volume already at its final sampling (.mha or .mhd, raw or compressed, either byte order, the element types
// fsio::read_metaimage lists).
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <string>
#include <vector>

#include "frogsurf.h"
#include "surf_io.h"

using std::cout;
using std::endl;

namespace {
double now() { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); }

int unsupported(const char* what) {
  std::cerr << fsio::unsupported_surf_message(what) << endl;
  return 7;
}

}  // namespace

int main(int argc, char* argv[]) {
  if (argc < 2) {
    cout << "Usage : surf3d file [options]" << endl;
    cout << "Available options:" << endl;
    cout << "-bin 0/1       : write points as bin file. Default : 0" << endl;
    cout << "-csv 0/1       : write points as csv file. Default : 0" << endl;
    cout << "-cmin value    : clamp values lower than specified value" << endl;
    cout << "-cmax value    : clamp values larger than specified value" << endl;
    cout << "-csvgz 0/1     : write points as csv.gz file. Default : 1" << endl;
    cout << "-gz opts       : set gz options such as compression level" << endl;
    cout << "-precision n   : set coefficients precision in csv.gz file" << endl;
    cout << "-n number      : maximum number of points" << endl;
    cout << "-normalize 0/1 : normalize descriptors (default : 1 )" << endl;
    cout << "-o basename    : set output file name. Default: \"points\"" << endl;
    cout << "-p file        : describe the points of a csv file (x,y,z,scale) instead of detecting" << endl;
    cout << "-r radius      : descriptor volume radius. Default : 5" << endl;
    cout << "-t threshold   : set detector threshold. Default: 0" << endl;
    cout << "-type 0/1      : set descriptor type :" << endl;
    cout << "       0 : SURF3D descriptor (default). Descriptor size : 48" << endl;
    cout << "       1 : subvolume HAAR coefficients. Descriptor size : 24 * radius^3" << endl;
    cout << "-gpu id        : CUDA device. Default : 0" << endl;
    exit(1);
  }

  fsio::SurfOptions o;
  fsio::parse_surf_options(argc, argv, 2, o);
  if (const char* what = fsio::unsupported_surf_option(o)) return unsupported(what);

  cout << "load : " << argv[1] << endl;
  double t0 = now();
  fsio::Volume vol;
  std::string err;
  if (!fsio::read_metaimage(argv[1], vol, err)) {
    std::cerr << "Cannot load file " << argv[1] << " as an image file; terminating.\n";
    std::cerr << err << endl;
    return 5;
  }
  fsio::clamp_volume(vol, o);
  cout << "Image loaded in " << now() - t0 << "s" << endl;
  fsio::write_bounds_json(o.outfilename + ".json", vol);

  fs_ctx* ctx = nullptr;
  if (fs_create(o.gpu, &ctx) != FS_OK) {
    std::cerr << "surf3d (B200): " << fs_last_error(nullptr) << endl;
    return 1;
  }
  auto die = [&](const char* what) {
    std::cerr << "surf3d (B200): " << what << ": " << fs_last_error(ctx) << endl;
    fs_destroy(ctx);
    return 1;
  };
  cout << "Image dimensions : " << vol.dims[0] << " " << vol.dims[1] << " " << vol.dims[2] << endl;
  cout << "Initial spacing  : " << vol.spacing[0] << " " << vol.spacing[1] << " " << vol.spacing[2] << endl;
  fs_stats st;
  t0 = now();
  if (fs_set_volume(ctx, vol.data.data(), vol.voxel_type, vol.dims[0], vol.dims[1], vol.dims[2]) != FS_OK) return die("volume");
  cout << "Integral computed in " << now() - t0 << "s" << endl;
  t0 = now();
  uint32_t n = 0;
  if (o.pointFile) {  // vtk3DSURF.cxx:183: ReadIPoints instead of the detector
    cout << "Use points in " << o.pointFile << endl;
    cout << "Read : " << o.pointFile << endl;
    std::vector<float> xyzs;
    size_t outside = 0;
    if (!fsio::read_points_file(o.pointFile, vol.spacing, vol.origin, vol.dims, xyzs, outside, err)) {
      std::cerr << "surf3d (B200): " << err << endl;
      fs_destroy(ctx);
      return 1;
    }
    if (outside) cout << "Error : " << outside << " points are outside image" << endl;
    n = (uint32_t)(xyzs.size() / 4);
    if (fs_set_points(ctx, xyzs.data(), n) != FS_OK) return die("points");
  } else {
    if (fs_detect(ctx, (float)o.threshold, &n) != FS_OK) return die("detector");
    cout << " Ipoints : " << n << endl;
    cout << "FastHessian computed in " << now() - t0 << "s" << endl;
  }
  t0 = now();
  if (fs_select(ctx, o.numberOfPoints) != FS_OK) return die("select");
  uint32_t dsize = 0;
  if (fs_describe(ctx, o.descriptorType, o.subVolumeRadius, o.normalize) != FS_OK) return die("descriptors");
  fs_num_points(ctx, &n, &dsize);
  cout << "Number of keypoints : " << n << endl;
  std::vector<fs_point> pts(n);
  std::vector<float> desc((size_t)n * dsize);
  if (fs_get_points(ctx, pts.data(), desc.data()) != FS_OK) return die("read back");
  cout << "Descriptors computed in " << now() - t0 << "s" << endl;
  fs_get_stats(ctx, &st);
  cout << "GPU ms : integral " << st.ms_integral << ", response map " << st.ms_response_map << ", extrema " << st.ms_extrema
       << ", descriptors " << st.ms_describe << endl;
  if (st.n_clamped) cout << "Warning : " << st.n_clamped << " keypoints have descriptor windows leaving the volume" << endl;
  fs_destroy(ctx);

  if (o.writeBIN) {
    t0 = now();
    fsio::write_points_bin(o.outfilename + ".bin", pts.data(), desc.data(), n, dsize, vol.spacing, vol.origin);
    cout << "bin written in " << now() - t0 << "s" << endl;
  }
  if (o.writeCSV) {
    t0 = now();
    fsio::write_points_csv(o.outfilename + ".csv", pts.data(), desc.data(), n, dsize, vol.spacing, vol.origin);
    cout << "csv written in " << now() - t0 << "s" << endl;
  }
  if (o.writeCSVGZ) {
    t0 = now();
    fsio::write_points_csvgz(o.outfilename + ".csv.gz", o.gzOpts, o.precision, pts.data(), desc.data(), n, dsize, vol.spacing, vol.origin);
    cout << "csvgz written in " << now() - t0 << "s" << endl;
  }
  return 0;
}
