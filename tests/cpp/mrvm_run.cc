// Drives MultiResolutionVoxelMapB200 (adapter/registrators_b200.h) with the stand-in headers of tests/stubs, the way
// MapBuilder::SaveMaps uses the reference class: Initialise, InsertPointCloud per frame, OutputToPointCloud.
// Reads  <in>:  int64 n_scans, then per scan: int64 n, float origin[3], InnerPointType points[n]
// writes <out>: the output records {x, y, z, intensity} as raw floats.  tests/test_gpu_mrvm.py compares them with the
// oracle.
#include <cstdint>
#include <cstdio>
#include <fstream>
#include <vector>

#include "registrators_b200.h"

using namespace static_map;

struct MrvmSettings {   // builder/multi_resolution_voxel_map.h:55-66
  bool output_average = false;
  bool output_rgb = false;
  bool use_max_intensity = true;
  float prob_threshold = 0.6f;
  float low_resolution = 1.f;
  float high_resolution = 0.1f;
  float hit_prob = 0.55f;
  float miss_prob = 0.48f;
  float z_offset = 0.f;
  int max_point_num_in_cell = 10;
};

int main(int argc, char** argv) {
  if (argc != 3) return 2;
  std::ifstream in(argv[1], std::ios::binary);
  int64_t n_scans = 0;
  in.read(reinterpret_cast<char*>(&n_scans), 8);
  MrvmSettings settings;
  settings.output_average = true;
  registrator::MultiResolutionVoxelMapB200 map;
  map.Initialise(settings);
  map.SetOffsetZ(0.f);
  for (int64_t s = 0; s < n_scans; ++s) {
    int64_t n = 0;
    float origin[3];
    in.read(reinterpret_cast<char*>(&n), 8);
    in.read(reinterpret_cast<char*>(origin), sizeof(origin));
    data::InnerCloudType cloud;
    cloud.points.resize(n);
    in.read(reinterpret_cast<char*>(cloud.points.data()), n * sizeof(data::InnerPointType));
    CHECK(in.good());
    map.InsertPointCloud(cloud, origin);
  }
  std::vector<float> out;
  map.OutputToPointCloud(settings.prob_threshold, settings.output_rgb, &out);
  std::ofstream o(argv[2], std::ios::binary);
  o.write(reinterpret_cast<const char*>(out.data()), out.size() * sizeof(float));
  fprintf(stderr, "voxels %zu, records %zu\n", map.size(), out.size() / 4);
  return 0;
}
