// Drives FilterFactoryB200 (adapter/registrators_b200.h) with the stand-in headers of tests/stubs, the way
// DataCollector::CloudPreProcessing uses the reference Factory: the <filters> block of static_mapping_default.xml
// (Range 4.5 - 75 m, RandomSampler 0.35), then Filter on each scan.
// Reads  <in>:  int64 n_scans, then per scan: int64 n, InnerPointType points[n]
// writes <out>: per scan int64 m, then the m filtered InnerPointType records.  tests/test_gpu_filters.py compares
// them with the oracle.
#include <cstdint>
#include <fstream>
#include <memory>
#include <vector>

#include "registrators_b200.h"

using namespace static_map;

int main(int argc, char** argv) {
  if (argc != 3) return 2;
  std::ifstream in(argv[1], std::ios::binary);
  std::ofstream out(argv[2], std::ios::binary);
  registrator::FilterFactoryB200 factory(0, 7);
  factory.AddFilter("Range", {{"min_range", 1, " 4.5 "}, {"max_range", 1, "75"}});
  factory.AddFilter("RandomSampler", {{"sampling_rate", 1, "0.35"}});
  int64_t n_scans = 0;
  in.read(reinterpret_cast<char*>(&n_scans), sizeof(n_scans));
  for (int64_t k = 0; k < n_scans; ++k) {
    int64_t n = 0;
    in.read(reinterpret_cast<char*>(&n), sizeof(n));
    auto cloud = std::make_shared<data::InnerCloudType>();
    cloud->points.resize(static_cast<size_t>(n));
    in.read(reinterpret_cast<char*>(cloud->points.data()), n * sizeof(data::InnerPointType));
    factory.Filter(cloud);
    const int64_t m = static_cast<int64_t>(cloud->points.size());
    out.write(reinterpret_cast<const char*>(&m), sizeof(m));
    out.write(reinterpret_cast<const char*>(cloud->points.data()), m * sizeof(data::InnerPointType));
  }
  return in && out ? 0 : 1;
}
