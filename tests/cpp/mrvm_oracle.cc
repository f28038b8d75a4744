// ORACLE — TEST INFRASTRUCTURE ONLY: only tests/ and profiles/time_mrvm.py load it (through tests/mrvm_oracle.py,
// which compiles this file with g++ -O2 -ffp-contract=off on first use); the product never does.
//
// builder::MultiResolutionVoxelMap (builder/multi_resolution_voxel_map.{h,cc}) restated serially: Initialise (:42-48),
// SetOffsetZ (:50-52), InsertPointCloud (:54-123) with its loop run by one thread in point order,
// OutputToPointCloud (:125-215) and common::VoxelCastingBresenham (common/math.cc:35-95) with its CHECK_EQ on the ray
// end.  The probability arithmetic is the reference's, expression by expression (.h:134-140, .cc:36-40, :63-69):
// float odds table, float log-odds sums, double OddToProbability rounded to float, clamp, `* kTableSize`, cast to
// uint8.  Three things differ from the reference on purpose, as in the engine (include/sm_b200.h): voxels are output
// in ascending key order, points with a non-finite coordinate are dropped, and an insert with a voxel index outside
// [-2^20, 2^20) is refused before anything changes.
//
// C API (all extern "C"):
//   sm_oracle_mrvm_create(settings) -> handle, NULL where map_builder_options.cc:66-68 CHECK-fails or
//       high_resolution <= 0;  settings = MrvmSettings (.h:55-66) in the layout of sm_mrvm_settings
//   sm_oracle_mrvm_insert(h, pts5, n, origin_3) -> dropped (non-finite) points, -1 index out of range (nothing
//       changed), -2 ray-end CHECK_EQ failure;  pts5 = packed InnerPointType
//   sm_oracle_mrvm_output(h, threshold, rgb, out4, capacity) -> number of {x, y, z, intensity or grey} records
//   sm_oracle_mrvm_state(h, keys, prob, max_intensity, npts, points4, capacity) -> voxel count, layout of
//       sm_debug_mrvm_state (include/sm_b200_debug.h)
//   sm_oracle_voxel_casting_bresenham(start_3, end_3, step, out3, capacity) -> voxel count, -1 / -2 as above
#include <math.h>
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <unordered_map>
#include <vector>

extern "C" {
typedef struct sm_oracle_mrvm_settings {
  int32_t output_average, output_rgb, use_max_intensity;
  float prob_threshold, low_resolution, high_resolution, hit_prob, miss_prob, z_offset;
  int32_t max_point_num_in_cell;
} sm_oracle_mrvm_settings;
}

namespace {

using Probability = uint8_t;
constexpr size_t kTableSize = 256;
constexpr Probability kUnknown = 128;
constexpr int kHalf = 1 << 20;

struct Point { float x, y, z, intensity, factor; };

struct Voxel {
  Probability probability = kUnknown;
  bool need_update = true;
  int max_intensity = 0;
  std::vector<Point> points;
};

template <typename T>
T Clamp(const T value, const T min, const T max) {
  if (value > max) return max;
  if (value < min) return min;
  return value;
}

float ProbabilityToOdd(float prob) { return std::log(prob / (1. - prob)); }
float OddToProbability(float odd) { return 1. - 1. / (1. + std::exp(odd)); }

struct Key {
  int x, y, z;
  bool operator==(const Key& o) const { return x == o.x && y == o.y && z == o.z; }
};
uint64_t key64(const Key& k) {
  return ((uint64_t)(k.x + kHalf) << 42) | ((uint64_t)(k.y + kHalf) << 21) | (uint64_t)(k.z + kHalf);
}
struct KeyHash {
  size_t operator()(const Key& k) const { return std::hash<uint64_t>()(key64(k)); }
};

// voxel index of one coordinate: lround(floor(v / step)) in float; false outside [-2^20, 2^20)
bool voxel_index(float v, float step, int* out) {
  const float f = std::floor(v / step);
  if (!(f >= -(float)kHalf && f < (float)kHalf)) return false;
  *out = (int)std::lround(f);
  return true;
}

// common::VoxelCastingBresenham; returns false where the reference's CHECK_EQ on the end voxel would fail
bool VoxelCastingBresenham(const Key& start, const Key& end, std::vector<Key>* visited) {
  visited->clear();
  int x0 = start.x, y0 = start.y, z0 = start.z;
  int x1 = end.x, y1 = end.y, z1 = end.z;
  const int dx = std::abs(x1 - x0), sx = x0 < x1 ? 1 : -1;
  const int dy = std::abs(y1 - y0), sy = y0 < y1 ? 1 : -1;
  const int dz = std::abs(z1 - z0), sz = z0 < z1 ? 1 : -1;
  const int dm = std::max({dx, dy, dz});
  x1 = y1 = z1 = (dm >> 1);
  int i = dm;
  visited->reserve(dm + 1);
  for (;;) {
    visited->push_back(Key{x0, y0, z0});
    if (i-- == 0) break;
    x1 -= dx;
    if (x1 < 0) { x1 += dm; x0 += sx; }
    y1 -= dy;
    if (y1 < 0) { y1 += dm; y0 += sy; }
    z1 -= dz;
    if (z1 < 0) { z1 += dm; z0 += sz; }
  }
  return x0 == end.x && y0 == end.y && z0 == end.z;
}

}  // namespace

struct sm_oracle_mrvm {
  sm_oracle_mrvm_settings settings;
  float odds_table[kTableSize];
  std::unordered_map<Key, Voxel, KeyHash> voxels;

  std::vector<std::pair<uint64_t, const Voxel*>> sorted() const {
    std::vector<std::pair<uint64_t, const Voxel*>> v;
    v.reserve(voxels.size());
    for (const auto& kv : voxels) v.emplace_back(key64(kv.first), &kv.second);
    std::sort(v.begin(), v.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
    return v;
  }
};

extern "C" sm_oracle_mrvm* sm_oracle_mrvm_create(const sm_oracle_mrvm_settings* s) {
  // map_builder_options.cc:66-68 CHECKs, and a usable voxel size
  if (!s || !(s->hit_prob > 0.5f) || !(s->miss_prob < 0.5f) || s->max_point_num_in_cell < 1 ||
      !(s->high_resolution > 0.f))
    return nullptr;
  sm_oracle_mrvm* m = new sm_oracle_mrvm;
  for (size_t i = 0; i < kTableSize; ++i) m->odds_table[i] = ProbabilityToOdd(static_cast<float>(i) / kTableSize);
  m->settings = *s;   // Initialise
  m->settings.hit_prob = Clamp(m->settings.hit_prob, 0.501f, 0.9f);
  m->settings.miss_prob = Clamp(m->settings.miss_prob, 0.1f, 0.499f);
  return m;
}

extern "C" void sm_oracle_mrvm_destroy(sm_oracle_mrvm* m) { delete m; }

extern "C" void sm_oracle_mrvm_set_offset_z(sm_oracle_mrvm* m, float offset) { m->settings.z_offset = offset; }

extern "C" int64_t sm_oracle_mrvm_size(const sm_oracle_mrvm* m) { return (int64_t)m->voxels.size(); }

extern "C" int64_t sm_oracle_mrvm_insert(sm_oracle_mrvm* m, const float* pts5, int64_t n, const float* origin) {
  if (n <= 0) return 0;                                   // "cloud is empty."
  const sm_oracle_mrvm_settings& st = m->settings;
  float offseted_origin[3] = {origin[0], origin[1], origin[2]};
  offseted_origin[2] += st.z_offset;
  const float resolution = st.high_resolution;
  Key start;
  if (!voxel_index(offseted_origin[0], resolution, &start.x) || !voxel_index(offseted_origin[1], resolution, &start.y) ||
      !voxel_index(offseted_origin[2], resolution, &start.z))
    return -1;
  // drop non-finite points; refuse the insert if a voxel index is out of range, before anything changes
  std::vector<int64_t> kept;
  std::vector<Key> ends;
  kept.reserve(n);
  ends.reserve(n);
  int64_t dropped = 0;
  for (int64_t i = 0; i < n; ++i) {
    const float* p = pts5 + 5 * i;
    if (!std::isfinite(p[0]) || !std::isfinite(p[1]) || !std::isfinite(p[2])) { ++dropped; continue; }
    Key e;
    if (!voxel_index(p[0], resolution, &e.x) || !voxel_index(p[1], resolution, &e.y) ||
        !voxel_index(p[2], resolution, &e.z))
      return -1;
    kept.push_back(i);
    ends.push_back(e);
  }
  const float hit_log_odd = ProbabilityToOdd(st.hit_prob);
  const float miss_log_odd = ProbabilityToOdd(st.miss_prob);
  auto update_prob = [&](Probability former_prob, bool hit) -> float {
    float odd = m->odds_table[former_prob];
    odd += hit ? hit_log_odd : miss_log_odd;
    return Clamp(OddToProbability(odd), 0.1f, 0.9f);
  };
  std::vector<Key> end_voxels;
  std::vector<Key> ray;
  for (size_t j = 0; j < kept.size(); ++j) {
    const float* pf = pts5 + 5 * kept[j];
    Point point{pf[0], pf[1], pf[2], pf[3], pf[4]};
    if (!VoxelCastingBresenham(start, ends[j], &ray)) return -2;   // CHECK_EQ(x0, x1_init) etc.
    if (ray.empty()) continue;
    const Key high_end_index = ray.back();
    Voxel& voxel = m->voxels[high_end_index];
    voxel.need_update = false;
    end_voxels.push_back(high_end_index);
    if (static_cast<int>(point.intensity) > static_cast<int>(voxel.max_intensity))
      voxel.max_intensity = static_cast<int>(point.intensity);
    voxel.probability = (Probability)(update_prob(voxel.probability, true) * kTableSize);
    if (voxel.points.size() < (size_t)st.max_point_num_in_cell) voxel.points.push_back(point);
    for (size_t i = 0; i + 1 < ray.size(); ++i) {
      auto it = m->voxels.find(ray[i]);
      if (it != m->voxels.end() && it->second.need_update) {
        Probability& prob = it->second.probability;
        prob = (Probability)(update_prob(prob, false) * kTableSize);
      }
    }
  }
  for (const Key& k : end_voxels) m->voxels[k].need_update = true;
  return dropped;
}

extern "C" int64_t sm_oracle_mrvm_output(const sm_oracle_mrvm* m, float threshold, int32_t rgb, float* out4,
                                         int64_t capacity) {
  const sm_oracle_mrvm_settings& st = m->settings;
  const Probability prob_threshold = threshold * kTableSize;
  int64_t k = 0;
  auto emit = [&](float x, float y, float z, float v) {
    if (k < capacity) { out4[4 * k] = x; out4[4 * k + 1] = y; out4[4 * k + 2] = z; out4[4 * k + 3] = v; }
    ++k;
  };
  for (const auto& kv : m->sorted()) {
    const Voxel& voxel = *kv.second;
    if (voxel.probability < prob_threshold) continue;
    if (voxel.points.empty()) return -2;                  // CHECK(!points.empty())
    uint32_t intensity = voxel.max_intensity;             // the PointXYZRGB overload, :182-187
    intensity *= 1.4;
    if (intensity > 255) intensity = 255;
    const uint8_t grey = intensity;
    if (st.output_average) {
      float x = 0.f, y = 0.f, z = 0.f;                    // pcl::PointXYZI / PointXYZRGB default to zero
      for (const Point& p : voxel.points) { x += p.x; y += p.y; z += p.z; }
      const float size = voxel.points.size();
      x /= size; y /= size; z /= size;
      emit(x, y, z, rgb ? (float)grey : (st.use_max_intensity ? (float)static_cast<int>(voxel.max_intensity) : 0.f));
    } else {
      for (const Point& p : voxel.points)
        emit(p.x, p.y, p.z,
             rgb ? (float)grey : (st.use_max_intensity ? (float)static_cast<int>(voxel.max_intensity) : p.intensity));
    }
  }
  return k;
}

extern "C" int64_t sm_oracle_mrvm_state(const sm_oracle_mrvm* m, int64_t* keys, uint8_t* prob, int32_t* max_intensity,
                                        int32_t* npts, float* points4, int64_t capacity) {
  const size_t mp = (size_t)m->settings.max_point_num_in_cell;
  int64_t i = 0;
  for (const auto& kv : m->sorted()) {
    if (i < capacity) {
      const Voxel& v = *kv.second;
      keys[i] = (int64_t)kv.first;
      prob[i] = v.probability;
      max_intensity[i] = v.max_intensity;
      npts[i] = (int32_t)v.points.size();
      for (size_t q = 0; q < mp; ++q) {
        float* o = points4 + 4 * (i * mp + q);
        if (q < v.points.size()) { o[0] = v.points[q].x; o[1] = v.points[q].y; o[2] = v.points[q].z; o[3] = v.points[q].intensity; }
        else { o[0] = o[1] = o[2] = o[3] = 0.f; }
      }
    }
    ++i;
  }
  return i;
}

extern "C" int64_t sm_oracle_voxel_casting_bresenham(const float* start, const float* end, float step, int32_t* out3,
                                                     int64_t capacity) {
  Key a, b;
  for (int d = 0; d < 3; ++d)
    if (!std::isfinite(start[d]) || !std::isfinite(end[d])) return -1;
  if (!voxel_index(start[0], step, &a.x) || !voxel_index(start[1], step, &a.y) || !voxel_index(start[2], step, &a.z) ||
      !voxel_index(end[0], step, &b.x) || !voxel_index(end[1], step, &b.y) || !voxel_index(end[2], step, &b.z))
    return -1;
  std::vector<Key> ray;
  if (!VoxelCastingBresenham(a, b, &ray)) return -2;
  for (size_t i = 0; i < ray.size() && (int64_t)i < capacity; ++i) {
    out3[3 * i] = ray[i].x; out3[3 * i + 1] = ray[i].y; out3[3 * i + 2] = ray[i].z;
  }
  return (int64_t)ray.size();
}
