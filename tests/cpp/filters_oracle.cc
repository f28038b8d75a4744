// Serial restatement of pre_processers::filter::Factory and its nine filters (pre_processors/filter_*.cc), the parity
// checker of the sm_filter_chain_* entry points.  TEST INFRASTRUCTURE, compiled with g++ by tests/filters_oracle.py.
//
// One thread, the reference's loops in the reference's order, with the engine's documented deviations
// (include/sm_b200.h): RandomSampler draws from the counter hash, StatisticRemoval is the identity, non-finite points
// are not binned by GroundRemoval / GroundRemoval2, invalid stages are refused.  angle_mode selects the angle
// function: 0 = the host C library's atan2f (the literal reference), 1 = the engine's (restated below), so that
// the logic downstream of the angles can be compared bit for bit.
#include <math.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <cfloat>
#include <climits>
#include <limits>
#include <map>
#include <string>
#include <tuple>
#include <vector>

namespace {

struct Pt { float x, y, z, intensity, factor; };

// ---- the engine's angle function: (float) of atan2 in double from +, -, *, /, sqrt ----
double atan_unit(double t) {
  int halvings = 0;
  while (t > 0.19891236737965800691) { t = t / (1.0 + sqrt(1.0 + t * t)); ++halvings; }
  const double t2 = t * t;
  double s = 0.0;
  for (int k = 23; k >= 1; k -= 2) s = 1.0 / (double)k - t2 * s;
  double a = t * s;
  for (int h = 0; h < halvings; ++h) a = a + a;
  return a;
}
float engine_atan2f(float y, float x) {
  const double dy = y, dx = x, ax = fabs(dx), ay = fabs(dy);
  if (ax != ax || ay != ay) return (float)(dx + dy);
  if (ax == 0.0 && ay == 0.0) return 0.0f;
  if (std::isinf(ax) && std::isinf(ay)) return (float)(dx + dy - dx);
  const bool swap = ay > ax;
  double a = atan_unit(swap ? ax / ay : ay / ax);
  if (swap) a = M_PI / 2 - a;
  if (dx < 0.0) a = M_PI - a;
  if (dy < 0.0) a = -a;
  return (float)a;
}

int g_angle_mode = 1;
float angle(float y, float x) { return g_angle_mode == 0 ? std::atan2(y, x) : engine_atan2f(y, x); }

uint64_t mix64(uint64_t z) {
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}

// ---- filters: each maps (input cloud, input kept indices) -> output, or returns false (refused) ----
struct Cloud { std::vector<Pt> p; std::vector<int32_t> kept; };

struct Param { std::string name; bool is_int; float f; int32_t i; };
struct Stage {
  std::string name;
  std::vector<Param> params;
  float F(const char* n) const { for (auto& q : params) if (q.name == n) return q.f; abort(); }
  int32_t I(const char* n) const { for (auto& q : params) if (q.name == n) return q.i; abort(); }
};

void keep_if(const Cloud& in, const std::vector<char>& keep, Cloud* out) {
  out->p.clear(); out->kept.clear();
  for (size_t i = 0; i < in.p.size(); ++i)
    if (keep[i]) { out->p.push_back(in.p[i]); out->kept.push_back(in.kept[i]); }
}

bool range_filter(const Stage& S, const Cloud& in, Cloud* out) {
  const float min_range = S.F("min_range"), max_range = S.F("max_range");
  std::vector<char> keep(in.p.size());
  for (size_t i = 0; i < in.p.size(); ++i) {
    const Pt& q = in.p[i];
    const float range = std::sqrt(q.x * q.x + q.y * q.y + q.z * q.z);
    keep[i] = range >= min_range && range <= max_range;
  }
  keep_if(in, keep, out);
  return true;
}

bool axis_range(const Stage& S, const Cloud& in, Cloud* out) {
  const float mn = S.F("min"), mx = S.F("max");
  const int axis = S.I("axis_index");
  if (!(mx > mn && axis >= 0 && axis <= 2)) return false;
  if (mn == -std::numeric_limits<float>::max() && mx == std::numeric_limits<float>::max()) { *out = in; return true; }
  std::vector<char> keep(in.p.size(), 1);
  for (size_t i = 0; i < in.p.size(); ++i) {
    const float v = axis == 0 ? in.p[i].x : (axis == 1 ? in.p[i].y : in.p[i].z);
    if (v < mn || v > mx) keep[i] = 0;
  }
  keep_if(in, keep, out);
  return true;
}

bool bounding_box(const Stage& S, const Cloud& in, Cloud* out) {
  const double lo[3] = {S.F("min_x"), S.F("min_y"), S.F("min_z")}, hi[3] = {S.F("max_x"), S.F("max_y"), S.F("max_z")};
  if (!(lo[0] < hi[0] && lo[1] < hi[1] && lo[2] < hi[2])) return false;
  std::vector<char> keep(in.p.size());
  for (size_t i = 0; i < in.p.size(); ++i) {
    const double v[3] = {in.p[i].x, in.p[i].y, in.p[i].z};
    const bool inside = (v[0] >= lo[0] && v[0] <= hi[0]) && (v[1] >= lo[1] && v[1] <= hi[1]) &&
                        (v[2] >= lo[2] && v[2] <= hi[2]);
    keep[i] = !inside;
  }
  keep_if(in, keep, out);
  return true;
}

bool random_sampler(const Stage& S, int stage, uint64_t seed, uint64_t call, const Cloud& in, Cloud* out) {
  const float rate = S.F("sampling_rate");
  if (!(rate >= 0.f && rate <= 1.f)) return false;
  if (rate > 0.999) { *out = in; return true; }
  std::vector<char> keep(in.p.size());
  for (size_t i = 0; i < in.p.size(); ++i) {
    const uint64_t key = in.kept[i] >= 0 ? (uint64_t)in.kept[i] : ((1ull << 32) | (uint64_t)i);
    const uint64_t h = mix64(mix64(mix64(mix64(seed) ^ call) ^ (uint64_t)stage) ^ key);
    const double u = (double)(h >> 11) * (1.0 / 9007199254740992.0);
    keep[i] = u <= rate;
  }
  keep_if(in, keep, out);
  return true;
}

bool range_image(const Stage& S, const Cloud& in, Cloud* out) {
  const float top = S.F("top_angle"), btm = S.F("btm_angle");
  const float ox = S.F("offset_x"), oy = S.F("offset_y"), oz = S.F("offset_z");
  const int V = S.I("vertical_line_num"), H = S.I("horizontal_line_num");
  if (V <= 0 || H <= 0) return false;
  const float image_horizontal_res = M_PI * 2 / static_cast<float>(H);
  const float image_vertical_res = (top - btm) / static_cast<float>(V) / 180.f * M_PI;
  std::vector<char> taken((size_t)V * H, 0), keep(in.p.size(), 0);
  for (size_t i = 0; i < in.p.size(); ++i) {
    Pt q = in.p[i];
    q.x += ox; q.y += oy; q.z += oz;
    const float distance_in_xy = std::sqrt(q.x * q.x + q.y * q.y);
    if (distance_in_xy < 0.01f) continue;
    const float vertical_rad = angle(q.z, distance_in_xy);
    const double row_q = (vertical_rad - btm / 180.f * M_PI) / image_vertical_res;
    if (!(row_q > -1.0 && row_q < (double)V)) continue;       // int conversion: toward zero; NaN -> INT_MIN on x86
    const int row = (int)row_q;
    float horizontal_rad = angle(q.y, q.x);
    if (horizontal_rad < 0.f) horizontal_rad += M_PI * 2;
    const float col_q = horizontal_rad / image_horizontal_res;
    if (!(fabsf(col_q) < 1.0e9f)) continue;
    long col = std::lround(col_q);
    if (col >= H) col -= H;
    if (col < 0 || col >= H) continue;
    char& t = taken[(size_t)row * H + col];
    if (!t) { t = 1; keep[i] = 1; }
  }
  keep_if(in, keep, out);
  return true;
}

bool ground_removal(const Stage& S, const Cloud& in, Cloud* out) {
  const float leaf = S.F("leaf_size"), height_threshold = S.F("height_threshold");
  const int min_pts = S.I("min_point_num_in_voxel");
  if (leaf == 0.f || leaf != leaf) return false;
  std::map<std::tuple<int, int, int>, std::vector<int>> voxels;
  std::vector<int> not_finite;
  for (size_t i = 0; i < in.p.size(); ++i) {
    const Pt& q = in.p[i];
    if (!std::isfinite(q.x) || !std::isfinite(q.y) || !std::isfinite(q.z)) { not_finite.push_back((int)i); continue; }
    const float v[3] = {q.x / leaf, q.y / leaf, q.z / leaf};
    for (float f : v) if (!(f > -2147483649.0f && f < 2147483648.0f)) return false;
    voxels[std::make_tuple(static_cast<int>(v[0]), static_cast<int>(v[1]), static_cast<int>(v[2]))].push_back((int)i);
  }
  out->p.clear(); out->kept.clear();
  for (auto& kv : voxels) {
    const auto& vec = kv.second;
    if ((int32_t)vec.size() < min_pts) continue;
    bool is_ground = false;
    if (std::get<2>(kv.first) <= 0) {
      float max_z = -1.e9, min_z = 1.e9;
      for (int i : vec) { if (in.p[i].z > max_z) max_z = in.p[i].z; if (in.p[i].z < min_z) min_z = in.p[i].z; }
      const float delta = max_z - min_z;
      if (delta >= 0. && delta <= height_threshold) is_ground = true;
    }
    if (!is_ground)
      for (int i : vec) { out->p.push_back(in.p[i]); out->kept.push_back(in.kept[i]); }
  }
  for (int i : not_finite) { out->p.push_back(in.p[i]); out->kept.push_back(in.kept[i]); }
  return true;
}

// ---- GroundRemoval2 ----
struct P2 { float d, z; };
struct Line { P2 start, end; };
struct LocalLine { float m = 0.f, b = 0.f; };

// least squares [d 1] [m b]^T = z: Householder QR with column pivoting, two columns, in double
LocalLine fit_local_line(const std::vector<P2>& pts) {
  const size_t k = pts.size();
  std::vector<double> A0(k), A1(k, 1.0), y(k);
  for (size_t i = 0; i < k; ++i) { A0[i] = pts[i].d; y[i] = pts[i].z; }
  double n0 = 0.0, n1 = 0.0;
  for (size_t i = 0; i < k; ++i) { n0 += A0[i] * A0[i]; n1 += 1.0; }
  const int piv = n1 > n0 ? 1 : 0;
  std::vector<double>& a = piv == 0 ? A0 : A1;        // pivot column
  std::vector<double>& w = piv == 0 ? A1 : A0;        // the other
  // reflection 1: H = I - tau v v^T, v = (1, a[1:] / (a0 - beta))
  auto reflect = [&](std::vector<double>& col, size_t r0, std::vector<std::vector<double>*> others) {
    double tail = 0.0;
    for (size_t i = r0 + 1; i < k; ++i) tail += col[i] * col[i];
    const double c0 = r0 < k ? col[r0] : 0.0;
    if (tail == 0.0) return c0;
    double beta = std::sqrt(c0 * c0 + tail);
    if (c0 >= 0.0) beta = -beta;
    const double den = c0 - beta, tau = (beta - c0) / beta;
    std::vector<double> v(k, 0.0);
    for (size_t i = r0 + 1; i < k; ++i) v[i] = col[i] / den;
    for (auto* o : others) {
      double s = (*o)[r0];
      for (size_t i = r0 + 1; i < k; ++i) s += v[i] * (*o)[i];
      (*o)[r0] = (*o)[r0] - tau * s;
      for (size_t i = r0 + 1; i < k; ++i) (*o)[i] = (*o)[i] - tau * s * v[i];
    }
    return beta;
  };
  const double r00 = reflect(a, 0, {&w, &y});
  const double r01 = w[0];
  const double r11 = reflect(w, 1, {&y});
  const double z1 = std::fabs(r11) > 4.4408920985006262e-16 * std::fabs(r00) ? y[1] / r11 : 0.0;
  const double z0 = r00 != 0.0 ? (y[0] - r01 * z1) / r00 : 0.0;
  LocalLine L;
  L.m = (float)(piv == 0 ? z0 : z1);
  L.b = (float)(piv == 0 ? z1 : z0);
  return L;
}

float get_max_error(const std::vector<P2>& pts, const LocalLine& line) {
  float max_error = 0.;
  for (auto& q : pts) {
    const float error = std::fabs(line.m * q.d + line.b - q.z);
    if (error > max_error) max_error = error;
  }
  return max_error;
}

Line local_line_to_line(const LocalLine& l, const std::vector<P2>& pts) {
  Line line;
  const float start_d = pts.front().d, end_d = pts.back().d;
  line.start = {start_d, l.m * start_d + l.b};
  line.end = {end_d, l.m * end_d + l.b};
  return line;
}

struct Gr2 {
  float r_max, r_min, start_ground_height, long_line_threshold, max_long_line_height, max_start_height, max_error,
      max_slope, max_b, max_dist_to_line, search_angle;
  int bin_num, segment_num;
};
struct Cell { P2 min_z_point{1.e6f, 1.e6f}; std::vector<std::pair<int, P2>> points; };

std::vector<Line> fit_lines(const Gr2& G, const std::vector<Cell>& cells, int s) {
  std::vector<Line> segment;
  auto cell = [&](int b) -> const Cell& { return cells[(size_t)s * G.bin_num + b]; };
  int start_index = 0;
  for (start_index = 0; start_index < G.bin_num; ++start_index)
    if (!cell(start_index).points.empty()) break;
  if (start_index >= G.bin_num - 1) return segment;
  std::vector<P2> cur_pts;
  cur_pts.push_back(cell(start_index).min_z_point);
  LocalLine current_line;
  bool is_long_line = false;
  float ground_height = G.start_ground_height;
  for (int i = start_index + 1; i < G.bin_num; ++i) {
    const Cell& c = cell(i);
    if (c.points.empty()) continue;
    const P2 current_point = c.min_z_point;
    if (current_point.d - cur_pts.back().d >= G.long_line_threshold) is_long_line = true;
    float expected_z = std::numeric_limits<float>::max();
    if (is_long_line && cur_pts.size() > 2) expected_z = current_line.m * current_point.d + current_line.b;
    if (cur_pts.size() >= 2) {
      cur_pts.push_back(current_point);
      current_line = fit_local_line(cur_pts);
      const float error = get_max_error(cur_pts, current_line);
      if (error > G.max_error || std::fabs(current_line.m) > G.max_slope ||
          (is_long_line && std::fabs(expected_z - current_point.z) > G.max_long_line_height)) {
        cur_pts.pop_back();
        if (cur_pts.size() >= 3) {
          const LocalLine new_line = fit_local_line(cur_pts);
          segment.push_back(local_line_to_line(new_line, cur_pts));
          ground_height = new_line.m * cur_pts.back().d + new_line.b;
        }
        is_long_line = false;
        cur_pts.erase(cur_pts.begin(), --cur_pts.end());
        --i;
      }
    } else {
      if (!is_long_line && std::fabs(cur_pts.back().z - ground_height) < G.max_start_height) {
        cur_pts.push_back(current_point);
      } else {
        cur_pts.clear();
        cur_pts.push_back(current_point);
      }
    }
  }
  if (cur_pts.size() > 2) segment.push_back(local_line_to_line(fit_local_line(cur_pts), cur_pts));
  return segment;
}

float vertical_distance(const P2& q, const std::vector<Line>& seg) {
  const float margin = 0.1;
  float distance = -1.;
  for (auto& line : seg) {
    if (line.start.d - margin < q.d && line.end.d + margin > q.d) {
      const float delta_z = line.end.z - line.start.z, delta_d = line.end.d - line.start.d;
      const float expected_z = (q.d - line.start.d) / delta_d * delta_z + line.start.z;
      distance = std::fabs(q.z - expected_z);
    }
  }
  return distance;
}

Gr2 gr2_of(const Stage& S) {
  return Gr2{S.F("r_max"), S.F("r_min"), S.F("start_ground_height"), S.F("long_line_threshold"),
             S.F("max_long_line_height"), S.F("max_start_height"), S.F("max_error"), S.F("max_slope"), S.F("max_b"),
             S.F("max_dist_to_line"), S.F("search_angle"), S.I("bin_num"), S.I("segment_num")};
}

// cells of SetInputCloud (:127-210); the binning with clamped indices
std::vector<Cell> gr2_cells(const Gr2& G, const Cloud& in) {
  std::vector<Cell> grids((size_t)G.bin_num * G.segment_num);
  const float double_pi = M_PI * 2;
  const float delta_alpha = double_pi / G.segment_num;
  const float delta_bin = (G.r_max - G.r_min) / G.bin_num;
  for (size_t i = 0; i < in.p.size(); ++i) {
    const Pt& q = in.p[i];
    if (!std::isfinite(q.x) || !std::isfinite(q.y) || !std::isfinite(q.z)) continue;
    const float range = std::sqrt(q.x * q.x + q.y * q.y);
    float rad = angle(q.y, q.x);
    if (rad < 0.) rad += double_pi;
    const float sq = rad / delta_alpha, bq = (range - G.r_min) / delta_bin;
    int32_t s_index = sq >= (float)G.segment_num ? G.segment_num : (sq <= -1.f ? -1 : (int32_t)sq);
    int32_t b_index = bq >= (float)G.bin_num ? G.bin_num : (bq <= -1.f ? -1 : (int32_t)bq);
    if (b_index >= G.bin_num) b_index = G.bin_num - 1; else if (b_index < 0) b_index = 0;
    if (s_index >= G.segment_num) s_index = G.segment_num - 1; else if (s_index < 0) s_index = 0;
    Cell& grid = grids[(size_t)s_index * G.bin_num + b_index];
    const P2 pt{range, q.z};
    if (grid.points.empty() || pt.z < grid.min_z_point.z) grid.min_z_point = pt;
    if (pt.z <= grid.min_z_point.z + 0.5) grid.points.push_back(std::make_pair((int)i, pt));
  }
  return grids;
}

bool ground_removal2(const Stage& S, const Cloud& in, Cloud* out) {
  const Gr2 G = gr2_of(S);
  if (G.bin_num <= 0 || G.segment_num <= 0) return false;
  const float delta_alpha = M_PI * 2 / G.segment_num;
  const double q = G.search_angle / 180. * M_PI / delta_alpha;
  if (!(q > -1.0 && q < (double)G.segment_num)) return false;
  const int search_max_step = (int)q;
  const std::vector<Cell> grids = gr2_cells(G, in);
  std::vector<std::vector<Line>> segments(G.segment_num);
  for (int s = 0; s < G.segment_num; ++s) segments[s] = fit_lines(G, grids, s);
  std::vector<int> cand;
  for (int i = search_max_step; i > 0; --i) { cand.push_back(i); cand.push_back(-i); }
  std::vector<char> is_outlier(in.p.size(), 0);
  for (int s = 0; s < G.segment_num; ++s)
    for (int b = 0; b < G.bin_num; ++b)
      for (auto& ip : grids[(size_t)s * G.bin_num + b].points) {
        float distance = vertical_distance(ip.second, segments[s]);
        if (distance < 0.) {
          for (int i : cand) {
            int cs = s + i;
            if (cs < 0) cs += G.segment_num; else if (cs >= G.segment_num) cs -= G.segment_num;
            distance = vertical_distance(ip.second, segments[cs]);
            if (distance > 0.) break;
          }
        }
        if (distance > 0. && distance <= G.max_dist_to_line) is_outlier[ip.first] = 1;
      }
  std::vector<char> keep(in.p.size());
  for (size_t i = 0; i < in.p.size(); ++i) keep[i] = !is_outlier[i];
  keep_if(in, keep, out);
  return true;
}

bool voxel_grid(const Stage& S, const Cloud& in, Cloud* out) {
  const float voxel_size = S.F("voxel_size");
  if (!(voxel_size > 1.e-6)) return false;
  struct Acc { double x = 0, y = 0, z = 0, i = 0; int n = 0; };
  std::map<std::tuple<long, long, long>, Acc> voxels;
  for (const Pt& q : in.p) {
    const float v[3] = {q.x / voxel_size, q.y / voxel_size, q.z / voxel_size};
    if (!(fabsf(v[0]) < 9.0e18f && fabsf(v[1]) < 9.0e18f && fabsf(v[2]) < 9.0e18f)) continue;
    Acc& a = voxels[std::make_tuple(std::lround(v[0]), std::lround(v[1]), std::lround(v[2]))];
    a.x += q.x; a.y += q.y; a.z += q.z; a.i += q.intensity; ++a.n;
  }
  out->p.clear(); out->kept.clear();
  for (auto& kv : voxels) {
    const Acc& a = kv.second;
    out->p.push_back(Pt{(float)(a.x / a.n), (float)(a.y / a.n), (float)(a.z / a.n), (float)(a.i / a.n), 0.f});
    out->kept.push_back(-1);
  }
  return true;
}

struct Def { const char* filter; const char* name; bool is_int; double init; };
const Def kDefs[] = {
    {"Range", "min_range", false, 0.0}, {"Range", "max_range", false, FLT_MAX},
    {"AxisRange", "min", false, -FLT_MAX}, {"AxisRange", "max", false, FLT_MAX}, {"AxisRange", "axis_index", true, 2},
    {"BoundingBoxRemoval", "min_x", false, -FLT_MAX}, {"BoundingBoxRemoval", "min_y", false, -FLT_MAX},
    {"BoundingBoxRemoval", "min_z", false, -FLT_MAX}, {"BoundingBoxRemoval", "max_x", false, FLT_MAX},
    {"BoundingBoxRemoval", "max_y", false, FLT_MAX}, {"BoundingBoxRemoval", "max_z", false, FLT_MAX},
    {"RandomSampler", "sampling_rate", false, 1.0},
    {"StatisticRemoval", "std_mul", false, 1.0}, {"StatisticRemoval", "point_num_meank", true, 30},
    {"RangeImage", "top_angle", false, 30.}, {"RangeImage", "btm_angle", false, -15.},
    {"RangeImage", "offset_x", false, 0.}, {"RangeImage", "offset_y", false, 0.}, {"RangeImage", "offset_z", false, 0.},
    {"RangeImage", "vertical_line_num", true, 40}, {"RangeImage", "horizontal_line_num", true, 1800},
    {"GroundRemoval", "leaf_size", false, 0.8}, {"GroundRemoval", "height_threshold", false, 0.15},
    {"GroundRemoval", "min_point_num_in_voxel", true, 10},
    {"GroundRemoval2", "r_max", false, 100.}, {"GroundRemoval2", "r_min", false, 1.},
    {"GroundRemoval2", "start_ground_height", false, -0.25}, {"GroundRemoval2", "long_line_threshold", false, 1.0},
    {"GroundRemoval2", "max_long_line_height", false, 0.1}, {"GroundRemoval2", "max_start_height", false, 0.2},
    {"GroundRemoval2", "max_error", false, 0.05}, {"GroundRemoval2", "max_slope", false, std::tan(M_PI / 12.)},
    {"GroundRemoval2", "max_b", false, 0.1}, {"GroundRemoval2", "max_dist_to_line", false, 0.05},
    {"GroundRemoval2", "search_angle", false, 10.}, {"GroundRemoval2", "bin_num", true, 200},
    {"GroundRemoval2", "segment_num", true, 180}, {"GroundRemoval2", "thread_num", true, 4},
    {"VoxelGrid", "voxel_size", false, 0.1},
};

struct Chain { std::vector<Stage> stages; std::vector<int64_t> counts; uint64_t seed = 0, call = 0; };

bool valid(const Stage& S) {
  if (S.name == "AxisRange") return S.F("max") > S.F("min") && S.I("axis_index") >= 0 && S.I("axis_index") <= 2;
  if (S.name == "BoundingBoxRemoval")
    return S.F("min_x") < S.F("max_x") && S.F("min_y") < S.F("max_y") && S.F("min_z") < S.F("max_z");
  if (S.name == "RandomSampler") return S.F("sampling_rate") >= 0.f && S.F("sampling_rate") <= 1.f;
  if (S.name == "VoxelGrid") return S.F("voxel_size") > 1.e-6;
  return true;
}

}  // namespace

extern "C" {

void* sm_oracle_filter_chain_create() { return new Chain; }
void sm_oracle_filter_chain_destroy(void* h) { delete (Chain*)h; }
void sm_oracle_filter_set_angle_mode(int mode) { g_angle_mode = mode; }

int sm_oracle_filter_chain_add(void* h, const char* name) {
  Stage S;
  S.name = name;
  for (const Def& d : kDefs)
    if (S.name == d.filter) S.params.push_back(Param{d.name, d.is_int, d.is_int ? 0.f : (float)d.init, (int32_t)d.init});
  if (S.params.empty()) return -11;
  Chain* c = (Chain*)h;
  c->stages.push_back(S);
  return (int)c->stages.size() - 1;
}

int sm_oracle_filter_chain_set_param(void* h, int stage, const char* name, int type, const char* text) {
  Chain* c = (Chain*)h;
  if (stage < 0 || stage >= (int)c->stages.size()) return -1;
  for (Param& q : c->stages[stage].params) {
    if (q.name != name) continue;
    if (type == 0) {
      const char* t = text;
      while (*t == ' ' || *t == '\t' || *t == '\n' || *t == '\r') ++t;
      const bool neg = *t == '-';
      if (*t == '-' || *t == '+') ++t;
      const long long a = strtoll(t, nullptr, (t[0] == '0' && (t[1] == 'x' || t[1] == 'X')) ? 16 : 10);
      const long long v = neg ? -a : a;
      const int32_t iv = (int32_t)(v > INT_MAX ? INT_MAX : (v < INT_MIN ? INT_MIN : v));
      if (q.is_int) q.i = iv; else q.f = (float)iv;
    } else if (type == 1) {
      const float v = (float)strtod(text, nullptr);
      if (q.is_int) q.i = (int32_t)v; else q.f = v;
    } else {
      return -1;
    }
    return 0;
  }
  return -10;
}

int sm_oracle_filter_chain_valid(void* h, int stage) {
  Chain* c = (Chain*)h;
  if (stage < 0 || stage >= (int)c->stages.size()) return -1;
  return valid(c->stages[stage]) ? 1 : 0;
}

void sm_oracle_filter_chain_set_seed(void* h, uint64_t seed) { ((Chain*)h)->seed = seed; ((Chain*)h)->call = 0; }

// points: n InnerPointType records; out / kept: capacity n.  Returns the output count, or -1 (a refused stage)
int64_t sm_oracle_filter_chain_filter(void* h, const float* points, int64_t n, float* out, int32_t* kept) {
  Chain* c = (Chain*)h;
  const uint64_t call = c->call++;
  c->counts.assign(c->stages.size(), 0);
  for (const Stage& S : c->stages) if (!valid(S)) return -1;
  Cloud cur, next;
  for (int64_t i = 0; i < n; ++i) {
    const float* p = points + 5 * i;
    cur.p.push_back(Pt{p[0], p[1], p[2], p[3], p[4]});
    cur.kept.push_back((int32_t)i);
  }
  for (size_t k = 0; k < c->stages.size(); ++k) {
    const Stage& S = c->stages[k];
    bool ok = true;
    if (cur.p.empty()) { next = cur; }
    else if (S.name == "Range") ok = range_filter(S, cur, &next);
    else if (S.name == "AxisRange") ok = axis_range(S, cur, &next);
    else if (S.name == "BoundingBoxRemoval") ok = bounding_box(S, cur, &next);
    else if (S.name == "RandomSampler") ok = random_sampler(S, (int)k, c->seed, call, cur, &next);
    else if (S.name == "RangeImage") ok = range_image(S, cur, &next);
    else if (S.name == "GroundRemoval") ok = ground_removal(S, cur, &next);
    else if (S.name == "GroundRemoval2") ok = ground_removal2(S, cur, &next);
    else if (S.name == "VoxelGrid") ok = voxel_grid(S, cur, &next);
    else next = cur;                                               // StatisticRemoval
    if (!ok) return -1;
    cur.p.swap(next.p); cur.kept.swap(next.kept);
    c->counts[k] = (int64_t)cur.p.size();
  }
  for (size_t i = 0; i < cur.p.size(); ++i) {
    const Pt& q = cur.p[i];
    float* o = out + 5 * i;
    o[0] = q.x; o[1] = q.y; o[2] = q.z; o[3] = q.intensity; o[4] = q.factor;
    kept[i] = cur.kept[i];
  }
  return (int64_t)cur.p.size();
}

int sm_oracle_filter_chain_stage_counts(void* h, int64_t* counts, int n) {
  Chain* c = (Chain*)h;
  for (int k = 0; k < n && k < (int)c->counts.size(); ++k) counts[k] = c->counts[k];
  return (int)c->stages.size();
}

// GroundRemoval2 pieces for the model tests: per point its cell (-1 not binned) and membership; per cell its
// min_z_point and whether `points` is non-empty; per segment its lines (lines4 capacity: cells / 2 + 2 per segment)
int sm_oracle_gr2_state(const float* points, int64_t n, const float* params, int32_t* cell, uint8_t* member,
                        float* cell_dz, uint8_t* cell_used, float* lines4, int32_t* nlines) {
  Stage S;
  S.name = "GroundRemoval2";
  for (const Def& d : kDefs)
    if (S.name == d.filter) S.params.push_back(Param{d.name, d.is_int, (float)d.init, (int32_t)d.init});
  const char* names[] = {"r_max", "r_min", "start_ground_height", "long_line_threshold", "max_long_line_height",
                         "max_start_height", "max_error", "max_slope", "max_b", "max_dist_to_line", "search_angle"};
  for (int k = 0; k < 11; ++k) for (Param& q : S.params) if (q.name == names[k]) q.f = params[k];
  for (Param& q : S.params) { if (q.name == "bin_num") q.i = (int)params[11]; if (q.name == "segment_num") q.i = (int)params[12]; }
  const Gr2 G = gr2_of(S);
  Cloud in;
  for (int64_t i = 0; i < n; ++i) { const float* p = points + 5 * i; in.p.push_back(Pt{p[0], p[1], p[2], p[3], p[4]}); in.kept.push_back((int32_t)i); }
  const std::vector<Cell> grids = gr2_cells(G, in);
  for (int64_t i = 0; i < n; ++i) { cell[i] = -1; member[i] = 0; }
  for (size_t c = 0; c < grids.size(); ++c) {
    cell_dz[2 * c] = grids[c].min_z_point.d; cell_dz[2 * c + 1] = grids[c].min_z_point.z;
    cell_used[c] = !grids[c].points.empty();
    for (auto& ip : grids[c].points) member[ip.first] = 1;
  }
  // cell of every binned point (members or not): recompute the index
  const float double_pi = M_PI * 2, delta_alpha = double_pi / G.segment_num, delta_bin = (G.r_max - G.r_min) / G.bin_num;
  for (int64_t i = 0; i < n; ++i) {
    const Pt& q = in.p[i];
    if (!std::isfinite(q.x) || !std::isfinite(q.y) || !std::isfinite(q.z)) continue;
    const float range = std::sqrt(q.x * q.x + q.y * q.y);
    float rad = angle(q.y, q.x);
    if (rad < 0.) rad += double_pi;
    const float sq = rad / delta_alpha, bq = (range - G.r_min) / delta_bin;
    int s = sq >= (float)G.segment_num ? G.segment_num - 1 : (sq <= -1.f ? 0 : (int)sq);
    int b = bq >= (float)G.bin_num ? G.bin_num - 1 : (bq <= -1.f ? 0 : (int)bq);
    s = s < 0 ? 0 : s; b = b < 0 ? 0 : b;
    cell[i] = s * G.bin_num + b;
  }
  const int cap = G.bin_num / 2 + 2;
  for (int s = 0; s < G.segment_num; ++s) {
    const std::vector<Line> L = fit_lines(G, grids, s);
    nlines[s] = (int32_t)L.size();
    for (size_t l = 0; l < L.size() && (int)l < cap; ++l) {
      float* o = lines4 + 4 * ((size_t)s * cap + l);
      o[0] = L[l].start.d; o[1] = L[l].start.z; o[2] = L[l].end.d; o[3] = L[l].end.z;
    }
  }
  return 0;
}

}  // extern "C"
