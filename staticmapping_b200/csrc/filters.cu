// pre_processers::filter::Factory and its nine filters (pre_processors/filter_*.cc) on the device: the chain every
// lidar scan goes through before motion compensation, Align and the static map.  Semantics and deviations:
// include/sm_b200.h (sm_filter_chain_*); formulation: DESIGN.md section 4i.
//
// The chain state is a cloud of 20-byte InnerPointType records plus, per record, its chain-input index (-1 behind
// a VoxelGrid).  Every stage writes a keep flag per record and one stable compaction (exclusive scan + scatter)
// moves the kept records into the other ping-pong buffer:
//   - a maximal run of point-wise stages (Range, AxisRange, BoundingBoxRemoval, RandomSampler, StatisticRemoval) is
//     one predicate kernel;
//   - RangeImage: atomicMin of the point's position on its pixel, then a point is kept iff it owns its pixel (the
//     first point in input order, like the reference's serial loop);
//   - GroundRemoval: 63-bit voxel keys, stable radix sort, per voxel count / min z / max z (order independent), and
//     the kept points gathered in sorted order (== std::map<Vector3i> order, input order inside a voxel);
//   - GroundRemoval2: cell keys, stable radix sort, one thread per cell walks its points in input order (running
//     minimum of z -> cell membership, first strict minimum), one thread per angular segment runs FitLines serially
//     (the line fit is a two-column Householder QR with column pivoting in double), one thread per point runs
//     ClusterGround;
//   - VoxelGrid: the kernels of voxel_filter.cu.
// Compiled with -fmad=false: every float expression rounds like the reference's.
#include <float.h>
#include <limits.h>
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <string>
#include <vector>

#include "../../include/sm_b200.h"
#include "../../include/sm_b200_debug.h"
#include "common.cuh"
#include "kernels.h"

namespace smb {

// ---- per-point functions shared by the kernels and the host test hooks ------------------------------------------
namespace {

constexpr double kPi = 3.14159265358979323846;   // M_PI

// The angle function of the product: atan2 in double from +, -, *, / and sqrt only (each correctly rounded under
// IEEE 754, no contraction), rounded once to float.  So the host build and the device build give the same bits on
// every machine.  libm's atan2f differs between C libraries (and CUDA's is a 2-ulp approximation); see the header.
__host__ __device__ __forceinline__ double atan_unit(double t) {     // atan(t) for 0 <= t <= 1
  int halvings = 0;
  while (t > 0.19891236737965800691) {                                // tan(pi / 16)
    t = t / (1.0 + sqrt(1.0 + t * t));                                  // atan(t) = 2 atan(t / (1 + sqrt(1 + t^2)))
    ++halvings;
  }
  const double t2 = t * t;
  double s = 0.0;
  for (int k = 23; k >= 1; k -= 2) s = 1.0 / (double)k - t2 * s;      // 1 - t^2/3 + t^4/5 - ... (Horner)
  double a = t * s;
  for (int h = 0; h < halvings; ++h) a = a + a;
  return a;
}

__host__ __device__ __forceinline__ float sm_atan2f(float y, float x) {
  const double dy = (double)y, dx = (double)x;
  const double ax = fabs(dx), ay = fabs(dy);
  if (ax != ax || ay != ay) return (float)(dx + dy);                  // NaN in, NaN out
  if (ax == 0.0 && ay == 0.0) return 0.0f;
  if (isinf(ax) && isinf(ay)) return (float)(dx + dy - dx);           // NaN: no angle
  const bool swap = ay > ax;
  double a = atan_unit(swap ? ax / ay : ay / ax);
  if (swap) a = kPi / 2 - a;
  if (dx < 0.0) a = kPi - a;
  if (dy < 0.0) a = -a;
  return (float)a;
}

// RangeImage::Filter (filter_range_image.cc:89-126): pixel of one point, -1 for an outlier
struct RiParams { float top, btm, ox, oy, oz; int V, H; };
__host__ __device__ __forceinline__ int64_t ri_pixel(const float* p, const RiParams& P) {
  const float image_horizontal_res = kPi * 2 / static_cast<float>(P.H);
  const float image_vertical_res = (P.top - P.btm) / static_cast<float>(P.V) / 180.f * kPi;
  const float x = p[0] + P.ox, y = p[1] + P.oy, z = p[2] + P.oz;
  const float distance_in_xy = sqrtf(x * x + y * y);
  if (distance_in_xy < 0.01f) return -1;
  const float vertical_rad = sm_atan2f(z, distance_in_xy);
  const double row_q = (vertical_rad - P.btm / 180.f * kPi) / image_vertical_res;
  // (int) truncates toward zero: a quotient in (-1, 0) is row 0; NaN (x86 gives INT_MIN) is an outlier
  if (!(row_q > -1.0 && row_q < (double)P.V)) return -1;
  const int row = (int)row_q;
  float horizontal_rad = sm_atan2f(y, x);
  if (horizontal_rad < 0.f) horizontal_rad += kPi * 2;
  const float col_q = horizontal_rad / image_horizontal_res;
  if (!(fabsf(col_q) < 1.0e9f)) return -1;
  long col = lroundf(col_q);
  if (col >= P.H) col -= P.H;
  if (col < 0 || col >= P.H) return -1;
  return (int64_t)row * P.H + col;
}

// GroundRemoval2::SetInputCloud (filter_ground_removal2.cc:144-192): cell of one point, -1 when it is not binned
struct Gr2Params {
  float r_max, r_min, start_ground_height, long_line_threshold, max_long_line_height, max_start_height, max_error,
      max_slope, max_b, max_dist_to_line, search_angle;
  int bin_num, segment_num;
};
__host__ __device__ __forceinline__ int64_t gr2_cell(const float* p, const Gr2Params& P, float* range_out) {
  if (!isfinite(p[0]) || !isfinite(p[1]) || !isfinite(p[2])) return -1;
  const float double_pi = kPi * 2;
  const float delta_alpha = double_pi / P.segment_num;
  const float delta_bin = (P.r_max - P.r_min) / P.bin_num;
  const float range = sqrtf(p[0] * p[0] + p[1] * p[1]);
  // `range < r_min_ && range > r_max_` is never true: every point is binned
  float rad = sm_atan2f(p[1], p[0]);
  if (rad < 0.) rad += double_pi;
  const float sq = rad / delta_alpha, bq = (range - P.r_min) / delta_bin;
  // int32_t index = quotient, then clamped; the clamp is applied to the quotient first so that no float outside
  // the int range is converted
  const int s = !(sq < (float)P.segment_num) ? P.segment_num - 1 : (sq <= -1.f ? 0 : (int)sq);
  const int b = !(bq < (float)P.bin_num) ? P.bin_num - 1 : (bq <= -1.f ? 0 : (int)bq);
  *range_out = range;
  return (int64_t)s * P.bin_num + b;
}

// FitLocalLine (:29-44): least squares z = m d + b by a two-column Householder QR with column pivoting, in double,
// computed on the fly from the points (no scratch).  Columns: 0 = d, 1 = 1.
__host__ __device__ __forceinline__ void gr2_fit(const float2* pts, int k, float* m_out, float* b_out) {
  double n0 = 0.0, n1 = 0.0;
  for (int i = 0; i < k; ++i) { const double d = pts[i].x; n0 += d * d; n1 += 1.0; }
  const int piv = n1 > n0 ? 1 : 0;                                    // ties: the first column
  auto col = [&](int c, int i) -> double { return c == 0 ? (double)pts[i].x : 1.0; };
  // first reflection, on the pivot column
  double tail = 0.0;
  for (int i = 1; i < k; ++i) { const double v = col(piv, i); tail += v * v; }
  const double c0 = col(piv, 0);
  double beta1 = c0, tau1 = 0.0, den1 = 1.0;
  if (tail != 0.0) {
    beta1 = sqrt(c0 * c0 + tail);
    if (c0 >= 0.0) beta1 = -beta1;
    den1 = c0 - beta1;
    tau1 = (beta1 - c0) / beta1;
  }
  auto v1 = [&](int i) -> double { return tail != 0.0 ? col(piv, i) / den1 : 0.0; };   // i >= 1
  double sw = col(1 - piv, 0), sy = (double)pts[0].y;
  for (int i = 1; i < k; ++i) { sw += v1(i) * col(1 - piv, i); sy += v1(i) * (double)pts[i].y; }
  auto w1 = [&](int i) -> double { return i == 0 ? col(1 - piv, 0) - tau1 * sw : col(1 - piv, i) - tau1 * sw * v1(i); };
  auto y1 = [&](int i) -> double { return i == 0 ? (double)pts[0].y - tau1 * sy : (double)pts[i].y - tau1 * sy * v1(i); };
  // second reflection, on rows 1.. of the other column
  double tail2 = 0.0;
  for (int i = 2; i < k; ++i) { const double v = w1(i); tail2 += v * v; }
  const double c1 = k > 1 ? w1(1) : 0.0;
  double beta2 = c1, tau2 = 0.0, den2 = 1.0;
  if (tail2 != 0.0) {
    beta2 = sqrt(c1 * c1 + tail2);
    if (c1 >= 0.0) beta2 = -beta2;
    den2 = c1 - beta2;
    tau2 = (beta2 - c1) / beta2;
  }
  double sy2 = k > 1 ? y1(1) : 0.0;
  if (tail2 != 0.0)
    for (int i = 2; i < k; ++i) sy2 += (w1(i) / den2) * y1(i);
  const double qy1 = (k > 1 ? y1(1) : 0.0) - tau2 * sy2, qy0 = y1(0);
  const double r00 = beta1, r01 = w1(0), r11 = beta2;
  // rank: a pivot counts when |r_ii| > 2 eps |r_00| (Eigen's default threshold); the other unknown is 0
  const double z1 = fabs(r11) > 4.4408920985006262e-16 * fabs(r00) ? qy1 / r11 : 0.0;
  const double z0 = r00 != 0.0 ? (qy0 - r01 * z1) / r00 : 0.0;
  *m_out = (float)(piv == 0 ? z0 : z1);
  *b_out = (float)(piv == 0 ? z1 : z0);
}

__host__ __device__ __forceinline__ float gr2_max_error(const float2* pts, int k, float m, float b) {
  float max_error = 0.f;
  for (int i = 0; i < k; ++i) {
    const float error = fabsf(m * pts[i].x + b - pts[i].y);
    if (error > max_error) max_error = error;
  }
  return max_error;
}

struct Line { float sd, sz, ed, ez; };

__host__ __device__ __forceinline__ Line gr2_line(const float2* pts, int k, float m, float b) {
  const float start_d = pts[0].x, end_d = pts[k - 1].x;
  return Line{start_d, m * start_d + b, end_d, m * end_d + b};
}

// GroundRemoval2::FitLines (:240-316) of one segment.  cell_d / cell_z / cell_used: the segment's bin_num cells
// (min_z_point, points non-empty); pts: bin_num scratch points; lines: room for cap lines.  Returns the number of
// lines (more than cap: only the first cap were written).
__host__ __device__ __forceinline__ int gr2_fit_lines(const float* cell_d, const float* cell_z,
                                                      const uint8_t* cell_used, const Gr2Params& P, float2* pts,
                                                      Line* lines, int cap) {
  int nl = 0;
  int start_index = 0;
  for (start_index = 0; start_index < P.bin_num; ++start_index)
    if (cell_used[start_index]) break;
  if (start_index >= P.bin_num - 1) return 0;
  int k = 0;
  pts[k++] = make_float2(cell_d[start_index], cell_z[start_index]);
  float cm = 0.f, cb = 0.f;                                           // current_line
  bool is_long_line = false;
  float ground_height = P.start_ground_height;
  for (int i = start_index + 1; i < P.bin_num; ++i) {
    if (!cell_used[i]) continue;
    const float2 cur = make_float2(cell_d[i], cell_z[i]);
    if (cur.x - pts[k - 1].x >= P.long_line_threshold) is_long_line = true;
    float expected_z = FLT_MAX;
    if (is_long_line && k > 2) expected_z = cm * cur.x + cb;        // the previous fit
    if (k >= 2) {
      pts[k++] = cur;
      gr2_fit(pts, k, &cm, &cb);
      const float error = gr2_max_error(pts, k, cm, cb);
      if (error > P.max_error || fabsf(cm) > P.max_slope ||
          (is_long_line && fabsf(expected_z - cur.y) > P.max_long_line_height)) {
        --k;
        if (k >= 3) {
          float nm, nb;
          gr2_fit(pts, k, &nm, &nb);
          if (nl < cap) lines[nl] = gr2_line(pts, k, nm, nb);
          ++nl;
          ground_height = nm * pts[k - 1].x + nb;
        }
        is_long_line = false;
        pts[0] = pts[k - 1];                                          // erase all but the last point
        k = 1;
        --i;
      }
    } else {
      if (!is_long_line && fabsf(pts[k - 1].y - ground_height) < P.max_start_height) {
        pts[k++] = cur;
      } else {
        k = 0;
        pts[k++] = cur;
      }
    }
  }
  if (k > 2) {
    float nm, nb;
    gr2_fit(pts, k, &nm, &nb);
    if (nl < cap) lines[nl] = gr2_line(pts, k, nm, nb);
    ++nl;
  }
  return nl;
}

// VerticalDistanceToSegment (:398-414): the last line that covers d (margin 0.1) decides; -1 if none
__host__ __device__ __forceinline__ float gr2_vertical_distance(float d, float z, const Line* seg, int n) {
  const float margin = 0.1;
  float distance = -1.;
  for (int l = 0; l < n; ++l) {
    const Line& line = seg[l];
    if (line.sd - margin < d && line.ed + margin > d) {
      const float delta_z = line.ez - line.sz;
      const float delta_d = line.ed - line.sd;
      const float expected_z = (d - line.sd) / delta_d * delta_z + line.sz;
      distance = fabsf(z - expected_z);
    }
  }
  return distance;
}

__host__ __device__ __forceinline__ int gr2_search_max_step(const Gr2Params& P) {
  const float delta_alpha = kPi * 2 / P.segment_num;
  const double q = P.search_angle / 180. * kPi / delta_alpha;
  return q > -1.0 && q < 2147483647.0 ? (int)q : -1;
}

// RandomSampler draw: a counter hash of (seed, call, stage, key) -> u uniform on [0, 1) with 53 bits
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z += 0x9e3779b97f4a7c15ull;
  z = (z ^ (z >> 30)) * 0xbf58476d1ce4e5b9ull;
  z = (z ^ (z >> 27)) * 0x94d049bb133111ebull;
  return z ^ (z >> 31);
}
__host__ __device__ __forceinline__ double rs_uniform(uint64_t seed, uint64_t call, int stage, uint64_t key) {
  const uint64_t h = mix64(mix64(mix64(mix64(seed) ^ call) ^ (uint64_t)stage) ^ key);
  return (double)(h >> 11) * (1.0 / 9007199254740992.0);
}

// ---- kernels ------------------------------------------------------------------------------------------------
enum StageType { kRange, kAxisRange, kBoundingBox, kRandomSampler, kStatisticRemoval, kRangeImage, kGroundRemoval,
                 kGroundRemoval2, kVoxelGrid, kStageTypes };
const char* const kNames[kStageTypes] = {"Range", "AxisRange", "BoundingBoxRemoval", "RandomSampler",
                                         "StatisticRemoval", "RangeImage", "GroundRemoval", "GroundRemoval2",
                                         "VoxelGrid"};

constexpr int kMaxFused = 16;
struct PwStage { int type; int index; float f[6]; int axis; };
struct PwRun { PwStage s[kMaxFused]; int n; uint64_t seed, call; };

__device__ __forceinline__ bool pw_keep(const PwStage& S, const float* p, int32_t kept, uint32_t pos, uint64_t seed,
                                        uint64_t call) {
  switch (S.type) {
    case kRange: {
      const float range = sqrtf(p[0] * p[0] + p[1] * p[1] + p[2] * p[2]);
      return range >= S.f[0] && range <= S.f[1];
    }
    case kAxisRange: {
      if (S.f[0] == -FLT_MAX && S.f[1] == FLT_MAX) return true;
      if (S.axis < 0 || S.axis > 2) return true;
      const float v = p[S.axis];
      return !(v < S.f[0] || v > S.f[1]);
    }
    case kBoundingBox: {
      const double x = p[0], y = p[1], z = p[2];
      return !((x >= (double)S.f[0] && x <= (double)S.f[3]) && (y >= (double)S.f[1] && y <= (double)S.f[4]) &&
               (z >= (double)S.f[2] && z <= (double)S.f[5]));
    }
    case kRandomSampler: {
      if ((double)S.f[0] > 0.999) return true;
      const uint64_t key = kept >= 0 ? (uint64_t)kept : ((1ull << 32) | pos);
      return rs_uniform(seed, call, S.index, key) <= (double)S.f[0];
    }
    default: return true;                                            // StatisticRemoval
  }
}

__global__ void __launch_bounds__(256)
pw_flag_kernel(const float* __restrict__ rec, const int32_t* __restrict__ kept, int n, PwRun R,
               uint32_t* __restrict__ flag, uint32_t* __restrict__ rejected) {
  // rejected[s]: points the run's stage s removes (the first stage that fails a point removes it), so that the
  // count after every stage of the run is known
  __shared__ uint32_t rej[kMaxFused];
  if (threadIdx.x < kMaxFused) rej[threadIdx.x] = 0;
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    const float* p = rec + 5 * (int64_t)i;
    int s = 0;
    while (s < R.n && pw_keep(R.s[s], p, kept[i], (uint32_t)i, R.seed, R.call)) ++s;
    flag[i] = s == R.n ? 1u : 0u;
    if (s < R.n) atomicAdd(&rej[s], 1u);
  }
  __syncthreads();
  if (threadIdx.x < R.n && rej[threadIdx.x]) atomicAdd(&rejected[threadIdx.x], rej[threadIdx.x]);
}

// flag: exclusive scan of the keep flags (n + 1 entries); order (optional): gather through a permutation
__global__ void __launch_bounds__(256)
compact_kernel(const float* __restrict__ rec, const int32_t* __restrict__ kept, const uint32_t* __restrict__ flag,
               const uint32_t* __restrict__ order, int n, float* __restrict__ out, int32_t* __restrict__ out_kept) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t pos = flag[k];
  if (flag[k + 1] == pos) return;
  const int64_t j = order ? (int64_t)order[k] : (int64_t)k;
  for (int c = 0; c < 5; ++c) out[5 * (int64_t)pos + c] = rec[5 * j + c];
  out_kept[pos] = kept[j];
}

__global__ void __launch_bounds__(256)
gather_input_kernel(const char* __restrict__ pts, int64_t stride, int n, float* __restrict__ rec,
                    int32_t* __restrict__ kept) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float* p = reinterpret_cast<const float*>(pts + (int64_t)i * stride);
  for (int c = 0; c < 5; ++c) rec[5 * (int64_t)i + c] = p[c];
  kept[i] = i;
}

__global__ void __launch_bounds__(256)
ri_claim_kernel(const float* __restrict__ rec, int n, RiParams P, int64_t* __restrict__ pix,
                unsigned int* __restrict__ image) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t q = ri_pixel(rec + 5 * (int64_t)i, P);
  pix[i] = q;
  if (q >= 0) atomicMin(&image[q], (unsigned int)i);
}

__global__ void __launch_bounds__(256)
ri_flag_kernel(const int64_t* __restrict__ pix, int n, const unsigned int* __restrict__ image,
               uint32_t* __restrict__ flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t q = pix[i];
  flag[i] = (q >= 0 && image[q] == (unsigned int)i) ? 1u : 0u;
}

// GroundRemoval voxel: static_cast<int>(v / leaf) per axis.  0 ok, 1 not finite, 2 outside the int range
__host__ __device__ __forceinline__ int gr_voxel(const float* p, float leaf, long long* ijk) {
  for (int d = 0; d < 3; ++d) {
    if (!isfinite(p[d])) return 1;
  }
  for (int d = 0; d < 3; ++d) {
    const float q = p[d] / leaf;
    if (!(q > -2147483649.0f && q < 2147483648.0f)) return 2;
    ijk[d] = (long long)(int)q;
  }
  return 0;
}

constexpr long long kSpan = 1ll << 21;

// meta[0..2]: minimum voxel index over the finite points; meta[4]: an index outside the int range or a span of 2^21
__global__ void __launch_bounds__(256)
gr_min_kernel(const float* __restrict__ rec, int n, float leaf, long long* __restrict__ meta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  long long v[3] = {LLONG_MAX, LLONG_MAX, LLONG_MAX};
  if (i < n) {
    long long a[3];
    const int rc = gr_voxel(rec + 5 * (int64_t)i, leaf, a);
    if (rc == 0) { v[0] = a[0]; v[1] = a[1]; v[2] = a[2]; }
    if (rc == 2) atomicExch((unsigned long long*)&meta[4], 1ull);
  }
  for (int o = 16; o > 0; o >>= 1)
    for (int d = 0; d < 3; ++d) v[d] = min(v[d], __shfl_xor_sync(0xffffffffu, v[d], o));
  if ((threadIdx.x & 31) == 0)
    for (int d = 0; d < 3; ++d) atomicMin(&meta[d], v[d]);
}

__global__ void __launch_bounds__(256)
gr_key_kernel(const float* __restrict__ rec, int n, float leaf, uint64_t* __restrict__ keys,
              uint32_t* __restrict__ vals, long long* __restrict__ meta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  long long a[3];
  uint64_t key = ~0ull;                                              // not finite: behind every voxel, kept
  if (gr_voxel(rec + 5 * (int64_t)i, leaf, a) == 0) {
    const unsigned long long ox = (unsigned long long)(a[0] - meta[0]), oy = (unsigned long long)(a[1] - meta[1]),
                             oz = (unsigned long long)(a[2] - meta[2]);
    if (ox < (unsigned long long)kSpan && oy < (unsigned long long)kSpan && oz < (unsigned long long)kSpan)
      key = (ox << 42) | (oy << 21) | oz;
    else
      atomicExch((unsigned long long*)&meta[4], 1ull);
  }
  keys[i] = key;
  vals[i] = (uint32_t)i;
}

__global__ void __launch_bounds__(256)
head_flag_kernel(const uint64_t* __restrict__ keys, int n, uint32_t* __restrict__ flag) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  flag[k] = (k == 0 || keys[k] != keys[k - 1]) ? 1u : 0u;
}

// starts[v] = first sorted position of segment v, starts[n_seg] = n
__global__ void __launch_bounds__(256)
head_scatter_kernel(const uint32_t* __restrict__ flag, int n, uint32_t* __restrict__ starts) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k > n) return;
  if (k == n) { starts[flag[n]] = (uint32_t)n; return; }
  if (flag[k + 1] != flag[k]) starts[flag[k]] = (uint32_t)k;
}

// one thread per voxel: the keep flag of each of its sorted positions
__global__ void __launch_bounds__(256)
gr_voxel_kernel(const float* __restrict__ rec, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ order,
                const uint32_t* __restrict__ starts, uint32_t n_seg, long long min_iz,
                int min_pts, float height_threshold, uint32_t* __restrict__ flag) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_seg) return;
  const uint32_t a = starts[v], b = starts[v + 1];
  uint32_t keep = 1;
  if (keys[a] != ~0ull) {
    if ((int64_t)(b - a) < (int64_t)min_pts) {
      keep = 0;                                                      // vanishes: neither inlier nor outlier
    } else if ((long long)(keys[a] & (kSpan - 1)) + min_iz <= 0) {   // index[2] <= 0
      float max_z = -1.e9f, min_z = 1.e9f;
      for (uint32_t k = a; k < b; ++k) {
        const float z = rec[5 * (int64_t)order[k] + 2];
        if (z > max_z) max_z = z;
        if (z < min_z) min_z = z;
      }
      const float delta = max_z - min_z;
      if (delta >= 0. && delta <= height_threshold) keep = 0;        // ground
    }
  }
  for (uint32_t k = a; k < b; ++k) flag[k] = keep;
}

__global__ void __launch_bounds__(256)
gr2_key_kernel(const float* __restrict__ rec, int n, Gr2Params P, uint64_t* __restrict__ keys,
               uint32_t* __restrict__ vals, float* __restrict__ range) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float r = 0.f;
  const int64_t c = gr2_cell(rec + 5 * (int64_t)i, P, &r);
  keys[i] = c < 0 ? 0xffffffffull : (uint64_t)c;
  vals[i] = (uint32_t)i;
  range[i] = r;
}

// one thread per cell: its points in input order; member[i]: the point entered the cell's `points`
__global__ void __launch_bounds__(256)
gr2_cell_kernel(const float* __restrict__ rec, const uint64_t* __restrict__ keys, const uint32_t* __restrict__ order,
                const uint32_t* __restrict__ starts, uint32_t n_seg, const float* __restrict__ range, float* __restrict__ cell_d, float* __restrict__ cell_z,
                uint8_t* __restrict__ cell_used, uint8_t* __restrict__ member) {
  const uint32_t v = blockIdx.x * blockDim.x + threadIdx.x;
  if (v >= n_seg) return;
  const uint32_t a = starts[v], b = starts[v + 1];
  const uint64_t c = keys[a];
  if (c == 0xffffffffull) return;
  float md = 1.e6f, mz = 1.e6f;
  for (uint32_t k = a; k < b; ++k) {
    const uint32_t i = order[k];
    const float z = rec[5 * (int64_t)i + 2];
    if (k == a || z < mz) { md = range[i]; mz = z; }
    member[i] = (double)z <= (double)mz + 0.5 ? 1 : 0;
  }
  cell_d[c] = md; cell_z[c] = mz; cell_used[c] = 1;
}

__global__ void __launch_bounds__(64)
gr2_fit_kernel(const float* __restrict__ cell_d, const float* __restrict__ cell_z,
               const uint8_t* __restrict__ cell_used, Gr2Params P, float2* __restrict__ scratch,
               Line* __restrict__ lines, int cap, int* __restrict__ nlines) {
  const int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= P.segment_num) return;
  const int64_t o = (int64_t)s * P.bin_num;
  nlines[s] = gr2_fit_lines(cell_d + o, cell_z + o, cell_used + o, P, scratch + o, lines + (int64_t)s * cap, cap);
}

// ClusterGround (:337-396) for one point: 1 = ground (outlier)
__global__ void __launch_bounds__(256)
gr2_cluster_kernel(const float* __restrict__ rec, int n, Gr2Params P, int search_max_step,
                   const uint64_t* __restrict__ keys, const uint32_t* __restrict__ order,
                   const uint8_t* __restrict__ member, const float* __restrict__ range, const Line* __restrict__ lines,
                   int cap, const int* __restrict__ nlines, uint32_t* __restrict__ flag) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const uint32_t i = order[k];
  const uint64_t c = keys[k];
  uint32_t keep = 1;
  if (c != 0xffffffffull && member[i]) {
    const int s = (int)(c / (uint64_t)P.bin_num);
    const float d = range[i], z = rec[5 * (int64_t)i + 2];
    float distance = gr2_vertical_distance(d, z, lines + (int64_t)s * cap, nlines[s]);
    if (distance < 0.) {
      for (int step = search_max_step; step > 0; --step) {
        for (int sign = 0; sign < 2; ++sign) {
          int cs = s + (sign ? -step : step);
          if (cs < 0) cs += P.segment_num;
          else if (cs >= P.segment_num) cs -= P.segment_num;
          distance = gr2_vertical_distance(d, z, lines + (int64_t)cs * cap, nlines[cs]);
          if (distance > 0.) break;
        }
        if (distance > 0.) break;
      }
    }
    if (distance > 0. && distance <= P.max_dist_to_line) keep = 0;
  }
  flag[i] = keep;
}

}  // namespace
}  // namespace smb

using namespace smb;

// ---- the handle ---------------------------------------------------------------------------------------------
namespace {

struct ParamDef { const char* name; int is_int; int slot; double init; };
// per stage type: the reference's registered parameters (INIT_*_PARAM) and constructor defaults
const std::vector<ParamDef>& param_defs(int type) {
  static const std::vector<ParamDef> defs[kStageTypes] = {
      {{"min_range", 0, 0, 0.0}, {"max_range", 0, 1, FLT_MAX}},
      {{"min", 0, 0, -FLT_MAX}, {"max", 0, 1, FLT_MAX}, {"axis_index", 1, 0, 2}},
      {{"min_x", 0, 0, -FLT_MAX}, {"min_y", 0, 1, -FLT_MAX}, {"min_z", 0, 2, -FLT_MAX},
       {"max_x", 0, 3, FLT_MAX}, {"max_y", 0, 4, FLT_MAX}, {"max_z", 0, 5, FLT_MAX}},
      {{"sampling_rate", 0, 0, 1.0}},
      {{"std_mul", 0, 0, 1.0}, {"point_num_meank", 1, 0, 30}},
      {{"top_angle", 0, 0, 30.0}, {"btm_angle", 0, 1, -15.0}, {"offset_x", 0, 2, 0.0}, {"offset_y", 0, 3, 0.0},
       {"offset_z", 0, 4, 0.0}, {"vertical_line_num", 1, 0, 40}, {"horizontal_line_num", 1, 1, 1800}},
      {{"leaf_size", 0, 0, 0.8}, {"height_threshold", 0, 1, 0.15}, {"min_point_num_in_voxel", 1, 0, 10}},
      {{"r_max", 0, 0, 100.0}, {"r_min", 0, 1, 1.0}, {"start_ground_height", 0, 2, -0.25},
       {"long_line_threshold", 0, 3, 1.0}, {"max_long_line_height", 0, 4, 0.1}, {"max_start_height", 0, 5, 0.2},
       {"max_error", 0, 6, 0.05}, {"max_slope", 0, 7, (float)std::tan(kPi / 12.)}, {"max_b", 0, 8, 0.1},
       {"max_dist_to_line", 0, 9, 0.05}, {"search_angle", 0, 10, 10.0}, {"bin_num", 1, 0, 200},
       {"segment_num", 1, 1, 180}, {"thread_num", 1, 2, 4}},
      {{"voxel_size", 0, 0, 0.1}},
  };
  return defs[type];
}

struct Stage {
  int type = 0;
  float f[12] = {};
  int32_t i[3] = {};
};

Gr2Params gr2_params(const Stage& S) {
  Gr2Params P;
  P.r_max = S.f[0]; P.r_min = S.f[1]; P.start_ground_height = S.f[2]; P.long_line_threshold = S.f[3];
  P.max_long_line_height = S.f[4]; P.max_start_height = S.f[5]; P.max_error = S.f[6]; P.max_slope = S.f[7];
  P.max_b = S.f[8]; P.max_dist_to_line = S.f[9]; P.search_angle = S.f[10];
  P.bin_num = S.i[0]; P.segment_num = S.i[1];
  return P;
}

RiParams ri_params(const Stage& S) { return RiParams{S.f[0], S.f[1], S.f[2], S.f[3], S.f[4], S.i[0], S.i[1]}; }

// ConfigsValid() of the reference, and (second) whether this engine can run the stage
bool configs_valid(const Stage& S) {
  const float* f = S.f;
  switch (S.type) {
    case kAxisRange: return f[1] > f[0] && S.i[0] >= 0 && S.i[0] <= 2;
    case kBoundingBox: return f[0] < f[3] && f[1] < f[4] && f[2] < f[5];
    case kRandomSampler: return f[0] >= 0.f && f[0] <= 1.f;
    case kVoxelGrid: return f[0] > 1.e-6;
    default: return true;
  }
}
bool runnable(const Stage& S) {
  if (!configs_valid(S)) return false;
  switch (S.type) {
    case kRangeImage: return S.i[0] > 0 && S.i[1] > 0 && (int64_t)S.i[0] * S.i[1] <= (1ll << 28);
    case kGroundRemoval: return S.f[0] != 0.f && !isnan(S.f[0]);
    case kGroundRemoval2: {
      const Gr2Params P = gr2_params(S);
      return P.bin_num > 0 && P.segment_num > 0 && (int64_t)P.bin_num * P.segment_num <= (1ll << 26) &&
             gr2_search_max_step(P) >= 0 && gr2_search_max_step(P) <= P.segment_num;
    }
    default: return true;
  }
}

int32_t parse_int(const char* t) {                 // pugixml as_int: decimal or 0x hex, saturated
  while (*t == ' ' || *t == '\t' || *t == '\n' || *t == '\r') ++t;
  const bool neg = *t == '-';
  const char* s = (*t == '-' || *t == '+') ? t + 1 : t;
  const int base = (s[0] == '0' && (s[1] == 'x' || s[1] == 'X')) ? 16 : 10;
  const long long v = strtoll(s, nullptr, base);
  const long long sv = neg ? -v : v;
  return (int32_t)std::min<long long>(INT_MAX, std::max<long long>(INT_MIN, sv));
}

}  // namespace

struct sm_filter_chain {
  int device = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev_caller = nullptr;
  std::vector<cudaEvent_t> ev;                     // one before the chain, one after each stage
  std::vector<Stage> stages;
  std::vector<int64_t> counts;                     // points after each stage of the last call
  std::vector<float> stage_ms;                     // device time of each stage of the last call
  uint64_t seed = 0, call = 0;
  char* ws = nullptr;
  size_t ws_bytes = 0;
};

namespace {

int reserve(sm_filter_chain* h, size_t need) {
  if (need <= h->ws_bytes) return SM_OK;
  cudaFree(h->ws);
  h->ws = nullptr; h->ws_bytes = 0;
  if (cudaMalloc(&h->ws, need) != cudaSuccess) return SM_ERR_CUDA;
  h->ws_bytes = need;
  return SM_OK;
}

size_t al(size_t b) { return (b + 255) & ~(size_t)255; }

// scan the n + 1 flags in place and read back the kept count
int scan_count(uint32_t* flag, int n, cudaStream_t s, uint32_t* m) {
  cudaMemsetAsync(flag + n, 0, sizeof(uint32_t), s);
  radix_scan_kernel_launch(flag, n + 1, 1, s);
  if (cudaMemcpyAsync(m, flag + n, sizeof(uint32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess)
    return SM_ERR_CUDA;
  return SM_OK;
}

int run(sm_filter_chain* h, const float* points, int64_t n, int64_t stride, float* out, int64_t capacity,
        int64_t* m_out, int32_t* kept_index, bool on_device, cudaStream_t caller) {
  if (!h || !m_out || n < 0 || n > (1 << 30) || stride < 20 || stride % 4 || capacity < 0 ||
      (n > 0 && !points) || (capacity > 0 && !out))
    return SM_ERR_BAD_ARGUMENT;
  *m_out = 0;
  const int ns = (int)h->stages.size();
  for (const Stage& S : h->stages)
    if (!runnable(S)) return SM_ERR_BAD_ARGUMENT;    // the reference would run an invalid stage anyway
  for (const Stage& S : h->stages)                   // a search step past segment_num: segments.at() throws
    if (S.type == kGroundRemoval2 && gr2_search_max_step(gr2_params(S)) >= gr2_params(S).segment_num) return SM_ERR_BAD_ARGUMENT;
  if (cudaSetDevice(h->device) != cudaSuccess) return SM_ERR_CUDA;
  const cudaStream_t s = h->stream;
  const uint64_t call = h->call++;
  h->counts.assign(ns, 0);
  h->stage_ms.assign(ns, 0.f);
  if (n == 0) return SM_OK;
  const int ni = (int)n;
  const int64_t st = (n + 63) & ~(int64_t)63;
  // workspace: input copy, 2 x (records, kept), flags, sort buffers, starts, per-point scratch, per-stage extras
  size_t extra = 0;
  for (const Stage& S : h->stages) {
    if (S.type == kRangeImage) extra = std::max(extra, al((size_t)S.i[0] * S.i[1] * 4) + al((size_t)n * 8));
    if (S.type == kGroundRemoval2) {
      const Gr2Params P = gr2_params(S);
      const size_t cells = (size_t)P.bin_num * P.segment_num, cap = (size_t)P.bin_num / 2 + 2;
      extra = std::max(extra, 2 * al(cells * 4) + al(cells) + al(cells * 8) + al((size_t)P.segment_num * cap * 16) +
                                  al((size_t)P.segment_num * 4) + al((size_t)n) + al((size_t)n * 4));
    }
  }
  const size_t in_bytes = on_device ? 0 : al((size_t)n * stride);
  const size_t need = in_bytes + 2 * (al(st * 20) + al(st * 4)) + al((st + 8) * 4) + 2 * al(st * 8) + 2 * al(st * 4) +
                      al(radix_sort_scratch_bytes(ni, 1)) + al((st + 8) * 4) + 2 * 256 + extra + 1024;
  int rc = reserve(h, need);
  if (rc) return rc;
  char* cur = h->ws;
  auto take = [&](size_t b) { char* p = cur; cur += al(b); return p; };
  const char* d_in = on_device ? (const char*)points : take((size_t)n * stride);
  float* rec[2] = {(float*)take(st * 20), (float*)take(st * 20)};
  int32_t* kept[2] = {(int32_t*)take(st * 4), (int32_t*)take(st * 4)};
  uint32_t* flag = (uint32_t*)take((st + 8) * 4);
  uint64_t* keys0 = (uint64_t*)take(st * 8);
  uint64_t* keys1 = (uint64_t*)take(st * 8);
  uint32_t* ord0 = (uint32_t*)take(st * 4);
  uint32_t* ord1 = (uint32_t*)take(st * 4);
  uint32_t* scratch = (uint32_t*)take(radix_sort_scratch_bytes(ni, 1));
  uint32_t* starts = (uint32_t*)take((st + 8) * 4);
  long long* meta = (long long*)take(256);
  uint32_t* rejected = (uint32_t*)take(kMaxFused * sizeof(uint32_t));
  uint32_t host_rejected[kMaxFused] = {};
  char* ex = cur;

  if (on_device) {
    if (cudaEventRecord(h->ev_caller, caller) != cudaSuccess || cudaStreamWaitEvent(s, h->ev_caller, 0) != cudaSuccess)
      return SM_ERR_CUDA;
  } else if (cudaMemcpyAsync((void*)d_in, points, (size_t)n * stride, cudaMemcpyHostToDevice, s) != cudaSuccess) {
    return SM_ERR_CUDA;
  }
  cudaEventRecord(h->ev[0], s);
  gather_input_kernel<<<ceil_div(n, 256), 256, 0, s>>>(d_in, stride, ni, rec[0], kept[0]);
  std::vector<int> steps;                            // first stage of each step (a fused run is one step)
  int c = 0;                                         // current buffer
  uint32_t m = (uint32_t)ni;
  int k = 0;
  while (k < ns && m > 0) {
    const Stage& S = h->stages[k];
    const int mi = (int)m;
    const int g = ceil_div(mi, 256);
    int done = 1;                                    // stages consumed by this step
    const uint32_t* order = nullptr;
    switch (S.type) {
      case kRange: case kAxisRange: case kBoundingBox: case kRandomSampler: case kStatisticRemoval: {
        PwRun R{};
        R.seed = h->seed; R.call = call; R.n = 0;
        for (int j = k; j < ns && R.n < kMaxFused; ++j) {
          const Stage& T = h->stages[j];
          if (T.type > kStatisticRemoval) break;
          PwStage& P = R.s[R.n++];
          P.type = T.type; P.index = j; P.axis = T.i[0];
          for (int q = 0; q < 6; ++q) P.f[q] = T.f[q];
        }
        done = R.n;
        cudaMemsetAsync(rejected, 0, kMaxFused * sizeof(uint32_t), s);
        pw_flag_kernel<<<g, 256, 0, s>>>(rec[c], kept[c], mi, R, flag, rejected);
        if (cudaMemcpyAsync(host_rejected, rejected, kMaxFused * sizeof(uint32_t), cudaMemcpyDeviceToHost, s) !=
            cudaSuccess)
          return SM_ERR_CUDA;                         // read once the scan below has synchronised the stream
        break;
      }
      case kRangeImage: {
        const RiParams P = ri_params(S);
        unsigned int* image = (unsigned int*)ex;
        int64_t* pix = (int64_t*)(ex + al((size_t)P.V * P.H * 4));
        cudaMemsetAsync(image, 0xff, (size_t)P.V * P.H * 4, s);
        ri_claim_kernel<<<g, 256, 0, s>>>(rec[c], mi, P, pix, image);
        ri_flag_kernel<<<g, 256, 0, s>>>(pix, mi, image, flag);
        break;
      }
      case kGroundRemoval: {
        const long long meta_init[8] = {LLONG_MAX, LLONG_MAX, LLONG_MAX, 0, 0, 0, 0, 0};
        long long hm[8];
        if (cudaMemcpyAsync(meta, meta_init, sizeof(meta_init), cudaMemcpyHostToDevice, s) != cudaSuccess)
          return SM_ERR_CUDA;
        gr_min_kernel<<<g, 256, 0, s>>>(rec[c], mi, S.f[0], meta);
        gr_key_kernel<<<g, 256, 0, s>>>(rec[c], mi, S.f[0], keys0, ord0, meta);
        if (radix_sort_pairs_u64(keys0, ord0, keys1, ord1, mi, 1, st, scratch, s, 8)) return SM_ERR_CUDA;
        uint32_t nseg = 0;
        head_flag_kernel<<<g, 256, 0, s>>>(keys0, mi, flag);
        if ((rc = scan_count(flag, mi, s, &nseg))) return rc;
        head_scatter_kernel<<<ceil_div(mi + 1, 256), 256, 0, s>>>(flag, mi, starts);
        if (cudaMemcpyAsync(hm, meta, sizeof(hm), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
            cudaStreamSynchronize(s) != cudaSuccess)
          return SM_ERR_CUDA;
        if (hm[4]) return SM_ERR_BAD_ARGUMENT;      // a voxel index outside the int range, or a span of 2^21
        const long long min_iz = hm[2] == LLONG_MAX ? 0 : hm[2];
        gr_voxel_kernel<<<ceil_div(nseg, 256), 256, 0, s>>>(rec[c], keys0, ord0, starts, nseg, min_iz, S.i[0],
                                                             S.f[1], flag);
        order = ord0;
        break;
      }
      case kGroundRemoval2: {
        const Gr2Params P = gr2_params(S);
        const size_t cells = (size_t)P.bin_num * P.segment_num;
        const int cap = P.bin_num / 2 + 2;
        char* e = ex;
        auto etake = [&](size_t b) { char* p = e; e += al(b); return p; };
        float* cell_d = (float*)etake(cells * 4);
        float* cell_z = (float*)etake(cells * 4);
        uint8_t* cell_used = (uint8_t*)etake(cells);
        float2* fit_scratch = (float2*)etake(cells * 8);
        Line* lines = (Line*)etake((size_t)P.segment_num * cap * 16);
        int* nlines = (int*)etake((size_t)P.segment_num * 4);
        uint8_t* member = (uint8_t*)etake((size_t)n);
        float* range = (float*)etake((size_t)n * 4);
        cudaMemsetAsync(cell_used, 0, cells, s);
        cudaMemsetAsync(member, 0, (size_t)mi, s);
        gr2_key_kernel<<<g, 256, 0, s>>>(rec[c], mi, P, keys0, ord0, range);
        if (radix_sort_pairs_u64(keys0, ord0, keys1, ord1, mi, 1, st, scratch, s, 4)) return SM_ERR_CUDA;
        uint32_t nseg = 0;
        head_flag_kernel<<<g, 256, 0, s>>>(keys0, mi, flag);
        if ((rc = scan_count(flag, mi, s, &nseg))) return rc;
        head_scatter_kernel<<<ceil_div(mi + 1, 256), 256, 0, s>>>(flag, mi, starts);
        gr2_cell_kernel<<<ceil_div(nseg, 256), 256, 0, s>>>(rec[c], keys0, ord0, starts, nseg, range, cell_d,
                                                             cell_z, cell_used, member);
        gr2_fit_kernel<<<ceil_div(P.segment_num, 64), 64, 0, s>>>(cell_d, cell_z, cell_used, P, fit_scratch, lines,
                                                                   cap, nlines);
        gr2_cluster_kernel<<<g, 256, 0, s>>>(rec[c], mi, P, gr2_search_max_step(P), keys0, ord0, member, range,
                                             lines, cap, nlines, flag);
        break;
      }
      case kVoxelGrid: {
        uint32_t mv = 0;
        if ((rc = voxel_grid_device((const char*)rec[c], 20, mi, S.f[0], rec[1 - c], &mv, s))) return rc;
        cudaMemsetAsync(kept[1 - c], 0xff, (size_t)mv * 4, s);
        c = 1 - c;
        m = mv;
        break;
      }
    }
    if (S.type != kVoxelGrid) {
      uint32_t mk = 0;
      if ((rc = scan_count(flag, mi, s, &mk))) return rc;
      compact_kernel<<<g, 256, 0, s>>>(rec[c], kept[c], flag, order, mi, rec[1 - c], kept[1 - c]);
      c = 1 - c;
      m = mk;
    }
    cudaEventRecord(h->ev[k + done], s);
    if (S.type <= kStatisticRemoval) {               // a fused point-wise run: count after each of its stages
      int64_t left = mi;
      for (int j = k; j < k + done; ++j) h->counts[j] = (left -= host_rejected[j - k]);
    } else {
      h->counts[k] = m;
    }
    steps.push_back(k);
    k += done;
  }
  steps.push_back(k);                                // the end of the last step that ran (stages after it saw 0 points)
  if (cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess) return SM_ERR_CUDA;
  for (size_t q = 0; q + 1 < steps.size(); ++q) {   // a fused run's time is reported on its first stage
    float ms = 0.f;
    const int a = steps[q], b = steps[q + 1];
    if (cudaEventElapsedTime(&ms, h->ev[q == 0 ? 0 : a], h->ev[b]) == cudaSuccess) h->stage_ms[a] = ms;
  }
  *m_out = m;
  if ((int64_t)m > capacity) return SM_ERR_BAD_ARGUMENT;
  if (m == 0) return SM_OK;
  const cudaMemcpyKind kind = on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  if (cudaMemcpyAsync(out, rec[c], (size_t)m * 20, kind, s) != cudaSuccess ||
      (kept_index && cudaMemcpyAsync(kept_index, kept[c], (size_t)m * 4, kind, s) != cudaSuccess) ||
      cudaStreamSynchronize(s) != cudaSuccess)
    return SM_ERR_CUDA;
  return SM_OK;
}

}  // namespace

extern "C" int sm_filter_chain_create(int device, sm_filter_chain** out) {
  if (!out) return SM_ERR_BAD_ARGUMENT;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return SM_ERR_NO_DEVICE;
  if (device < 0 || device >= ndev || cudaSetDevice(device) != cudaSuccess) return SM_ERR_BAD_ARGUMENT;
  sm_filter_chain* h = new sm_filter_chain;
  h->device = device;
  h->ev.assign(1, nullptr);
  if (cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->ev_caller, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreate(&h->ev[0]) != cudaSuccess) {
    sm_filter_chain_destroy(h);
    return SM_ERR_CUDA;
  }
  *out = h;
  return SM_OK;
}

extern "C" int sm_filter_chain_destroy(sm_filter_chain* h) {
  if (!h) return SM_ERR_BAD_ARGUMENT;
  cudaSetDevice(h->device);
  cudaFree(h->ws);
  for (cudaEvent_t e : h->ev) if (e) cudaEventDestroy(e);
  if (h->ev_caller) cudaEventDestroy(h->ev_caller);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
  return SM_OK;
}

extern "C" int sm_filter_chain_add(sm_filter_chain* h, const char* name) {
  if (!h || !name) return SM_ERR_BAD_ARGUMENT;
  for (int t = 0; t < kStageTypes; ++t) {
    if (strcmp(name, kNames[t]) != 0) continue;
    Stage S;
    S.type = t;
    for (const ParamDef& d : param_defs(t)) {
      if (d.is_int) S.i[d.slot] = (int32_t)d.init;
      else S.f[d.slot] = (float)d.init;
    }
    cudaEvent_t e = nullptr;
    if (cudaSetDevice(h->device) != cudaSuccess || cudaEventCreate(&e) != cudaSuccess) return SM_ERR_CUDA;
    h->ev.push_back(e);
    h->stages.push_back(S);
    return (int)h->stages.size() - 1;
  }
  return SM_ERR_UNSUPPORTED_TYPE;
}

extern "C" int sm_filter_chain_set_param(sm_filter_chain* h, int32_t stage, const char* name, int32_t type,
                                         const char* text) {
  if (!h || !name || !text || stage < 0 || stage >= (int)h->stages.size()) return SM_ERR_BAD_ARGUMENT;
  Stage& S = h->stages[stage];
  for (const ParamDef& d : param_defs(S.type)) {
    if (strcmp(name, d.name) != 0) continue;
    if (type == 0) {                                 // as_int, then static_cast to the parameter's type
      const int32_t v = parse_int(text);
      if (d.is_int) S.i[d.slot] = v; else S.f[d.slot] = (float)v;
    } else if (type == 1) {                          // as_float (strtod, rounded to float)
      const float v = (float)strtod(text, nullptr);
      if (d.is_int) {
        if (!(v > -2147483649.f && v < 2147483648.f)) return SM_ERR_BAD_ARGUMENT;
        S.i[d.slot] = (int32_t)v;
      } else {
        S.f[d.slot] = v;
      }
    } else {
      return SM_ERR_BAD_ARGUMENT;                    // no / unknown type attribute: CHECK(all_right) fails
    }
    return SM_OK;
  }
  return SM_ERR_UNKNOWN_OPTION;
}

extern "C" int sm_filter_chain_valid(const sm_filter_chain* h, int32_t stage) {
  if (!h || stage < 0 || stage >= (int)h->stages.size()) return SM_ERR_BAD_ARGUMENT;
  return configs_valid(h->stages[stage]) ? 1 : 0;
}

extern "C" int sm_filter_chain_set_seed(sm_filter_chain* h, uint64_t seed) {
  if (!h) return SM_ERR_BAD_ARGUMENT;
  h->seed = seed;
  h->call = 0;
  return SM_OK;
}

extern "C" int sm_filter_chain_filter(sm_filter_chain* h, const float* points, int64_t n, int64_t stride_bytes,
                                      float* out, int64_t capacity, int64_t* m_out, int32_t* kept_index) {
  return run(h, points, n, stride_bytes, out, capacity, m_out, kept_index, false, nullptr);
}

extern "C" int sm_filter_chain_filter_device(sm_filter_chain* h, const float* dev_points, int64_t n,
                                             int64_t stride_bytes, float* dev_out, int64_t capacity, int64_t* m_out,
                                             int32_t* dev_kept_index, void* cuda_stream) {
  return run(h, dev_points, n, stride_bytes, dev_out, capacity, m_out, dev_kept_index, true,
             (cudaStream_t)cuda_stream);
}

extern "C" int sm_filter_chain_stage_counts(const sm_filter_chain* h, int64_t* counts, int32_t n) {
  if (!h || n < 0 || (n > 0 && !counts)) return SM_ERR_BAD_ARGUMENT;
  for (int k = 0; k < std::min(n, (int32_t)h->counts.size()); ++k) counts[k] = h->counts[k];
  return (int)h->stages.size();
}

extern "C" int sm_filter_chain_stage_ms(const sm_filter_chain* h, float* ms, int32_t n) {
  if (!h || n < 0 || (n > 0 && !ms)) return SM_ERR_BAD_ARGUMENT;
  for (int k = 0; k < std::min(n, (int32_t)h->stage_ms.size()); ++k) ms[k] = h->stage_ms[k];
  return (int)h->stages.size();
}

// ---- test hooks (include/sm_b200_debug.h) ---------------------------------------------------------------------
extern "C" int sm_debug_filter_points(int32_t op, const float* points, int64_t n, int64_t stride_bytes,
                                      const float* params, int64_t* out) {
  if (!points || !params || !out || n < 0 || stride_bytes < 12 || stride_bytes % 4) return SM_ERR_BAD_ARGUMENT;
  for (int64_t k = 0; k < n; ++k) {
    const float* p = (const float*)((const char*)points + k * stride_bytes);
    if (op == 0) {
      const float a = sm_atan2f(p[1], p[0]);
      uint32_t u; memcpy(&u, &a, 4); out[k] = u;
    } else if (op == 1) {
      const RiParams P{params[0], params[1], params[2], params[3], params[4], (int)params[5], (int)params[6]};
      if (P.V <= 0 || P.H <= 0) return SM_ERR_BAD_ARGUMENT;
      out[k] = ri_pixel(p, P);
    } else if (op == 2) {
      Gr2Params P{params[0], params[1], 0, 0, 0, 0, 0, 0, 0, 0, 0, (int)params[2], (int)params[3]};
      if (P.bin_num <= 0 || P.segment_num <= 0) return SM_ERR_BAD_ARGUMENT;
      float r;
      out[k] = gr2_cell(p, P, &r);
    } else if (op == 3) {
      long long a[3] = {0, 0, 0};
      const int rc = gr_voxel(p, params[0], a);
      out[4 * k] = rc; out[4 * k + 1] = a[0]; out[4 * k + 2] = a[1]; out[4 * k + 3] = a[2];
    } else {
      return SM_ERR_BAD_ARGUMENT;
    }
  }
  return SM_OK;
}

extern "C" int sm_debug_filter_fit_lines(const float* cell_dz, const uint8_t* cell_used, const float* params,
                                         float* lines4, int64_t capacity, int64_t* n_out) {
  if (!cell_dz || !cell_used || !params || !n_out || capacity < 0 || (capacity > 0 && !lines4))
    return SM_ERR_BAD_ARGUMENT;
  Gr2Params P{params[0], params[1], params[2], params[3], params[4], params[5], params[6], params[7], params[8],
              params[9], params[10], (int)params[11], 1};
  if (P.bin_num <= 0) return SM_ERR_BAD_ARGUMENT;
  std::vector<float> d(P.bin_num), z(P.bin_num);
  for (int b = 0; b < P.bin_num; ++b) { d[b] = cell_dz[2 * b]; z[b] = cell_dz[2 * b + 1]; }
  std::vector<float2> scratch(P.bin_num);
  std::vector<Line> lines((size_t)P.bin_num / 2 + 2);
  const int nl = gr2_fit_lines(d.data(), z.data(), cell_used, P, scratch.data(), lines.data(), (int)lines.size());
  *n_out = nl;
  if (nl > capacity) return SM_ERR_BAD_ARGUMENT;
  for (int l = 0; l < nl; ++l) {
    lines4[4 * l] = lines[l].sd; lines4[4 * l + 1] = lines[l].sz; lines4[4 * l + 2] = lines[l].ed;
    lines4[4 * l + 3] = lines[l].ez;
  }
  return SM_OK;
}

extern "C" int sm_debug_filter_line_fit(const float* dz, int64_t k, float* mb) {
  if (!dz || !mb || k < 1 || k > (1 << 20)) return SM_ERR_BAD_ARGUMENT;
  std::vector<float2> p(k);
  for (int64_t i = 0; i < k; ++i) p[i] = make_float2(dz[2 * i], dz[2 * i + 1]);
  gr2_fit(p.data(), (int)k, &mb[0], &mb[1]);
  mb[2] = gr2_max_error(p.data(), (int)k, mb[0], mb[1]);
  return SM_OK;
}
