// MultiResolutionVoxelMap (builder/multi_resolution_voxel_map.{h,cc}) on the device: the ray-casting occupancy map
// behind static_map.pcd.  Semantics and deviations: include/sm_b200.h; formulation: DESIGN.md section 4h.
//
// Read serially, one InsertPointCloud gives voxel V m(V) misses and then h(V) hits, where h(V) = points of the scan
// ending in V and m(V) = rays j < first_end(V) through V, counted only when V existed before the scan.  So an insert
// is: end keys -> stable radix sort (key, point index) -> segments (one per end voxel: first_end, h, the points to
// append) -> insert-or-find of the segment keys into an open-addressing table -> one thread per ray walks its
// Bresenham ray and counts misses on voxels born before the scan -> one thread per voxel applies m misses and h hits
// by binary lifting over the reference's uint8 -> uint8 update maps, then max_intensity and the appended points.
// Voxel ids are dense and allocated in increasing order, so "born before this scan" is id < voxel count before it.
// Compiled with -fmad=false (the averaged output is compared bit for bit with the oracle).
#include <math.h>
#include <string.h>

#include <algorithm>
#include <cmath>
#include <vector>

#include "../../include/sm_b200.h"
#include "../../include/sm_b200_debug.h"
#include "common.cuh"
#include "kernels.h"

namespace smb {
namespace {

constexpr int kAxisHalf = 1 << 20;             // voxel index range per axis: [-2^20, 2^20)
constexpr uint64_t kEmpty = ~0ull;             // empty table slot / dropped point (a voxel key has bit 63 clear)
constexpr uint32_t kNone = 0xffffffffu;
constexpr int kLift = 32;                      // binary-lifting levels: counts < 2^32
constexpr uint8_t kUnknown = 128;

// voxel of one point: lround(floor(v / step)) per axis in float (common/math.cc:42-52).
// 0: ok, 1: a coordinate is not finite (dropped), 2: an index is outside [-2^20, 2^20) (insert refused)
__host__ __device__ __forceinline__ int mrvm_voxel(const float* p, float step, int* ijk) {
  int rc = 0;
  for (int d = 0; d < 3; ++d) {
    if (!isfinite(p[d])) return 1;
    const float f = floorf(p[d] / step);
    if (!(f >= -(float)kAxisHalf && f < (float)kAxisHalf)) rc = 2;
    else ijk[d] = (int)f;
  }
  return rc;
}

__host__ __device__ __forceinline__ uint64_t mrvm_key(int x, int y, int z) {
  return ((uint64_t)(x + kAxisHalf) << 42) | ((uint64_t)(y + kAxisHalf) << 21) | (uint64_t)(z + kAxisHalf);
}

// common::VoxelCastingBresenham (math.cc:35-95): visits (x0, y0, z0) .. (x1, y1, z1), dm + 1 voxels, each once;
// the last one only if with_end
template <class F>
__host__ __device__ __forceinline__ void mrvm_walk(int x0, int y0, int z0, int x1, int y1, int z1, bool with_end,
                                                   F&& visit) {
  const int dx = abs(x1 - x0), sx = x0 < x1 ? 1 : -1;
  const int dy = abs(y1 - y0), sy = y0 < y1 ? 1 : -1;
  const int dz = abs(z1 - z0), sz = z0 < z1 ? 1 : -1;
  const int dm = max(dx, max(dy, dz));
  int ex = dm >> 1, ey = ex, ez = ex;
  for (int i = dm; i > 0; --i) {
    visit(x0, y0, z0);
    ex -= dx; if (ex < 0) { ex += dm; x0 += sx; }
    ey -= dy; if (ey < 0) { ey += dm; y0 += sy; }
    ez -= dz; if (ez < 0) { ez += dm; z0 += sz; }
  }
  if (with_end) visit(x0, y0, z0);
}

// p after m applications of a map whose 2^k-th powers are tab[k * 256 ..]
__host__ __device__ __forceinline__ uint8_t mrvm_lift(const uint8_t* tab, uint8_t p, uint32_t m) {
  for (int k = 0; m; ++k, m >>= 1)
    if (m & 1u) p = tab[k * 256 + p];
  return p;
}

// the reference's probability arithmetic, literally (.h:134-140, .cc:30-40, :63-69)
float prob_to_odd(float prob) { return std::log(prob / (1. - prob)); }
float odd_to_prob(float odd) { return 1. - 1. / (1. + std::exp(odd)); }
float clampf_ref(float v, float lo, float hi) { return v > hi ? hi : (v < lo ? lo : v); }

// tab[0 .. 32*256): miss^(2^k), tab[32*256 ..): hit^(2^k); one_step (optional): hit map, then miss map
void mrvm_tables(float hit_prob, float miss_prob, uint8_t* tab, uint8_t* one_step) {
  hit_prob = clampf_ref(hit_prob, 0.501f, 0.9f);
  miss_prob = clampf_ref(miss_prob, 0.1f, 0.499f);
  const float hit_log_odd = prob_to_odd(hit_prob), miss_log_odd = prob_to_odd(miss_prob);
  for (int w = 0; w < 2; ++w) {
    uint8_t* t = tab + w * kLift * 256;
    const float add = w ? hit_log_odd : miss_log_odd;
    for (int p = 0; p < 256; ++p) {
      float odd = prob_to_odd(static_cast<float>(p) / 256);
      odd += add;
      t[p] = (uint8_t)(clampf_ref(odd_to_prob(odd), 0.1f, 0.9f) * 256);
      if (one_step) one_step[(1 - w) * 256 + p] = t[p];
    }
    for (int k = 1; k < kLift; ++k)
      for (int p = 0; p < 256; ++p) t[k * 256 + p] = t[(k - 1) * 256 + t[(k - 1) * 256 + p]];
  }
}

__device__ __forceinline__ uint32_t slot_of(uint64_t k, uint32_t mask) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (uint32_t)k & mask;
}

__device__ __forceinline__ uint32_t table_find(const uint64_t* __restrict__ tkeys, const uint32_t* __restrict__ tids,
                                               uint32_t mask, uint64_t k) {
  for (uint32_t s = slot_of(k, mask);; s = (s + 1) & mask) {
    const uint64_t t = tkeys[s];
    if (t == k) return tids[s];
    if (t == kEmpty) return kNone;
  }
}

// keys inserted by one launch are distinct: a slot taken by another thread holds another key
__device__ __forceinline__ uint32_t table_insert(uint64_t* tkeys, uint32_t* tids, uint32_t mask, uint64_t k,
                                                 uint32_t* next_id, bool* created) {
  for (uint32_t s = slot_of(k, mask);; s = (s + 1) & mask) {
    uint64_t t = tkeys[s];
    if (t == k) { *created = false; return tids[s]; }
    if (t == kEmpty) {
      t = atomicCAS((unsigned long long*)&tkeys[s], (unsigned long long)kEmpty, (unsigned long long)k);
      if (t == kEmpty) {
        const uint32_t id = atomicAdd(next_id, 1u);
        tids[s] = id;
        *created = true;
        return id;
      }
    }
  }
}

struct Voxels {            // indexed by voxel id
  uint64_t* key;
  uint8_t* prob;
  int32_t* max_int;
  int32_t* npts;
  uint32_t* miss;          // misses of the current insert
  uint32_t* hits;          // hits of the current insert
  uint32_t* first;         // first_end of the current insert (kNone: no point ends here)
  uint32_t* seg;           // sorted position of the first point ending here
  float4* pts;             // max_point_num_in_cell records per voxel
};

// meta[3]: points with a non-finite coordinate, meta[4]: points outside the index range
__global__ void __launch_bounds__(256)
mrvm_key_kernel(const char* __restrict__ pts, int64_t stride, int n, float step, uint64_t* __restrict__ keys,
                uint32_t* __restrict__ vals, long long* __restrict__ meta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int v[3];
  const int rc = mrvm_voxel(reinterpret_cast<const float*>(pts + (int64_t)i * stride), step, v);
  keys[i] = rc ? kEmpty : mrvm_key(v[0], v[1], v[2]);
  vals[i] = (uint32_t)i;
  if (rc) atomicAdd((unsigned long long*)&meta[rc == 1 ? 3 : 4], 1ull);
}

// one thread per segment (= end voxel of this insert)
__global__ void __launch_bounds__(256)
mrvm_segment_kernel(const uint64_t* __restrict__ keys, const uint32_t* __restrict__ order,
                    const uint32_t* __restrict__ starts, const uint32_t* __restrict__ n_seg, uint64_t* tkeys,
                    uint32_t* tids, uint32_t mask, uint32_t* next_id, Voxels V) {
  const uint32_t s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= *n_seg) return;
  const uint32_t a = starts[s], b = starts[s + 1];
  const uint64_t k = keys[a];
  bool created = false;
  const uint32_t id = table_insert(tkeys, tids, mask, k, next_id, &created);
  if (created) { V.key[id] = k; V.prob[id] = kUnknown; V.max_int[id] = 0; V.npts[id] = 0; }
  V.first[id] = order[a];
  V.hits[id] = b - a;
  V.seg[id] = a;
}

__global__ void __launch_bounds__(256)
mrvm_rehash_kernel(const uint64_t* __restrict__ vkeys, uint32_t nvox, uint64_t* tkeys, uint32_t* tids, uint32_t mask) {
  const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= nvox) return;
  const uint64_t k = vkeys[id];
  for (uint32_t s = slot_of(k, mask);; s = (s + 1) & mask)
    if (atomicCAS((unsigned long long*)&tkeys[s], (unsigned long long)kEmpty, (unsigned long long)k) == kEmpty) {
      tids[s] = id;
      return;
    }
}

// one thread per ray: misses on the voxels before its end that were born before this insert, if no point before
// this one ended there
__global__ void __launch_bounds__(256)
mrvm_ray_kernel(const char* __restrict__ pts, int64_t stride, int n, float step, int ox, int oy, int oz,
                const uint64_t* __restrict__ tkeys, const uint32_t* __restrict__ tids, uint32_t mask,
                uint32_t nvox_before, const uint32_t* __restrict__ first, uint32_t* __restrict__ miss) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  int e[3];
  if (mrvm_voxel(reinterpret_cast<const float*>(pts + (int64_t)j * stride), step, e)) return;
  mrvm_walk(ox, oy, oz, e[0], e[1], e[2], false, [&](int x, int y, int z) {
    const uint32_t id = table_find(tkeys, tids, mask, mrvm_key(x, y, z));
    if (id < nvox_before && (uint32_t)j < first[id]) atomicAdd(&miss[id], 1u);
  });
}

// one thread per voxel: misses, then hits, max_intensity, appended points; counters reset for the next insert
__global__ void __launch_bounds__(256)
mrvm_update_kernel(const char* __restrict__ pts, int64_t stride, const uint32_t* __restrict__ order,
                   const uint32_t* __restrict__ nvox, const uint8_t* __restrict__ tab, int max_pts, Voxels V) {
  const uint32_t id = blockIdx.x * blockDim.x + threadIdx.x;
  if (id >= *nvox) return;
  const uint32_t m = V.miss[id], h = V.hits[id];
  if (!m && !h) return;
  V.prob[id] = mrvm_lift(tab + kLift * 256, mrvm_lift(tab, V.prob[id], m), h);
  if (h) {
    const uint32_t a = V.seg[id];
    int mi = V.max_int[id], c = V.npts[id];
    for (uint32_t k = 0; k < h; ++k) {
      const float* q = reinterpret_cast<const float*>(pts + (int64_t)order[a + k] * stride);
      mi = max(mi, (int)q[3]);
      if (c < max_pts) V.pts[(int64_t)id * max_pts + c++] = make_float4(q[0], q[1], q[2], q[3]);
    }
    V.max_int[id] = mi;
    V.npts[id] = c;
  }
  V.miss[id] = 0; V.hits[id] = 0; V.first[id] = kNone;
}

// ---- output ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
mrvm_out_keys_kernel(const uint64_t* __restrict__ vkeys, uint32_t nvox, uint64_t* __restrict__ keys,
                     uint32_t* __restrict__ vals) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nvox) return;
  keys[i] = vkeys[i];
  vals[i] = i;
}

__global__ void __launch_bounds__(256)
mrvm_out_count_kernel(const uint32_t* __restrict__ ids, uint32_t nvox, const uint8_t* __restrict__ prob,
                      const int32_t* __restrict__ npts, uint8_t thr, int average, uint32_t* __restrict__ cnt) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nvox) return;
  const uint32_t id = ids[i];
  cnt[i] = prob[id] >= thr ? (average ? 1u : (uint32_t)npts[id]) : 0u;
}

__global__ void __launch_bounds__(256)
mrvm_out_write_kernel(const uint32_t* __restrict__ ids, uint32_t nvox, const uint32_t* __restrict__ off,
                      const uint8_t* __restrict__ prob, const int32_t* __restrict__ npts,
                      const int32_t* __restrict__ max_int, const float4* __restrict__ vpts, int max_pts, uint8_t thr,
                      int average, int rgb, int use_max, float4* __restrict__ out) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= nvox) return;
  const uint32_t id = ids[i];
  if (prob[id] < thr) return;
  const int c = npts[id];
  const float4* p = vpts + (int64_t)id * max_pts;
  uint32_t grey = (uint32_t)max_int[id];                  // OutputToPointCloud(PointXYZRGB), :182-187
  grey = (uint32_t)(grey * 1.4);
  if (grey > 255) grey = 255;
  const float mi = (float)max_int[id];
  float4* o = out + off[i];
  if (average) {
    float x = 0.f, y = 0.f, z = 0.f;
    for (int k = 0; k < c; ++k) { x += p[k].x; y += p[k].y; z += p[k].z; }
    const float size = (float)c;
    *o = make_float4(x / size, y / size, z / size, rgb ? (float)(uint8_t)grey : (use_max ? mi : 0.f));
  } else {
    for (int k = 0; k < c; ++k)
      o[k] = make_float4(p[k].x, p[k].y, p[k].z, rgb ? (float)(uint8_t)grey : (use_max ? mi : p[k].w));
  }
}

}  // namespace
}  // namespace smb

using namespace smb;

struct sm_mrvm {
  int device = 0;
  sm_mrvm_settings st{};
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[6] = {};
  cudaEvent_t ev_caller = nullptr;
  float phase_ms[5] = {0, 0, 0, 0, 0};
  int64_t inserts = 0;
  uint8_t* tab = nullptr;            // 2 x 32 x 256 lifting tables
  // voxels
  Voxels V{};
  uint32_t nvox = 0, vcap = 0;
  uint32_t* d_next = nullptr;        // device voxel counter
  // table
  uint64_t* tkeys = nullptr;
  uint32_t* tids = nullptr;
  uint32_t tcap = 0;
  // per-insert workspace
  char* ws = nullptr;
  size_t ws_bytes = 0;
};

namespace {

template <class T>
int grow_array(T** p, uint32_t old_n, size_t new_n, size_t per, cudaStream_t s, int fill) {
  T* q = nullptr;
  if (cudaMalloc(&q, new_n * per * sizeof(T)) != cudaSuccess) return SM_ERR_CUDA;
  if (old_n && cudaMemcpyAsync(q, *p, (size_t)old_n * per * sizeof(T), cudaMemcpyDeviceToDevice, s) != cudaSuccess)
    return SM_ERR_CUDA;
  if (cudaMemsetAsync(q + (size_t)old_n * per, fill, (new_n - old_n) * per * sizeof(T), s) != cudaSuccess)
    return SM_ERR_CUDA;
  if (cudaStreamSynchronize(s) != cudaSuccess) return SM_ERR_CUDA;
  cudaFree(*p);
  *p = q;
  return SM_OK;
}

// room for `need` voxels in the arrays and at most half of the table's slots in use
int reserve_voxels(sm_mrvm* h, uint64_t need) {
  if (need >= (1ull << 31)) return SM_ERR_BAD_ARGUMENT;
  const cudaStream_t s = h->stream;
  if (need > h->vcap) {
    const size_t cap = std::max<uint64_t>(need, 2ull * h->vcap);
    const size_t mp = (size_t)h->st.max_point_num_in_cell;
    Voxels& V = h->V;
    int rc = SM_OK;
    if ((rc = grow_array(&V.key, h->nvox, cap, 1, s, 0)) || (rc = grow_array(&V.prob, h->nvox, cap, 1, s, 0)) ||
        (rc = grow_array(&V.max_int, h->nvox, cap, 1, s, 0)) || (rc = grow_array(&V.npts, h->nvox, cap, 1, s, 0)) ||
        (rc = grow_array(&V.miss, h->nvox, cap, 1, s, 0)) || (rc = grow_array(&V.hits, h->nvox, cap, 1, s, 0)) ||
        (rc = grow_array(&V.first, h->nvox, cap, 1, s, 0xff)) || (rc = grow_array(&V.seg, h->nvox, cap, 1, s, 0)) ||
        (rc = grow_array(&V.pts, h->nvox, cap, mp, s, 0)))
      return rc;
    h->vcap = (uint32_t)cap;
  }
  if (2 * need > h->tcap) {
    uint64_t cap = std::max<uint32_t>(h->tcap, 1024u);
    while (cap < 2 * need) cap *= 2;
    cudaFree(h->tkeys); cudaFree(h->tids);
    h->tkeys = nullptr; h->tids = nullptr; h->tcap = 0;
    if (cudaMalloc(&h->tkeys, cap * sizeof(uint64_t)) != cudaSuccess ||
        cudaMalloc(&h->tids, cap * sizeof(uint32_t)) != cudaSuccess ||
        cudaMemsetAsync(h->tkeys, 0xff, cap * sizeof(uint64_t), s) != cudaSuccess)
      return SM_ERR_CUDA;
    h->tcap = (uint32_t)cap;
    if (h->nvox)
      mrvm_rehash_kernel<<<ceil_div(h->nvox, 256), 256, 0, s>>>(h->V.key, h->nvox, h->tkeys, h->tids, h->tcap - 1);
    if (cudaGetLastError() != cudaSuccess) return SM_ERR_CUDA;
  }
  return SM_OK;
}

int insert(sm_mrvm* h, const float* points, int64_t n, int64_t stride, const float* origin, bool on_device,
           cudaStream_t caller) {
  if (!h || !origin || n < 0 || n > (1 << 30) || stride < 16 || stride % 4 || (n > 0 && !points))
    return SM_ERR_BAD_ARGUMENT;
  if (n == 0) return 0;                                   // "cloud is empty.": nothing changes (:56-59)
  float o[3] = {origin[0], origin[1], origin[2]};
  o[2] += h->st.z_offset;
  int ov[3];
  if (mrvm_voxel(o, h->st.high_resolution, ov)) return SM_ERR_BAD_ARGUMENT;
  if (cudaSetDevice(h->device) != cudaSuccess) return SM_ERR_CUDA;
  const cudaStream_t s = h->stream;
  const int ni = (int)n;
  const int nblk = ceil_div(n, 2048);
  const int64_t st = (n + 63) & ~(int64_t)63;
  const size_t in_bytes = on_device ? 0 : (size_t)n * (size_t)stride;
  const size_t need = in_bytes + 2 * st * (sizeof(uint64_t) + sizeof(uint32_t)) + radix_sort_scratch_bytes(ni, 1) +
                      ((size_t)nblk + 8 + (size_t)n + 8) * sizeof(uint32_t) + 16 * 256;
  if (need > h->ws_bytes) {
    cudaFree(h->ws);
    h->ws = nullptr; h->ws_bytes = 0;
    if (cudaMalloc(&h->ws, need) != cudaSuccess) return SM_ERR_CUDA;
    h->ws_bytes = need;
  }
  char* cur = h->ws;
  auto take = [&](size_t b) { char* p = cur; cur += (b + 255) & ~(size_t)255; return p; };
  char* d_in = on_device ? (char*)points : take(in_bytes);
  uint64_t* keys0 = (uint64_t*)take(st * sizeof(uint64_t));
  uint64_t* keys1 = (uint64_t*)take(st * sizeof(uint64_t));
  uint32_t* ord0 = (uint32_t*)take(st * sizeof(uint32_t));
  uint32_t* ord1 = (uint32_t*)take(st * sizeof(uint32_t));
  uint32_t* scratch = (uint32_t*)take(radix_sort_scratch_bytes(ni, 1));
  uint32_t* block_sum = (uint32_t*)take(((size_t)nblk + 8) * sizeof(uint32_t));
  uint32_t* starts = (uint32_t*)take(((size_t)n + 8) * sizeof(uint32_t));
  long long* meta = (long long*)take(256);

  cudaEventRecord(h->ev[0], s);
  if (on_device) {
    if (cudaEventRecord(h->ev_caller, caller) != cudaSuccess || cudaStreamWaitEvent(s, h->ev_caller, 0) != cudaSuccess)
      return SM_ERR_CUDA;
  } else if (cudaMemcpyAsync(d_in, points, in_bytes, cudaMemcpyHostToDevice, s) != cudaSuccess) {
    return SM_ERR_CUDA;
  }
  cudaEventRecord(h->ev[1], s);
  cudaMemsetAsync(meta, 0, 256, s);
  const float step = h->st.high_resolution;
  mrvm_key_kernel<<<ceil_div(n, 256), 256, 0, s>>>(d_in, stride, ni, step, keys0, ord0, meta);
  if (radix_sort_pairs_u64(keys0, ord0, keys1, ord1, ni, 1, st, scratch, s, 8)) return SM_ERR_CUDA;
  segment_heads_launch(keys0, ni, block_sum, starts, meta, s);
  cudaEventRecord(h->ev[2], s);
  long long hm[8] = {0};
  uint32_t nseg = 0;
  if (cudaMemcpyAsync(hm, meta, sizeof(hm), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaMemcpyAsync(&nseg, block_sum + nblk, sizeof(uint32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess)
    return SM_ERR_CUDA;
  if (hm[4]) return SM_ERR_BAD_ARGUMENT;                  // a voxel index outside [-2^20, 2^20): map unchanged
  const int dropped = (int)hm[3];
  if (nseg == 0) return dropped;
  int rc = reserve_voxels(h, (uint64_t)h->nvox + nseg);
  if (rc) return rc;
  const uint32_t nvox_before = h->nvox;
  mrvm_segment_kernel<<<ceil_div(nseg, 256), 256, 0, s>>>(keys0, ord0, starts, block_sum + nblk, h->tkeys, h->tids,
                                                          h->tcap - 1, h->d_next, h->V);
  cudaEventRecord(h->ev[3], s);
  if (nvox_before > 0)                                    // an empty map has nothing to miss
    mrvm_ray_kernel<<<ceil_div(n, 256), 256, 0, s>>>(d_in, stride, ni, step, ov[0], ov[1], ov[2], h->tkeys, h->tids,
                                                     h->tcap - 1, nvox_before, h->V.first, h->V.miss);
  cudaEventRecord(h->ev[4], s);
  mrvm_update_kernel<<<ceil_div((int64_t)nvox_before + nseg, 256), 256, 0, s>>>(
      d_in, stride, ord0, h->d_next, h->tab, h->st.max_point_num_in_cell, h->V);
  cudaEventRecord(h->ev[5], s);
  uint32_t nvox = 0;
  if (cudaMemcpyAsync(&nvox, h->d_next, sizeof(uint32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess)
    return SM_ERR_CUDA;
  h->nvox = nvox;
  for (int k = 0; k < 5; ++k) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->ev[k], h->ev[k + 1]);
    h->phase_ms[k] += ms;
  }
  ++h->inserts;
  return dropped;
}

void destroy(sm_mrvm* h) {
  Voxels& V = h->V;
  cudaFree(V.key); cudaFree(V.prob); cudaFree(V.max_int); cudaFree(V.npts); cudaFree(V.miss); cudaFree(V.hits);
  cudaFree(V.first); cudaFree(V.seg); cudaFree(V.pts);
  cudaFree(h->tkeys); cudaFree(h->tids); cudaFree(h->ws); cudaFree(h->tab); cudaFree(h->d_next);
  for (auto& e : h->ev) if (e) cudaEventDestroy(e);
  if (h->ev_caller) cudaEventDestroy(h->ev_caller);
  if (h->stream) cudaStreamDestroy(h->stream);
  delete h;
}

}  // namespace

extern "C" int sm_mrvm_create(int device, const sm_mrvm_settings* settings, int64_t expected_voxels, sm_mrvm** out) {
  if (!settings || !out || expected_voxels < 0) return SM_ERR_BAD_ARGUMENT;
  *out = nullptr;
  const sm_mrvm_settings& s = *settings;
  // map_builder_options.cc:66-68, and a voxel size the index arithmetic can use
  if (!(s.hit_prob > 0.5f) || !(s.miss_prob < 0.5f) || s.max_point_num_in_cell < 1 ||
      !(s.high_resolution > 0.f) || !isfinite(s.high_resolution) || !isfinite(s.z_offset))
    return SM_ERR_BAD_ARGUMENT;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return SM_ERR_NO_DEVICE;
  if (device < 0 || device >= ndev || cudaSetDevice(device) != cudaSuccess) return SM_ERR_BAD_ARGUMENT;
  sm_mrvm* h = new sm_mrvm;
  h->device = device;
  h->st = s;
  uint8_t tab[2 * kLift * 256];
  mrvm_tables(s.hit_prob, s.miss_prob, tab, nullptr);
  bool ok = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking) == cudaSuccess &&
            cudaEventCreateWithFlags(&h->ev_caller, cudaEventDisableTiming) == cudaSuccess;
  for (auto& e : h->ev) ok = ok && cudaEventCreate(&e) == cudaSuccess;
  ok = ok && cudaMalloc(&h->tab, sizeof(tab)) == cudaSuccess && cudaMalloc(&h->d_next, 256) == cudaSuccess &&
       cudaMemcpy(h->tab, tab, sizeof(tab), cudaMemcpyHostToDevice) == cudaSuccess &&
       cudaMemset(h->d_next, 0, 256) == cudaSuccess;
  const int rc = ok ? reserve_voxels(h, (uint64_t)std::max<int64_t>(expected_voxels, 1024)) : SM_ERR_CUDA;
  if (rc) { destroy(h); return rc; }
  *out = h;
  return SM_OK;
}

extern "C" int sm_mrvm_destroy(sm_mrvm* h) {
  if (!h) return SM_ERR_BAD_ARGUMENT;
  cudaSetDevice(h->device);
  destroy(h);
  return SM_OK;
}

extern "C" int sm_mrvm_set_offset_z(sm_mrvm* h, float offset) {
  if (!h || !isfinite(offset)) return SM_ERR_BAD_ARGUMENT;
  h->st.z_offset = offset;
  return SM_OK;
}

extern "C" int sm_mrvm_insert(sm_mrvm* h, const float* points, int64_t n, int64_t stride_bytes, const float* origin_3) {
  return insert(h, points, n, stride_bytes, origin_3, false, nullptr);
}

extern "C" int sm_mrvm_insert_device(sm_mrvm* h, const float* dev_points, int64_t n, int64_t stride_bytes,
                                     const float* origin_3, void* cuda_stream) {
  return insert(h, dev_points, n, stride_bytes, origin_3, true, (cudaStream_t)cuda_stream);
}

extern "C" int64_t sm_mrvm_size(const sm_mrvm* h) { return h ? (int64_t)h->nvox : SM_ERR_BAD_ARGUMENT; }

extern "C" int sm_mrvm_phase_ms(const sm_mrvm* h, float* ms_6) {
  if (!h || !ms_6) return SM_ERR_BAD_ARGUMENT;
  for (int k = 0; k < 5; ++k) ms_6[k] = h->phase_ms[k];
  ms_6[5] = (float)h->inserts;
  return SM_OK;
}

extern "C" int sm_mrvm_output(sm_mrvm* h, float threshold, int32_t rgb, float* out4, int64_t capacity,
                              int64_t* m_out) {
  if (!h || !m_out || capacity < 0 || (capacity > 0 && !out4)) return SM_ERR_BAD_ARGUMENT;
  const float t = threshold * 256;                        // `Probability prob_threshold = threshold * kTableSize`
  if (!(t > -1.f && t < 256.f)) return SM_ERR_BAD_ARGUMENT;
  const uint8_t thr = (uint8_t)t;
  *m_out = 0;
  const uint32_t nv = h->nvox;
  if (nv == 0) return SM_OK;
  if (cudaSetDevice(h->device) != cudaSuccess) return SM_ERR_CUDA;
  const cudaStream_t s = h->stream;
  const int64_t st = ((int64_t)nv + 63) & ~(int64_t)63;
  const size_t bytes = 2 * st * (sizeof(uint64_t) + sizeof(uint32_t)) + radix_sort_scratch_bytes((int)nv, 1) +
                       ((size_t)nv + 8) * sizeof(uint32_t) + 4096;
  char* base = nullptr;
  if (cudaMalloc(&base, bytes) != cudaSuccess) return SM_ERR_CUDA;
  char* cur = base;
  auto take = [&](size_t b) { char* p = cur; cur += (b + 255) & ~(size_t)255; return p; };
  uint64_t* k0 = (uint64_t*)take(st * sizeof(uint64_t));
  uint64_t* k1 = (uint64_t*)take(st * sizeof(uint64_t));
  uint32_t* v0 = (uint32_t*)take(st * sizeof(uint32_t));
  uint32_t* v1 = (uint32_t*)take(st * sizeof(uint32_t));
  uint32_t* scratch = (uint32_t*)take(radix_sort_scratch_bytes((int)nv, 1));
  uint32_t* cnt = (uint32_t*)take(((size_t)nv + 8) * sizeof(uint32_t));
  float4* d_out = nullptr;
  auto fail = [&](int code) { cudaFree(base); cudaFree(d_out); return code; };
  const Voxels& V = h->V;
  mrvm_out_keys_kernel<<<ceil_div(nv, 256), 256, 0, s>>>(V.key, nv, k0, v0);
  if (radix_sort_pairs_u64(k0, v0, k1, v1, (int)nv, 1, st, scratch, s, 8)) return fail(SM_ERR_CUDA);
  mrvm_out_count_kernel<<<ceil_div(nv, 256), 256, 0, s>>>(v0, nv, V.prob, V.npts, thr, h->st.output_average, cnt);
  cudaMemsetAsync(cnt + nv, 0, sizeof(uint32_t), s);
  radix_scan_kernel_launch(cnt, (int)nv + 1, 1, s);
  uint32_t m = 0;
  if (cudaMemcpyAsync(&m, cnt + nv, sizeof(uint32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess)
    return fail(SM_ERR_CUDA);
  *m_out = (int64_t)m;
  if ((int64_t)m > capacity) return fail(SM_ERR_BAD_ARGUMENT);
  if (m == 0) return fail(SM_OK);
  if (cudaMalloc(&d_out, (size_t)m * sizeof(float4)) != cudaSuccess) return fail(SM_ERR_CUDA);
  mrvm_out_write_kernel<<<ceil_div(nv, 256), 256, 0, s>>>(v0, nv, cnt, V.prob, V.npts, V.max_int, V.pts,
                                                          h->st.max_point_num_in_cell, thr, h->st.output_average,
                                                          rgb ? 1 : 0, h->st.use_max_intensity, d_out);
  if (cudaMemcpyAsync(out4, d_out, (size_t)m * sizeof(float4), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess || cudaGetLastError() != cudaSuccess)
    return fail(SM_ERR_CUDA);
  return fail(SM_OK);
}

// ---- test hooks (include/sm_b200_debug.h) ---------------------------------------------------------------------
extern "C" int sm_debug_mrvm_ray(const float* origin_3, const float* point_3, float step, int32_t* voxels_3n,
                                 int64_t capacity, int64_t* n_out) {
  if (!origin_3 || !point_3 || !n_out || !(step > 0.f) || capacity < 0 || (capacity > 0 && !voxels_3n))
    return SM_ERR_BAD_ARGUMENT;
  int a[3], b[3];
  if (mrvm_voxel(origin_3, step, a) || mrvm_voxel(point_3, step, b)) return SM_ERR_BAD_ARGUMENT;
  int64_t k = 0;
  mrvm_walk(a[0], a[1], a[2], b[0], b[1], b[2], true, [&](int x, int y, int z) {
    if (k < capacity) { voxels_3n[3 * k] = x; voxels_3n[3 * k + 1] = y; voxels_3n[3 * k + 2] = z; }
    ++k;
  });
  *n_out = k;
  return k > capacity ? SM_ERR_BAD_ARGUMENT : SM_OK;
}

extern "C" int sm_debug_mrvm_update(float hit_prob, float miss_prob, const uint8_t* probs, const int64_t* misses,
                                    const int64_t* hits, int64_t n, uint8_t* out, uint8_t* tables_out) {
  if (n < 0 || (n > 0 && (!probs || !misses || !hits || !out))) return SM_ERR_BAD_ARGUMENT;
  std::vector<uint8_t> tab(2 * kLift * 256);
  mrvm_tables(hit_prob, miss_prob, tab.data(), tables_out);
  for (int64_t i = 0; i < n; ++i) {
    if (misses[i] < 0 || hits[i] < 0 || misses[i] >= (1ll << 32) || hits[i] >= (1ll << 32)) return SM_ERR_BAD_ARGUMENT;
    out[i] = mrvm_lift(tab.data() + kLift * 256, mrvm_lift(tab.data(), probs[i], (uint32_t)misses[i]),
                       (uint32_t)hits[i]);
  }
  return SM_OK;
}

extern "C" int sm_debug_mrvm_state(sm_mrvm* h, int64_t* keys, uint8_t* prob, int32_t* max_intensity, int32_t* npts,
                                   float* points4, int64_t capacity, int64_t* n_out) {
  if (!h || !n_out) return SM_ERR_BAD_ARGUMENT;
  const uint32_t nv = h->nvox;
  *n_out = nv;
  if ((int64_t)nv > capacity) return SM_ERR_BAD_ARGUMENT;
  if (nv == 0) return SM_OK;
  if (!keys || !prob || !max_intensity || !npts || !points4) return SM_ERR_BAD_ARGUMENT;
  const size_t mp = (size_t)h->st.max_point_num_in_cell;
  std::vector<uint64_t> k(nv);
  std::vector<uint8_t> p(nv);
  std::vector<int32_t> mi(nv), c(nv);
  std::vector<float4> pts((size_t)nv * mp);
  if (cudaSetDevice(h->device) != cudaSuccess ||
      cudaMemcpy(k.data(), h->V.key, nv * sizeof(uint64_t), cudaMemcpyDeviceToHost) != cudaSuccess ||
      cudaMemcpy(p.data(), h->V.prob, nv, cudaMemcpyDeviceToHost) != cudaSuccess ||
      cudaMemcpy(mi.data(), h->V.max_int, nv * sizeof(int32_t), cudaMemcpyDeviceToHost) != cudaSuccess ||
      cudaMemcpy(c.data(), h->V.npts, nv * sizeof(int32_t), cudaMemcpyDeviceToHost) != cudaSuccess ||
      cudaMemcpy(pts.data(), h->V.pts, pts.size() * sizeof(float4), cudaMemcpyDeviceToHost) != cudaSuccess)
    return SM_ERR_CUDA;
  std::vector<uint32_t> ord(nv);
  for (uint32_t i = 0; i < nv; ++i) ord[i] = i;
  std::sort(ord.begin(), ord.end(), [&](uint32_t a, uint32_t b) { return k[a] < k[b]; });
  for (uint32_t i = 0; i < nv; ++i) {
    const uint32_t id = ord[i];
    keys[i] = (int64_t)k[id]; prob[i] = p[id]; max_intensity[i] = mi[id]; npts[i] = c[id];
    for (size_t q = 0; q < mp; ++q) {
      const float4 v = pts[id * mp + q];
      float* o = points4 + 4 * (i * mp + q);
      o[0] = v.x; o[1] = v.y; o[2] = v.z; o[3] = v.w;
    }
  }
  return SM_OK;
}
