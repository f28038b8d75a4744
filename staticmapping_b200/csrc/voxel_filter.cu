// pre_processers::filter::VoxelGrid::Filter on the device
// (pre_processors/filter_voxel_grid.cc:37-78; used by Submap::InsertFrame's down-sampling,
// builder/submap.cc:144-158, the step that produces the ICP / NDT targets).
//
// Reference: every point goes into std::unordered_map<Vector3i, vector<point>> under the key
// (lround(x / s), lround(y / s), lround(z / s)); each voxel emits the mean of x, y, z, intensity,
// accumulated in double in insertion order (== input order), cast to float; factor = 0.
// Here: 63-bit voxel key per point -> stable radix sort (points of a voxel stay in input order)
// -> segment heads -> points gathered into voxel order -> one warp per voxel adds the four double
// chains in order (addends staged through shared memory, like ndt_leaf_kernel) -> one output
// point per voxel.  Every output value is bit-identical to the reference's; the ORDER of the
// output points is ascending (ix, iy, iz), whereas the reference's is the iteration order of a
// libstdc++ unordered_map (an accident of its rehash history; nothing downstream depends on it
// beyond summation order).  Compiled with -fmad=false.
#include <limits.h>
#include <math.h>

#include "../../include/sm_b200.h"
#include "common.cuh"
#include "kernels.h"

namespace smb {
namespace {

constexpr long long kSpan = 1ll << 21;   // voxel indices of one axis must span < 2^21 (3 x 21-bit key)
constexpr int kT = 256, kItems = 8, kTile = kT * kItems;

// meta[0..2]: per-axis minimum voxel index over the finite points; meta[3]: dropped (non-finite) points;
// meta[4]: 1 if an axis spans 2^21 voxels or more
__host__ __device__ __forceinline__ bool vf_index(const float* p, float voxel, long long* ix, long long* iy, long long* iz) {
  const float qx = p[0] / voxel, qy = p[1] / voxel, qz = p[2] / voxel;
  // std::lround of a NaN / inf quotient is unspecified in the reference: such points are dropped here
  if (!(fabsf(qx) < 9.0e18f && fabsf(qy) < 9.0e18f && fabsf(qz) < 9.0e18f)) return false;
  *ix = llroundf(qx); *iy = llroundf(qy); *iz = llroundf(qz);
  return true;
}

__global__ void __launch_bounds__(256)
vf_min_kernel(const char* __restrict__ pts, int64_t stride, int n, float voxel, long long* __restrict__ meta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  long long ix = LLONG_MAX, iy = LLONG_MAX, iz = LLONG_MAX;
  if (i < n) {
    long long a, b, c;
    if (vf_index(reinterpret_cast<const float*>(pts + (int64_t)i * stride), voxel, &a, &b, &c)) { ix = a; iy = b; iz = c; }
  }
  for (int o = 16; o > 0; o >>= 1) {
    ix = min(ix, __shfl_xor_sync(0xffffffffu, ix, o));
    iy = min(iy, __shfl_xor_sync(0xffffffffu, iy, o));
    iz = min(iz, __shfl_xor_sync(0xffffffffu, iz, o));
  }
  if ((threadIdx.x & 31) == 0) { atomicMin(&meta[0], ix); atomicMin(&meta[1], iy); atomicMin(&meta[2], iz); }
}

__global__ void __launch_bounds__(256)
vf_key_kernel(const char* __restrict__ pts, int64_t stride, int n, float voxel, uint64_t* __restrict__ keys,
              uint32_t* __restrict__ vals, long long* __restrict__ meta) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  long long ix, iy, iz;
  uint64_t key = ~0ull;                      // dropped points sort behind every voxel
  if (vf_index(reinterpret_cast<const float*>(pts + (int64_t)i * stride), voxel, &ix, &iy, &iz)) {
    // offsets from the cloud's own minimum: the key order stays ascending (ix, iy, iz)
    const unsigned long long ox = (unsigned long long)(ix - meta[0]), oy = (unsigned long long)(iy - meta[1]),
                             oz = (unsigned long long)(iz - meta[2]);
    if (ox < (unsigned long long)kSpan && oy < (unsigned long long)kSpan && oz < (unsigned long long)kSpan)
      key = (ox << 42) | (oy << 21) | oz;
    else
      atomicExch((unsigned long long*)&meta[4], 1ull);
  } else {
    atomicAdd((unsigned long long*)&meta[3], 1ull);
  }
  keys[i] = key;
  vals[i] = (uint32_t)i;
}

__device__ __forceinline__ uint32_t vf_is_head(const uint64_t* keys, int i) {
  return (keys[i] != ~0ull && (i == 0 || keys[i] != keys[i - 1])) ? 1u : 0u;
}

__global__ void __launch_bounds__(kT)
vf_heads_count_kernel(const uint64_t* __restrict__ keys, int n, uint32_t* __restrict__ block_sum) {
  __shared__ uint32_t ws[kT / 32];
  uint32_t c = 0;
  const int base = blockIdx.x * kTile + threadIdx.x * kItems;
  for (int r = 0; r < kItems; ++r) if (base + r < n) c += vf_is_head(keys, base + r);
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = c;
  __syncthreads();
  if (threadIdx.x == 0) { uint32_t t = 0; for (int w = 0; w < kT / 32; ++w) t += ws[w]; block_sum[blockIdx.x] = t; }
}

// voxel_start[v] = first sorted position of voxel v; voxel_start[n_voxels] = n
__global__ void __launch_bounds__(kT)
vf_heads_scatter_kernel(const uint64_t* __restrict__ keys, int n, const uint32_t* __restrict__ block_off,
                        uint32_t* __restrict__ voxel_start, const long long* __restrict__ meta) {
  __shared__ uint32_t ws[kT / 32];
  const int base = blockIdx.x * kTile + threadIdx.x * kItems;
  uint32_t f[kItems], c = 0;
  for (int r = 0; r < kItems; ++r) { f[r] = (base + r < n) ? vf_is_head(keys, base + r) : 0u; c += f[r]; }
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  uint32_t incl = c;
  for (int o = 1; o < 32; o <<= 1) { const uint32_t t = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += t; }
  if (lane == 31) ws[w] = incl;
  __syncthreads();
  uint32_t wb = 0;
  for (int ww = 0; ww < w; ++ww) wb += ws[ww];
  uint32_t pos = block_off[blockIdx.x] + wb + incl - c;
  for (int r = 0; r < kItems; ++r) if (f[r]) voxel_start[pos++] = (uint32_t)(base + r);
  if (blockIdx.x == 0 && threadIdx.x == 0) voxel_start[block_off[gridDim.x]] = (uint32_t)(n - (int)meta[3]);   // sentinel: first dropped point
}

__global__ void __launch_bounds__(256)
vf_gather_kernel(const char* __restrict__ pts, int64_t stride, const uint32_t* __restrict__ order, int n,
                 float4* __restrict__ sorted) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const float* p = reinterpret_cast<const float*>(pts + (int64_t)order[k] * stride);
  sorted[k] = make_float4(p[0], p[1], p[2], p[3]);
}

// one warp per voxel; lanes 0..3 own the running sums of x, y, z, intensity
__global__ void __launch_bounds__(256)
vf_mean_kernel(const float4* __restrict__ sorted, const uint32_t* __restrict__ voxel_start,
               const uint32_t* __restrict__ n_voxels_dev, float* __restrict__ out) {
  constexpr int kPad = 33;
  __shared__ double s_d[8][4 * kPad];
  const int64_t v = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;    // n may exceed 2^27: 64-bit
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  if (v >= (int64_t)*n_voxels_dev) return;
  const uint32_t s0 = voxel_start[v], s1 = voxel_start[v + 1];
  double* sd = s_d[wib];
  const double* mine = sd + min(lane, 3) * kPad;
  double acc = 0.0;
  for (uint32_t base = s0; base < s1; base += 32) {
    const uint32_t i = min(base + (uint32_t)lane, s1 - 1);
    const float4 p = sorted[i];
    sd[0 * kPad + lane] = (double)p.x; sd[1 * kPad + lane] = (double)p.y;
    sd[2 * kPad + lane] = (double)p.z; sd[3 * kPad + lane] = (double)p.w;
    __syncwarp();
    const int cnt = (int)min(32u, s1 - base);
    if (cnt == 32) {
      double t[32];
#pragma unroll
      for (int u = 0; u < 32; ++u) t[u] = mine[u];
#pragma unroll
      for (int u = 0; u < 32; ++u) acc += t[u];
    } else {
      for (int u = 0; u < cnt; ++u) acc += mine[u];
    }
    __syncwarp();
  }
  if (lane < 4) out[5 * v + lane] = (float)(acc / (double)(int)(s1 - s0));   // sum / size, size is an int
  if (lane == 4) out[5 * v + 4] = 0.0f;                                      // factor keeps its default
}

}  // namespace

// segment heads of sorted keys (~0 = dropped point, sorted behind every voxel): starts[v] = first sorted position of
// segment v, starts[count] = n - meta[3]; block_sum[ceil(n / 2048)] = count.  Also used by mrvm.cu.
void segment_heads_launch(const uint64_t* keys, int n, uint32_t* block_sum, uint32_t* starts, const long long* meta,
                          cudaStream_t s) {
  const int nblk = ceil_div(n, kTile);
  vf_heads_count_kernel<<<nblk, kT, 0, s>>>(keys, n, block_sum);
  cudaMemsetAsync(block_sum + nblk, 0, sizeof(uint32_t), s);
  radix_scan_kernel_launch(block_sum, nblk + 1, 1, s);                                // block_sum[nblk] = number of voxels
  vf_heads_scatter_kernel<<<nblk, kT, 0, s>>>(keys, n, block_sum, starts, meta);
}

// host build of the voxel index of one point (test hook sm_debug_voxel_index op 0)
bool vf_debug_index_host(const float* p, float voxel, long long* ixyz) { return vf_index(p, voxel, &ixyz[0], &ixyz[1], &ixyz[2]); }
// VoxelGrid::Filter over a device cloud (records `stride` >= 16 bytes apart): d_out receives *m_out records of 5 floats
// (capacity n), in ascending voxel order.  Returns after the stream has finished.  Also used by filters.cu.
int voxel_grid_device(const char* d_in, int64_t stride, int n, float voxel_size, float* d_out, uint32_t* m_out,
                      cudaStream_t s) {
  *m_out = 0;
  if (n == 0) return SM_OK;
  const int ni = n;
  const int nblk = ceil_div(n, kTile);
  const int64_t st = ((int64_t)n + 63) & ~(int64_t)63;
  size_t bytes = 256;
  bytes += 2 * st * sizeof(uint64_t) + 2 * st * sizeof(uint32_t);            // keys, order (ping-pong)
  bytes += radix_sort_scratch_bytes(ni, 1) + 256;
  bytes += ((size_t)nblk + 8) * sizeof(uint32_t) + ((size_t)n + 8) * sizeof(uint32_t);   // block sums, voxel_start
  bytes += (size_t)n * sizeof(float4) + 1024;
  char* base = nullptr;
  if (cudaMalloc(&base, bytes) != cudaSuccess) return SM_ERR_CUDA;
  char* cur = base;
  auto take = [&](size_t b) { char* p = cur; cur += (b + 255) & ~(size_t)255; return p; };
  uint64_t* keys0 = (uint64_t*)take(st * sizeof(uint64_t));
  uint64_t* keys1 = (uint64_t*)take(st * sizeof(uint64_t));
  uint32_t* ord0 = (uint32_t*)take(st * sizeof(uint32_t));
  uint32_t* ord1 = (uint32_t*)take(st * sizeof(uint32_t));
  uint32_t* scratch = (uint32_t*)take(radix_sort_scratch_bytes(ni, 1));
  uint32_t* block_sum = (uint32_t*)take(((size_t)nblk + 8) * sizeof(uint32_t));
  uint32_t* voxel_start = (uint32_t*)take(((size_t)n + 8) * sizeof(uint32_t));
  float4* sorted = (float4*)take((size_t)n * sizeof(float4));
  long long* meta = (long long*)take(256);
  int rc = SM_OK;
  auto fail = [&](int code) { cudaFree(base); return code; };
  const long long meta_init[8] = {LLONG_MAX, LLONG_MAX, LLONG_MAX, 0, 0, 0, 0, 0};
  if (cudaMemcpyAsync(meta, meta_init, sizeof(meta_init), cudaMemcpyHostToDevice, s) != cudaSuccess)
    return fail(SM_ERR_CUDA);
  vf_min_kernel<<<ceil_div(n, 256), 256, 0, s>>>(d_in, stride, ni, voxel_size, meta);
  vf_key_kernel<<<ceil_div(n, 256), 256, 0, s>>>(d_in, stride, ni, voxel_size, keys0, ord0, meta);
  rc = radix_sort_pairs_u64(keys0, ord0, keys1, ord1, ni, 1, st, scratch, s, 8);   // 8 passes: result back in [0]
  if (rc) return fail(rc == -100 ? SM_ERR_CUDA : rc);
  segment_heads_launch(keys0, ni, block_sum, voxel_start, meta, s);                   // block_sum[nblk] = number of voxels
  vf_gather_kernel<<<ceil_div(n, 256), 256, 0, s>>>(d_in, stride, ord0, ni, sorted);
  vf_mean_kernel<<<ceil_div((int64_t)n * 32, 256), 256, 0, s>>>(sorted, voxel_start, block_sum + nblk, d_out);
  uint32_t m = 0;
  long long host_meta[8] = {0};
  if (cudaGetLastError() != cudaSuccess ||
      cudaMemcpyAsync(&m, block_sum + nblk, sizeof(uint32_t), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaMemcpyAsync(host_meta, meta, sizeof(host_meta), cudaMemcpyDeviceToHost, s) != cudaSuccess ||
      cudaStreamSynchronize(s) != cudaSuccess)
    return fail(SM_ERR_CUDA);
  if (host_meta[4]) return fail(SM_ERR_BAD_ARGUMENT);   // the finite points span 2^21 voxels or more along an axis
  *m_out = m;
  return fail(SM_OK);
}
}  // namespace smb

using namespace smb;

extern "C" int sm_voxel_grid_filter(int device, const float* points, int64_t n, int64_t stride_bytes,
                                    float voxel_size, float* out, int64_t* m_out) {
  if (!points || !out || !m_out || n < 0 || n > (1 << 30) || stride_bytes < 16 || stride_bytes % 4 ||
      !(voxel_size > 1.e-6f))       // ConfigsValid(), filter_voxel_grid.cc:35
    return SM_ERR_BAD_ARGUMENT;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0) return SM_ERR_NO_DEVICE;
  SMB_CUDA_OK(cudaSetDevice(device));
  *m_out = 0;
  if (n == 0) return SM_OK;
  const size_t in_bytes = (size_t)n * (size_t)stride_bytes;
  char* d_in = nullptr;
  float* d_out = nullptr;
  auto fail = [&](int code) { cudaFree(d_in); cudaFree(d_out); return code; };
  cudaStream_t s = nullptr;
  if (cudaMalloc(&d_in, in_bytes) != cudaSuccess || cudaMalloc(&d_out, (size_t)n * 5 * sizeof(float)) != cudaSuccess ||
      cudaMemcpyAsync(d_in, points, in_bytes, cudaMemcpyHostToDevice, s) != cudaSuccess)
    return fail(SM_ERR_CUDA);
  uint32_t m = 0;
  const int rc = voxel_grid_device(d_in, stride_bytes, (int)n, voxel_size, d_out, &m, s);
  if (rc) return fail(rc);
  if (m > 0 && cudaMemcpy(out, d_out, (size_t)m * 5 * sizeof(float), cudaMemcpyDeviceToHost) != cudaSuccess)
    return fail(SM_ERR_CUDA);
  *m_out = (int64_t)m;
  return fail(SM_OK);
}
