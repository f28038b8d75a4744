// Internal host-side launch API shared by the .cu translation units of libsm_b200.
#ifndef SM_B200_KERNELS_H_
#define SM_B200_KERNELS_H_

#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace smb {

// ---- radix_sort.cu ---------------------------------------------------------------------
size_t radix_sort_scratch_bytes(int n, int batch);
int radix_sort_pairs_u64(uint64_t* keys_a, uint32_t* vals_a, uint64_t* keys_b, uint32_t* vals_b,
                         int n, int batch, int64_t stride, uint32_t* scratch,
                         cudaStream_t stream, int passes = 8);
// exclusive scan of `count` u32 per batch (in place), one block per batch
void radix_scan_kernel_launch(uint32_t* data, int count, int batch, cudaStream_t stream);

// ---- kdtree.cu -------------------------------------------------------------------------
int kd_num_levels(int n, int bucket);
struct KdWorkspace {
  uint64_t* keys[2];
  uint32_t* lists[2];
  uint32_t* gloc;
  uint8_t* flag;
  uint32_t* scratch;
  double* bounds[2];
  int* level_dim;
  int64_t lstride;
  static size_t bytes_needed(int n, int bucket);
  void carve(void* base, int n, int bucket);
};
// ccut / cdim (optional): the compact search layout's node arrays, see KdCompact
// coords_are_float: every coordinate is exactly a float (clouds uploaded as float): 32-bit sort keys
int kd_build(const double* coord, int64_t cstride, int n, int bucket, KdWorkspace& ws,
             KdNode* nodes, uint32_t* leaf_order, cudaStream_t stream, double* ccut = nullptr,
             uint8_t* cdim = nullptr, bool coords_are_float = false, double2* cnode = nullptr);

// Compact search layout of the same tree, shaped for a shared-memory resident traversal:
//   cut[h], dim[h]  heap order (children of h: 2h+1, 2h+2) for the levels above the deepest
//                   leaf level; dim 3 = leaf.  8 + 1 bytes per node: the 14 inner levels of a
//                   ~107 k-point target are 144 KB and are staged into shared memory with bulk
//                   async copies (cp.async.bulk + mbarrier) once per CTA;
//   pb              padded buckets, x[8] y[8] z[8] doubles per leaf slot of the deepest level
//                   (+inf padding), so a leaf's bucket address is pure index arithmetic and a
//                   bucket scan is 12 aligned 16-byte loads;
//   pn, pid         normals / original ids per padded entry (entry = bucket * 8 + k).
struct KdCompact {
  const double* cut;
  const uint8_t* dim;
  const double2* node;    // {cut, dim as a 64-bit integer} of heap node h at slot h + 1, 2^levels slots: the
                          // search reads the levels below the shared-memory ones with one 16-byte load per node
  const double* pb;
  const BucketNormal* pn;
  const int32_t* pid;
  int levels;
};
size_t kd_compact_node_slots(int levels);     // entries of cut[] / dim[] (multiple of 16)
inline size_t kd_compact_bucket_entries(int levels) { return (size_t)8 << levels; }
int kd_compact_buckets(const double* coord, int64_t cstride, const double* nrm, int64_t nstride,
                       const uint32_t* leaf_order, int n, int bucket, int levels, double* pb,
                       BucketNormal* pn, int32_t* pid, cudaStream_t stream);

// ---- icp.cu ----------------------------------------------------------------------------
constexpr int kKnnItemSlack = 4096;   // a warp's item list may extend past the last query of the last batch
constexpr int kHistBins = 2048;

// Device-resident state of one IcpFast::Align call (one per handle).
struct IcpState {
  double T_iter[16];      // column-major, accumulated iteration transform
  double G0[16];          // T_mean^-1 * guess
  double T_mean[16];
  double result[16];
  double mean[3];
  double final_score;
  double quat_hist[5][4]; // ring of the last 5 rotations (w,x,y,z)
  double trans_hist[5][3];
  double limit;           // last quantile limit (debug / parity)
  long long kept;         // last K
  int hist_len;           // number of entries pushed (incl. the initial identity)
  int iteration;
  int done;               // 1 once converged or max_iteration reached
  int status;             // 0 ok, <0 error (-2 no finite distance, -3 nothing kept)
  int solve_path;         // 0 LLT, 1 min-norm, 2 SVD (last iteration)
  int pad;
  long long stamps[12];   // clock64 at the section boundaries of the last finish kernel (diagnostics)
};
static_assert(sizeof(IcpState) % 8 == 0, "IcpState is copied as 8-byte words");

struct IcpParams {
  int n_source, n_target;
  int max_iteration;
  float dist_outlier_ratio;
  double max_error2;       // (1+eps)^2
  int disable_convergence;
  int tree_levels;         // kd_num_levels(n_target, 8): depth of the root-to-leaf path
  int knn_queries_per_cta; // phase A: 0 = one query per thread, else queries per 256-thread CTA
};

struct IcpBuffers {
  // target (caller order, SoA, centred in place by the prologue)
  double* tgt;            // [3][tstride]
  double* tgt_raw;        // [3][tstride] as uploaded (un-centred)
  double* nrm;            // [3][tstride]
  int64_t tstride;
  // tree: build-time node array (blocked layout), leaf order, and the compact search layout
  KdNode* nodes;
  uint32_t* leaf_order;
  double* ccut;           // writable views of kc.cut / kc.dim / kc.pb / kc.pn (filled by the prologue)
  uint8_t* cdim;
  double2* cnode;
  double* cpb;
  BucketNormal* cpn;
  KdCompact kc;
  // source
  double* src_raw;        // [3][sstride] as uploaded
  double* src_g0;         // [3][sstride] after G0, caller order
  double* src0;           // [3][sstride] after G0, Morton order (what the iterations read)
  uint64_t* src_keys[2];  // Morton keys (ping-pong)
  uint32_t* src_vals[2];  // permutation (ping-pong)
  uint32_t* src_scratch;  // radix scratch
  int64_t sstride;
  // per-iteration
  int32_t* slot;          // [n_source] padded bucket entry of the match (kc.pb / kc.pn index)
  int4* knn_items;        // [n_source + kKnnItemSlack] parked searches of the k-NN kernel's second phase (16 B each)
  double* d2;             // [n_source]
  uint32_t* hist;         // [kHistBins] first-level histogram of dist^2 (phase A)
  uint32_t* hist2;        // [kHistBins] second-level histogram inside the quantile bin (phase B)
  double* sums;           // [32] reduced normal-equation sums of the iteration (phase C1 -> C2)
  double* cand_terms;     // [blocks*tile][8] per-block compacted candidates (members of the quantile bin):
                          // the 6 Jacobian terms, the residual and sqrt(d2) of the match (phase B -> C)
  unsigned long long* cand_key;  // [blocks*tile] bit pattern of the candidate's dist^2
  uint32_t* cand_cnt;     // [accum blocks]
  double* partials;       // [accum blocks][32]
  double* mean_partials;  // [blocks][4]
  IcpState* state;
};

int icp_accum_blocks(int n_source);
int icp_prologue(const IcpBuffers& b, const IcpParams& p, const double* guess_dev,
                 KdWorkspace& ws, cudaStream_t stream);
// events (optional): 4 per iteration — before A, after A, after B, after C
int icp_enqueue_iterations(const IcpBuffers& b, const IcpParams& p, int start_iteration, int count,
                           cudaStream_t stream, cudaEvent_t* events);
void icp_finish_launch(const IcpBuffers& b, const IcpParams& p, int nblocks_b, cudaStream_t stream);
// stand-alone k-NN over an already built tree (compact layout incl. pid): ids = original indices
int knn_query(const KdCompact& kc, const double* query, int64_t qstride, int nq, double max_error2,
              int32_t* ids, double* d2, cudaStream_t stream, int queries_per_cta = 0, int4* items = nullptr);
int kd_fill_buckets(const double* coord, int64_t cstride, const double* nrm, int64_t nstride,
                    const uint32_t* leaf_order, int n, BucketPoint* bpts, BucketNormal* bnrm,
                    cudaStream_t stream);

// ---- ndt.cu ------------------------------------------------------------------------------
struct NdtGrid {            // VoxelGridCovariance bookkeeping (_impl.hpp:88-103)
  float inv_leaf;
  int min_b[3], div_b[3], mul[3];
  int n_voxels;
};
struct NdtLeaf {            // VoxelGridCovariance::Leaf (voxel_grid_covariance_omp.h:92-186)
  double mean[3];
  double icov[9];           // zero for leaves that failed the eigenvalue test
  float centroid[3];
  int nr_points;            // -1: invalid covariance (still searchable, like the reference)
  int searchable;           // >= min_points_per_voxel: centroid is in the search cloud
  int pad;
};
struct NdtEvalParams {      // everything one computeDerivatives call needs, by value
  float T[16];              // final_transformation_, column-major
  float j_ang[8][3];        // computeAngleDerivatives (ndt_omp_impl.hpp:288-393)
  float h_ang[15][3];
  double gauss_d1, gauss_d2;
  float radius;             // resolution_
  int f64_math;             // 1: stock pcl::NormalDistributionsTransform term math (double), the
                            //    class NdtWithGicp uses; 0: pclomp's single-precision math
  double j_ang_d[8][3];     // the same tables in double (stock PCL keeps them as Vector3d)
  double h_ang_d[15][3];
};
uint32_t ndt_table_size(int nt);
// host build of the leaf plane fit of normals.cu (test hook sm_debug_normals_leaf): 1 kept, 0 dropped, < 0 bad count
int normals_debug_leaf_host(const double* members, int count, double* mean, double* unit);
// host build of one target-grid leaf of ndt.cu (test hook sm_debug_ndt_leaf)
void ndt_debug_leaf_host(const float* pts, int n, int min_points, double eig_mult, double* mean3, double* icov9,
                         float* centroid3, int* nr_points, int* searchable);
// host build of the per-(point, voxel) derivative term of ndt.cu (test hook sm_debug_ndt_term)
void ndt_debug_term_host(const NdtEvalParams& P, const float* x_orig, const float* x_trans, const double* mean,
                         const double* icov, double* out43);
int ndt_blocks(int n);
struct NdtWorkspace {
  uint64_t* keys[2];
  uint32_t* order[2];
  uint32_t* scratch;
  uint32_t* voxel_start;
  int* voxel_key;
  NdtLeaf* leaves;
  int* table_key;
  int* table_val;
  uint32_t table_size;
  double* partials;
  double* sums;             // [64] reduced outputs
  float* minmax;
  float* sorted_pts;        // target points gathered into voxel order (packed xyz)
  NdtGrid* grid;
  int64_t stride;
  static size_t bytes_needed(int nt, int ns);
  void carve(void* base, int nt, int ns);
};
int ndt_build_grid(const float* tgt, int nt, float resolution, NdtWorkspace& ws, cudaStream_t stream);
int ndt_eval(const float* src, int ns, const NdtEvalParams& P, NdtWorkspace& ws, cudaStream_t stream);
int ndt_float_to_soa(const float* pts, int n, double* soa, int64_t stride, cudaStream_t stream);
int ndt_fitness(const float* src, int ns, const NdtEvalParams& P, const KdNode* nodes,
                const BucketPoint* bpts, const float* tgt, NdtWorkspace& ws, cudaStream_t stream);

// ---- gicp.cu -----------------------------------------------------------------------------
struct GicpIterParams {     // one outer GICP iteration (gicp_omp_impl.hpp:414-461)
  float guess[16];          // base transformation (NDT result), column-major
  float transformation[16]; // transformation_ of this iteration
  double R[9];              // rotation of transformation_ * guess, row-major, double
  double dist_threshold;    // corr_dist_threshold_^2
};
struct GicpCostParams {     // one BFGS function evaluation (:255-377)
  float T[16];              // base with applyState(x)
  float base[16];
};
// voxel_filter.cu: segment heads of radix-sorted keys (~0 = dropped, meta[3] of them), shared with mrvm.cu
void segment_heads_launch(const uint64_t* keys, int n, uint32_t* block_sum, uint32_t* starts, const long long* meta,
                          cudaStream_t s);
// VoxelGrid::Filter of a device cloud into d_out (capacity n records of 5 floats); shared with filters.cu
int voxel_grid_device(const char* d_in, int64_t stride, int n, float voxel_size, float* d_out, uint32_t* m_out,
                      cudaStream_t s);
// host builds of the three voxel-index functions (test hook sm_debug_voxel_index)
bool vf_debug_index_host(const float* p, float voxel, long long* ixyz);
int ndt_debug_voxel_coord_host(float v, float inv_leaf, int min_b);
void gicp_debug_approx_cell_host(const float* p, float inv, int* ixyz, uint32_t* slot);
// host builds of gicp.cu's per-point arithmetic (test hook sm_debug_gicp_point)
void gicp_debug_mahalanobis_host(const double* R, const double* C1, const double* C2, double* out9);
void gicp_debug_cost_terms_host(const float* T, const float* base, const float* ps, const float* pt, const double* M,
                                double* acc13);
size_t approx_ws_bytes(int n);
int approx_voxel_grid(const float* pts, int n, float leaf, void* ws_base, float* out, uint32_t* n_out_dev,
                      cudaStream_t stream);
int approx_voxel_grid_emit(int n, int n_runs, void* ws_base, float* out, const uint32_t* n_out_dev,
                           cudaStream_t stream);
int gicp_covariances(const float* cloud, int n, const KdNode* nodes, const BucketPoint* bpts, double eps,
                     double* covs, cudaStream_t stream);
int gicp_correspond(const float* src, int ns, const float* tgt, const GicpIterParams& P, const KdNode* nodes,
                    const BucketPoint* bpts, const double* cov_s, const double* cov_t, int32_t* match,
                    double* maha, uint32_t* count, cudaStream_t stream);
int gicp_cost_blocks(int ns);
// ticket: a zeroed u32; host_sums_dev / host_flag_dev: device views of mapped pinned host memory (13 doubles and a
// sequence word the kernel sets to `seq` after the sums), or null
int gicp_cost(const float* src, int ns, const float* tgt, const GicpCostParams& P, const int32_t* match,
              const double* maha, double* partials, double* sums, uint32_t* ticket, double* host_sums_dev,
              long long* host_flag_dev, long long seq, cudaStream_t stream);

// ---- normals.cu ------------------------------------------------------------------------
int normals_scratch_blocks(int n);
int normals_run(const double* coord, int64_t cstride, int n, KdWorkspace& ws, KdNode* nodes,
                uint32_t* leaf_order, double* tmp_pts, double* tmp_nrm, uint32_t* keep,
                uint32_t* block_sums, double* out_pts, double* out_nrm, uint32_t* m_dev,
                cudaStream_t stream);

}  // namespace smb

#endif  // SM_B200_KERNELS_H_
