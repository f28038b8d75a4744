/* sm_b200_debug.h — TEST HOOKS of libsm_b200.so.  Not part of the drop-in boundary (include/sm_b200.h):
 * nothing in the reference binds these.  They let tests/ drive pieces of PRODUCT code that have no entry point of
 * their own against INDEPENDENT implementations (numpy / scipy / tests/pyref.py), so that a transcription error
 * shared by the product and the oracle cannot pass unnoticed — most of them without a GPU (DESIGN.md section 2a):
 *   host code of the product, over caller-supplied evaluations
 *     sm_debug_bfgs_minimize   the BFGS minimiser of the GICP stage (csrc/gicp_host.h: PCL's port of GSL
 *                              vector_bfgs2 with the Fletcher line search, gicp_omp_impl.hpp:218-224)
 *     sm_debug_ndt_newton      the NDT Newton loop (csrc/ndt_host.h newton_loop, ndt_omp_impl.hpp:81-171)
 *     sm_debug_gicp_outer      the GICP outer loop (csrc/gicp_host.h outer_loop, gicp_omp_impl.hpp:381-514, :187-246)
 *     sm_debug_ndt_host        6x6 Jacobi-SVD solve, pose <-> 6-vector with Eigen's eulerAngles(0,1,2), Gauss constants
 *     sm_debug_gicp_host       applyState, computeRDerivative
 *   device math of the product compiled for the host (the same __host__ __device__ source the kernels call)
 *     sm_debug_solve6_host     SolvePossiblyUnderdeterminedLinearSystem (csrc/linalg_dev.cuh, icp_fast.cc:204-254)
 *     sm_debug_icp_host        per-match normal-equation terms, AngleAxis / quaternion / angularDistance helpers
 *     sm_debug_ndt_leaf        one leaf of the NDT target grid: covariance, eigenvalue inflation, inverse
 *     sm_debug_ndt_term        one (point, voxel) term of computeDerivatives, pclomp float and stock-PCL double forms
 *     sm_debug_gicp_point      Mahalanobis matrix of a correspondence, one correspondence's cost / gradient terms
 *     sm_debug_voxel_index     the voxel index of a point in the submap filter, the NDT grid and ApproximateVoxelGrid
 *     sm_debug_motion_host     InterpolateTransform(Identity, delta, factor) applied to a point
 *     sm_debug_normals_leaf    the leaf plane fit of CalculateNormals (cloud_types.cc:73-103)
 *     sm_debug_mrvm_ray        the Bresenham ray of one point of MultiResolutionVoxelMap::InsertPointCloud
 *     sm_debug_mrvm_update     its per-voxel probability update (misses, then hits, by binary lifting)
 *   on the device
 *     sm_debug_mrvm_state      the full state of a MultiResolutionVoxelMap, for bit-level comparison with the oracle
 *     sm_debug_solve6          the 6x6 solver exactly as icp_finish_kernel calls it
 *     sm_debug_knn1_batched    sm_knn1 with the scheduling the ICP iteration uses when many alignments are in flight
 *                              (queries_per_cta > 256: lockstep root visits, then the lanes of a warp pull parked
 *                              searches), so that path's index sets and squared distances meet the oracle's directly */
#ifndef SM_B200_DEBUG_H_
#define SM_B200_DEBUG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* A: row-major 6x6 (symmetric in the ICP use), b: 6.  path: 0 LLT, 1 rank-reduced min-norm, 2 SVD. */
int sm_debug_solve6(int device, const double* A_36, const double* b_6, double* x_6, int32_t* path);

/* the same routine compiled for the host (no GPU needed): the source both builds share is csrc/linalg_dev.cuh */
int sm_debug_solve6_host(const double* A_36, const double* b_6, double* x_6, int32_t* path);

/* f and/or g may be NULL (value-only / gradient-only evaluations of the line search); return < 0 to abort. */
typedef int (*sm_debug_fdf)(const double* x_6, double* f, double* g_6, void* user);
/* Runs the GICP inner loop (gicp_omp_impl.hpp:225-240): set, then iterate + test_gradient(grad_tol) until
 * it reports success / no progress or max_iterations.  status: 0 success, 1 still running (iteration cap),
 * 2 no progress, -1 error. */
int sm_debug_bfgs_minimize(sm_debug_fdf fn, void* user, double* x_6_inout, double grad_tol,
                           int32_t max_iterations, int32_t* iterations, int32_t* evaluations, int32_t* status);

/* sm_knn1 (include/sm_b200.h) with `queries_per_cta` queries per 256-thread CTA (rounded up to a multiple of
 * 256; 0 = sm_knn1's own one query per thread). */
int sm_debug_knn1_batched(int device, const double* target_3xn, int64_t n_target, const double* query_3xn,
                          int64_t n_query, double epsilon, int bucket_size, int32_t queries_per_cta,
                          int32_t* ids, double* dists2);

/* The host-side scalar pieces of registrator::Ndt's Newton loop (csrc/ndt_host.h), runnable without a GPU, so that
 * product code is compared with numpy directly (tests/test_independent_checks.py):
 *   op 0: JacobiSVD(H).solve(b), ndt_omp_impl.hpp:127-129     in = H[36] row-major, b[6]       out = x[6]
 *   op 1: Translation * AngleAxis(X) * AngleAxis(Y) * AngleAxis(Z) in float, :146-149 / :797-800
 *                                                              in = p[6]                        out = T[16] col-major
 *   op 2: translation + rotation().eulerAngles(0, 1, 2) in float, :103-111
 *                                                              in = T[16] col-major             out = p[6]
 *   op 3: Gauss constants d1, d2, :86-93                       in = {outlier_ratio, resolution} out = {d1, d2}
 * Returns 0, or SM_ERR_BAD_ARGUMENT for an unknown op / null pointer. */
int sm_debug_ndt_host(int32_t op, const double* in, double* out);

/* The ICP iteration's per-match arithmetic and pose-update helpers compiled for the host (csrc/icp_dev.cuh,
 * csrc/linalg_dev.cuh; ErrorElements + ComputePointToPlane, icp_fast.cc:268-313, CheckConvergence :377-405):
 *   op 0: in = n records {p[3], q[3], normal[3], d2}  out = 29 sums: upper triangle of A = sum F F^T (21, row by row),
 *         sum F (n . (p - q)) (6), sum sqrt(d2), count;  F = [p x normal; normal]
 *   op 1: in = {angle, axis[3]}        out = R[9] row-major   (Eigen::AngleAxis::toRotationMatrix)
 *   op 2: in = R[9] row-major          out = {w, x, y, z}     (Eigen::Quaterniond(Matrix3d))
 *   op 3: in = two quaternions {w,x,y,z}  out[0] = angularDistance
 *   op 4: in = two column-major 4x4    out = their product */
int sm_debug_icp_host(int32_t op, const double* in, int64_t n, double* out);

/* The Newton loop of registrator::Ndt (NormalDistributionsTransform::computeTransformation, ndt_omp_impl.hpp:81-171,
 * with the step-length routine whose More-Thuente loop never runs, :757-916) as the product runs it: csrc/ndt_host.h
 * newton_loop, the function that drives the device evaluations in sm_align.  Here the evaluation is the caller's:
 * fn(T, p, sums, user) receives final_transformation_ (column-major 4x4, float-valued) and the pose vector p[6] it
 * was built from (the angle-derivative tables belong to p) and fills sums[0] = score, [1..6] = gradient, [7..42] = Hessian row-major, [43] = neighbour count
 * summed over the points; it returns < 0 to abort. */
typedef int (*sm_debug_ndt_eval)(const double* T_4x4, const double* p_6, double* sums_44, void* user);
int sm_debug_ndt_newton(sm_debug_ndt_eval fn, void* user, const double* guess_4x4, int32_t n_source, float resolution,
                        double step_size, double outlier_ratio, double transformation_epsilon, int32_t max_iterations,
                        double* final_4x4, int32_t* iterations, int32_t* evaluations, double* score);

/* The outer loop of the GICP stage as the product runs it (csrc/gicp_host.h outer_loop =
 * GeneralizedIterativeClosestPoint::computeTransformation + estimateRigidTransformationBFGS, gicp_omp_impl.hpp:381-514,
 * :187-246, with the options of ndt_gicp.cc:50-51), over the caller's per-point work:
 *   correspond(transformation_4x4, R_9, &m, user): correspondences and Mahalanobis matrices for transformation_ (column-
 *       major, float-valued) with R = rot(transformation_ * guess) row-major in double; m = number of correspondences
 *   cost(T_4x4, S_13, user): S[0] = sum res^T M res, S[1..3] = sum M res, S[4..12] = sum (guess p)(M res)^T row-major
 *       for T = guess with applyState(x) (column-major, float-valued)
 * both return < 0 to abort. */
typedef int (*sm_debug_gicp_correspond)(const double* transformation_4x4, const double* R_9, int32_t* m, void* user);
typedef int (*sm_debug_gicp_cost)(const double* T_4x4, double* S_13, void* user);
int sm_debug_gicp_outer(sm_debug_gicp_correspond correspond, sm_debug_gicp_cost cost, void* user,
                        const double* guess_4x4, double* final_4x4, int32_t* iterations, int32_t* bfgs_evaluations);

/* The voxel index of one point {x, y, z} as the three voxelisations compute it (device functions compiled for the host):
 *   op 0: submap filter, lround(x / voxel) (filter_voxel_grid.cc:50-52), param = voxel size; out[3] = 0: point dropped
 *   op 1: NDT grid, int(floor(x * inv) - float(min_b)) per axis (voxel_grid_covariance_omp_impl.hpp:218-220), param = inv
 *   op 2: ApproximateVoxelGrid, floor(x * inv) per axis, out[3] = hash slot (ix * 7171 + iy * 3079 + iz * 4231) & 511 */
int sm_debug_voxel_index(int32_t op, const float* p_3, float param, int32_t min_b, int64_t* out_4);

/* The per-point arithmetic of the GICP kernels compiled for the host (csrc/gicp.cu mahalanobis / cost_terms):
 *   op 0: M = (R C1 R^T + C2)^-1, gicp_omp_impl.hpp:450-457    in = R[9], C1[9], C2[9] row-major     out = M[9]
 *   op 1: one correspondence of the functor, :341-377          in = T[16], base[16] col-major, p_src[3], p_tgt[3], M[9]
 *         out = {res^T M res, (M res)[3], ((base p_src)(M res)^T)[9] row-major} */
int sm_debug_gicp_point(int32_t op, const double* in, double* out);

/* Host pieces of the GICP stage besides the minimiser (csrc/gicp_host.h):
 *   op 0: applyState, gicp_omp_impl.hpp:516-527   in = T[16] col-major, x[6]      out = T'[16] (float arithmetic)
 *   op 1: computeRDerivative, :133-183            in = x[6], R[9] row-major       out = {g[3], g[4], g[5]} */
int sm_debug_gicp_host(int32_t op, const double* in, double* out);

/* The leaf routine of EigenPointCloud::CalculateNormals (cloud_types.cc:73-103; csrc/normals.cu leaf_plane_fit compiled
 * for the host): count (1..7) members {x, y, z} in member order -> mean, unit normal of the plane n . p = 1, kept = 0
 * when rank(covariance) + 1 < 3. */
int sm_debug_normals_leaf(const double* members_3k, int32_t count, double* mean_3, double* normal_3, int32_t* kept);

/* sm_motion_compensation's arithmetic on the host (csrc/motion.cu make_params + motion_point): packed
 * {x, y, z, intensity, factor} float records in and out; SM_ERR_BAD_ARGUMENT if a factor is outside [0, 1]. */
int sm_debug_motion_host(const float* points_5n, int64_t n, const double* delta_4x4, float* out_5n);

/* One leaf of VoxelGridCovariance::applyFilter (voxel_grid_covariance_omp_impl.hpp:209-366; csrc/ndt.cu finish_leaf
 * compiled for the host): the n points of a voxel in input order -> mean, inverse covariance (zero when the leaf has
 * fewer than min_points points or fails the eigenvalue test), float centroid, nr_points (-1 = invalid covariance),
 * searchable. */
int sm_debug_ndt_leaf(const float* points_3n, int32_t n, int32_t min_points, double eig_mult, double* mean_3,
                      double* icov_9, float* centroid_3, int32_t* nr_points, int32_t* searchable);

/* One (point, voxel) term of computeDerivatives (ndt_omp_impl.hpp:397-438 + :483-535; f64_math = 1: the stock PCL
 * double form NdtWithGicp uses): csrc/ndt.cu's update_derivatives compiled for the host, evaluation tables built by
 * csrc/ndt_host.h for the pose vector p.  out43 = {score increment, gradient term[6], Hessian term[36] row-major}. */
int sm_debug_ndt_term(const double* p_6, double outlier_ratio, float resolution, int32_t f64_math,
                      const float* x_orig_3, const float* x_trans_3, const double* voxel_mean_3,
                      const double* voxel_icov_9, double* out43);

/* The ray of one point of MultiResolutionVoxelMap::InsertPointCloud (csrc/mrvm.cu mrvm_voxel + mrvm_walk compiled for
 * the host, common::VoxelCastingBresenham math.cc:35-95): the voxels from origin's to point's, both included,
 * 3 int32 each.  *n_out = number of voxels; SM_ERR_BAD_ARGUMENT for a non-finite or out-of-range coordinate, or when
 * it exceeds `capacity`. */
int sm_debug_mrvm_ray(const float* origin_3, const float* point_3, float step, int32_t* voxels_3n, int64_t capacity,
                      int64_t* n_out);
/* The per-voxel probability update of an insert (csrc/mrvm.cu mrvm_tables + mrvm_lift): probs[i] after misses[i]
 * misses and then hits[i] hits (each < 2^32), for hit_prob / miss_prob as sm_mrvm_create takes them.  tables_out
 * (optional, 512 bytes): the one-step hit and miss maps. */
int sm_debug_mrvm_update(float hit_prob, float miss_prob, const uint8_t* probs, const int64_t* misses,
                         const int64_t* hits, int64_t n, uint8_t* out, uint8_t* tables_out);
/* Full state of a map in ascending key order (for bit-level comparison): key = ((ix + 2^20) << 42) |
 * ((iy + 2^20) << 21) | (iz + 2^20), probability, max_intensity, number of stored points, and the stored points
 * {x, y, z, intensity} (max_point_num_in_cell records per voxel, unused ones zero).  *n_out = number of voxels;
 * SM_ERR_BAD_ARGUMENT if it exceeds `capacity`. */
int sm_debug_mrvm_state(struct sm_mrvm* h, int64_t* keys, uint8_t* prob, int32_t* max_intensity, int32_t* npts,
                        float* points4, int64_t capacity, int64_t* n_out);

/* The per-point functions of the filter chain (csrc/filters.cu), compiled for the host, over n points `stride_bytes`
 * apart:
 *   op 0: the product's atan2f(y, x), out[k] = its float bits                       params unused
 *   op 1: RangeImage pixel row * H + col, -1 outlier      params = top, btm, offset_x, offset_y, offset_z, V, H
 *   op 2: GroundRemoval2 cell s * bin_num + b, -1 not binned   params = r_max, r_min, bin_num, segment_num
 *   op 3: GroundRemoval voxel, out[4k..4k+3] = rc (0 ok, 1 not finite, 2 outside int), ix, iy, iz   params = leaf */
int sm_debug_filter_points(int32_t op, const float* points, int64_t n, int64_t stride_bytes, const float* params,
                           int64_t* out);
/* GroundRemoval2::FitLines of one segment: cell_dz = bin_num (d, z) min_z_points, cell_used = bin_num flags (the
 * cell's `points` is not empty); params = r_max, r_min, start_ground_height, long_line_threshold, max_long_line_height,
 * max_start_height, max_error, max_slope, max_b, max_dist_to_line, search_angle, bin_num.  lines4: (start d, start z,
 * end d, end z) per line; *n_out = number of lines. */
int sm_debug_filter_fit_lines(const float* cell_dz, const uint8_t* cell_used, const float* params, float* lines4,
                              int64_t capacity, int64_t* n_out);
/* FitLocalLine + GetMaxError over k (d, z) points: mb = m, b, max error. */
int sm_debug_filter_line_fit(const float* dz, int64_t k, float* mb);

#ifdef __cplusplus
}
#endif
#endif /* SM_B200_DEBUG_H_ */
