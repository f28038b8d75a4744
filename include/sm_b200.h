/* sm_b200.h — C ABI of libsm_b200.so, the B200-native scan-matching engine that stands in
 * for StaticMapping's registrators/ hot path.
 *
 * Drop-in boundary: the reference has no FFI of its own (it is one C++ process); the
 * interface a maintainer binds is registrator::Interface
 * (/root/reference/registrators/interface.h:67-119).  Each entry point below names the
 * reference member it replaces.  INTEGRATION.md shows the C++ adapter
 * (adapter/registrators_b200.h) that maps these 1:1 onto that class.
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types; never throws across the ABI;
 *   - 4x4 transforms are 16 doubles, COLUMN-major (Eigen::Matrix4d storage);
 *   - clouds are 3xN column-major doubles (x0,y0,z0,x1,...) == Eigen::MatrixXd of
 *     data::EigenPointCloud::points / ::normals (builder/data/cloud_types.h:143-146);
 *   - return value: >= 0 success, < 0 error (sm_last_error gives the text).  Where the
 *     reference would glog-CHECK-abort the C++ adapter turns the negative code into the
 *     same CHECK failure (SURVEY.md section 5 "failure detection");
 *   - one handle is used by one thread at a time; different handles may run concurrently
 *     from different threads (map_builder.cc:655,706-708; loop_detector.cc:224-228).  Each
 *     handle owns its CUDA stream and workspace.
 */
#ifndef SM_B200_H_
#define SM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct sm_handle sm_handle;

/* registrator::Type (interface.h:41-50); values match the XML `type="N"` attribute. */
enum sm_matcher_type {
  SM_TYPE_ICP_PM = 1,
  SM_TYPE_NDT_WITH_GICP = 3,
  SM_TYPE_NDT = 5,
  SM_TYPE_FAST_ICP = 6
};

enum sm_error {
  SM_OK = 0,
  SM_ERR_BAD_ARGUMENT = -1,
  SM_ERR_NO_FINITE_MATCH = -2,   /* CHECK(!values.empty())            icp_fast.cc:81  */
  SM_ERR_NOTHING_TO_MINIMIZE = -3, /* CHECK_GT(points_count, 0)        icp_fast.cc:114 */
  SM_ERR_MISSING_INPUT = -4,     /* CHECK(cloud) / missing normals    icp_fast.cc:422-430 */
  SM_ERR_UNKNOWN_OPTION = -10,   /* "Init an unknown option"          interface.cc:66-67 */
  SM_ERR_UNSUPPORTED_TYPE = -11, /* CreateMatcher default branch      interface.cc:158-160 */
  SM_ERR_NO_DEVICE = -20,        /* no CUDA device: the engine has no CPU fallback */
  SM_ERR_CUDA = -100
};

/* CreateMatcher(options) (interface.cc:139-173) + the concrete constructors
 * (IcpFast::IcpFast icp_fast.cc:407-419).  `device` is the CUDA ordinal. */
int sm_create(int type, int device, sm_handle** out);
int sm_destroy(sm_handle* h);

/* Interface::InitWithXml (interface.cc:62-90): one <param name=...>text</param> entry.
 * `text` is parsed like pugixml's as_int / as_float / as_bool for the registered type.
 * Registered names, IcpFast (icp_fast.cc:411-418): knn_normal_estimate (int, unused),
 * max_iteration (int, 100), dist_outlier_ratio (float, 0.7).  Added by this engine:
 * knn_epsilon (float, 3.16 = icp_fast.cc:174), knn_queries_per_cta (int, 0 = one query per
 * thread; 1024 suits many alignments in flight), disable_convergence_check (bool, false;
 * fixed-iteration throughput runs), profile_kernels (bool, false; CUDA events around
 * every phase kernel, reported by sm_get_align_info), use_graphs (bool, true; replay the
 * launch sequence of an Align as CUDA graphs).  Unknown name -> SM_ERR_UNKNOWN_OPTION.
 * registrator::Ndt registers NO option (ndt.cc:28-34) — the reference-facing mirrors reject
 * every <param> for type 5; the engine itself accepts the pclomp setters hard-coded by the
 * reference: resolution (1.0), step_size (0.1), outlier_ratio (0.55),
 * transformation_epsilon (0.1), max_iterations (35).
 * SM_TYPE_ICP_PM is NOT a bit-level parity implementation of registrator::IcpUsingPointMatcher: libpointmatcher
 * 1.3.1 is an external float library whose RandomSampling filter draws from the process-global std::rand stream
 * (two Align calls on the same clouds give poses ~0.5 mm apart: the reference's result is not a function of its
 * inputs) and whose surface-normal filter uses eigenvector normals.  Type 1 is a deterministic matcher with the
 * same module chain (DESIGN.md section 4e): bit-checked against a composition of this repository's oracle
 * pieces, and shown to lie within the literal chain's own call-to-call variation by a restatement of
 * libpointmatcher's filters (tests/pyref.py icp_pm_literal, tests/test_oracle_vs_python_restatement.py).
 * SM_TYPE_ICP_PM (stand-in for IcpUsingPointMatcher's default libpointmatcher chain,
 * icp_pointmatcher.cc:166-247; float clouds through the _f32 setters) registers no option in the
 * reference either; the engine accepts the IcpFast names (max_iteration defaults to 150, :214)
 * plus reading_sample_prob (0.9, :173), accept_min_score (0.6, :145) and sample_seed (1). */
int sm_set_option(sm_handle* h, const char* name, const char* text);
/* Interface::PrintOptions (interface.cc:115-137): writes "name -> value\n" lines. */
int sm_print_options(sm_handle* h, char* buf, int64_t buf_len);
/* Interface::GetType (interface.h:106). */
int sm_get_type(const sm_handle* h);

/* IcpFast::SetInputSource / SetInputTarget (icp_fast.cc:421-431): deep copy into the
 * engine (host pointers are not retained).  The target must carry unit normals
 * (CHECK(HasNormals()), icp_fast.cc:430) — the caller computed them with
 * EigenPointCloud::CalculateNormals (map_builder.cc:286,389) or sm_calculate_normals. */
int sm_set_input_source(sm_handle* h, const double* points_3xn, int64_t n);
int sm_set_input_target(sm_handle* h, const double* points_3xn, const double* normals_3xn,
                        int64_t n);
/* Ndt / NdtWithGicp keep the caller's float cloud (Interface::SetInputSource/Target,
 * interface.cc:38-60, converted by ToPclPointCloud at Align, ndt.cc:48-51).  `xyz` points at
 * the first x; consecutive points are `stride_bytes` apart (sizeof(InnerPointType) == 20 for
 * the reference's std::vector<InnerPointType>, 12 for packed xyz). */
int sm_set_input_source_f32(sm_handle* h, const float* xyz, int64_t n, int64_t stride_bytes);
int sm_set_input_target_f32(sm_handle* h, const float* xyz, int64_t n, int64_t stride_bytes);
int sm_set_input_source_f32_device(sm_handle* h, const float* dev_xyz, int64_t n, int64_t stride_bytes);
int sm_set_input_target_f32_device(sm_handle* h, const float* dev_xyz, int64_t n, int64_t stride_bytes);

/* Same, for clouds already resident in this device's memory (same layout). */
int sm_set_input_source_device(sm_handle* h, const double* dev_points_3xn, int64_t n);
int sm_set_input_target_device(sm_handle* h, const double* dev_points_3xn,
                               const double* dev_normals_3xn, int64_t n);

/* Interface::Align(const Matrix4d& guess, Matrix4d& result) (interface.h:103-104;
 * IcpFast::Align icp_fast.cc:455-529).  Returns 1 (true) / 0 (false) like the
 * reference's bool, or a negative sm_error. */
int sm_align(sm_handle* h, const double* guess_4x4, double* result_4x4);
/* The same Align in two halves, so ONE host thread can keep several matcher instances in
 * flight (the reference gets its concurrency from a thread pool / TBB tasks calling Align on
 * distinct instances: map_builder.cc:655,706-708; loop_detector.cc:224-228):
 * sm_align_async enqueues everything and returns; sm_align_wait blocks for the result (and,
 * with the convergence test enabled, keeps enqueuing 8-iteration chunks until it fires).
 * IcpFast only; sm_align == async + wait. */
int sm_align_async(sm_handle* h, const double* guess_4x4);
int sm_align_wait(sm_handle* h, double* result_4x4);
/* Batched Align.  The reference fans independent Align calls out to a thread pool / TBB tasks
 * (back_end/loop_detector.cc:216-228 one task per loop-closure candidate; builder/map_builder.cc:
 * 655,706-708 submap pairs); here ONE host thread keeps many alignments in flight on the GPU.
 *
 * sm_align_batch: `n` matcher instances whose SetInputSource / SetInputTarget have been called.
 * IcpFast instances are all enqueued before the first result is awaited; the other matcher types
 * (host-driven Newton / BFGS loops) run on up to 16 internal worker threads.  guesses / results:
 * n x 16 doubles; rc_n[i] = what sm_align would have returned for instance i.  Returns SM_OK or the
 * most negative rc.
 *
 * sm_align_pairs: `n_pairs` independent IcpFast alignments pipelined over `n_handles` instances
 * (pair k runs on instance k % n_handles; an instance's previous result is collected right before
 * it is given its next pair).  Host clouds are uploaded asynchronously on the instance's stream —
 * unlike sm_set_input_*, the arrays of a pair must stay valid until sm_align_pairs returns (pinned
 * host memory makes the copies overlap the other pipelines' kernels).  scores_n (optional) receives
 * GetFitnessScore per pair. */
typedef struct sm_pair {
  const double* source_3xn;          /* SetInputSource */
  int64_t n_source;
  const double* target_3xn;          /* SetInputTarget (points + unit normals) */
  const double* target_normals_3xn;
  int64_t n_target;
  const double* guess_4x4;           /* NULL = identity */
  int32_t on_device;                 /* 1: the three cloud pointers are device pointers */
  int32_t reserved;
} sm_pair;
int sm_align_batch(sm_handle* const* handles, int32_t n, const double* guesses_16n, double* results_16n,
                   int32_t* rc_n);
int sm_align_pairs(sm_handle* const* handles, int32_t n_handles, const sm_pair* pairs, int32_t n_pairs,
                   double* results_16n, double* scores_n, int32_t* rc_n);
/* Interface::GetFitnessScore (interface.h:100). */
double sm_get_fitness_score(const sm_handle* h);

typedef struct sm_align_info {
  int32_t iterations;      /* ICP iterations executed */
  int32_t status;          /* 0 or sm_error */
  int32_t solve_path;      /* last 6x6 solve: 0 Cholesky, 1 rank-reduced, 2 SVD */
  int32_t reserved;
  int64_t kept;            /* matches kept by the 70 % trim in the last iteration */
  double limit;            /* its squared-distance limit */
  float ms_upload;         /* device time of the last SetInput* copies */
  float ms_prologue;       /* centre + tree build + G0 (icp_fast.cc:456-480) */
  float ms_iterations;     /* all ICP iterations */
  int32_t kernel_launches; /* kernels launched by the last sm_align */
  /* filled only when option profile_kernels=1: summed device time of each phase kernel */
  float ms_knn;            /* transform + k-NN + histogram        (icp_fast.cc:486-493) */
  float ms_accum;          /* quantile bin + normal equations      (icp_fast.cc:496-503) */
  float ms_finish;         /* exact limit, solve, pose update      (icp_fast.cc:506-523) */
  int32_t profiled_iterations;
  /* NDT only */
  int32_t evaluations;        /* computeDerivatives calls (ndt_omp_impl.hpp:180) */
  double trans_probability;   /* score / N_source (ndt_omp_impl.hpp:170) */
  double mean_neighbors;      /* mean number of neighbour voxels per source point */
  /* IcpUsingPointMatcher stand-in (type 1): [0] IcpFast's own score of the last iteration,
   * [1] matches kept by the trim in the final score pass, [2] reading / [3] reference points after
   * the data filters.
   * NdtWithGicp only: [0] NDT fitness (the <= 1.0 gate, ndt_gicp.cc:92), [1] GICP fitness,
   * [2] source points after ApproximateVoxelGrid, [3] target points after it;
   * iterations = GICP outer iterations, profiled_iterations = BFGS cost evaluations */
  double aux[4];
} sm_align_info;
int sm_get_align_info(const sm_handle* h, sm_align_info* out);

/* Run this handle's work on the caller's CUDA stream (a cudaStream_t passed as void*;
 * NULL restores the handle's own stream).  Lets a host that already owns a stream —
 * e.g. the bench's torch stream — order and time the engine's kernels with its own
 * events.  No reference counterpart (the reference is CPU-only). */
int sm_set_stream(sm_handle* h, void* cuda_stream);

const char* sm_last_error(const sm_handle* h);

/* ---- building blocks exposed for parity tests and for callers that hold clouds ------- */

/* libnabo-compatible tree build + 1-NN (NNS::create + knn, icp_fast.cc:466-467,177-178).
 * ids: original target column, -1 if none; dists2: squared distances.  bucket_size 2..8
 * (libnabo's default is 8; one padded bucket of the search layout holds 8 points). */
int sm_knn1(int device, const double* target_3xn, int64_t n_target, const double* query_3xn,
            int64_t n_query, double epsilon, int bucket_size, int32_t* ids, double* dists2);

/* EigenPointCloud::CalculateNormals (builder/data/cloud_types.cc:347-368): median-split
 * the cloud into leaves of <= 7 points, fit n.p = 1 per leaf, keep one point (the leaf
 * mean) + unit normal per valid leaf, survivors in ascending order of the smallest
 * original index of their leaf.  out_points / out_normals: capacity 3*n doubles;
 * *m_out receives the number of survivors.  Called by the reference right before
 * IcpFast::SetInputTarget (map_builder.cc:286,389; submap.cc:161).
 * DEVIATION from the reference (cloud_types.cc:79-100): there a leaf is represented by
 * indices[first] and summed in the member order std::nth_element happens to leave, both of which
 * depend on the standard library's partition internals; here the representative is the member
 * with the smallest original index and members are summed in ascending index.  The SET of surviving
 * leaves is identical (the split is order independent for distinct coordinates); the column order
 * of the output and the last bits of a mean / normal may differ from a run of the real reference. */
int sm_calculate_normals(int device, const double* points_3xn, int64_t n, double* out_points,
                         double* out_normals, int64_t* m_out);

/* MotionCompensation (builder/map_builder.cc:232-257; called either side of Align at :320-352
 * when motion_compensation_options.enable is set): every point is moved by
 * common::InterpolateTransform(Identity, delta, point.factor) (common/math.h:198-211 — slerp of
 * the rotation, linear translation).  `points` / `out` are arrays of the reference's
 * data::InnerPointType {float x, y, z, intensity, factor} (builder/data/cloud_types.h:46-52),
 * consecutive points `stride_bytes` (>= 20) apart; intensity and factor are copied.  `delta` is
 * 16 doubles, column-major.  Returns SM_ERR_BAD_ARGUMENT where the reference CHECK-fails
 * (a factor outside [0, 1], common/math.h:201); `out` is still written in that case.
 * The _device form takes device pointers (in and out may not overlap) and runs on
 * `cuda_stream` (a cudaStream_t, NULL = default stream); it returns after the stream has
 * finished. */
int sm_motion_compensation(int device, const float* points, int64_t n, int64_t stride_bytes,
                           const double* delta_4x4, float* out);
int sm_motion_compensation_device(int device, const float* dev_points, int64_t n,
                                  int64_t stride_bytes, const double* delta_4x4, float* dev_out,
                                  void* cuda_stream);

/* pre_processers::filter::VoxelGrid::Filter (pre_processors/filter_voxel_grid.cc:37-78), the
 * down-sampling Submap::InsertFrame applies before CalculateNormals (builder/submap.cc:144-161):
 * one output point per occupied voxel, voxel index = lround(coordinate / voxel_size) per axis
 * (:47-49), x / y / z / intensity = mean of the voxel's points accumulated in double in input
 * order (:58-70), factor = 0.  `points`: data::InnerPointType records (x, y, z, intensity, ...)
 * `stride_bytes` (>= 16) apart; `out`: capacity n records of 5 packed floats; *m_out = number of
 * voxels.  Every value is bit-identical to the reference's; the ORDER of the output points is
 * ascending (ix, iy, iz), where the reference emits them in std::unordered_map iteration order.
 * Points with a NaN / inf coordinate are dropped (std::lround of such a value is unspecified in the
 * reference; one bad lidar return must not stop the mapper).  SM_ERR_BAD_ARGUMENT: voxel_size <= 1e-6
 * (ConfigsValid, :35), or finite points that span 2^21 voxels or more along one axis (209 km at the
 * reference's 0.1 m voxels). */
int sm_voxel_grid_filter(int device, const float* points, int64_t n, int64_t stride_bytes,
                         float voxel_size, float* out, int64_t* m_out);

/* descriptor::M2dp (descriptor/m2dp.cc:37-172; parameters of the constructor, m2dp.h:50-51: r = 0.1,
 * max_distance = 100, t = 16, p = 4, q = 16), the loop-closure descriptor of a submap:
 * M2dp::setInputCloud + getFinalDescriptor.  `points`: float x, y, z records `stride_bytes` (>= 12) apart
 * (data::InnerPointType = 20).  descriptor: p*q + l*t floats, l = ceil(sqrt(max_distance / r)) — [u1; v1],
 * the first left / right singular vectors of the p*q x l*t signature matrix (:148-152); A_out (optional):
 * that matrix as counts, row-major.  Returns 1 (true), 0 for an empty cloud (setInputCloud returns false,
 * :130-133), SM_ERR_BAD_ARGUMENT for r < 1e-6 (:64-67) or a too small `capacity`.
 * Two orientations are Eigen-internal in the reference and fixed here: each of the first two PCA axes has
 * its component of largest magnitude positive, and so has u1 (v1 follows).  sm_m2dp_match does not depend
 * on the second; the first decides which points the reference's |.| projections fold together.
 * sm_m2dp_match: matchTwoM2dpDescriptors (:155-170) = |Pearson correlation|, -1 for n < 10. */
int64_t sm_m2dp_descriptor_length(double r, double max_distance, int32_t t, int32_t p, int32_t q);
int sm_m2dp(int device, const float* points, int64_t n, int64_t stride_bytes, double r, double max_distance,
            int32_t t, int32_t p, int32_t q, float* descriptor, int64_t capacity, int32_t* A_out);
double sm_m2dp_match(const float* P, const float* Q, int64_t n);

/* MultiResolutionVoxelMap (builder/multi_resolution_voxel_map.{h,cc}), the ray-casting occupancy map that
 * MapBuilder::SaveMaps fills with every frame to write static_map.pcd.  The map lives on the device across inserts.
 * Points are data::InnerPointType records (x, y, z, intensity, ...) `stride_bytes` (>= 16) apart.
 * Semantics: those of the reference run by ONE thread.  Per insert, each point casts a Bresenham ray
 * (common::VoxelCastingBresenham, math.cc:35-95) from origin + (0, 0, z_offset) to its voxel
 * lround(floor(v / high_resolution)) (float); its end voxel is created if absent and gets one hit (probability,
 * max_intensity = max(., int(intensity)), the point appended while fewer than max_point_num_in_cell are stored);
 * every other voxel of the ray gets one miss if it existed before this insert and no earlier point of this insert
 * ended in it.  Updates are the reference's uint8 -> uint8 maps (float / double expressions of .h:134-140,
 * .cc:36-40, :63-69).  Deviations from the reference:
 *   1. InsertPointCloud runs its loop on 10 OpenMP threads (:75-77) with a non-atomic read-modify-write of each
 *      voxel's probability and unordered point appends (:93-114): its result is not reproducible.  This map
 *      computes the one-thread result, exactly, whatever the scheduling.
 *   2. Output is in ascending voxel order (ix, iy, iz), not tbb::concurrent_unordered_map order.
 *   3. Points with a NaN / inf coordinate are dropped and counted (the reference reaches lround(NaN) and then
 *      FATAL_CHECK_POINT).
 *   4. Voxel indices must lie in [-2^20, 2^20) per axis (+-104 km at 0.1 m): an insert with a point or an origin
 *      outside returns SM_ERR_BAD_ARGUMENT and leaves the map unchanged.
 * Intensities must be within the int range (the reference converts them with static_cast<int>).
 * One handle is used by one thread at a time; it owns its CUDA stream.  Every call returns after its device work
 * has finished. */
typedef struct sm_mrvm sm_mrvm;
typedef struct sm_mrvm_settings {   /* MrvmSettings, multi_resolution_voxel_map.h:55-66 (defaults in brackets) */
  int32_t output_average;           /* [0] one mean point per voxel instead of every stored point */
  int32_t output_rgb;               /* [0] not read by this API: the caller picks the record type in sm_mrvm_output */
  int32_t use_max_intensity;        /* [1] */
  float prob_threshold;             /* [0.6] not read by this API: sm_mrvm_output takes the threshold */
  float low_resolution;             /* [1.0] unused, like in the reference */
  float high_resolution;            /* [0.1] voxel size, > 0 */
  float hit_prob;                   /* [0.55] > 0.5, clamped to [0.501, 0.9] */
  float miss_prob;                  /* [0.48] < 0.5, clamped to [0.1, 0.499] */
  float z_offset;                   /* [0] added to the ray origin's z */
  int32_t max_point_num_in_cell;    /* [10] >= 1 */
} sm_mrvm_settings;
/* Constructor + Initialise (:36-48).  SM_ERR_BAD_ARGUMENT where map_builder_options.cc:66-68 CHECK-fails
 * (hit_prob <= 0.5, miss_prob >= 0.5, max_point_num_in_cell < 1) and for high_resolution <= 0.  expected_voxels
 * sizes the first allocation; the map grows past it as needed. */
int sm_mrvm_create(int device, const sm_mrvm_settings* settings, int64_t expected_voxels, sm_mrvm** out);
int sm_mrvm_destroy(sm_mrvm* h);
/* SetOffsetZ (:50-52). */
int sm_mrvm_set_offset_z(sm_mrvm* h, float offset);
/* InsertPointCloud (:54-123); origin = the sensor position, 3 floats.  An empty cloud leaves the map unchanged.
 * Returns the number of points dropped for a non-finite coordinate (>= 0), or an sm_error.  The _device form
 * reads device memory and orders itself after the work already queued on `cuda_stream` (a cudaStream_t, NULL = the
 * legacy default stream). */
int sm_mrvm_insert(sm_mrvm* h, const float* points, int64_t n, int64_t stride_bytes, const float* origin_3);
int sm_mrvm_insert_device(sm_mrvm* h, const float* dev_points, int64_t n, int64_t stride_bytes,
                          const float* origin_3, void* cuda_stream);
/* Number of voxels in the map (high_resolution_voxels_.size()). */
int64_t sm_mrvm_size(const sm_mrvm* h);
/* OutputToPointCloud (:125-215): voxels with probability >= (uint8)(threshold * 256) in ascending voxel order.
 * out4: records {x, y, z, value}; with output_average one record per voxel (the float mean of its stored points,
 * summed in stored order), otherwise one per stored point.  value: rgb = 0 (the PointXYZI overload):
 * max_intensity if use_max_intensity, else 0 for a mean and the point's own intensity for a stored point;
 * rgb = 1 (the PointXYZRGB overload): the grey level min(255, (uint32)(max_intensity * 1.4)).  *m_out = number of
 * records; SM_ERR_BAD_ARGUMENT if it exceeds `capacity` (out4 untouched) or threshold * 256 is outside (-1, 256). */
int sm_mrvm_output(sm_mrvm* h, float threshold, int32_t rgb, float* out4, int64_t capacity, int64_t* m_out);
/* Cumulative device time of the insert phases, from CUDA events: [0] upload, [1] end keys + sort + segments,
 * [2] table insert (and growth), [3] rays, [4] voxel update; [5] = number of inserts. */
int sm_mrvm_phase_ms(const sm_mrvm* h, float* ms_6);

/* pre_processers::filter::Factory (pre_processors/filter_factory.cc:63-123) and its nine filters, the <filters> chain
 * DataCollector::CloudPreProcessing runs on every scan (builder/data/data_collector.cc:120-156).  A handle holds the
 * stages in XML order; sm_filter_chain_add takes the filter's name (RandomSampler, RangeImage, GroundRemoval,
 * GroundRemoval2, Range, StatisticRemoval, VoxelGrid, AxisRange, BoundingBoxRemoval) and returns the stage index,
 * SM_ERR_UNSUPPORTED_TYPE for any other name (the reference skips it with a log line).  sm_filter_chain_set_param is
 * one <param type=... name=...>text</param>: type 0 parses text like pugixml's as_int, type 1 like as_float, and the
 * value is cast to the parameter's own type; SM_ERR_UNKNOWN_OPTION for a name the filter does not register (a CHECK
 * failure in the reference), SM_ERR_BAD_ARGUMENT for another type.  Parameters keep their values until set again.
 * sm_filter_chain_valid: the filter's ConfigsValid() (1 / 0).
 * Points are data::InnerPointType records {x, y, z, intensity, factor} `stride_bytes` (>= 20) apart; `out` receives
 * records of 5 packed floats, `kept_index` (optional) the chain-input index of each output record (-1 behind a
 * VoxelGrid).  *m_out = number of output records; SM_ERR_BAD_ARGUMENT if it exceeds `capacity` (out untouched).
 * Every filter keeps the reference's semantics, quirks included:
 *   Range: r = sqrtf(x*x + y*y + z*z), kept iff min_range <= r <= max_range (a NaN point is removed).
 *   AxisRange: removed iff v < min || v > max on axis_index; the identity at min = -FLT_MAX and max = FLT_MAX, and for
 *     an axis_index outside 0..2; a NaN coordinate is kept.
 *   BoundingBoxRemoval: removes the points inside the box, bounds included (the default box removes every finite point).
 *   RangeImage: the first point in input order that lands in a pixel is kept; rows truncate toward zero (a point up to
 *     one row below btm_angle lands in row 0), columns are lround of a float quotient wrapped once; xy < 0.01 and a
 *     row or column outside the image are outliers.
 *   GroundRemoval: voxels static_cast<int>(v / leaf_size); voxels with fewer than min_point_num_in_voxel points vanish;
 *     a voxel with iz <= 0 and max z - min z <= height_threshold is ground.  Output in std::map order: ascending
 *     (ix, iy, iz), input order inside a voxel.
 *   GroundRemoval2: the reference's binning, FitLines and ClusterGround, serially per segment.
 *   VoxelGrid: sm_voxel_grid_filter.
 * Deviations from the reference:
 *   1. RandomSampler seeds std::mt19937 from std::random_device on every call, so its result is not a function of its
 *      inputs.  Here a point is kept iff u <= sampling_rate, u uniform on [0, 1) from a counter hash of (seed, call
 *      number, stage index, chain-input index); the call number starts at 0 at sm_filter_chain_set_seed and advances
 *      once per filter call.  A rate above 0.999 is the identity, as in the reference.
 *   2. Angles (RangeImage's pixel, GroundRemoval2's segment) use one atan2: a double-precision evaluation from
 *      correctly rounded +, -, *, / and sqrt, rounded to float, the same bits on the host and the device.  libm's
 *      atan2f is not the same function on every C library (glibc's differs from (float)atan2((double)y, x) on about
 *      16 % of random points), so pixel and cell indices equal a reference run's only given the same angle function.
 *   3. GroundRemoval2's line fit is a two-column Householder QR with column pivoting in double; Eigen's
 *      colPivHouseholderQr rounds through vectorised reductions, so m and b agree to float rounding, not bit for bit.
 *   4. StatisticRemoval (its body is commented out in the reference) is the identity.  As the FIRST stage the
 *      reference's Factory returns an empty cloud (the untouched intermediate cloud); that bug is not reproduced.
 *   5. A stage whose ConfigsValid() is false, or that this engine cannot run (RangeImage with a line count <= 0,
 *      GroundRemoval with leaf_size 0, GroundRemoval2 with bin_num or segment_num <= 0 or a search angle of a full
 *      turn), makes the call return SM_ERR_BAD_ARGUMENT without output; the reference runs it anyway (or divides by 0).
 *   6. Non-finite points: RangeImage drops a point whose row is NaN; GroundRemoval and GroundRemoval2 do not bin them:
 *      they stay inliers (GroundRemoval emits them after every voxel) and are never ground.  GroundRemoval returns
 *      SM_ERR_BAD_ARGUMENT for a voxel index outside the int range or finite points spanning 2^21 voxels on one axis.
 *   7. thread_num of GroundRemoval2 is accepted and ignored.
 * The _device form takes device pointers (in, out and kept_index), orders itself after the work queued on
 * `cuda_stream` and reads back only the count.  Every call returns after its device work has finished.  One handle is
 * used by one thread at a time; it owns its CUDA stream. */
typedef struct sm_filter_chain sm_filter_chain;
int sm_filter_chain_create(int device, sm_filter_chain** out);
int sm_filter_chain_destroy(sm_filter_chain* h);
int sm_filter_chain_add(sm_filter_chain* h, const char* name);
int sm_filter_chain_set_param(sm_filter_chain* h, int32_t stage, const char* name, int32_t type, const char* text);
int sm_filter_chain_valid(const sm_filter_chain* h, int32_t stage);
int sm_filter_chain_set_seed(sm_filter_chain* h, uint64_t seed);
int sm_filter_chain_filter(sm_filter_chain* h, const float* points, int64_t n, int64_t stride_bytes, float* out,
                           int64_t capacity, int64_t* m_out, int32_t* kept_index);
int sm_filter_chain_filter_device(sm_filter_chain* h, const float* dev_points, int64_t n, int64_t stride_bytes,
                                  float* dev_out, int64_t capacity, int64_t* m_out, int32_t* dev_kept_index,
                                  void* cuda_stream);
/* Points after each stage of the last call (counts[k] for k < n); returns the number of stages. */
int sm_filter_chain_stage_counts(const sm_filter_chain* h, int64_t* counts, int32_t n);
/* Device time of each stage of the last call, from CUDA events (a fused run of point-wise stages is reported on its
 * first stage, the initial gather on the first step); returns the number of stages. */
int sm_filter_chain_stage_ms(const sm_filter_chain* h, float* ms, int32_t n);

int sm_device_count(void);
const char* sm_version(void);

#ifdef __cplusplus
}
#endif
#endif /* SM_B200_H_ */
