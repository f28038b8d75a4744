// registrators_b200.h — drop-in C++ matcher for the StaticMapping tree, backed by
// libsm_b200.so (C ABI: include/sm_b200.h).
//
// Compile this header INSIDE the reference tree (it needs the reference's own headers:
// registrators/interface.h, builder/data/cloud_types.h, Eigen, glog).  It is not compiled in
// the sm_b200 repository, where those dependencies do not exist; tests/test_adapter_syntax.py
// checks its syntax against minimal stand-in headers.
//
//   registrator::IcpFastB200 replaces registrator::IcpFast (registrators/icp_fast.h:37-62):
//   same base class, same overrides, same option names, same CHECK behaviour.
#ifndef ADAPTER_REGISTRATORS_B200_H_
#define ADAPTER_REGISTRATORS_B200_H_

#include <stdio.h>

#include <algorithm>
#include <memory>
#include <string>
#include <vector>

#include "registrators/interface.h"
#include "sm_b200.h"

namespace static_map {
namespace registrator {

// float option -> text without losing bits (std::to_string prints 6 fixed decimals)
inline std::string OptionText(float v) {
  char buf[32];
  snprintf(buf, sizeof(buf), "%.9g", static_cast<double>(v));
  return buf;
}

class IcpFastB200 : public Interface {
 public:
  USE_REGISTRATOR_CLOUDS;

  explicit IcpFastB200(int device = 0) : Interface() {
    this->type_ = kFastIcp;
    const int rc = sm_create(SM_TYPE_FAST_ICP, device, &handle_);
    CHECK_EQ(rc, 0) << "sm_create failed (" << rc << "): no CUDA device / no CPU fallback";
    // same registry as IcpFast::IcpFast (icp_fast.cc:411-418): InitWithXml writes through
    // these pointers, InitWithOptions forwards the values to the engine.
    REG_REGISTRATOR_INNER_OPTION("knn_normal_estimate", OptionItemDataType::kInt32,
                                 options_.knn_for_normal_estimate);
    REG_REGISTRATOR_INNER_OPTION("max_iteration", OptionItemDataType::kInt32,
                                 options_.max_iteration);
    REG_REGISTRATOR_INNER_OPTION("dist_outlier_ratio", OptionItemDataType::kFloat32,
                                 options_.dist_outlier_ratio);
  }
  ~IcpFastB200() override { sm_destroy(handle_); }

  PROHIBIT_COPY_AND_ASSIGN(IcpFastB200);

  void InitWithOptions() override {
    Check(sm_set_option(handle_, "max_iteration", std::to_string(options_.max_iteration).c_str()));
    Check(sm_set_option(handle_, "dist_outlier_ratio", OptionText(options_.dist_outlier_ratio).c_str()));
  }

  // icp_fast.cc:421-425
  void SetInputSource(InnerCloudPtr cloud) override {
    CHECK(cloud);
    CHECK(cloud->GetEigenCloud());
    const auto& pts = cloud->GetEigenCloud()->points;          // 3xN, column-major doubles
    Check(sm_set_input_source(handle_, pts.data(), pts.cols()));
  }

  // icp_fast.cc:427-431
  void SetInputTarget(InnerCloudPtr cloud) override {
    CHECK(cloud);
    CHECK(cloud->GetEigenCloud());
    CHECK(cloud->GetEigenCloud()->HasNormals());
    const auto& ec = *cloud->GetEigenCloud();
    Check(sm_set_input_target(handle_, ec.points.data(), ec.normals.data(), ec.points.cols()));
  }

  // icp_fast.cc:455-529
  bool Align(const Eigen::Matrix4d& guess, Eigen::Matrix4d& result) override {  // NOLINT
    const int rc = sm_align(handle_, guess.data(), result.data());  // both column-major
    Check(rc);
    this->final_score_ = sm_get_fitness_score(handle_);
    return rc == 1;
  }

  // hooks of AlignBatch (below)
  sm_handle* handle() const { return handle_; }
  void PrepareBatch() {}
  void SetFinalScore(double score) { this->final_score_ = score; }

 private:
  void Check(int rc) const {
    CHECK_GE(rc, 0) << "sm_b200: " << sm_last_error(handle_);   // reference aborts via glog
  }

  sm_handle* handle_ = nullptr;
  struct {
    int32_t knn_for_normal_estimate = 7;
    int32_t max_iteration = 100;
    float dist_outlier_ratio = 0.7;
  } options_;
};

// registrator::Ndt (registrators/ndt.h, ndt.cc:28-64) and registrator::NdtWithGicp
// (ndt_gicp.h, ndt_gicp.cc:28-112) keep the caller's float cloud (base-class SetInput*,
// interface.cc:38-60) and hand it over at Align: std::vector<InnerPointType>, 20-byte stride.
template <int kType>
class FloatCloudMatcherB200 : public Interface {
 public:
  USE_REGISTRATOR_CLOUDS;
  explicit FloatCloudMatcherB200(int device = 0) : Interface() {
    this->type_ = static_cast<Type>(kType);
    const int rc = sm_create(kType, device, &handle_);
    CHECK_EQ(rc, 0) << "sm_create failed (" << rc << ")";
  }
  ~FloatCloudMatcherB200() override { sm_destroy(handle_); }

  bool Align(const Eigen::Matrix4d& guess, Eigen::Matrix4d& result) override {  // NOLINT
    if (!this->source_cloud_ || !this->target_cloud_) {
      if (kType == SM_TYPE_NDT) return false;                 // ndt.cc:40-42
      CHECK(this->source_cloud_ && this->target_cloud_);      // NdtWithGicp dereferences them
    }
    PrepareBatch();
    const int rc = sm_align(handle_, guess.data(), result.data());
    CheckRc(rc);
    this->final_score_ = sm_get_fitness_score(handle_);
    return rc == 1;
  }

  // hooks of AlignBatch (below): the clouds kept by the base class go to the engine
  sm_handle* handle() const { return handle_; }
  void PrepareBatch() {
    CHECK(this->source_cloud_ && this->target_cloud_);
    const auto& s = this->source_cloud_->GetInnerCloud()->points;
    const auto& t = this->target_cloud_->GetInnerCloud()->points;
    CheckRc(sm_set_input_source_f32(handle_, &s[0].x, static_cast<int64_t>(s.size()),
                                    sizeof(data::InnerPointType)));
    CheckRc(sm_set_input_target_f32(handle_, &t[0].x, static_cast<int64_t>(t.size()),
                                    sizeof(data::InnerPointType)));
  }
  void SetFinalScore(double score) { this->final_score_ = score; }

 protected:
  void CheckRc(int rc) const { CHECK_GE(rc, 0) << "sm_b200: " << sm_last_error(handle_); }
  sm_handle* handle_ = nullptr;
};

class NdtB200 : public FloatCloudMatcherB200<SM_TYPE_NDT> {   // registers no option, like Ndt
 public:
  explicit NdtB200(int device = 0) : FloatCloudMatcherB200<SM_TYPE_NDT>(device) {}
};

class NdtWithGicpB200 : public FloatCloudMatcherB200<SM_TYPE_NDT_WITH_GICP> {
 public:
  explicit NdtWithGicpB200(int device = 0) : FloatCloudMatcherB200<SM_TYPE_NDT_WITH_GICP>(device) {
    REG_REGISTRATOR_INNER_OPTION("use_ndt", OptionItemDataType::kBool, options_.use_ndt);            // ndt_gicp.cc:31-36
    REG_REGISTRATOR_INNER_OPTION("using_voxel_filter", OptionItemDataType::kBool, options_.using_voxel_filter);
    REG_REGISTRATOR_INNER_OPTION("voxel_resolution", OptionItemDataType::kFloat32, options_.voxel_resolution);
  }
  void InitWithOptions() override {
    CheckRc(sm_set_option(handle_, "use_ndt", options_.use_ndt ? "1" : "0"));
    CheckRc(sm_set_option(handle_, "using_voxel_filter", options_.using_voxel_filter ? "1" : "0"));
    CheckRc(sm_set_option(handle_, "voxel_resolution", OptionText(options_.voxel_resolution).c_str()));
  }

 private:
  struct { float voxel_resolution = 0.2; bool using_voxel_filter = true; bool use_ndt = true; } options_;
};

// Stand-in for registrator::IcpUsingPointMatcher (icp_pointmatcher.h, .cc:125-247): the default
// libpointmatcher chain (random reading filter 0.9, surface-normal reference filter knn 7, k-d
// tree eps 3.16, trimmed 0.7, point-to-plane, 150 iterations / differential checker) run by the
// IcpFast kernels; Align() is false below score 0.6 (.cc:145).  Registers no option.  It is what
// loop_detector.cc:304-308 would construct instead of `new IcpUsingPointMatcher`.
class IcpUsingPointMatcherB200 : public FloatCloudMatcherB200<SM_TYPE_ICP_PM> {
 public:
  explicit IcpUsingPointMatcherB200(int device = 0) : FloatCloudMatcherB200<SM_TYPE_ICP_PM>(device) {}
};

// MotionCompensation (builder/map_builder.cc:232-257) on the GPU: same signature as the static
// function it replaces, so the two call sites (:325-327, :344-347) stay as they are.
inline void MotionCompensationB200(const data::InnerCloudType& raw_cloud, const Eigen::Matrix4d& delta_transform,
                                   data::InnerCloudType* const output_cloud, int device = 0) {
  CHECK(output_cloud);
  output_cloud->stamp = raw_cloud.stamp;
  output_cloud->points.resize(raw_cloud.points.size());
  if (raw_cloud.points.empty()) return;
  const int rc = sm_motion_compensation(device, &raw_cloud.points[0].x, static_cast<int64_t>(raw_cloud.points.size()),
                                        sizeof(data::InnerPointType), delta_transform.data(),
                                        &output_cloud->points[0].x);
  CHECK_EQ(rc, 0) << "MotionCompensation: factor outside [0, 1] (common/math.h:201) or CUDA failure";
}

// Batched CloseLoop / SubmapPairMatch: the reference starts one task (TBB / thread pool) per candidate
// pair, each constructing a matcher and calling Align (back_end/loop_detector.cc:216-228,304-308;
// builder/map_builder.cc:655,706-708).  With the engine ONE thread aligns all the candidates: the
// matchers have their clouds set as usual, AlignBatch enqueues every Align before it waits for the
// first result.  ok[i] / results[i] are what matchers[i]->Align(guesses[i], results[i]) would give.
template <typename MatcherB200>
inline void AlignBatch(const std::vector<MatcherB200*>& matchers, const std::vector<Eigen::Matrix4d>& guesses,
                       std::vector<Eigen::Matrix4d>* results, std::vector<bool>* ok) {
  CHECK(results && ok);
  CHECK_EQ(matchers.size(), guesses.size());
  const size_t n = matchers.size();
  std::vector<sm_handle*> handles(n);
  std::vector<double> g(16 * n), r(16 * n);
  std::vector<int32_t> rc(n);
  for (size_t i = 0; i < n; ++i) {
    matchers[i]->PrepareBatch();
    handles[i] = matchers[i]->handle();
    std::copy(guesses[i].data(), guesses[i].data() + 16, g.begin() + 16 * i);   // column-major, like Eigen
  }
  sm_align_batch(handles.data(), static_cast<int32_t>(n), g.data(), r.data(), rc.data());
  results->resize(n); ok->resize(n);
  for (size_t i = 0; i < n; ++i) {
    CHECK_GE(rc[i], 0) << "sm_b200: " << sm_last_error(handles[i]);               // reference aborts via glog
    std::copy(r.begin() + 16 * i, r.begin() + 16 * (i + 1), (*results)[i].data());
    (*ok)[i] = rc[i] != 0;
    matchers[i]->SetFinalScore(sm_get_fitness_score(handles[i]));
  }
}

// pre_processers::filter::VoxelGrid::Filter (pre_processors/filter_voxel_grid.cc:37-78) on the GPU:
// the body of that member becomes
//   this->FilterPrepare(cloud); registrator::VoxelGridFilterB200(*this->inner_cloud_, voxel_size_, cloud.get());
// Output points come in ascending voxel order instead of unordered_map iteration order.
inline void VoxelGridFilterB200(const data::InnerCloudType& input, float voxel_size,
                                data::InnerCloudType* const output, int device = 0) {
  CHECK(output);
  output->points.resize(input.points.size());
  int64_t m = 0;
  if (!input.points.empty()) {
    const int rc = sm_voxel_grid_filter(device, &input.points[0].x, static_cast<int64_t>(input.points.size()),
                                        sizeof(data::InnerPointType), voxel_size, &output->points[0].x, &m);
    // non-finite points are dropped by the engine (the reference keeps running on such input too).
    // SM_ERR_BAD_ARGUMENT is left for a cloud spanning >= 2^21 voxels along an axis or an invalid voxel
    // size (the reference refuses that one in ConfigsValid()): report and pass the cloud through
    // unfiltered rather than abort the mapper; only CUDA failures are fatal.
    CHECK_NE(rc, SM_ERR_CUDA) << "sm_voxel_grid_filter: CUDA failure";
    CHECK_NE(rc, SM_ERR_NO_DEVICE) << "sm_voxel_grid_filter: no CUDA device (no CPU fallback)";
    if (rc != 0) {
      LOG(ERROR) << "sm_voxel_grid_filter refused the cloud (" << rc << "): passing it through unfiltered";
      output->points = input.points;
      return;
    }
  }
  output->points.resize(m);
}

// descriptor::M2dp::setInputCloud + getFinalDescriptor on the GPU (descriptor/m2dp.cc:129-153): the body of
// setInputCloud becomes   return registrator::M2dpB200(*source, r_, max_distance_, t_, p_, q_, &descriptor_);
inline bool M2dpB200(const data::InnerCloudType& source, double r, double max_distance, int32_t t, int32_t p,
                     int32_t q, std::vector<float>* descriptor, int device = 0) {
  CHECK(descriptor);
  const int64_t len = sm_m2dp_descriptor_length(r, max_distance, t, p, q);
  if (len < 0) return false;                              // "r is too small" (m2dp.cc:64-67)
  if (source.points.empty()) return false;                // "source is empty" (:130-133)
  descriptor->assign(static_cast<size_t>(len), 0.f);
  const int rc = sm_m2dp(device, &source.points[0].x, static_cast<int64_t>(source.points.size()),
                         sizeof(data::InnerPointType), r, max_distance, t, p, q, descriptor->data(), len, nullptr);
  CHECK_GE(rc, 0) << "sm_m2dp failed (" << rc << ")";
  return rc == 1;
}

// EigenPointCloud::CalculateNormals on the GPU (cloud_types.cc:347-368); call sites
// map_builder.cc:286,389 and submap.cc:161.
inline void CalculateNormalsB200(data::EigenPointCloud* cloud, int device = 0) {
  CHECK(cloud);
  const int64_t n = cloud->points.cols();
  Eigen::MatrixXd pts(3, n), nrm(3, n);
  int64_t m = 0;
  const int rc = sm_calculate_normals(device, cloud->points.data(), n, pts.data(), nrm.data(), &m);
  CHECK_EQ(rc, 0) << "sm_calculate_normals failed";
  cloud->points = pts.leftCols(m);
  cloud->normals = nrm.leftCols(m);
}

// builder::MultiResolutionVoxelMap (builder/multi_resolution_voxel_map.{h,cc}) on the GPU: the map stays on the
// device across inserts.  Semantics are the reference's run by one thread; output comes in ascending voxel order
// (include/sm_b200.h lists the deviations).  INTEGRATION.md shows the members of the reference class forwarding here.
class MultiResolutionVoxelMapB200 {
 public:
  explicit MultiResolutionVoxelMapB200(int device = 0, int64_t expected_voxels = 1 << 22)
      : device_(device), expected_voxels_(expected_voxels) {}
  ~MultiResolutionVoxelMapB200() { if (handle_) sm_mrvm_destroy(handle_); }
  MultiResolutionVoxelMapB200(const MultiResolutionVoxelMapB200&) = delete;
  MultiResolutionVoxelMapB200& operator=(const MultiResolutionVoxelMapB200&) = delete;

  // Initialise (:42-48), from the reference's MrvmSettings (or anything with its field names)
  template <typename Settings>
  void Initialise(const Settings& s) {
    sm_mrvm_settings st;
    st.output_average = s.output_average; st.output_rgb = s.output_rgb; st.use_max_intensity = s.use_max_intensity;
    st.prob_threshold = s.prob_threshold; st.low_resolution = s.low_resolution; st.high_resolution = s.high_resolution;
    st.hit_prob = s.hit_prob; st.miss_prob = s.miss_prob; st.z_offset = s.z_offset;
    st.max_point_num_in_cell = s.max_point_num_in_cell;
    if (handle_) sm_mrvm_destroy(handle_);
    handle_ = nullptr;
    const int rc = sm_mrvm_create(device_, &st, expected_voxels_, &handle_);
    CHECK_EQ(rc, 0) << "sm_mrvm_create failed (" << rc << "): invalid MrvmSettings or no CUDA device";
  }

  void SetOffsetZ(const float& offset) { CHECK_EQ(sm_mrvm_set_offset_z(handle_, offset), 0); }

  // InsertPointCloud (:54-123); origin = the sensor position (x, y, z)
  void InsertPointCloud(const data::InnerCloudType& cloud, const float* origin) {
    CHECK(handle_);
    if (cloud.points.empty()) {                               // "cloud is empty." (:56-59)
      LOG(ERROR) << "cloud is empty.";
      return;
    }
    const int rc = sm_mrvm_insert(handle_, &cloud.points[0].x, static_cast<int64_t>(cloud.points.size()),
                                  sizeof(data::InnerPointType), origin);
    CHECK_GE(rc, 0) << "sm_mrvm_insert failed (" << rc << "): voxel index outside +-2^20 or CUDA failure";
    if (rc > 0) LOG(ERROR) << rc << " points with a non-finite coordinate dropped";
  }

  size_t size() const { return handle_ ? static_cast<size_t>(sm_mrvm_size(handle_)) : 0; }

  // OutputToPointCloud (:125-215): {x, y, z, intensity} records (rgb = false, the PointXYZI overload) or
  // {x, y, z, grey level} (rgb = true, PointXYZRGB with r = g = b = grey)
  void OutputToPointCloud(float threshold, bool rgb, std::vector<float>* xyzv) const {
    CHECK(handle_ && xyzv);
    int64_t m = 0;
    int rc = sm_mrvm_output(handle_, threshold, rgb ? 1 : 0, nullptr, 0, &m);
    xyzv->assign(static_cast<size_t>(4 * m), 0.f);
    if (m > 0) rc = sm_mrvm_output(handle_, threshold, rgb ? 1 : 0, xyzv->data(), m, &m);
    CHECK_EQ(rc, 0) << "sm_mrvm_output failed (" << rc << ")";
  }

 private:
  int device_;
  int64_t expected_voxels_;
  sm_mrvm* handle_ = nullptr;
};

// pre_processers::filter::Factory (pre_processors/filter_factory.cc:63-123) on the GPU.  Stages come in XML order as
// (filter name, [(param name, type attribute, text)]); Filter runs them on a data::InnerCloudType.  Semantics and
// deviations: include/sm_b200.h (sm_filter_chain_*).
class FilterFactoryB200 {
 public:
  struct Param { std::string name; int type; std::string text; };
  explicit FilterFactoryB200(int device = 0, uint64_t seed = 0) {
    const int rc = sm_filter_chain_create(device, &handle_);
    CHECK_EQ(rc, 0) << "sm_filter_chain_create failed (" << rc << "): no CUDA device";
    sm_filter_chain_set_seed(handle_, seed);
  }
  ~FilterFactoryB200() { if (handle_) sm_filter_chain_destroy(handle_); }
  FilterFactoryB200(const FilterFactoryB200&) = delete;
  FilterFactoryB200& operator=(const FilterFactoryB200&) = delete;

  // Factory::InitFromXmlNode for one <filter>: an unknown name or parameter is a CHECK failure here
  void AddFilter(const std::string& name, const std::vector<Param>& params) {
    const int stage = sm_filter_chain_add(handle_, name.c_str());
    CHECK_GE(stage, 0) << name << " not supported";
    for (const Param& p : params)
      CHECK_EQ(sm_filter_chain_set_param(handle_, stage, p.name.c_str(), p.type, p.text.c_str()), 0)
          << name << ": cannot set " << p.name;
  }

  // Factory::Filter: `cloud` (a data::InnerCloudType::Ptr, or any pointer to one) in, the filtered cloud out
  template <typename CloudPtr>
  void Filter(const CloudPtr& cloud) {
    CHECK(cloud);
    const int64_t n = static_cast<int64_t>(cloud->points.size());
    if (n == 0) return;
    std::vector<data::InnerPointType> out(static_cast<size_t>(n));
    int64_t m = 0;
    const int rc = sm_filter_chain_filter(handle_, &cloud->points[0].x, n, sizeof(data::InnerPointType), &out[0].x, n,
                                          &m, nullptr);
    CHECK_EQ(rc, 0) << "sm_filter_chain_filter failed (" << rc << "): invalid stage or CUDA failure";
    out.resize(static_cast<size_t>(m));
    cloud->points.assign(out.begin(), out.end());
  }

 private:
  sm_filter_chain* handle_ = nullptr;
};

}  // namespace registrator
}  // namespace static_map

#endif  // ADAPTER_REGISTRATORS_B200_H_
