// nano_gicp.hpp — drop-in C++ facade: the class surface of the reference's
// nano_gicp::NanoGICP<PointSource,PointTarget> (reference include/nano_gicp/nano_gicp.hpp:58-137 on top of
// include/nano_gicp/lsq_registration.hpp:54-116 and pcl::Registration), implemented as a thin forwarder to the C ABI
// of libnanogicp_b200.so (include/nanogicp_c.h).  OdomNode's call sites (reference src/dlo/odom.cc:100-120,
// 472-528, 792-852, 1160-1174) compile against it unchanged, including the public members they poke:
//   gicp.source_kdtree_ = gicp_s2s.source_kdtree_;      -> ngicp_share_source      (no rebuild, no copy)
//   gicp.source_covs_.clear();                          -> ngicp_clear_covs
//   gicp.source_covs_   = gicp_s2s.source_covs_;        -> ngicp_share_source_covs (stays in HBM)
//   keyframe_normals.push_back(gicp_s2s.getSourceCovariances());   host vector materialised on demand
//   gicp.setTargetCovariances(submap_normals);          -> ngicp_set_target_covs   (H2D of Matrix4d records)
//
// Host code only (C++14, no CUDA headers needed).  With PCL and Eigen on the include path their types are
// used; otherwise the minimal stand-ins of compat/pcl_eigen_min.hpp (same layouts).
#ifndef NANO_GICP_NANO_GICP_HPP
#define NANO_GICP_NANO_GICP_HPP

#include <cfloat>
#include <cstdio>
#include <cstring>
#include <limits>
#include <memory>
#include <stdexcept>
#include <string>
#include <vector>

#if defined(__has_include)
#if __has_include(<pcl/point_cloud.h>) && __has_include(<Eigen/Core>) && !defined(NANO_GICP_B200_FORCE_COMPAT)
#define NANO_GICP_B200_HAVE_PCL 1
#endif
#endif
#ifdef NANO_GICP_B200_HAVE_PCL
#include <Eigen/Core>
#include <Eigen/Geometry>
#include <pcl/point_cloud.h>
#include <pcl/point_types.h>
#else
#include "compat/pcl_eigen_min.hpp"
#endif

#include "../nanogicp_c.h"

namespace nano_gicp {

// include/nano_gicp/gicp/gicp_settings.hpp:47
enum class RegularizationMethod { NONE, MIN_EIG, NORMALIZED_MIN_EIG, PLANE, FROBENIUS };
// include/nano_gicp/lsq_registration.hpp:54
enum class LSQ_OPTIMIZER_TYPE { GaussNewton, LevenbergMarquardt };

typedef std::vector<Eigen::Matrix4d, Eigen::aligned_allocator<Eigen::Matrix4d>> CovarianceVectorHost;

namespace detail {
struct Handle {
  ngicp_t* h = nullptr;
  Handle(int device) {
    int rc = ngicp_create(device, &h);
    if (rc != NGICP_OK || !h) {
      std::fprintf(stderr, "[NanoGICP-B200] ngicp_create failed (rc=%d): no CUDA device; this library has no CPU fallback\n", rc);
      h = nullptr;
    }
  }
  ~Handle() { if (h) ngicp_destroy(h); }
  Handle(const Handle&) = delete;
  Handle& operator=(const Handle&) = delete;
};
inline void report(ngicp_t* h, int rc, const char* where) {
  if (rc < 0) std::fprintf(stderr, "[NanoGICP-B200] %s: %s\n", where, h ? ngicp_last_error(h) : "no handle");
}
}  // namespace detail

// What `source_covs_` / `target_covs_` are in this build: a vector of Matrix4d that lives in HBM and is
// mirrored to the host only when somebody reads it.  Assigning one to another shares the device buffer.
class CovarianceVector {
 public:
  CovarianceVector() {}
  void bind(ngicp_t* h, int which) { h_ = h; which_ = which; }

  size_t size() const { return h_ ? ngicp_covs_size(h_, which_) : 0; }
  bool empty() const { return size() == 0; }
  void clear() {
    if (h_) ngicp_clear_covs(h_, which_);
    host_valid_ = false;
  }
  // device -> device (gicp.source_covs_ = gicp_s2s.source_covs_)
  CovarianceVector& operator=(const CovarianceVector& o) {
    if (this == &o || !h_) return *this;
    if (which_ == NGICP_SOURCE && o.which_ == NGICP_SOURCE && o.h_) detail::report(h_, ngicp_share_source_covs(h_, o.h_), "source_covs_ =");
    else *this = o.host();
    host_valid_ = false;
    return *this;
  }
  // host -> device
  CovarianceVector& operator=(const CovarianceVectorHost& v) {
    if (!h_) return *this;
    const double* p = v.empty() ? nullptr : reinterpret_cast<const double*>(v.data());
    int rc = which_ == NGICP_SOURCE ? ngicp_set_source_covs(h_, p, v.size()) : ngicp_set_target_covs(h_, p, v.size());
    detail::report(h_, rc, "set covariances");
    host_valid_ = false;
    return *this;
  }
  // device -> host, on demand
  const CovarianceVectorHost& host() const {
    const size_t n = size();
    if (!host_valid_ || host_.size() != n) {
      host_.resize(n);
      if (n) {
        int rc = which_ == NGICP_SOURCE ? ngicp_get_source_covs(h_, reinterpret_cast<double*>(host_.data()), n)
                                        : ngicp_get_target_covs(h_, reinterpret_cast<double*>(host_.data()), n);
        detail::report(h_, rc, "get covariances");
      }
      host_valid_ = true;
    }
    return host_;
  }
  operator const CovarianceVectorHost&() const { return host(); }
  CovarianceVectorHost::const_iterator begin() const { return host().begin(); }
  CovarianceVectorHost::const_iterator end() const { return host().end(); }
  const Eigen::Matrix4d& operator[](size_t i) const { return host()[i]; }
  void invalidate_host() { host_valid_ = false; }
  void swap_binding(CovarianceVector& o) { std::swap(host_valid_, o.host_valid_); host_.swap(o.host_); }

 private:
  ngicp_t* h_ = nullptr;
  int which_ = NGICP_SOURCE;
  mutable CovarianceVectorHost host_;
  mutable bool host_valid_ = false;
};

}  // namespace nano_gicp

namespace nanoflann {
// Stand-in for the reference's kd-tree wrapper type (include/nano_gicp/nanoflann.hpp:54-108): in this build the
// search index is the uniform grid inside the handle; this object only names "the index of that handle's
// source/target cloud" so that the reference's shared_ptr assignments keep working.
template <typename PointT>
class KdTreeFLANN {
 public:
  typedef typename pcl::PointCloud<PointT>::ConstPtr PointCloudConstPtr;
  ngicp_t* owner = nullptr;
  PointCloudConstPtr cloud;
  PointCloudConstPtr getInputCloud() const { return cloud; }
};
}  // namespace nanoflann

namespace nano_gicp {

// `source_kdtree_` / `target_kdtree_`: behaves like the reference's std::shared_ptr<KdTreeFLANN> for the
// operations OdomNode performs; assigning another object's source index shares the device index at once.
template <typename PointT>
class IndexSlot {
 public:
  typedef nanoflann::KdTreeFLANN<PointT> Tree;
  void bind(ngicp_t* h, int which) { h_ = h; which_ = which; p_.reset(new Tree()); p_->owner = h; }
  IndexSlot& operator=(const IndexSlot& o) {
    if (this == &o) return *this;
    p_ = o.p_;
    if (h_ && o.h_ && which_ == NGICP_SOURCE && o.which_ == NGICP_SOURCE && h_ != o.h_) detail::report(h_, ngicp_share_source(h_, o.h_), "source_kdtree_ =");
    return *this;
  }
  Tree* operator->() const { return p_.get(); }
  Tree& operator*() const { return *p_; }
  Tree* get() const { return p_.get(); }
  explicit operator bool() const { return (bool)p_; }
  void reset(Tree* t = nullptr) { p_.reset(t); if (t) t->owner = h_; }
  void swap(IndexSlot& o) { p_.swap(o.p_); }

 private:
  std::shared_ptr<Tree> p_;
  ngicp_t* h_ = nullptr;
  int which_ = NGICP_SOURCE;
};

template <typename PointSource, typename PointTarget>
class NanoGICP {
 public:
  using Scalar = float;
  using Matrix4 = Eigen::Matrix4f;
  using PointCloudSource = pcl::PointCloud<PointSource>;
  using PointCloudSourcePtr = typename PointCloudSource::Ptr;
  using PointCloudSourceConstPtr = typename PointCloudSource::ConstPtr;
  using PointCloudTarget = pcl::PointCloud<PointTarget>;
  using PointCloudTargetPtr = typename PointCloudTarget::Ptr;
  using PointCloudTargetConstPtr = typename PointCloudTarget::ConstPtr;

  EIGEN_MAKE_ALIGNED_OPERATOR_NEW

  explicit NanoGICP(int device = 0) : handle_(new detail::Handle(device)) {
    ngicp_params_default(&prm_);   // k 20, FLT_MAX, PLANE (nano_gicp_impl.hpp:57-61); 64, 2e-3, 5e-4, LM, 10, 1e-9 (lsq_registration_impl.hpp:52-59)
    source_kdtree_.bind(h(), NGICP_SOURCE);
    target_kdtree_.bind(h(), NGICP_TARGET);
    source_covs_.bind(h(), NGICP_SOURCE);
    target_covs_.bind(h(), NGICP_TARGET);
    final_transformation_ = Matrix4::Identity();
    final_hessian_.setIdentity();
  }
  virtual ~NanoGICP() {}
  NanoGICP(const NanoGICP&) = delete;
  NanoGICP& operator=(const NanoGICP&) = delete;

  // ---- nano_gicp.hpp:82-84 ----------------------------------------------------------------------
  void setNumThreads(int) {}   // OpenMP knob; nothing to do on the GPU
  // Every setter changes ONE field and keeps it only if the library accepts it (a rejected value used to stay in prm_
  // and make every later setter fail as well).  A value the GPU path cannot honour is a configuration error and is
  // reported where it is made: the reference accepts any k, this build k in [1, 128] (k <= 32: warp-wide
  // result set, the tuned kernels; 33..128: a shared-memory result set on the warp-search path).
  void setCorrespondenceRandomness(int k) {
    if (!set_field(&ngicp_params::k_correspondences, k))
      throw std::invalid_argument("NanoGICP-B200: setCorrespondenceRandomness(" + std::to_string(k) + "): this build supports 1 <= k <= 128");
  }
  void setRegularizationMethod(RegularizationMethod m) { set_field(&ngicp_params::regularization_method, (int)m); }

  // ---- pcl::Registration setters used at odom.cc:100-120 -----------------------------------------
  void setMaxCorrespondenceDistance(double d) { set_field(&ngicp_params::max_correspondence_distance, d); }
  void setMaximumIterations(int n) { set_field(&ngicp_params::max_iterations, n); }
  void setTransformationEpsilon(double e) { set_field(&ngicp_params::transformation_epsilon, e); }
  void setEuclideanFitnessEpsilon(double) {}               // never read by NanoGICP (SURVEY A8)
  void setRANSACIterations(int) {}
  void setRANSACOutlierRejectionThreshold(double) {}
  template <class TreePtr> void setSearchMethodSource(const TreePtr&, bool = false) {}
  template <class TreePtr> void setSearchMethodTarget(const TreePtr&, bool = false) {}
  double getMaxCorrespondenceDistance() const { return prm_.max_correspondence_distance; }
  int getMaximumIterations() const { return prm_.max_iterations; }

  // ---- lsq_registration.hpp:81-85 ---------------------------------------------------------------
  void setRotationEpsilon(double e) { set_field(&ngicp_params::rotation_epsilon, e); }
  void setInitialLambdaFactor(double f) { set_field(&ngicp_params::lm_init_lambda_factor, f); }
  void setDebugPrint(bool) {}
  const Eigen::Matrix<double, 6, 6>& getFinalHessian() const { return final_hessian_; }

  // ---- B200-side knobs ---------------------------------------------------------------------------
  void setGridCellSize(float c) { set_field(&ngicp_params::grid_cell_size, c); }
  void setAlignMode(int mode) { set_field(&ngicp_params::align_mode, mode); }
  void setKnnPath(int path) { set_field(&ngicp_params::knn_path, path); }
  void setVoxelPath(int path) { set_field(&ngicp_params::voxel_path, path); }
  void setIndexPath(int path) { set_field(&ngicp_params::index_path, path); }
  void setFillOutputCloud(bool f) { fill_output_ = f; }
  ngicp_t* handle() const { return h(); }

  // ---- clouds (nano_gicp_impl.hpp:90-139) --------------------------------------------------------
  virtual void swapSourceAndTarget() {
    input_.swap(target_);
    source_kdtree_.swap(target_kdtree_);
    source_covs_.swap_binding(target_covs_);
    if (h()) ngicp_swap(h());
  }
  virtual void clearSource() { input_.reset(); if (h()) ngicp_clear_source(h()); source_covs_.invalidate_host(); }
  virtual void clearTarget() { target_.reset(); device_target_ = false; if (h()) ngicp_clear_target(h()); target_covs_.invalidate_host(); }
  // the target was replaced behind the facade (KeyframeStore::setTarget): drop the cached host pointer and host covariances
  void forgetTarget() { target_.reset(); target_covs_.invalidate_host(); device_target_ = true; }

  virtual void setInputSource(const PointCloudSourceConstPtr& cloud) {
    if (input_ == cloud) return;
    if (!check_cloud(cloud, "setInputSource")) return;
    input_ = cloud;
    detail::report(h(), ngicp_set_source(h(), cloud->points.data(), cloud->points.size(), sizeof(PointSource)), "setInputSource");
    source_kdtree_->cloud = cloud;
    source_covs_.invalidate_host();
  }
  virtual void registerInputSource(const PointCloudSourceConstPtr& cloud) {
    if (input_ == cloud) return;
    if (!check_cloud(cloud, "setInputSource")) return;
    input_ = cloud;
    detail::report(h(), ngicp_register_source(h(), cloud->points.data(), cloud->points.size(), sizeof(PointSource)), "registerInputSource");
  }
  virtual void setInputTarget(const PointCloudTargetConstPtr& cloud) {
    if (target_ == cloud) return;
    if (!check_cloud(cloud, "setInputTarget")) return;
    target_ = cloud;
    device_target_ = false;
    detail::report(h(), ngicp_set_target(h(), cloud->points.data(), cloud->points.size(), sizeof(PointTarget)), "setInputTarget");
    target_kdtree_->cloud = cloud;
    target_covs_.invalidate_host();
  }
  PointCloudSourceConstPtr getInputSource() const { return input_; }
  PointCloudTargetConstPtr getInputTarget() const { return target_; }

  // ---- covariances (nano_gicp_impl.hpp:141-159) --------------------------------------------------
  virtual void setSourceCovariances(const CovarianceVectorHost& covs) { source_covs_ = covs; }
  virtual void setTargetCovariances(const CovarianceVectorHost& covs) { target_covs_ = covs; }
  // the reference returns true unconditionally (nano_gicp_impl.hpp:151-159); here false means "no covariances were made"
  virtual bool calculateSourceCovariances() {
    const int rc = h() ? ngicp_calc_source_covs(h()) : NGICP_E_STATE;
    detail::report(h(), rc, "calculateSourceCovariances");
    source_covs_.invalidate_host();
    return rc >= 0;
  }
  virtual bool calculateTargetCovariances() {
    const int rc = h() ? ngicp_calc_target_covs(h()) : NGICP_E_STATE;
    detail::report(h(), rc, "calculateTargetCovariances");
    target_covs_.invalidate_host();
    return rc >= 0;
  }
  const CovarianceVectorHost& getSourceCovariances() const { return source_covs_.host(); }
  const CovarianceVectorHost& getTargetCovariances() const { return target_covs_.host(); }

  // ---- pcl::Registration::align (SURVEY App. B2) -------------------------------------------------
  void align(PointCloudSource& output) { align(output, Matrix4::Identity()); }
  void align(PointCloudSource& output, const Matrix4& guess) {
    converged_ = false;
    final_transformation_ = Matrix4::Identity();
    if (!target_ && !device_target_) { std::fprintf(stderr, "[pcl::Registration::align] No input target dataset was given!\n"); return; }
    if (!input_) { std::fprintf(stderr, "[pcl::Registration::align] No input source dataset was given!\n"); return; }
    ngicp_result res;
    int rc = ngicp_align(h(), guess.data(), &res);
    detail::report(h(), rc, "align");
    // PCL's own early-outs (missing cloud / index) print and return with converged_ = false, like above.  Anything else
    // (a CUDA failure, fewer points than k, a sharded peer that never arrived) has no counterpart in the reference, and
    // returning silently would make OdomNode integrate an identity transform: raise instead.
    if (rc == NGICP_E_STATE) return;
    if (rc < 0) throw std::runtime_error(std::string("NanoGICP-B200: align failed: ") + (h() ? ngicp_last_error(h()) : "no handle"));
    std::memcpy(final_transformation_.data(), res.final_transformation, sizeof(float) * 16);
    std::memcpy(final_hessian_.data(), res.final_hessian, sizeof(double) * 36);
    converged_ = res.converged != 0;
    nr_iterations_ = res.nr_iterations;
    last_result_ = res;
    source_covs_.invalidate_host();   // lazily computed covariances may now exist
    target_covs_.invalidate_host();
    if (fill_output_) {
      // pcl::transformPointCloud(*input_, output, final_transformation_) (lsq_registration_impl.hpp:114)
      const size_t n = input_->points.size();
      if (&output != input_.get()) output = *input_;
      scratch_.resize(n * 4);
      if (n && ngicp_transform_source(h(), final_transformation_.data(), scratch_.data(), n) == NGICP_OK)
        for (size_t i = 0; i < n; i++) { output.points[i].x = scratch_[4 * i]; output.points[i].y = scratch_[4 * i + 1]; output.points[i].z = scratch_[4 * i + 2]; }
    }
  }
  Matrix4 getFinalTransformation() const { return final_transformation_; }
  // pcl::Registration::getFitnessScore(max_range): the mean squared distance from the source, transformed by
  // final_transformation_ (in float, as pcl::transformPointCloud), to its nearest target point, over the points whose
  // SQUARED distance is <= max_range — PCL compares the squared distance with max_range as given.  DBL_MAX when no point
  // qualifies.  PCL searches its own tree_, which DLO never builds (it calls setSearchMethodTarget(null, true)); this
  // version searches the handle's device index, so it works in every configuration, also after
  // KeyframeStore::setTarget.  A missing source, target or index prints and returns DBL_MAX; CUDA errors throw.
  double getFitnessScore(double max_range = std::numeric_limits<double>::max()) {
    double score = DBL_MAX;
    const int rc = ngicp_fitness_score(h(), final_transformation_.data(), max_range, &score, nullptr);
    if (rc == NGICP_E_STATE) {
      std::fprintf(stderr, "[pcl::Registration::getFitnessScore] %s\n", ngicp_last_error(h()));
      return DBL_MAX;
    }
    if (rc < 0) throw std::runtime_error(std::string("NanoGICP-B200: getFitnessScore failed: ") + (h() ? ngicp_last_error(h()) : "no handle"));
    return score;
  }
  bool hasConverged() const { return converged_; }
  const ngicp_result& getLastResult() const { return last_result_; }

 public:
  // public data members of the reference class (nano_gicp.hpp:121-125)
  IndexSlot<PointSource> source_kdtree_;
  IndexSlot<PointTarget> target_kdtree_;
  CovarianceVector source_covs_;
  CovarianceVector target_covs_;

 protected:
  ngicp_t* h() const { return handle_ ? handle_->h : nullptr; }
  // change one parameter; the handle is the judge: a rejected value is rolled back and reported
  template <class F, class V> bool set_field(F ngicp_params::*field, V value) {
    const F old = prm_.*field;
    prm_.*field = (F)value;
    if (!h()) return true;
    const int rc = ngicp_set_params(h(), &prm_);
    if (rc < 0) { detail::report(h(), rc, "set parameter"); prm_.*field = old; return false; }
    return true;
  }
  template <class CloudPtr> bool check_cloud(const CloudPtr& c, const char* who) const {
    if (!c || c->points.empty()) { std::fprintf(stderr, "[pcl::Registration::%s] Invalid or empty point cloud dataset given!\n", who); return false; }
    return h() != nullptr;
  }

  std::unique_ptr<detail::Handle> handle_;
  ngicp_params prm_;
  PointCloudSourceConstPtr input_;
  PointCloudTargetConstPtr target_;
  Matrix4 final_transformation_;
  Eigen::Matrix<double, 6, 6> final_hessian_;
  ngicp_result last_result_;
  bool converged_ = false;
  int nr_iterations_ = 0;
  bool fill_output_ = true;
  bool device_target_ = false;   // target assembled on the device by KeyframeStore::setTarget (no host cloud)
  std::vector<float> scratch_;
};

// pcl::VoxelGrid<PointT> with the three calls DLO makes (odom.cc:126-127, 460-463): setLeafSize, setInputCloud, filter
template <typename PointT>
class VoxelGrid {
 public:
  explicit VoxelGrid(int device = 0) : handle_(new detail::Handle(device)) {}
  void setLeafSize(float lx, float, float) { leaf_ = lx; }   // DLO always passes (r, r, r)
  void setInputCloud(const typename pcl::PointCloud<PointT>::ConstPtr& c) { in_ = c; }
  void filter(pcl::PointCloud<PointT>& out) {
    if (!in_ || !handle_->h) return;
    const size_t n = in_->points.size();
    std::vector<PointT> tmp(n ? n : 1);
    size_t m = 0;
    int rc = ngicp_voxel_filter(handle_->h, in_->points.data(), n, sizeof(PointT), leaf_, tmp.data(), tmp.size(), &m);
    detail::report(handle_->h, rc, "VoxelGrid::filter");
    if (rc == NGICP_W_VOXEL_OVERFLOW) std::fprintf(stderr, "[pcl::VoxelGrid::applyFilter] Leaf size is too small for the input dataset. Integer indices would overflow.\n");
    tmp.resize(m);
    out.points.swap(tmp);
    out.width = (uint32_t)m; out.height = 1; out.is_dense = true;
  }
 private:
  std::unique_ptr<detail::Handle> handle_;
  typename pcl::PointCloud<PointT>::ConstPtr in_;
  float leaf_ = 0.25f;
};

// ---- additive helpers (not part of the reference class; INTEGRATION.md section 5) ---------------------------------

// OdomNode::preprocessPoints (odom.cc:443-465) in one device pass: removeNaN + negative CropBox(+-crop_size; <= 0 skips
// it) + scan voxel grid (leaf <= 0 skips it)
template <typename PointT>
class Preprocessor {
 public:
  explicit Preprocessor(int device = 0) : handle_(new detail::Handle(device)) {}
  void setCropSize(float s) { crop_ = s; }
  void setLeafSize(float l) { leaf_ = l; }
  void filter(const pcl::PointCloud<PointT>& in, pcl::PointCloud<PointT>& out) {
    if (!handle_->h) return;
    const size_t n = in.points.size();
    std::vector<PointT> tmp(n ? n : 1);
    size_t m = 0;
    const float lo[3] = {-crop_, -crop_, -crop_}, hi[3] = {crop_, crop_, crop_};
    int rc = ngicp_preprocess(handle_->h, in.points.data(), n, sizeof(PointT), crop_ > 0.f ? lo : nullptr, crop_ > 0.f ? hi : nullptr, leaf_,
                              tmp.data(), tmp.size(), &m);
    detail::report(handle_->h, rc, "Preprocessor::filter");
    tmp.resize(m);
    out.points.swap(tmp);
    out.width = (uint32_t)m; out.height = 1; out.is_dense = true;
  }
  // pcl::fromROSMsg(*pc, *current_scan) (odom.cc:636-637) + preprocessPoints in the same device pass.  Msg is
  // sensor_msgs::PointCloud2 or anything with its members (width, height, point_step, row_step, is_bigendian, data,
  // fields[] with name / offset / datatype / count); the members of PointXYZI are matched as PCL does: same name,
  // datatype FLOAT32 (7), count 1.
  template <class Msg>
  void filterMsg(const Msg& msg, pcl::PointCloud<PointT>& out) {
    if (!handle_->h) return;
    ngicp_pc2_layout lay;
    lay.width = (unsigned)msg.width; lay.height = (unsigned)msg.height;
    lay.point_step = (unsigned)msg.point_step; lay.row_step = (unsigned)msg.row_step;
    lay.offset_x = lay.offset_y = lay.offset_z = lay.offset_intensity = -1;
    lay.is_bigendian = msg.is_bigendian ? 1 : 0;
    for (const auto& f : msg.fields) {
      if ((int)f.datatype != 7 || ((int)f.count != 1 && (int)f.count != 0)) continue;
      int* dst = f.name == "x" ? &lay.offset_x : f.name == "y" ? &lay.offset_y : f.name == "z" ? &lay.offset_z
                 : f.name == "intensity" ? &lay.offset_intensity : nullptr;
      if (dst && *dst < 0) *dst = (int)f.offset;
    }
    const size_t n = (size_t)lay.width * lay.height;
    std::vector<PointT> tmp(n ? n : 1);
    size_t m = 0;
    const float lo[3] = {-crop_, -crop_, -crop_}, hi[3] = {crop_, crop_, crop_};
    int rc = ngicp_preprocess_pointcloud2(handle_->h, msg.data.data(), &lay, crop_ > 0.f ? lo : nullptr, crop_ > 0.f ? hi : nullptr, leaf_,
                                          tmp.data(), tmp.size(), &m);
    detail::report(handle_->h, rc, "Preprocessor::filterMsg");
    tmp.resize(m);
    out.points.swap(tmp);
    out.width = (uint32_t)m; out.height = 1; out.is_dense = true;
  }
 private:
  std::unique_ptr<detail::Handle> handle_;
  float crop_ = 1.0f, leaf_ = 0.25f;
};

// Device-resident keyframes: what OdomNode keeps in `keyframes` / `keyframe_normals` and concatenates on the host
// (odom.cc:498-504, 1172-1178, 1315-1328), kept on the GPU (ngicp_kfstore_*).
class KeyframeStore {
 public:
  explicit KeyframeStore(int device = 0) { if (ngicp_kfstore_create(device, &s_) != NGICP_OK) s_ = nullptr; }
  ~KeyframeStore() { if (s_) ngicp_kfstore_destroy(s_); }
  KeyframeStore(const KeyframeStore&) = delete;
  KeyframeStore& operator=(const KeyframeStore&) = delete;
  size_t size() const { return s_ ? ngicp_kfstore_size(s_) : 0; }
  // after gicp_s2s.setInputSource(keyframe_cloud); gicp_s2s.calculateSourceCovariances();
  template <class Gicp> int push(Gicp& gicp_s2s) {
    size_t idx = 0;
    detail::report(gicp_s2s.handle(), ngicp_kfstore_push(s_, gicp_s2s.handle(), &idx), "KeyframeStore::push");
    return (int)idx;
  }
  // instead of gicp.setInputTarget(submap_cloud); gicp.setTargetCovariances(submap_normals);
  template <class Gicp> void setTarget(Gicp& gicp, const std::vector<int>& keyframe_indices) {
    detail::report(gicp.handle(), ngicp_kfstore_set_target(s_, gicp.handle(), keyframe_indices.data(), keyframe_indices.size()),
                   "KeyframeStore::setTarget");
    gicp.forgetTarget();
  }
 private:
  ngicp_kfstore_t* s_ = nullptr;
};

}  // namespace nano_gicp

#endif
