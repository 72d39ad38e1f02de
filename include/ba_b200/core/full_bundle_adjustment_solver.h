// Drop-in for core/full_bundle_adjustment_solver.h (reference :127-146).  Same namespace, class name,
// _BA_* aliases and public signatures; the body is a thin host shim over the C-ABI of ba_b200.h:
// registration keeps the reference's pointer-keyed bookkeeping (full_bundle_adjustment_solver.cpp:72-206),
// Solve packs the scaled copies into SoA host buffers, runs the device LM loop (ba_solve) and writes the
// results back through the user's pointers (:1011-1022).  Link with -lba_b200.
//
// Differences from the reference, all deliberate and documented in INTEGRATION.md:
//  * FinalizeParameters() is public and idempotent (README.md:39-57 calls it publicly; the header has it
//    private, :153) and Solve() invokes it itself, like the reference (:663);
//  * free parameters are numbered in insertion order (the reference uses unordered_map order);
//  * AddObservation is accepted before and after FinalizeParameters().
#ifndef _FULL_BUNDLE_ADJUSTMENT_SOLVER_H_
#define _FULL_BUNDLE_ADJUSTMENT_SOLVER_H_

#include <chrono>
#include <cstdint>
#include <iomanip>
#include <ios>
#include <iostream>
#include <limits>
#include <sstream>
#include <stdexcept>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "../../ba_b200.h"
#include "../eigen_shim.h"
#include "solver_option_and_summary.h"

namespace visual_navigation {
namespace analytic_solver {
using _BA_Numeric = double;
using _BA_Index = int;
using _BA_Size_t = int;
using _BA_Pixel = Eigen::Matrix<_BA_Numeric, 2, 1>;
using _BA_Point = Eigen::Matrix<_BA_Numeric, 3, 1>;
using _BA_Rotation3 = Eigen::Matrix<_BA_Numeric, 3, 3>;
using _BA_Position3 = Eigen::Matrix<_BA_Numeric, 3, 1>;
using _BA_Pose = Eigen::Transform<_BA_Numeric, 3, 1>;

struct _BA_Camera {
  _BA_Camera() {}
  _BA_Camera(const _BA_Camera &camera) {
    fx = camera.fx; fy = camera.fy; cx = camera.cx; cy = camera.cy;
    pose_this_to_cam0 = camera.pose_this_to_cam0;
  }
  _BA_Camera &operator=(const _BA_Camera &) = default;
  _BA_Numeric fx{0.0};
  _BA_Numeric fy{0.0};
  _BA_Numeric cx{0.0};
  _BA_Numeric cy{0.0};
  _BA_Pose pose_this_to_cam0;
};

struct _BA_Observation {
  int camera_index{-1};
  _BA_Pose *related_pose{nullptr};
  _BA_Point *related_point{nullptr};
  _BA_Pixel pixel{-1.0, -1.0};
};

class FullBundleAdjustmentSolver {
 public:
  FullBundleAdjustmentSolver() {  // full...cpp:6-42
    scaler_ = 0.01;
    inverse_scaler_ = 1.0 / scaler_;
    std::cout << "SparseBundleAdjustmentSolver() - initialize.\n";
  }
  ~FullBundleAdjustmentSolver() {
    if (handle_) ba_destroy(handle_);
  }
  FullBundleAdjustmentSolver(const FullBundleAdjustmentSolver &) = delete;
  FullBundleAdjustmentSolver &operator=(const FullBundleAdjustmentSolver &) = delete;

  void Reset() {  // :44-70
    camera_ids_.clear(); cam_intr_.clear(); cam_T_.clear(); camera_slot_.clear();
    pose_ptrs_.clear(); pose_index_.clear(); T_jw_.clear(); pose_fixed_.clear();
    point_ptrs_.clear(); point_index_.clear(); X_.clear(); point_fixed_.clear();
    obs_cam_.clear(); obs_pose_.clear(); obs_point_.clear(); obs_uv_.clear();
    num_fixed_poses_ = num_fixed_points_ = 0;
    is_parameter_finalized_ = false;
    if (handle_) ba_reset(handle_);
  }

  void AddCamera(const _BA_Index camera_index, const _BA_Camera &camera) {  // :72-85
    if (camera_slot_.count(camera_index) == 0) {  // unordered_map::insert keeps the first
      camera_slot_[camera_index] = static_cast<int>(camera_ids_.size());
      camera_ids_.push_back(camera_index);
      cam_intr_.push_back(camera.fx * scaler_); cam_intr_.push_back(camera.fy * scaler_);
      cam_intr_.push_back(camera.cx * scaler_); cam_intr_.push_back(camera.cy * scaler_);
      PushPose12(camera.pose_this_to_cam0, scaler_, &cam_T_);
    }
    std::cout << "New camera is added.\n";
    std::cout << "  fx: " << camera.fx * scaler_ << ", fy: " << camera.fy * scaler_ << ", cx: " << camera.cx * scaler_
              << ", cy: " << camera.cy * scaler_ << "\n";
  }

  void AddPose(_BA_Pose *original_pose) {  // :87-101
    if (is_parameter_finalized_) {
      std::cerr << TEXT_YELLOW("Cannot enroll parameter. (is_parameter_finalized_ == true)") << std::endl;
      return;
    }
    if (pose_index_.count(original_pose) == 0) {
      pose_index_[original_pose] = static_cast<int>(pose_ptrs_.size());
      pose_ptrs_.push_back(original_pose);
      const _BA_Pose T_jw = original_pose->inverse();
      PushPose12(T_jw, scaler_, &T_jw_);
      pose_fixed_.push_back(0);
    }
  }

  void AddPoint(_BA_Point *original_point) {  // :103-117
    if (is_parameter_finalized_) {
      std::cerr << TEXT_YELLOW("Cannot enroll parameter. (is_parameter_finalized_ == true)\n");
      return;
    }
    if (point_index_.count(original_point) == 0) {
      point_index_[original_point] = static_cast<int>(point_ptrs_.size());
      point_ptrs_.push_back(original_point);
      for (int k = 0; k < 3; ++k) X_.push_back((*original_point)(k) * scaler_);
      point_fixed_.push_back(0);
    }
  }

  void AddObservation(const _BA_Index index_camera, _BA_Pose *related_pose, _BA_Point *related_point,
                      const _BA_Pixel &pixel) {  // :155-180
    if (camera_slot_.count(index_camera) == 0) { std::cerr << TEXT_RED("Invalid camera index.\n"); return; }
    auto pj = pose_index_.find(related_pose);
    if (pj == pose_index_.end()) { std::cerr << TEXT_RED("Nonexisting pose.\n"); return; }
    auto pi = point_index_.find(related_point);
    if (pi == point_index_.end()) { std::cerr << TEXT_RED("Nonexisting point.\n"); return; }
    obs_cam_.push_back(index_camera);
    obs_pose_.push_back(pj->second);
    obs_point_.push_back(pi->second);
    obs_uv_.push_back(pixel(0) * scaler_);
    obs_uv_.push_back(pixel(1) * scaler_);
    device_dirty_ = true;
  }

  void MakePoseFixed(_BA_Pose *original_pose_to_be_fixed) {  // :119-134
    if (is_parameter_finalized_) {
      std::cerr << TEXT_YELLOW("Cannot enroll parameter. (is_parameter_finalized_ == true)\n");
      return;
    }
    if (original_pose_to_be_fixed == nullptr) { std::cerr << "Empty pointer is conveyed. Skip this one.\n"; return; }
    auto it = pose_index_.find(original_pose_to_be_fixed);
    if (it == pose_index_.end()) throw std::runtime_error("There is no pointer in the BA pose pool.");
    pose_fixed_[it->second] = 1;
    ++num_fixed_poses_;
  }

  void MakePointFixed(_BA_Point *original_point_to_be_fixed) {  // :136-153
    if (is_parameter_finalized_) {
      std::cerr << TEXT_YELLOW("Cannot enroll parameter. (is_parameter_finalized_ == true)\n");
      return;
    }
    if (original_point_to_be_fixed == nullptr) { std::cerr << "Empty pointer is conveyed. Skip this one.\n"; return; }
    auto it = point_index_.find(original_point_to_be_fixed);
    if (it == point_index_.end()) throw std::runtime_error("There is no pointer in the BA point pool.");
    point_fixed_[it->second] = 1;
    ++num_fixed_points_;
  }

  // :182-206.  Public + idempotent here; only freezes the parameter set (observations may still be added).
  void FinalizeParameters() { is_parameter_finalized_ = true; }

  bool Solve(Options options, Summary *summary = nullptr) {  // :630-1044 (always LM: solver_type is not read)
    return SolveWithMethod(options, summary, BA_METHOD_LEVENBERG_MARQUARDT);
  }

 protected:
  // one Solve of the device engine with the loop selected by `method` (BA_METHOD_*); shared with the refactor
  // front-end (core/full_bundle_adjustment_solver_refactor.h)
  bool SolveWithMethod(Options options, Summary *summary, int method) {
    const auto t_start = std::chrono::high_resolution_clock::now();
    if (summary != nullptr) {
      summary->max_iteration_ = options.iteration_handle.max_num_iterations;
      summary->threshold_cost_change_ = options.convergence_handle.threshold_cost_change;
      summary->threshold_step_size_ = options.convergence_handle.threshold_step_size;
      summary->convergence_status_ = true;
    }
    FinalizeParameters();
    GetSolverStatistics();
    CheckPoseAndPointConnectivity();
    Upload();

    ba_options o{};
    o.solver_type = static_cast<int>(options.solver_type);
    o.threshold_step_size = options.convergence_handle.threshold_step_size;
    o.threshold_cost_change = options.convergence_handle.threshold_cost_change;
    o.threshold_huber_loss = options.outlier_handle.threshold_huber_loss;
    o.threshold_outlier_rejection = options.outlier_handle.threshold_outlier_rejection;
    o.max_num_iterations = options.iteration_handle.max_num_iterations;
    o.initial_lambda = options.trust_region_handle.initial_lambda;
    o.decrease_ratio_lambda = options.trust_region_handle.decrease_ratio_lambda;
    o.increase_ratio_lambda = options.trust_region_handle.increase_ratio_lambda;
    o.b_accumulate = options.accumulate_offdiagonal_blocks ? 1 : 0;
    o.inverse_scaler = inverse_scaler_;
    o.check_every = 0;
    o.use_graph = 1;
    o.method = method;
    const int cap = o.max_num_iterations > 0 ? o.max_num_iterations : 1;
    std::vector<ba_iter_info> infos(cap);
    ba_result result{};
    Check(ba_solve(handle_, &o, infos.data(), cap, &result), "ba_solve");

    // write back (:1011-1022): free parameters only
    std::vector<double> T(pose_ptrs_.size() * 12), X(point_ptrs_.size() * 3);
    Check(ba_get_poses(handle_, T.data()), "ba_get_poses");
    Check(ba_get_points(handle_, X.data()), "ba_get_points");
    T_jw_ = T;
    X_ = X;
    for (size_t j = 0; j < pose_ptrs_.size(); ++j) {
      if (pose_fixed_[j]) continue;
      _BA_Pose T_jw = _BA_Pose::Identity();
      _BA_Rotation3 R;
      for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) R(r, c) = T[j * 12 + r * 3 + c];
      T_jw.linear() = R;
      T_jw.translation() = _BA_Position3(T[j * 12 + 9] * inverse_scaler_, T[j * 12 + 10] * inverse_scaler_,
                                         T[j * 12 + 11] * inverse_scaler_);
      *pose_ptrs_[j] = T_jw.inverse();
    }
    for (size_t i = 0; i < point_ptrs_.size(); ++i) {
      if (point_fixed_[i]) continue;
      *point_ptrs_[i] = _BA_Point(X[i * 3] * inverse_scaler_, X[i * 3 + 1] * inverse_scaler_, X[i * 3 + 2] * inverse_scaler_);
    }
    const double total_time =
        std::chrono::duration<double, std::milli>(std::chrono::high_resolution_clock::now() - t_start).count();
    if (summary != nullptr) {
      for (int k = 0; k < result.n_iterations && k < cap; ++k) {
        OptimizationInfo info;
        info.cost = infos[k].cost;
        info.cost_change = infos[k].cost_change;
        info.average_reprojection_error = infos[k].average_reprojection_error;
        info.abs_step = infos[k].abs_step;
        info.abs_gradient = infos[k].abs_gradient;
        info.damping_term = infos[k].damping_term;
        info.iter_time = infos[k].iter_time;
        info.iteration_status = static_cast<IterationStatus>(infos[k].iteration_status);
        summary->optimization_info_list_.push_back(info);  // never cleared: repeated solves append (:1002)
      }
      summary->convergence_status_ = result.converged != 0;
      summary->total_time_in_millisecond_ = total_time;
    }
    last_result_ = result;
    return true;  // always (:666,1043)
  }

  // cameras, the parameters (T_jw_ / X_: the initial values, or the accepted internal values written back by the
  // last Solve) and the observation rows, then ba_finalize
  void Upload() {
    EnsureHandle();
    Check(ba_set_cameras(handle_, static_cast<int>(camera_ids_.size()), camera_ids_.data(), cam_intr_.data(), cam_T_.data()),
          "ba_set_cameras");
    Check(ba_set_poses(handle_, static_cast<int>(pose_ptrs_.size()), T_jw_.data(), pose_fixed_.data()), "ba_set_poses");
    Check(ba_set_points(handle_, static_cast<int>(point_ptrs_.size()), X_.data(), point_fixed_.data()), "ba_set_points");
    long long kept = 0;
    Check(ba_set_observations(handle_, static_cast<long long>(obs_cam_.size()), obs_cam_.data(), obs_pose_.data(),
                              obs_point_.data(), obs_uv_.data(), &kept), "ba_set_observations");
    Check(ba_finalize(handle_), "ba_finalize");
    device_dirty_ = false;
  }

 public:
  std::string GetSolverStatistics() const {  // :208-239 (prints; returns an empty string like the reference)
    std::stringstream ss;
    int n_opt_poses = 0, n_opt_points = 0;
    for (auto f : pose_fixed_) n_opt_poses += f ? 0 : 1;
    for (auto f : point_fixed_) n_opt_points += f ? 0 : 1;
    const long long n_obs = static_cast<long long>(obs_cam_.size());
    std::cout << "| Bundle Adjustment Statistics:" << std::endl;
    std::cout << "| # cameras in rigid body system: " << camera_ids_.size() << std::endl;
    std::cout << "|   " << TEXT_CYAN("(Note: The reference camera is 'camera_list_[0]'.)") << std::endl;
    std::cout << "|             # of total poses: " << pose_ptrs_.size() << std::endl;
    std::cout << "|               - # fix  poses: " << num_fixed_poses_ << std::endl;
    std::cout << "|               - # opt. poses: " << n_opt_poses << std::endl;
    std::cout << "|            # of total points: " << point_ptrs_.size() << std::endl;
    std::cout << "|              - # fix  points: " << num_fixed_points_ << std::endl;
    std::cout << "|              - # opt. points: " << n_opt_points << std::endl;
    std::cout << "|            # of observations: " << n_obs << std::endl;
    std::cout << "|                Jacobian size: " << 6 * n_obs << " rows x " << 3 * n_opt_points + 6 * n_opt_poses
              << " cols" << std::endl;
    std::cout << "|                Residual size: " << 2 * n_obs << " rows" << std::endl;
    std::cout << std::endl;
    return ss.str();
  }

  // extension: device-side result of the last Solve (phase times need ba_set_profile)
  const ba_result &last_result() const { return last_result_; }
  ba_solver *native_handle() { EnsureHandle(); return handle_; }

  // extension: residual (projection - pixel, caller's pixels) and status (BA_OBS_INLIER / _OUTLIER /
  // _BEHIND_CAMERA, ba_b200.h) of every accepted AddObservation call, in call order, at the parameters of the last
  // Solve (the initial ones before it).  threshold_px is in the caller's pixels, on |r_u| + |r_v| as the Huber weight
  // measures it; +inf classifies depth only.  Either output may be null.
  void GetObservationResiduals(double threshold_px, std::vector<_BA_Pixel> *residuals, std::vector<int> *status) {
    FinalizeParameters();
    if (device_dirty_ || !handle_) Upload();
    const size_t n = obs_cam_.size();
    std::vector<double> r(residuals ? 2 * n : 0);
    std::vector<uint8_t> st(status ? n : 0);
    Check(ba_observation_residuals(handle_, threshold_px * scaler_, residuals ? r.data() : nullptr,
                                   status ? st.data() : nullptr, nullptr), "ba_observation_residuals");
    if (residuals) {
      residuals->resize(n);
      for (size_t k = 0; k < n; ++k) (*residuals)[k] = _BA_Pixel(r[2 * k] * inverse_scaler_, r[2 * k + 1] * inverse_scaler_);
    }
    if (status) status->assign(st.begin(), st.end());
  }

  // extension: removes every observation that is not BA_OBS_INLIER at threshold_px (caller's pixels) and returns how
  // many were removed.  The next Solve starts from the accepted parameters of the last one.
  int RemoveOutlierObservations(double threshold_px) {
    std::vector<int> status;
    GetObservationResiduals(threshold_px, nullptr, &status);
    size_t w = 0;
    for (size_t k = 0; k < status.size(); ++k) {
      if (status[k] != BA_OBS_INLIER) continue;
      obs_cam_[w] = obs_cam_[k]; obs_pose_[w] = obs_pose_[k]; obs_point_[w] = obs_point_[k];
      obs_uv_[2 * w] = obs_uv_[2 * k]; obs_uv_[2 * w + 1] = obs_uv_[2 * k + 1];
      ++w;
    }
    const int removed = static_cast<int>(status.size() - w);
    obs_cam_.resize(w); obs_pose_.resize(w); obs_point_.resize(w); obs_uv_.resize(2 * w);
    if (removed > 0) device_dirty_ = true;
    return removed;
  }
  void SetDevice(int device) { device_ = device; }

 protected:
  bool is_finalized() const { return is_parameter_finalized_; }
  bool has_camera(int id) const { return camera_slot_.count(id) > 0; }
  bool has_pose(_BA_Pose *p) const { return pose_index_.count(p) > 0; }
  bool has_point(_BA_Point *p) const { return point_index_.count(p) > 0; }
  long long num_observations() const { return static_cast<long long>(obs_cam_.size()); }

 private:
  static void PushPose12(const _BA_Pose &T, double t_scale, std::vector<double> *out) {
    const _BA_Rotation3 R = T.linear();
    const _BA_Position3 t = T.translation();
    for (int r = 0; r < 3; ++r) for (int c = 0; c < 3; ++c) out->push_back(R(r, c));
    for (int r = 0; r < 3; ++r) out->push_back(t(r) * t_scale);
  }
  void EnsureHandle() {
    if (handle_) return;
    if (ba_create(&handle_, device_) != BA_OK || !handle_)
      throw std::runtime_error("ba_create failed: no CUDA device (the engine has no CPU fallback)");
  }
  void Check(int rc, const char *what) {
    if (rc != BA_OK) throw std::runtime_error(std::string(what) + " failed: " + (handle_ ? ba_last_error(handle_) : ""));
  }
  void CheckPoseAndPointConnectivity() {  // :310-341, warnings only
    static constexpr int kMinNumObservedPoints = 5;
    static constexpr int kMinNumRelatedPoses = 2;
    std::vector<std::unordered_set<int>> pose_points(pose_ptrs_.size()), point_poses(point_ptrs_.size());
    for (size_t k = 0; k < obs_cam_.size(); ++k) {
      pose_points[obs_pose_[k]].insert(obs_point_[k]);
      point_poses[obs_point_[k]].insert(obs_pose_[k]);
    }
    int j_opt = 0;
    for (size_t j = 0; j < pose_ptrs_.size(); ++j) {
      if (pose_fixed_[j]) continue;
      if (static_cast<int>(pose_points[j].size()) < kMinNumObservedPoints)
        std::cerr << TEXT_YELLOW(std::to_string(j_opt) + "-th pose: It might diverge because some frames have insufficient related points.") << std::endl;
      ++j_opt;
    }
    int i_opt = 0;
    for (size_t i = 0; i < point_ptrs_.size(); ++i) {
      if (point_fixed_[i]) continue;
      if (static_cast<int>(point_poses[i].size()) < kMinNumRelatedPoses)
        std::cerr << TEXT_YELLOW(std::to_string(i_opt) + "-th point: It might diverge because some points have insufficient related poses.") << std::endl;
      ++i_opt;
    }
  }

  _BA_Numeric scaler_, inverse_scaler_;
  bool is_parameter_finalized_{false};
  bool device_dirty_{true};
  int device_{0};
  int num_fixed_poses_{0}, num_fixed_points_{0};
  ba_solver *handle_{nullptr};
  ba_result last_result_{};
  // cameras
  std::vector<int> camera_ids_;
  std::unordered_map<int, int> camera_slot_;
  std::vector<double> cam_intr_, cam_T_;
  // parameters, keyed by the caller's object addresses (full...h:205-220)
  std::vector<_BA_Pose *> pose_ptrs_;
  std::unordered_map<_BA_Pose *, int> pose_index_;
  std::vector<double> T_jw_;
  std::vector<uint8_t> pose_fixed_;
  std::vector<_BA_Point *> point_ptrs_;
  std::unordered_map<_BA_Point *, int> point_index_;
  std::vector<double> X_;
  std::vector<uint8_t> point_fixed_;
  // observations in insertion order
  std::vector<int> obs_cam_, obs_pose_, obs_point_;
  std::vector<double> obs_uv_;
};

}  // namespace analytic_solver
}  // namespace visual_navigation
#endif
