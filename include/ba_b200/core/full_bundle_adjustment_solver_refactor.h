// Drop-in for core/full_bundle_adjustment_solver_refactor.h (reference :31-136): the refactored front-end of the
// same analytic solver -- Register* names, exceptions instead of console warnings, and a solver_type switch
// (LEVENBERG_MARQUARDT / GAUSS_NEWTON in Solve, full_bundle_adjustment_solver_refactor.cpp:944-982) plus
// SolveByGradientDescent (:1075-1367).  The arithmetic of the linearisation, the Schur solve and the update is
// identical to FullBundleAdjustmentSolver (same scaling by 0.01, same T_jw = pose^-1 convention,
// `camera_to_body_pose` applied as Xc = camera_to_body_pose * Xb, :758), so this class is a thin adapter over the
// other shim: same C-ABI engine, loop selected through ba_options.method.
//
// Error behaviour follows the reference: std::runtime_error for registration after finalisation (:99,114), null or
// unknown pointers in Make*Fixed (:128-153), unknown camera / pose / point in AddObservation (:223-229) and a Solve
// without observations (:851); a duplicate camera id is a yellow warning (:71-75).
// Not reproduced: Solve with solver_type GRADIENT_DESCENT or UNDEFINED, which in the reference runs the loop without
// ever applying a step (:944-982 has no branch for them); here GRADIENT_DESCENT is routed to SolveByGradientDescent
// and UNDEFINED throws.
#ifndef _FULL_BUNDLE_ADJUSTMENT_SOLVER_REFACTOR_H_
#define _FULL_BUNDLE_ADJUSTMENT_SOLVER_REFACTOR_H_

#include <stdexcept>
#include <string>

#include "full_bundle_adjustment_solver.h"

namespace visual_navigation {
namespace analytic_solver {

using SolverNumeric = double;
using Index = int;
using Pixel = Eigen::Matrix<SolverNumeric, 2, 1>;
using Point = Eigen::Matrix<SolverNumeric, 3, 1>;
using Rotation3D = Eigen::Matrix<SolverNumeric, 3, 3>;
using Translation3D = Eigen::Matrix<SolverNumeric, 3, 1>;
using Pose = Eigen::Transform<SolverNumeric, 3, 1>;

struct OptimizerCamera {  // refactor.h:49-64
  OptimizerCamera() {}
  OptimizerCamera(const OptimizerCamera &camera) {
    fx = camera.fx; fy = camera.fy; cx = camera.cx; cy = camera.cy;
    camera_to_body_pose = camera.camera_to_body_pose;
  }
  OptimizerCamera &operator=(const OptimizerCamera &) = default;
  SolverNumeric fx{0.0};
  SolverNumeric fy{0.0};
  SolverNumeric cx{0.0};
  SolverNumeric cy{0.0};
  Pose camera_to_body_pose;
};

struct PointObservation {  // refactor.h:66-71
  int related_camera_id{-1};
  Pose *related_pose{nullptr};
  Point *related_point{nullptr};
  Pixel pixel{-1.0, -1.0};
};

class FullBundleAdjustmentSolverRefactor : private FullBundleAdjustmentSolver {
  using Base = FullBundleAdjustmentSolver;

 public:
  FullBundleAdjustmentSolverRefactor() {}

  void Reset() { Base::Reset(); }

  void RegisterCamera(const Index camera_id, const OptimizerCamera &camera) {  // refactor.cpp:69-94
    if (has_camera(camera_id)) {
      std::cerr << TEXT_YELLOW(std::string(__func__) + ": " + "WANNING: existing camera\n");
      return;
    }
    _BA_Camera cam;
    cam.fx = camera.fx; cam.fy = camera.fy; cam.cx = camera.cx; cam.cy = camera.cy;
    cam.pose_this_to_cam0 = camera.camera_to_body_pose;   // both are applied as Xc = T * Xb (:758 / full...cpp:747)
    Base::AddCamera(camera_id, cam);
  }

  void RegisterWorldToBodyPose(Pose *original_pose) {  // refactor.cpp:96-109
    if (is_finalized())
      throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " +
                                        "Cannot enroll parameter. (is_parameter_finalized_ == true)\n"));
    Base::AddPose(original_pose);
  }

  void RegisterWorldPoint(Point *original_point) {  // refactor.cpp:111-124
    if (is_finalized())
      throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " +
                                        "Cannot enroll parameter. (is_parameter_finalized_ == true)\n"));
    Base::AddPoint(original_point);
  }

  void MakePoseFixed(Pose *original_pose) {  // refactor.cpp:126-140
    if (is_finalized())
      throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " +
                                        "Cannot enroll parameter. (is_parameter_finalized_ == true)\n"));
    if (original_pose == nullptr)
      throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " + "Empty pose pointer is conveyed. Skip this one.\n"));
    Base::MakePoseFixed(original_pose);   // unknown pointer: "There is no pointer in the BA pose pool."
  }

  void MakePointFixed(Point *original_point) {  // refactor.cpp:142-159
    if (is_finalized())
      throw std::runtime_error(TEXT_RED(std::string(__func__) +
                                        "Cannot enroll parameter. (is_parameter_finalized_ == true)\n"));
    if (original_point == nullptr)
      throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " + "Empty point pointer is conveyed.\n"));
    if (!has_point(original_point))
      throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " + "There is no pointer in the BA point pool."));
    Base::MakePointFixed(original_point);
  }

  void AddObservation(const Index camera_id, Pose *related_pose, Point *related_point, const Pixel &pixel) {  // :218-239
    if (!has_camera(camera_id)) throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " + "Invalid camera index.\n"));
    if (!has_pose(related_pose)) throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " + "Nonexisting pose.\n"));
    if (!has_point(related_point)) throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " + "Nonexisting point.\n"));
    Base::AddObservation(camera_id, related_pose, related_point, pixel);
  }

  bool Solve(Options options, Summary *summary = nullptr) {  // refactor.cpp:641-1073
    if (num_observations() < 1) throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " + "num_observations < 1\n"));
    switch (options.solver_type) {
      case SolverType::LEVENBERG_MARQUARDT: return SolveWithMethod(options, summary, BA_METHOD_LEVENBERG_MARQUARDT);
      case SolverType::GAUSS_NEWTON: return SolveWithMethod(options, summary, BA_METHOD_GAUSS_NEWTON);
      case SolverType::GRADIENT_DESCENT: return SolveWithMethod(options, summary, BA_METHOD_GRADIENT_DESCENT);
      default: throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " + "solver_type is UNDEFINED.\n"));
    }
  }

  bool SolveByGradientDescent(Options options, Summary *summary = nullptr) {  // refactor.cpp:1075-1367
    if (num_observations() < 1) throw std::runtime_error(TEXT_RED(std::string(__func__) + ": " + "num_observations < 1\n"));
    return SolveWithMethod(options, summary, BA_METHOD_GRADIENT_DESCENT);
  }

  std::string GetSolverStatistics() const { return Base::GetSolverStatistics(); }

  // extensions shared with the other shim
  using Base::last_result;
  using Base::native_handle;
  using Base::SetDevice;
  using Base::GetObservationResiduals;
  using Base::RemoveOutlierObservations;
};

}  // namespace analytic_solver
}  // namespace visual_navigation
#endif
