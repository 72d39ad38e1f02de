// GPU test driver for the outlier extensions of the drop-in C++ API: AddObservation (with refused calls in between),
// GetObservationResiduals before the first Solve, Solve, GetObservationResiduals, RemoveOutlierObservations, Solve,
// GetObservationResiduals.  The scene file has the layout test_ba_dropin.cpp reads.
// usage: test_ba_outliers_dropin scene.bin result.bin max_iterations threshold_px huber_threshold
#include <cstdio>
#include <cstdlib>
#include <limits>
#include <unordered_map>
#include <vector>

#include "core/full_bundle_adjustment_solver.h"
#include "core/full_bundle_adjustment_solver_refactor.h"

using namespace visual_navigation::analytic_solver;

// the refactor front-end exposes the same two extensions
[[maybe_unused]] static auto kRefactorResiduals = &FullBundleAdjustmentSolverRefactor::GetObservationResiduals;
[[maybe_unused]] static auto kRefactorRemove = &FullBundleAdjustmentSolverRefactor::RemoveOutlierObservations;

template <typename T>
static void rd(FILE *f, T *p, size_t n) { if (fread(p, sizeof(T), n, f) != n) { std::perror("read"); std::exit(2); } }

static void write_rows(FILE *o, const std::vector<_BA_Pixel> &res, const std::vector<int> &status) {
  const int n = static_cast<int>(status.size());
  std::fwrite(&n, sizeof(int), 1, o);
  for (int s : status) std::fwrite(&s, sizeof(int), 1, o);
  for (const auto &r : res) std::fwrite(r.data(), sizeof(double), 2, o);
}

static void write_internal(FILE *o, ba_solver *h, int n_pose, int n_point) {
  std::vector<double> T(12 * n_pose), X(3 * n_point);
  if (ba_get_poses(h, T.data()) != BA_OK || ba_get_points(h, X.data()) != BA_OK) std::exit(4);
  std::fwrite(T.data(), sizeof(double), T.size(), o);
  std::fwrite(X.data(), sizeof(double), X.size(), o);
}

int main(int argc, char **argv) {
  if (argc < 6) return 2;
  FILE *f = std::fopen(argv[1], "rb");
  if (!f) return 2;
  int hdr[5];
  rd(f, hdr, 5);
  const int n_cam = hdr[0], n_pose = hdr[1], n_point = hdr[2], n_fixed = hdr[3], n_obs = hdr[4];
  FullBundleAdjustmentSolver ba_solver;
  for (int c = 0; c < n_cam; ++c) {
    int id; double intr[4], T[16];
    rd(f, &id, 1); rd(f, intr, 4); rd(f, T, 16);
    _BA_Camera cam;
    cam.fx = intr[0]; cam.fy = intr[1]; cam.cx = intr[2]; cam.cy = intr[3];
    _BA_Rotation3 R;
    for (int r = 0; r < 3; ++r) for (int k = 0; k < 3; ++k) R(r, k) = T[k * 4 + r];
    cam.pose_this_to_cam0 = _BA_Pose::Identity();
    cam.pose_this_to_cam0.linear() = R;
    cam.pose_this_to_cam0.translation() = _BA_Position3(T[12], T[13], T[14]);
    ba_solver.AddCamera(id, cam);
  }
  std::unordered_map<int, _BA_Pose> pose_pool;
  std::unordered_map<int, _BA_Point> point_pool;
  for (int j = 0; j < n_pose; ++j) {
    double T[16];
    rd(f, T, 16);
    _BA_Pose P = _BA_Pose::Identity();
    _BA_Rotation3 R;
    for (int r = 0; r < 3; ++r) for (int k = 0; k < 3; ++k) R(r, k) = T[k * 4 + r];
    P.linear() = R;
    P.translation() = _BA_Position3(T[12], T[13], T[14]);
    pose_pool[j] = P;
  }
  for (int i = 0; i < n_point; ++i) { double X[3]; rd(f, X, 3); point_pool[i] = _BA_Point(X[0], X[1], X[2]); }
  for (int j = 0; j < n_pose; ++j) ba_solver.AddPose(&pose_pool[j]);
  for (int i = 0; i < n_point; ++i) ba_solver.AddPoint(&point_pool[i]);
  for (int k = 0; k < n_fixed; ++k) { int j; rd(f, &j, 1); ba_solver.MakePoseFixed(&pose_pool[j]); }
  _BA_Pose stranger_pose = _BA_Pose::Identity();
  _BA_Point stranger_point(0.0, 0.0, 1.0);
  for (int k = 0; k < n_obs; ++k) {
    int ids[3]; double uv[2];
    rd(f, ids, 3); rd(f, uv, 2);
    if (k % 1000 == 17) {   // refused calls: not rows
      ba_solver.AddObservation(12345, &pose_pool[ids[1]], &point_pool[ids[2]], _BA_Pixel(uv[0], uv[1]));
      ba_solver.AddObservation(ids[0], &stranger_pose, &point_pool[ids[2]], _BA_Pixel(uv[0], uv[1]));
      ba_solver.AddObservation(ids[0], &pose_pool[ids[1]], &stranger_point, _BA_Pixel(uv[0], uv[1]));
    }
    ba_solver.AddObservation(ids[0], &pose_pool[ids[1]], &point_pool[ids[2]], _BA_Pixel(uv[0], uv[1]));
  }
  std::fclose(f);

  const int max_it = std::atoi(argv[3]);
  const double thr = std::atof(argv[4]);
  Options options;
  options.iteration_handle.max_num_iterations = max_it;
  options.convergence_handle.threshold_cost_change = 1e-6f;
  options.convergence_handle.threshold_step_size = 1e-6f;
  options.outlier_handle.threshold_huber_loss = static_cast<float>(std::atof(argv[5]));

  FILE *o = std::fopen(argv[2], "wb");
  if (!o) return 2;
  std::vector<_BA_Pixel> res;
  std::vector<int> status;
  // before the first Solve: the initial parameters (internal units as uploaded)
  ba_solver.GetObservationResiduals(thr, &res, &status);
  write_rows(o, res, status);
  write_internal(o, ba_solver.native_handle(), n_pose, n_point);
  ba_solver.Solve(options);
  ba_solver.GetObservationResiduals(thr, &res, &status);
  write_rows(o, res, status);
  const int removed = ba_solver.RemoveOutlierObservations(thr);
  std::fwrite(&removed, sizeof(int), 1, o);
  ba_solver.Solve(options);
  ba_solver.GetObservationResiduals(std::numeric_limits<double>::infinity(), &res, &status);
  write_rows(o, res, status);
  write_internal(o, ba_solver.native_handle(), n_pose, n_point);
  std::fclose(o);
  std::cout << "OUTLIERS_DROPIN_OK removed " << removed << std::endl;
  return 0;
}
