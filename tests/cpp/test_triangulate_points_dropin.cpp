// GPU test driver for TriangulatePoints of the drop-in C++ API: registration (the scene file's points, e.g. all at the
// origin), an unknown pointer in `select` (must throw), an empty selection (nothing written), TriangulatePoints on every
// free landmark, then Solve.  Writes the internal parameters at the start, the triangulated count and statuses, the
// points through the caller's _BA_Point objects, the internal points after the triangulation and the internal
// parameters after the Solve.  The scene file has the layout test_ba_dropin.cpp reads.
// usage: test_triangulate_points_dropin scene.bin result.bin max_iterations min_parallax_deg max_residual_px
#include <cstdio>
#include <cstdlib>
#include <limits>
#include <stdexcept>
#include <unordered_map>
#include <vector>

#include "core/full_bundle_adjustment_solver.h"
#include "core/full_bundle_adjustment_solver_refactor.h"

using namespace visual_navigation::analytic_solver;

// the refactor front-end exposes the extension too
[[maybe_unused]] static auto kRefactorTriangulate = &FullBundleAdjustmentSolverRefactor::TriangulatePoints;

template <typename T>
static void rd(FILE *f, T *p, size_t n) { if (fread(p, sizeof(T), n, f) != n) { std::perror("read"); std::exit(2); } }

static void write_internal(FILE *o, ba_solver *h, int n_pose, int n_point, bool poses) {
  std::vector<double> T(12 * n_pose), X(3 * n_point);
  if (ba_get_poses(h, T.data()) != BA_OK || ba_get_points(h, X.data()) != BA_OK) std::exit(4);
  if (poses) std::fwrite(T.data(), sizeof(double), T.size(), o);
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
  for (int k = 0; k < n_obs; ++k) {
    int ids[3]; double uv[2];
    rd(f, ids, 3); rd(f, uv, 2);
    ba_solver.AddObservation(ids[0], &pose_pool[ids[1]], &point_pool[ids[2]], _BA_Pixel(uv[0], uv[1]));
  }
  std::fclose(f);

  Options options;
  options.iteration_handle.max_num_iterations = std::atoi(argv[3]);
  options.convergence_handle.threshold_cost_change = 1e-6f;
  options.convergence_handle.threshold_step_size = 1e-6f;
  const double min_parallax_deg = std::atof(argv[4]), max_residual_px = std::atof(argv[5]);

  FILE *o = std::fopen(argv[2], "wb");
  if (!o) return 2;
  // the internal parameters the triangulation starts from (GetObservationResiduals uploads them)
  ba_solver.GetObservationResiduals(std::numeric_limits<double>::infinity(), nullptr, nullptr);
  write_internal(o, ba_solver.native_handle(), n_pose, n_point, true);
  // a point that was never added: std::runtime_error, nothing runs
  _BA_Point stranger(1.0, 2.0, 3.0);
  const std::vector<_BA_Point *> bad{&point_pool[0], &stranger};
  bool threw = false;
  try { ba_solver.TriangulatePoints(min_parallax_deg, max_residual_px, &bad); } catch (const std::runtime_error &) { threw = true; }
  if (!threw) return 6;
  // an empty selection: every landmark skipped, nothing written
  const std::vector<_BA_Point *> none;
  std::vector<int> status;
  if (ba_solver.TriangulatePoints(min_parallax_deg, max_residual_px, &none, &status) != 0) return 7;
  for (int s : status) if (s != BA_TRI_SKIPPED) return 8;
  const int triangulated = ba_solver.TriangulatePoints(min_parallax_deg, max_residual_px, nullptr, &status);
  std::fwrite(&triangulated, sizeof(int), 1, o);
  if (static_cast<int>(status.size()) != n_point) return 5;
  std::fwrite(status.data(), sizeof(int), status.size(), o);
  for (int i = 0; i < n_point; ++i) std::fwrite(point_pool[i].data(), sizeof(double), 3, o);
  write_internal(o, ba_solver.native_handle(), n_pose, n_point, false);
  ba_solver.Solve(options);
  write_internal(o, ba_solver.native_handle(), n_pose, n_point, true);
  std::fclose(o);
  std::cout << "TRIANGULATE_DROPIN_OK triangulated " << triangulated << std::endl;
  return 0;
}
