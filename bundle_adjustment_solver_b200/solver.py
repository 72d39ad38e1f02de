"""Host-side Python mirror of the reference's solver classes over the C-ABI.

The reference's host language is C++ (the drop-in C++ classes are in include/ba_b200/); this module
mirrors the same interface for Python callers, tests and bench.py:
  FullBundleAdjustmentSolver      core/full_bundle_adjustment_solver.h:127-146
  PoseOnlyBundleAdjustmentSolver  core/pose_only_bundle_adjustment_solver.h:19-67
  Options / Summary               core/solver_option_and_summary.h:47-93
Parameters are identified by the integer handle the Add* call returns (the reference keys them by
object address).  All arithmetic runs on the GPU; this file only converts units and copies buffers.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import BaError, IterInfo, Options, PoseOnlyOptions, PoseOnlyResult, Result, default_options, ptr

STATUS_NAMES = {0: "UPDATE", 1: "UPDATE_TRUST_MORE", 2: "SKIPPED"}


def _check(rc, L, h, what):
    if rc != 0:
        msg = L.ba_last_error(h).decode() if h else ""
        raise BaError(f"{what} failed (rc={rc}): {msg}")


def _inv_T(T):
    T = np.asarray(T, dtype=np.float64)
    out = np.zeros_like(T)
    Rt = np.swapaxes(T[..., :3, :3], -1, -2)
    out[..., :3, :3] = Rt
    out[..., :3, 3] = -np.einsum("...ij,...j->...i", Rt, T[..., :3, 3])
    out[..., 3, 3] = 1.0
    return out


def _to12(T):
    """(...,4,4) -> (...,12): R row-major | t."""
    T = np.asarray(T, dtype=np.float64)
    return np.concatenate([T[..., :3, :3].reshape(T.shape[:-2] + (9,)), T[..., :3, 3]], axis=-1)


def _from12(p):
    p = np.asarray(p, dtype=np.float64)
    T = np.zeros(p.shape[:-1] + (4, 4))
    T[..., :3, :3] = p[..., :9].reshape(p.shape[:-1] + (3, 3))
    T[..., :3, 3] = p[..., 9:]
    T[..., 3, 3] = 1.0
    return T


class Summary:
    """Mirrors Summary (core/solver_option_and_summary.h:74-93, .cpp:12-84)."""

    def __init__(self):
        self.optimization_info_list = []
        self.max_iteration = 0
        self.total_time_in_millisecond = 0.0
        self.threshold_step_size = 0.0
        self.threshold_cost_change = 0.0
        self.convergence_status = True
        self.result = None

    def get_total_time_in_second(self):
        return self.total_time_in_millisecond * 0.001

    def brief_report(self):
        out = ["itr   total_cost    avg.reproj.  cost_change  |step|    |gradient|  damp_term  itr_time[ms] itr_stat"]
        for k, it in enumerate(self.optimization_info_list):
            stat = {0: "UPDATE", 1: "\033[0;32mUPDATE\033[0m", 2: "\033[0;33m SKIP \033[0m"}.get(it.iteration_status, "")
            out.append(f"{k:3d}  {it.cost:.6e}    {it.average_reprojection_error:.2e}    {it.cost_change:.2e}   "
                       f"{it.abs_step:.2e}   {it.abs_gradient:.2e}    {it.damping_term:.2e}   {it.iter_time:.2e}     {stat}")
        n = len(self.optimization_info_list)
        out.append("Analytic Solver Report:")
        out.append(f"  Iterations      : {n}")
        out.append(f"  Total time      : {self.total_time_in_millisecond * 0.001:.5g} [second]")
        if n:
            first, last = self.optimization_info_list[0], self.optimization_info_list[-1]
            out.append(f"  Initial cost    : {first.cost:.5g}")
            out.append(f"  Final cost      : {last.cost:.5g}")
            out.append(f"  Initial reproj. : {first.average_reprojection_error:.5g} [pixel]")
            out.append(f"  Final reproj.   : {last.average_reprojection_error:.5g} [pixel]")
        out.append(", Termination     : " + ("\033[0;32mCONVERGENCE\033[0m" if self.convergence_status
                                             else "\033[0;33mNO_CONVERGENCE\033[0m"))
        if self.max_iteration == n:
            out.append("\033[0;33m WARNIING: MAX ITERATION is reached ! The solution could be local minima.\033[0m")
        return "\n".join(out) + "\n"


class FullBundleAdjustmentSolver:
    """GPU drop-in for analytic_solver::FullBundleAdjustmentSolver (integer handles)."""

    def __init__(self, device=0, stream=None):
        self.L = capi.lib()
        self.h = C.c_void_p()
        rc = self.L.ba_create(C.byref(self.h), device)
        if rc != 0:
            self.h = None
            raise BaError("ba_create failed: no CUDA device / engine unavailable (there is no CPU fallback)")
        if stream is not None:
            self.L.ba_set_stream(self.h, C.c_void_p(stream))
        self.scaler = 0.01                      # full...cpp:38
        self.inverse_scaler = 1.0 / self.scaler
        self._reset_host()

    def _reset_host(self):
        self.cam_ids, self.cam_intr, self.cam_T = [], [], []
        self.poses = np.zeros((0, 4, 4))       # user-facing camera-to-world 4x4
        self.points = np.zeros((0, 3))
        self.pose_fixed = np.zeros(0, dtype=np.uint8)
        self.point_fixed = np.zeros(0, dtype=np.uint8)
        self._obs = [[], [], [], []]
        self._obs_chunks = []
        self.is_parameter_finalized = False
        self._uploaded = False
        self._engine_has_parameters = False
        self._carried_internal = None   # accepted internal parameters the next upload starts from (remove_observations)

    def __del__(self):
        if getattr(self, "h", None):
            self.L.ba_destroy(self.h)
            self.h = None

    def reset(self):
        self.L.ba_reset(self.h)
        self._reset_host()

    # --- registration (full...cpp:72-180) -------------------------------------------------
    def add_camera(self, camera_index, fx, fy, cx, cy, pose_this_to_cam0):
        if camera_index in self.cam_ids:
            return  # unordered_map::insert ignores duplicates (:80)
        self.cam_ids.append(int(camera_index))
        self.cam_intr.append([fx, fy, cx, cy])
        self.cam_T.append(np.asarray(pose_this_to_cam0, dtype=np.float64).copy())

    def add_pose(self, T_wc):
        if self.is_parameter_finalized:
            print("\033[0;33mCannot enroll parameter. (is_parameter_finalized_ == true)\033[0m")
            return -1
        return self.add_poses(np.asarray(T_wc, dtype=np.float64).reshape(1, 4, 4))[0]

    def add_poses(self, T_wc):
        if self.is_parameter_finalized:
            print("\033[0;33mCannot enroll parameter. (is_parameter_finalized_ == true)\033[0m")
            return []
        T_wc = np.asarray(T_wc, dtype=np.float64).reshape(-1, 4, 4)
        base = len(self.poses)
        self.poses = np.concatenate([self.poses, T_wc])
        self.pose_fixed = np.concatenate([self.pose_fixed, np.zeros(len(T_wc), dtype=np.uint8)])
        return list(range(base, base + len(T_wc)))

    def add_point(self, X):
        if self.is_parameter_finalized:
            print("\033[0;33mCannot enroll parameter. (is_parameter_finalized_ == true)\033[0m")
            return -1
        return self.add_points(np.asarray(X, dtype=np.float64).reshape(1, 3))[0]

    def add_points(self, X):
        if self.is_parameter_finalized:
            print("\033[0;33mCannot enroll parameter. (is_parameter_finalized_ == true)\033[0m")
            return []
        X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
        base = len(self.points)
        self.points = np.concatenate([self.points, X])
        self.point_fixed = np.concatenate([self.point_fixed, np.zeros(len(X), dtype=np.uint8)])
        return range(base, base + len(X))

    def make_pose_fixed(self, pose_id):
        if self.is_parameter_finalized:
            print("\033[0;33mCannot enroll parameter. (is_parameter_finalized_ == true)\033[0m")
            return
        if pose_id is None:
            print("Empty pointer is conveyed. Skip this one.")
            return
        if not (0 <= pose_id < len(self.poses)):
            raise RuntimeError("There is no pointer in the BA pose pool.")
        self.pose_fixed[pose_id] = 1

    def make_point_fixed(self, point_id):
        if self.is_parameter_finalized:
            print("\033[0;33mCannot enroll parameter. (is_parameter_finalized_ == true)\033[0m")
            return
        if point_id is None:
            print("Empty pointer is conveyed. Skip this one.")
            return
        if not (0 <= point_id < len(self.points)):
            raise RuntimeError("There is no pointer in the BA point pool.")
        self.point_fixed[point_id] = 1

    def add_observation(self, camera_index, pose_id, point_id, pixel):
        if camera_index not in self.cam_ids:
            print("\033[0;31mInvalid camera index.\033[0m")
            return
        if not (0 <= pose_id < len(self.poses)):
            print("\033[0;31mNonexisting pose.\033[0m")
            return
        if not (0 <= point_id < len(self.points)):
            print("\033[0;31mNonexisting point.\033[0m")
            return
        self._obs[0].append(camera_index); self._obs[1].append(pose_id); self._obs[2].append(point_id)
        self._obs[3].append((float(pixel[0]), float(pixel[1])))
        self._uploaded = False

    def add_observations(self, cam, pose, point, uv):
        """Bulk AddObservation (insertion order preserved); invalid rows are dropped by the engine."""
        self._flush_scalar_obs()
        self._obs_chunks.append((np.asarray(cam, dtype=np.int32), np.asarray(pose, dtype=np.int32),
                                 np.asarray(point, dtype=np.int32), np.asarray(uv, dtype=np.float64).reshape(-1, 2)))
        self._uploaded = False

    def _flush_scalar_obs(self):
        if self._obs[0]:
            self._obs_chunks.append((np.asarray(self._obs[0], dtype=np.int32), np.asarray(self._obs[1], dtype=np.int32),
                                     np.asarray(self._obs[2], dtype=np.int32), np.asarray(self._obs[3], dtype=np.float64)))
            self._obs = [[], [], [], []]

    # --- FinalizeParameters (:182-206) -----------------------------------------------------
    def internal_parameters(self):
        """User units -> the reference's internal units (Add*: inverse pose, x0.01)."""
        T_jw = _inv_T(np.asarray(self.poses).reshape(-1, 4, 4))
        T_jw[:, :3, 3] = T_jw[:, :3, 3] * self.scaler
        X = np.asarray(self.points, dtype=np.float64).reshape(-1, 3) * self.scaler
        return np.ascontiguousarray(_to12(T_jw)), np.ascontiguousarray(X)

    def finalize_parameters(self):
        self.is_parameter_finalized = True
        self._upload()

    def _upload(self, internal_override=None):
        if self._uploaded:
            return
        L, h = self.L, self.h
        ids = np.asarray(self.cam_ids, dtype=np.int32)
        intr = np.ascontiguousarray(np.asarray(self.cam_intr, dtype=np.float64) * self.scaler)
        cT = np.asarray(self.cam_T, dtype=np.float64).reshape(-1, 4, 4).copy()
        cT[:, :3, 3] *= self.scaler
        cT12 = np.ascontiguousarray(_to12(cT))
        _check(L.ba_set_cameras(h, len(ids), ptr(ids), ptr(intr), ptr(cT12)), L, h, "ba_set_cameras")
        if internal_override is not None:
            T12, X = internal_override
        elif self._carried_internal is not None:
            T12, X = self._carried_internal
        else:
            T12, X = self.internal_parameters()
        pf = np.ascontiguousarray(self.pose_fixed, dtype=np.uint8)
        qf = np.ascontiguousarray(self.point_fixed, dtype=np.uint8)
        _check(L.ba_set_poses(h, len(pf), ptr(T12), ptr(pf)), L, h, "ba_set_poses")
        _check(L.ba_set_points(h, len(qf), ptr(X), ptr(qf)), L, h, "ba_set_points")
        self._flush_scalar_obs()
        if len(self._obs_chunks) == 1:       # one bulk AddObservation call: no host copy, the engine scales while it copies
            cam, pose, point, uv = (np.ascontiguousarray(a) for a in self._obs_chunks[0])
        elif self._obs_chunks:
            cam, pose, point, uv = (np.ascontiguousarray(np.concatenate([c[k] for c in self._obs_chunks])) for k in range(4))
        else:
            cam = pose = point = np.zeros(0, dtype=np.int32)
            uv = np.zeros((0, 2))
        kept = C.c_longlong(0)
        _check(L.ba_set_observations_scaled(h, len(cam), ptr(cam), ptr(pose), ptr(point), ptr(uv), self.scaler, C.byref(kept)),
               L, h, "ba_set_observations_scaled")
        self.num_total_observations = kept.value
        _check(L.ba_finalize(h), L, h, "ba_finalize")
        self._uploaded = True
        self._engine_has_parameters = True
        self._carried_internal = None

    # --- Solve (:630-1044) -------------------------------------------------------------------
    def solve(self, options=None, summary=None):
        options = options or default_options()
        if options.inverse_scaler == 0.0:
            options.inverse_scaler = self.inverse_scaler
        self.is_parameter_finalized = True
        self._upload()
        cap = max(1, options.max_num_iterations)
        infos = (IterInfo * cap)()
        res = Result()
        _check(self.L.ba_solve(self.h, C.byref(options), infos, cap, C.byref(res)), self.L, self.h, "ba_solve")
        self.last_result = res
        if summary is not None:
            summary.max_iteration = options.max_num_iterations
            summary.threshold_cost_change = options.threshold_cost_change
            summary.threshold_step_size = options.threshold_step_size
            summary.optimization_info_list.extend(infos[k] for k in range(res.n_iterations))
            summary.convergence_status = bool(res.converged)
            summary.total_time_in_millisecond = res.total_time_ms
            summary.result = res
        # write-back (:1011-1022)
        T12 = np.zeros((len(self.poses), 12))
        X = np.zeros((len(self.points), 3))
        _check(self.L.ba_get_poses(self.h, ptr(T12)), self.L, self.h, "ba_get_poses")
        _check(self.L.ba_get_points(self.h, ptr(X)), self.L, self.h, "ba_get_points")
        T = _from12(T12)
        T[:, :3, 3] *= self.inverse_scaler
        Twc = _inv_T(T)
        free_j = self.pose_fixed == 0
        free_i = self.point_fixed == 0
        self.poses[free_j] = Twc[free_j]
        self.points[free_i] = X[free_i] * self.inverse_scaler
        return True

    def get_poses(self):
        return np.asarray(self.poses).reshape(-1, 4, 4)

    def get_points(self):
        return np.asarray(self.points).reshape(-1, 3)

    def get_internal(self):
        """Accepted parameters in the engine's internal units (T_jw as 12 doubles, X), as ba_get_poses / ba_get_points
        return them; same layout as the oracle's get_internal()."""
        n_p, n_x = len(np.asarray(self.poses).reshape(-1, 16)), len(np.asarray(self.points).reshape(-1, 3))
        T = np.zeros((n_p, 12))
        X = np.zeros((n_x, 3))
        _check(self.L.ba_get_poses(self.h, ptr(T)), self.L, self.h, "ba_get_poses")
        _check(self.L.ba_get_points(self.h, ptr(X)), self.L, self.h, "ba_get_points")
        return T, X

    def sizes(self):
        out = np.zeros(6, dtype=np.int64)
        _check(self.L.ba_get_sizes(self.h, ptr(out)), self.L, self.h, "ba_get_sizes")
        return dict(N=int(out[0]), M=int(out[1]), P=int(out[2]), n_obs=int(out[3]), N_total=int(out[4]),
                    M_total=int(out[5]))

    def get_solver_statistics(self):
        s = self.sizes()
        lines = ["| Bundle Adjustment Statistics:",
                 f"| # cameras in rigid body system: {len(self.cam_ids)}",
                 "|   \033[0;36m(Note: The reference camera is 'camera_list_[0]'.)\033[0m",
                 f"|             # of total poses: {s['N_total']}",
                 f"|               - # fix  poses: {s['N_total'] - s['N']}",
                 f"|               - # opt. poses: {s['N']}",
                 f"|            # of total points: {s['M_total']}",
                 f"|              - # fix  points: {s['M_total'] - s['M']}",
                 f"|              - # opt. points: {s['M']}",
                 f"|            # of observations: {s['n_obs']}",
                 f"|                Jacobian size: {6 * s['n_obs']} rows x {3 * s['M'] + 6 * s['N']} cols",
                 f"|                Residual size: {2 * s['n_obs']} rows", ""]
        return "\n".join(lines)

    # --- debug / parity helpers ---------------------------------------------------------------
    DUMP = dict(A=0, a=1, C=2, b=3, Cinv=4, B=5, S=6, rhs=7, x=8, y=9, scalars=10, factor=11)

    def set_debug(self, keep=True):
        self.L.ba_set_debug(self.h, int(keep))

    def set_profile(self, enable=True):
        self.L.ba_set_profile(self.h, int(enable))

    def build_only(self, options, lam, do_solve=False):
        self._upload()
        _check(self.L.ba_build_only(self.h, C.byref(options), float(lam), int(do_solve)), self.L, self.h,
               "ba_build_only")

    def cost(self):
        self._upload()
        c = C.c_double(0)
        _check(self.L.ba_cost(self.h, C.byref(c)), self.L, self.h, "ba_cost")
        return c.value

    # --- per-observation residuals and outlier removal ---------------------------------------------
    def observation_residuals(self, threshold=np.inf):
        """Residuals (projection - pixel) of every observation row at the accepted parameters, with a status per row.

        Rows are every observation this mirror sent to the engine, in order: bulk rows the engine dropped are rows
        (status OBS_DROPPED, NaN residuals); scalar add_observation calls refused here never were.  threshold is in
        the caller's pixels, on |r_u| + |r_v| as in the Huber weight; a row above it is OBS_OUTLIER, a row behind its
        camera (or with a non-finite residual) OBS_BEHIND_CAMERA.  Returns (residuals (n, 2) in the caller's pixels,
        status uint8 (n,), counts (4,) rows per status)."""
        threshold = float(threshold)
        self.is_parameter_finalized = True
        self._upload()
        n = self._num_rows()
        res = np.zeros((n, 2))
        status = np.zeros(n, dtype=np.uint8)
        counts = np.zeros(4, dtype=np.int64)
        _check(self.L.ba_observation_residuals(self.h, threshold * self.scaler, ptr(res), ptr(status), ptr(counts)),
               self.L, self.h, "ba_observation_residuals")
        return res * self.inverse_scaler, status, counts

    def remove_observations(self, keep):
        """Keep only the observation rows where `keep` (bool, one per row of observation_residuals) is true.  The next
        solve uploads the kept rows and starts from the engine's accepted parameters, bit for bit."""
        self._flush_scalar_obs()
        keep = np.asarray(keep, dtype=bool)
        if keep.shape != (self._num_rows(),):
            raise ValueError(f"keep has shape {keep.shape}, expected ({self._num_rows()},)")
        if self._engine_has_parameters and self._carried_internal is None:
            self._carried_internal = self.get_internal()
        self.is_parameter_finalized = True
        rows = [np.concatenate([c[k] for c in self._obs_chunks]) for k in range(4)] if self._obs_chunks else None
        self._obs_chunks = [tuple(np.ascontiguousarray(a[keep]) for a in rows)] if rows is not None else []
        self._uploaded = False

    def reject_outliers(self, threshold):
        """Removes every row that is not OBS_INLIER at `threshold` (caller's pixels); returns how many were removed."""
        _, status, _ = self.observation_residuals(threshold)
        keep = status == capi.OBS_INLIER
        self.remove_observations(keep)
        return int((~keep).sum())

    def _num_rows(self):
        return sum(len(c[0]) for c in self._obs_chunks) + len(self._obs[0])

    def dump(self, name):
        n = self.L.ba_debug_dump(self.h, self.DUMP[name], None)
        if n < 0:
            raise BaError(f"ba_debug_dump({name}) rc={n}")
        buf = np.zeros(n, dtype=np.float64)
        self.L.ba_debug_dump(self.h, self.DUMP[name], ptr(buf))
        return buf

    def pairs(self):
        P = self.sizes()["P"]
        pj = np.zeros(P, dtype=np.int32)
        pi = np.zeros(P, dtype=np.int32)
        self.L.ba_debug_pairs(self.h, ptr(pj), ptr(pi))
        return pj, pi

    def update_parameters_internal(self, T12, X):
        _check(self.L.ba_update_parameters(self.h, ptr(np.ascontiguousarray(T12)), ptr(np.ascontiguousarray(X))),
               self.L, self.h, "ba_update_parameters")


def load_scene(solver, sc, init=True):
    """Feed a scenes.FullScene into a solver-like object (this class or the oracle mirror)."""
    for k, cid in enumerate(sc.cam_ids):
        solver.add_camera(cid, *sc.cam_intr[k], sc.cam_T[k])
    solver.add_poses(sc.poses_init if init else sc.poses_true)
    solver.add_points(sc.points_init if init else sc.points_true)
    for j in sc.fixed_poses:
        solver.make_pose_fixed(int(j))
    for i in sc.fixed_points:
        solver.make_point_fixed(int(i))
    solver.add_observations(sc.obs_cam, sc.obs_pose, sc.obs_point, sc.obs_uv)
    return solver


class PoseOnlyBundleAdjustmentSolver:
    """GPU drop-in for analytic_solver::PoseOnlyBundleAdjustmentSolver.

    Poses are 12 float32 (R row-major | t).  The per-frame Solve_* methods of the reference map to
    solve(kind, ...) with one frame; solve_batched runs many independent frames in one launch."""

    def __init__(self, device=0):
        self.L = capi.lib()
        self.device = device
        self.debug_poses = np.zeros((0, 12), dtype=np.float32)

    def get_debug_poses(self):
        return self.debug_poses

    def solve_batched(self, kind, offsets, points, px_left, px_right, intr_left, intr_right, poses_io, options,
                      left_to_right=None, base_to_camera=None, world_to_last=None, want_history=False):
        f32 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float32)
        offsets = np.ascontiguousarray(offsets, dtype=np.int32)
        nf = len(offsets) - 1
        points, px_left, px_right = f32(points), f32(px_left), f32(px_right)
        n = len(points)
        if len(px_left) != n or (px_right is not None and len(px_right) != n):
            raise RuntimeError("world_position_list.size() != current_pixel_list.size()")  # pose_only...cpp:31-37
        intr_left = f32(intr_left)
        intr_right = f32(intr_left if intr_right is None else intr_right)
        l2r, b2c, w2l = f32(left_to_right), f32(base_to_camera), f32(world_to_last)
        poses = f32(poses_io).reshape(nf, 12).copy()
        ml = np.zeros(n, dtype=np.uint8)
        mr = np.zeros(n, dtype=np.uint8)
        results = (PoseOnlyResult * max(nf, 1))()
        K = max(1, options.max_num_iterations)
        hc = np.zeros((nf, K), dtype=np.float32) if want_history else None
        hs = np.zeros((nf, K), dtype=np.float32) if want_history else None
        dbg = np.zeros((nf, K, 12), dtype=np.float32) if want_history else None
        rc = self.L.ba_poseonly_solve_batched(self.device, kind, nf, ptr(offsets), ptr(points), ptr(px_left),
                                              ptr(px_right), ptr(intr_left), ptr(intr_right), ptr(l2r), ptr(b2c),
                                              ptr(w2l), ptr(poses), ptr(ml), ptr(mr), C.byref(options), results,
                                              ptr(hc), ptr(hs), ptr(dbg))
        if rc != 0:
            raise BaError(f"ba_poseonly_solve_batched failed rc={rc} (no CPU fallback)")
        out = dict(poses=poses, mask_left=ml.astype(bool), mask_right=mr.astype(bool),
                   results=[results[k] for k in range(nf)])
        if want_history:
            out.update(hist_cost=hc, hist_step=hs, debug_poses=dbg)
        return out

    def solve(self, kind, points, px_left, px_right, intr_left, intr_right, pose_io, options, **kw):
        """One frame: Solve_Monocular_6Dof (kind 0), Solve_Stereo_6Dof (1), Solve_Monocular_Planar3Dof (2),
        Solve_Stereo_Planar3Dof (3).  Returns (success, pose, mask_left, mask_right, result)."""
        n = len(points)
        w2l = kw.pop("world_to_last", None)
        out = self.solve_batched(kind, [0, n], points, px_left, px_right, intr_left, intr_right,
                                 np.asarray(pose_io, dtype=np.float32).reshape(1, 12), options,
                                 world_to_last=None if w2l is None else np.asarray(w2l, dtype=np.float32).reshape(1, 12),
                                 want_history=True, **kw)
        r = out["results"][0]
        self.debug_poses = out["debug_poses"][0][:r.n_iterations]
        out1 = dict(success=bool(r.success), pose=out["poses"][0], mask_left=out["mask_left"],
                    mask_right=out["mask_right"], result=r, hist_cost=out["hist_cost"][0][:r.n_summary],
                    hist_step=out["hist_step"][0][:r.n_summary])
        return out1
