"""Per-observation residuals and outlier status of the full-BA engine (ba_observation_residuals, k_obs_residuals) and
the solve / reject outliers / solve loop built on them (FullBundleAdjustmentSolver.observation_residuals,
remove_observations, reject_outliers).

The residual is checked against a numpy restatement of the projection (full_bundle_adjustment_solver.cpp:744-760) at
the engine's own internal parameters, row by row and in the caller's row order; the rows the engine drops, the status
rules and the absence of side effects on the solver are checked directly; removal is checked bit for bit against a
fresh solver given only the kept rows and the same starting parameters."""
import copy
import struct
import subprocess

import numpy as np
import pytest

from bundle_adjustment_solver_b200 import scenes
from bundle_adjustment_solver_b200.capi import OBS_BEHIND_CAMERA, OBS_DROPPED, OBS_INLIER, OBS_OUTLIER, ptr
from bundle_adjustment_solver_b200.solver import BaError, Summary
from helpers import launched_kernels, load_engine, options_pair
from test_cpp_dropin import _compile, _write_scene

pytestmark = pytest.mark.gpu

PARITY_RTOL = 1e-12


# ------------------------------------------------------------------------------------------------ scenes
def _mixed_scene():
    # tile landmarks next to by-point landmarks (tracks wider than the tile window, loop closures), fixed poses inside
    # the tracks and fixed landmarks
    sc = scenes.scene_trajectory(120, 6000, 6, stereo=True, seed=5, n_fixed=3, heavy_tail=True, loop_fraction=0.03)
    sc.fixed_poses = np.array([0, 1, 2, 40, 41, 77])
    sc.fixed_points = np.arange(0, 6000, 97)
    return sc


def _scene(name):
    return scenes.scene_test_ba(seed=3) if name == "test_ba" else _mixed_scene()


def _outlier_scene(frac=0.02, shift=30.0, seed=11):
    """sigma = 0.5 px pixel noise and about frac of the rows shifted by `shift` px along u or v (random sign).  Tracks of
    6 to 10 poses: tile landmarks only, so solves of the same problem are bit-identical."""
    sc = scenes.scene_trajectory(100, 4000, 8, stereo=True, seed=seed, n_fixed=2, pixel_sigma=0.5)
    rng = np.random.default_rng(seed + 1)
    bad = np.sort(rng.choice(sc.n_obs, int(frac * sc.n_obs), replace=False))
    axis = rng.integers(0, 2, len(bad))
    sc.obs_uv[bad, axis] += shift * rng.choice([-1.0, 1.0], len(bad))
    return sc, bad


def _subset(sc, keep):
    out = copy.deepcopy(sc)
    out.obs_cam, out.obs_pose, out.obs_point = sc.obs_cam[keep], sc.obs_pose[keep], sc.obs_point[keep]
    out.obs_uv = sc.obs_uv[keep]
    return out


# ------------------------------------------------------------------------------------------------ reference
def _reference(sc, T12, X, scaler=0.01):
    """(residuals (n, 2), depth (n,)) in internal units from the internal parameters, as the reference computes them
    (full...cpp:744-760): Xb = R_jw X + t_jw, Xc = R_c Xb + t_c, r = (fx x/z + cx - u, fy y/z + cy - v)."""
    ids = np.asarray(sc.cam_ids)
    order = np.argsort(ids)
    slot = order[np.searchsorted(ids[order], sc.obs_cam)]
    intr = np.asarray(sc.cam_intr, dtype=np.float64) * scaler
    cT = np.asarray(sc.cam_T, dtype=np.float64).reshape(-1, 4, 4).copy()
    cT[:, :3, 3] *= scaler
    R = T12[sc.obs_pose, :9].reshape(-1, 3, 3)
    Xb = np.einsum("nij,nj->ni", R, X[sc.obs_point]) + T12[sc.obs_pose, 9:]
    Xc = np.einsum("nij,nj->ni", cT[slot, :3, :3], Xb) + cT[slot, :3, 3]
    invz = 1.0 / Xc[:, 2]
    f = intr[slot]
    uv = sc.obs_uv * scaler
    r = np.stack([f[:, 0] * (Xc[:, 0] * invz) + f[:, 2] - uv[:, 0], f[:, 1] * (Xc[:, 1] * invz) + f[:, 3] - uv[:, 1]],
                 axis=1)
    scale = np.abs(f[:, 0:2] * Xc[:, 0:2] * invz[:, None]) + np.abs(f[:, 2:4]) + np.abs(uv)   # size of the terms
    return r, Xc[:, 2], scale


def _raw(e, threshold=np.inf, want=(True, True, True)):
    """ba_observation_residuals in internal units (after the mirror has sent its rows)."""
    e._upload()
    n = e._num_rows()
    res = np.full((n, 2), -7.0) if want[0] else None
    st = np.full(n, 255, dtype=np.uint8) if want[1] else None
    cnt = np.full(4, -1, dtype=np.int64) if want[2] else None
    rc = e.L.ba_observation_residuals(e.h, float(threshold), ptr(res), ptr(st), ptr(cnt))
    if rc != 0:
        raise BaError(f"ba_observation_residuals rc={rc}: {e.L.ba_last_error(e.h).decode()}")
    return res, st, cnt


def _check_parity(sc, e):
    T, X = e.get_internal()
    ref, depth, scale = _reference(sc, T, X)
    res, st, cnt = _raw(e)
    err = np.abs(res - ref) / scale
    assert err.max() <= PARITY_RTOL, err.max()
    want = np.where(depth > 0, OBS_INLIER, OBS_BEHIND_CAMERA)
    np.testing.assert_array_equal(st, want)
    np.testing.assert_array_equal(cnt, np.bincount(st, minlength=4))
    # EvaluateCurrentCost is the sum of the residual norms (full...cpp:381-433)
    total = np.sqrt((res ** 2).sum(axis=1)).sum()
    assert abs(total - e.cost()) <= PARITY_RTOL * abs(total), (total, e.cost())
    # the Python mirror: the same rows in the caller's pixels
    res_px, st_px, cnt_px = e.observation_residuals()
    np.testing.assert_array_equal(res_px, res * e.inverse_scaler)
    np.testing.assert_array_equal(st_px, st)
    np.testing.assert_array_equal(cnt_px, cnt)
    return res, st


# ------------------------------------------------------------------------------------------------ 1. parity
@pytest.mark.parametrize("scene", ["test_ba", "mixed"])
def test_residuals_match_the_reference_projection(scene, engine_lib):
    sc = _scene(scene)
    e = load_engine(sc)
    _check_parity(sc, e)                                   # initial parameters
    _, eo = options_pair(max_num_iterations=10, threshold_cost_change=0.0, threshold_step_size=0.0)
    e.solve(eo)
    res, _ = _check_parity(sc, e)                          # accepted parameters of the solve
    assert np.abs(res).max() > 0


def test_residuals_on_a_c3_sized_scene(engine_lib):
    """About a million rows: every row through the grid stride and the row map."""
    sc = scenes.scene_c3(seed=4, pixel_sigma=0.3)
    assert sc.n_obs > 900_000
    e = load_engine(sc)
    _check_parity(sc, e)
    _, eo = options_pair(max_num_iterations=3, threshold_cost_change=0.0, threshold_step_size=0.0)
    e.solve(eo)
    _check_parity(sc, e)


# ------------------------------------------------------------------------------------------------ 2. rows
def test_dropped_rows_keep_their_place(engine_lib):
    sc = scenes.scene_test_ba(seed=2)
    rng = np.random.default_rng(0)
    n, nb = sc.n_obs, 60
    bad = np.stack([rng.integers(0, n, nb), rng.integers(0, 3, nb)], axis=1)
    cam, pose, point, uv = (list(a) for a in (sc.obs_cam, sc.obs_pose, sc.obs_point, sc.obs_uv))
    is_bad = [False] * n
    for at, kind in sorted(bad.tolist(), reverse=True):     # unknown camera id, pose out of range, point out of range
        row = [5 if kind == 0 else 0, len(sc.poses_init) + 3 if kind == 1 else 0, -1 if kind == 2 else 0]
        cam.insert(at, row[0]); pose.insert(at, row[1]); point.insert(at, row[2]); uv.insert(at, np.array([1.0, 2.0]))
        is_bad.insert(at, True)
    is_bad = np.array(is_bad)
    dirty = copy.deepcopy(sc)
    dirty.obs_cam, dirty.obs_pose, dirty.obs_point = (np.array(a, dtype=np.int32) for a in (cam, pose, point))
    dirty.obs_uv = np.array(uv)
    e = load_engine(dirty)
    # a scalar AddObservation refused by the mirror is not a row; an accepted one is the last row
    e.add_observation(9, 0, 0, (1.0, 1.0))
    e.add_observation(sc.obs_cam[0], sc.obs_pose[0], sc.obs_point[0], sc.obs_uv[0])
    res, st, cnt = _raw(e)
    assert len(st) == len(is_bad) + 1
    assert (st[:-1][is_bad] == OBS_DROPPED).all() and np.isnan(res[:-1][is_bad]).all()
    assert cnt[OBS_DROPPED] == nb and (st[:-1][~is_bad] != OBS_DROPPED).all()
    np.testing.assert_array_equal(cnt, np.bincount(st, minlength=4))
    clean = load_engine(sc)
    res_c, st_c, _ = _raw(clean)
    np.testing.assert_array_equal(res[:-1][~is_bad], res_c)
    np.testing.assert_array_equal(st[:-1][~is_bad], st_c)
    np.testing.assert_array_equal(res[-1], res_c[0])
    # the row map follows a re-finalisation that keeps the observations (new parameters, same rows)
    T, X = e.get_internal()
    e.L.ba_set_poses(e.h, len(T), ptr(np.ascontiguousarray(T)), ptr(np.ascontiguousarray(e.pose_fixed)))
    res2, st2, _ = _raw(e)
    np.testing.assert_array_equal(res2, res)
    np.testing.assert_array_equal(st2, st)


# ------------------------------------------------------------------------------------------------ 3. status
def test_point_behind_one_camera(engine_lib):
    sc = scenes.scene_test_ba(seed=1)
    e = load_engine(sc)
    T, X = e.get_internal()
    i0 = int(sc.obs_point[len(sc.obs_point) // 2])
    j0 = int(sc.obs_pose[len(sc.obs_pose) // 2])
    # reflect the landmark through the centre of pose j0: it goes behind that pose's cameras
    R, t = T[j0, :9].reshape(3, 3), T[j0, 9:]
    centre = -R.T @ t
    X = X.copy()
    X[i0] = 2.0 * centre - X[i0]
    e.update_parameters_internal(T, X)
    _, depth, _ = _reference(sc, T, X)
    res, st, cnt = _raw(e)
    behind = depth <= 0
    rows_i0 = sc.obs_point == i0
    assert behind[rows_i0 & (sc.obs_pose == j0)].all() and (behind <= rows_i0).all()
    np.testing.assert_array_equal(st == OBS_BEHIND_CAMERA, behind)
    np.testing.assert_array_equal(cnt, np.bincount(st, minlength=4))
    # BEHIND_CAMERA wins over OUTLIER
    _, st0, _ = _raw(e, 0.0)
    np.testing.assert_array_equal(st0[behind], OBS_BEHIND_CAMERA)


def test_threshold_boundary_and_validation(engine_lib):
    sc = scenes.scene_test_ba(seed=0, pixel_sigma=1.0)
    e = load_engine(sc)
    res, _, _ = _raw(e)
    l1 = np.abs(res[:, 0]) + np.abs(res[:, 1])
    k = int(np.argsort(l1)[len(l1) // 2])
    _, st, cnt = _raw(e, l1[k])                             # equal to the row's norm: inlier (the Huber test is `>`)
    assert st[k] == OBS_INLIER
    np.testing.assert_array_equal(st, np.where(l1 > l1[k], OBS_OUTLIER, OBS_INLIER))
    np.testing.assert_array_equal(cnt, np.bincount(st, minlength=4))
    _, st, _ = _raw(e, np.nextafter(l1[k], 0.0))
    assert st[k] == OBS_OUTLIER
    # outputs may be left out; a status-only call classifies the same way
    _, st_only, _ = _raw(e, l1[k], want=(False, True, False))
    np.testing.assert_array_equal(st_only, np.where(l1 > l1[k], OBS_OUTLIER, OBS_INLIER))
    for bad in (np.nan, -1.0):
        with pytest.raises(BaError):
            _raw(e, bad)
        with pytest.raises(BaError):
            e.observation_residuals(bad)


def test_shifted_rows_are_the_outliers(engine_lib):
    sc, bad = _outlier_scene()
    e = load_engine(sc)
    _, eo = options_pair(max_num_iterations=30, threshold_huber_loss=0.02)
    e.solve(eo)
    res, st, cnt = e.observation_residuals(5.0)
    is_bad = np.zeros(sc.n_obs, dtype=bool)
    is_bad[bad] = True
    np.testing.assert_array_equal(st == OBS_OUTLIER, is_bad)
    assert (st[~is_bad] == OBS_INLIER).all()
    np.testing.assert_array_equal(cnt, np.bincount(st, minlength=4))


# ------------------------------------------------------------------------------------------------ 4. no side effects
def test_residuals_leave_the_solve_unchanged(engine_lib):
    # tile landmarks only: no FP64 reds in the iteration, so two solves of the same problem are bit-identical
    sc = scenes.scene_trajectory(120, 20_000, 8, stereo=True, seed=31, n_fixed=2)
    _, eo = options_pair(max_num_iterations=10, threshold_cost_change=0.0, threshold_step_size=0.0)

    def run(between):
        e = load_engine(sc)
        rows, launches = [], []
        for k in range(2):
            s = Summary()
            e.solve(eo, s)
            rows += [(i.cost, i.cost_change, i.abs_step, i.abs_gradient, i.damping_term, i.iteration_status)
                     for i in s.optimization_info_list]
            launches.append(e.last_result.kernel_launches)
            if k == 0 and between:
                e.observation_residuals(3.0)
        T, X = e.get_internal()
        return rows, launches, T, X

    a, b = run(False), run(True)
    assert a[0] == b[0] and a[1] == b[1]
    np.testing.assert_array_equal(a[2], b[2])
    np.testing.assert_array_equal(a[3], b[3])
    # the solve never launches the residual kernel; the residual call does
    e = load_engine(sc)
    assert launched_kernels(lambda: e.solve(eo), ("k_obs_residuals",)) == set()
    assert launched_kernels(lambda: e.observation_residuals(), ("k_obs_residuals",)) == {"k_obs_residuals"}


# ------------------------------------------------------------------------------------------------ 5. removal
def test_reject_then_solve_equals_a_fresh_solver_on_the_kept_rows(engine_lib):
    sc, bad = _outlier_scene()
    # the first solve is the one of test_shifted_rows_are_the_outliers: exactly the shifted rows are not inliers
    _, eo = options_pair(max_num_iterations=30, threshold_huber_loss=0.02)
    e = load_engine(sc)
    e.solve(eo)
    T1, X1 = e.get_internal()
    _, st, _ = e.observation_residuals(5.0)
    keep = st == OBS_INLIER
    assert e.reject_outliers(5.0) == int((~keep).sum()) == len(bad)
    s = Summary()
    e.solve(eo, s)
    fresh = load_engine(_subset(sc, keep), identical_internal=(T1, X1))
    s_f = Summary()
    fresh.solve(eo, s_f)
    assert [i.cost for i in s.optimization_info_list] == [i.cost for i in s_f.optimization_info_list]
    for a, b in zip(e.get_internal(), fresh.get_internal()):
        np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(e.get_poses(), fresh.get_poses())
    res, st2, cnt = e.observation_residuals(5.0)
    assert len(st2) == int(keep.sum()) and cnt[OBS_OUTLIER] == 0
    # Rejection pays off when the next solve is not robust itself: from the same robust first solve, a squared-loss
    # solve (the default Huber threshold, 100 px, is far above every residual here) on the kept rows ends closer to the
    # true poses than the same solve on all rows.  (After a robust Huber solve the absolute pose error is dominated by
    # the drift of the trajectory away from its two fixed poses, which removing the shifted rows does not change.)
    _, eo_l2 = options_pair(max_num_iterations=200, threshold_cost_change=0.0, threshold_step_size=0.0)
    free = np.setdiff1d(np.arange(len(sc.poses_true)), sc.fixed_poses)

    def pose_err(reject):
        s_ = load_engine(sc)
        s_.solve(eo)
        if reject:
            s_.reject_outliers(5.0)
        s_.solve(eo_l2)
        return np.abs(s_.get_poses()[free, :3, 3] - sc.poses_true[free, :3, 3]).mean()

    with_rejection, without = pose_err(True), pose_err(False)
    assert with_rejection < 0.9 * without, (with_rejection, without)


def test_remove_observations_validates_the_mask(engine_lib):
    sc = scenes.scene_test_ba(seed=0)
    e = load_engine(sc)
    with pytest.raises(ValueError):
        e.remove_observations(np.ones(sc.n_obs + 1, dtype=bool))
    keep = np.arange(sc.n_obs) % 3 != 0
    e.remove_observations(keep)
    res, st, _ = e.observation_residuals()
    ref = load_engine(_subset(sc, keep))
    np.testing.assert_array_equal(res, ref.observation_residuals()[0])
    np.testing.assert_array_equal(st, ref.observation_residuals()[1])


# ------------------------------------------------------------------------------------------------ 7. C++ shim
def test_cpp_dropin_matches_the_mirror(tmp_path, engine_lib):
    """The drop-in sequence (tests/cpp/test_ba_outliers_dropin.cpp) and the Python mirror on the same scene, from the
    same internal parameters: the same statuses and removals, residuals and parameters to 1e-12."""
    sc, bad = _outlier_scene(seed=23)
    iters, thr, huber = 12, 5.0, 0.02
    exe = _compile("test_ba_outliers_dropin.cpp", tmp_path / "outliers")
    _write_scene(sc, tmp_path / "scene.bin")
    out = subprocess.run([exe, str(tmp_path / "scene.bin"), str(tmp_path / "res.bin"), str(iters), str(thr), str(huber)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "OUTLIERS_DROPIN_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
    raw = open(tmp_path / "res.bin", "rb").read()
    at = 0

    def rows():
        nonlocal at
        n = struct.unpack_from("<i", raw, at)[0]
        st = np.frombuffer(raw, "<i4", n, at + 4)
        res = np.frombuffer(raw, "<f8", 2 * n, at + 4 + 4 * n).reshape(n, 2)
        at += 4 + 4 * n + 16 * n
        return res, st

    def internal():
        nonlocal at
        N, M = len(sc.poses_init), len(sc.points_init)
        T = np.frombuffer(raw, "<f8", 12 * N, at).reshape(N, 12)
        X = np.frombuffer(raw, "<f8", 3 * M, at + 96 * N).reshape(M, 3)
        at += 96 * N + 24 * M
        return T, X

    res0, st0 = rows()
    T0, X0 = internal()
    res1, st1 = rows()
    removed = struct.unpack_from("<i", raw, at)[0]
    at += 4
    res2, st2 = rows()
    T2, X2 = internal()
    assert len(st0) == sc.n_obs                             # refused AddObservation calls are not rows

    def close(a, b):
        assert np.abs(a - b).max() <= 1e-12 * np.abs(b).max(), np.abs(a - b).max()

    e = load_engine(sc, identical_internal=(T0, X0))
    r, s, _ = e.observation_residuals(thr)
    np.testing.assert_array_equal(st0, s)
    close(res0, r)
    _, eo = options_pair(max_num_iterations=iters, threshold_cost_change=1e-6, threshold_step_size=1e-6,
                         threshold_huber_loss=huber)
    e.solve(eo)
    r, s, _ = e.observation_residuals(thr)
    np.testing.assert_array_equal(st1, s)
    close(res1, r)
    # a shorter solve than test_shifted_rows_are_the_outliers: every shifted row is out, a few clean rows may be too
    assert e.reject_outliers(thr) == removed == int((st1 != OBS_INLIER).sum())
    assert (st1[bad] == OBS_OUTLIER).all()
    e.solve(eo)
    r, s, _ = e.observation_residuals()
    np.testing.assert_array_equal(st2, s)
    close(res2, r)
    T, X = e.get_internal()
    close(T2, T)
    close(X2, X)
