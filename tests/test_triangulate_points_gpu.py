"""Triangulation on the device (ba_triangulate_points, k_triangulate_points): every selected free landmark is placed
at the multi-view midpoint of its viewing rays from the accepted poses, with parallax, depth and residual checks.

The reference is the float64 numpy restatement in triangulation_reference.py, given the engine's internal parameters.
Statuses must be identical and positions within 1e-9 relative; thresholds are moved (by 0.1 % steps) until no landmark
lies within 1e-6 relative of either, so ties are excluded by construction.  The solver's state after the call, the
consistency with ba_observation_residuals, determinism, a triangulate-then-solve workflow and the C++ drop-in are
checked directly."""
import copy
import math
import subprocess

import numpy as np
import pytest

from bundle_adjustment_solver_b200 import scenes
from bundle_adjustment_solver_b200.capi import (OBS_INLIER, TRI_BEHIND_CAMERA, TRI_LARGE_RESIDUAL, TRI_LOW_PARALLAX,
                                                TRI_SKIPPED, TRI_TOO_FEW_OBSERVATIONS, TRI_TRIANGULATED, ptr)
from bundle_adjustment_solver_b200.solver import Summary
from helpers import launched_kernels, load_engine, options_pair
from test_cpp_dropin import _compile, _write_scene
import triangulation_reference as R

pytestmark = pytest.mark.gpu

POINT_RTOL = 1e-9
BA_ERR_INVALID = -1


# ------------------------------------------------------------------------------------------------ helpers
def _true_poses(sc):
    sc = copy.deepcopy(sc)
    sc.poses_init = sc.poses_true.copy()
    return sc


def _nan_points(sc):
    """Every free landmark registered without a position."""
    sc = copy.deepcopy(sc)
    free = np.ones(len(sc.points_init), dtype=bool)
    free[np.asarray(sc.fixed_points, dtype=np.int64)] = False
    sc.points_init = sc.points_init.copy()
    sc.points_init[free] = np.nan
    return sc


def _bits(a):
    return np.ascontiguousarray(a).view(np.uint64)


def _call(e, select=None, deg=1.0, px=np.inf):
    """ba_triangulate_points through the C-ABI: (rc, status, counts)."""
    M = len(e.get_points())
    sel = None if select is None else np.ascontiguousarray(np.asarray(select, dtype=bool).astype(np.uint8))
    status = np.full(M, 255, dtype=np.uint8)
    counts = np.full(6, -1, dtype=np.int64)
    rc = e.L.ba_triangulate_points(e.h, ptr(sel), math.radians(deg), float(px) * e.scaler, ptr(status), ptr(counts))
    return rc, status, counts


def _check(e, sc, select=None, deg=1.0, px=np.inf, clear=True):
    """Engine against the reference from the engine's accepted parameters; returns (status, X after, reference)."""
    e.finalize_parameters()
    T0, X0 = (a.copy() for a in e.get_internal())
    pb = R.problem_from_scene(sc, T0, X0)
    if clear:
        deg, px = R.clear_thresholds(pb, deg, px, select)
    ref = R.triangulate(pb, select, math.radians(deg), px * R.SCALER)
    rc, status, counts = _call(e, select, deg, px)
    assert rc == 0, e.L.ba_last_error(e.h).decode()
    T, X = e.get_internal()
    np.testing.assert_array_equal(status, ref.status)
    np.testing.assert_array_equal(counts, np.bincount(status, minlength=6))
    np.testing.assert_array_equal(_bits(T), _bits(T0))
    kept = status != TRI_TRIANGULATED
    np.testing.assert_array_equal(_bits(X[kept]), _bits(X0[kept]))
    tri = ~kept
    err = np.linalg.norm(X[tri] - ref.points[tri], axis=1)
    bad = np.flatnonzero(err > POINT_RTOL * np.linalg.norm(ref.points[tri], axis=1))
    assert len(bad) == 0, (np.flatnonzero(tri)[bad[:5]], X[tri][bad[:5]], ref.points[tri][bad[:5]])
    return status, X, ref, (deg, px)


# ------------------------------------------------------------------------------------------------ 1. exact recovery
@pytest.mark.parametrize("stereo", [True, False])
def test_exact_recovery_from_noise_free_pixels(engine_lib, stereo):
    # float64 pixels at the true poses; every landmark registered as NaN
    sc = _nan_points(_true_poses(scenes.scene_trajectory(80, 3000, 6, stereo=stereo, seed=11)))
    e = load_engine(sc)
    status, X, _, _ = _check(e, sc)
    tri = status == TRI_TRIANGULATED
    assert tri.mean() > 0.95, np.bincount(status, minlength=6)
    truth = sc.points_true * R.SCALER
    err = np.linalg.norm(X[tri] - truth[tri], axis=1) / np.linalg.norm(truth[tri], axis=1)
    assert err.max() <= POINT_RTOL, err.max()
    assert np.isnan(X[~tri]).all()


# ------------------------------------------------------------------------------------------------ 2. parity
def _test_ba(at_true):
    sc = scenes.scene_test_ba(seed=0, pixel_sigma=0.5)
    return _true_poses(sc) if at_true else sc


@pytest.mark.parametrize("case", ["test_ba_true_poses", "test_ba_poses_init", "c3_shaped"])
def test_parity_with_the_reference(engine_lib, case):
    if case == "c3_shaped":
        sc = _true_poses(scenes.scene_c3(seed=0, pixel_sigma=0.5, scale=0.2))
        px = 2.0
    else:
        sc = _test_ba(case == "test_ba_true_poses")
        px = 3.0 if case == "test_ba_true_poses" else 10.0
    e = load_engine(sc)
    status, _, _, _ = _check(e, sc, deg=1.0, px=px)
    n = np.bincount(status, minlength=6)
    assert n[TRI_TRIANGULATED] > 0 and n[TRI_LARGE_RESIDUAL] > 0, n


# ------------------------------------------------------------------------------------------------ 3. constructed cases
def _constructed_scene():
    """A noise-free stereo trajectory at its true poses (fixed landmarks 2 and 3) plus, registered as NaN:
    U unobserved, O one observation, D two identical rows, B a point behind the cameras (projected from behind two
    poses), L a landmark seen more than 256 times (landmark 0's rows repeated with 0.5 px noise), and an injected 20 px
    outlier on one row of landmark 1."""
    sc = _true_poses(scenes.scene_trajectory(40, 600, 8, stereo=True, seed=4))
    rng = np.random.default_rng(4)
    M = len(sc.points_init)
    # L: landmark 0's rows repeated
    rows0 = np.flatnonzero(sc.obs_point == 0)
    rep = np.tile(rows0, 300 // len(rows0) + 1)
    extra = dict(cam=list(sc.obs_cam[rep]), pose=list(sc.obs_pose[rep]), point=list(sc.obs_point[rep]),
                 uv=list(sc.obs_uv[rep] + rng.normal(0.0, 0.5, (len(rep), 2))))
    # the outlier: 20 px on the u of one of landmark 1's rows
    rows1 = np.flatnonzero(sc.obs_point == 1)
    assert len(rows1) >= 6
    sc.obs_uv = sc.obs_uv.copy()
    sc.obs_uv[rows1[2], 0] += 20.0
    U, O, D, B = M, M + 1, M + 2, M + 3
    intr = sc.cam_intr[0]

    def pixel(j, Xw):
        T_cw = scenes.inv_T(sc.poses_true[j])
        Xc = T_cw[:3, :3] @ Xw + T_cw[:3, 3]
        return [intr[0] * Xc[0] / Xc[2] + intr[2], intr[1] * Xc[1] / Xc[2] + intr[3]]

    def add(point, pose, uv):
        extra["cam"].append(0); extra["pose"].append(pose); extra["point"].append(point); extra["uv"].append(uv)

    add(O, 5, [300.0, 200.0])
    add(D, 7, [310.0, 250.0])
    add(D, 7, [310.0, 250.0])
    # B: 5 m behind pose 10's camera; poses 10 and 14 both see it from the front of the lines through it
    Xb = sc.poses_true[10][:3, :3] @ np.array([0.3, 0.2, -5.0]) + sc.poses_true[10][:3, 3]
    add(B, 10, pixel(10, Xb))
    add(B, 14, pixel(14, Xb))
    sc.points_true = np.concatenate([sc.points_true, np.full((4, 3), np.nan)])
    sc.points_true[B] = Xb
    sc.points_init = np.concatenate([sc.points_init, np.full((4, 3), np.nan)])
    sc.obs_cam = np.concatenate([sc.obs_cam, np.asarray(extra["cam"])]).astype(np.int32)
    sc.obs_pose = np.concatenate([sc.obs_pose, np.asarray(extra["pose"])]).astype(np.int32)
    sc.obs_point = np.concatenate([sc.obs_point, np.asarray(extra["point"])]).astype(np.int32)
    sc.obs_uv = np.concatenate([sc.obs_uv, np.asarray(extra["uv"], dtype=np.float64)])
    sc.fixed_points = np.array([2, 3])
    return sc, dict(U=U, O=O, D=D, B=B, L=0, outlier=1, fixed=[2, 3])


@pytest.mark.parametrize("masked", [False, True])
def test_constructed_cases(engine_lib, masked):
    sc, ids = _constructed_scene()
    M = len(sc.points_init)
    assert np.bincount(sc.obs_point, minlength=M)[ids["L"]] > 256
    select = None
    if masked:
        select = np.random.default_rng(5).random(M) < 0.5
        select[[ids[k] for k in ("U", "O", "D", "B", "L", "outlier")]] = True
        select[ids["fixed"]] = True                    # selected but fixed: still skipped
    e = load_engine(sc)
    status, X, ref, (deg, px) = _check(e, sc, select, deg=1.0, px=5.0)
    assert status[ids["U"]] == TRI_TOO_FEW_OBSERVATIONS and status[ids["O"]] == TRI_TOO_FEW_OBSERVATIONS
    assert status[ids["D"]] == TRI_LOW_PARALLAX
    assert status[ids["B"]] == TRI_BEHIND_CAMERA
    np.testing.assert_allclose(ref.X[ids["B"]], sc.points_true[ids["B"]] * R.SCALER, rtol=1e-9)
    assert status[ids["outlier"]] == TRI_LARGE_RESIDUAL
    assert status[ids["L"]] == TRI_TRIANGULATED
    assert (status[ids["fixed"]] == TRI_SKIPPED).all()
    if masked:
        assert (status[~select] == TRI_SKIPPED).all()
    assert np.isnan(X[[ids["U"], ids["O"], ids["D"], ids["B"]]]).all()
    # +inf disables the residual rule: the outlier landmark is placed
    f = load_engine(sc)
    status_inf, _, _, _ = _check(f, sc, select, deg=deg, px=np.inf, clear=False)
    assert status_inf[ids["outlier"]] == TRI_TRIANGULATED
    changed = status != status_inf
    assert (status[changed] == TRI_LARGE_RESIDUAL).all()


# ------------------------------------------------------------------------------------------------ 4. residual report
def test_triangulated_rows_are_inliers_of_the_residual_report(engine_lib):
    sc = _test_ba(True)
    e = load_engine(sc)
    e.finalize_parameters()
    pb = R.problem_from_scene(sc, *e.get_internal())
    deg, tau = R.clear_thresholds(pb, 1.0, 2.0)
    P0 = e.get_points().copy()
    status, counts = e.triangulate_points(min_parallax_deg=deg, max_residual_px=tau)
    np.testing.assert_array_equal(counts, np.bincount(status, minlength=6))
    tri = status == TRI_TRIANGULATED
    assert tri.any() and (status == TRI_LARGE_RESIDUAL).any()
    _, obs_status, _ = e.observation_residuals(tau)
    assert (obs_status[tri[sc.obs_point]] == OBS_INLIER).all()
    # the mirror wrote the triangulated landmarks only, in the caller's units
    np.testing.assert_array_equal(e.get_points()[~tri], P0[~tri])
    np.testing.assert_array_equal(e.get_points()[tri], e.get_internal()[1][tri] * e.inverse_scaler)


# ------------------------------------------------------------------------------------------------ 5. state after
def _iter_rows(summ):
    return [(i.cost, i.cost_change, i.average_reprojection_error, i.abs_step, i.damping_term, i.iteration_status)
            for i in summ.optimization_info_list]


@pytest.mark.parametrize("solve_first", [False, True])
@pytest.mark.parametrize("follow", ["solve", "refine"])
def test_state_after_the_call_equals_a_fresh_solver(engine_lib, follow, solve_first):
    # tracks of 6 to 10 poses: tile landmarks only, whose solves are bit-reproducible
    sc = scenes.scene_trajectory(100, 4000, 8, stereo=True, seed=7, n_fixed=2, pixel_sigma=0.5)
    e = load_engine(sc)
    if solve_first:
        _, eo3 = options_pair(max_num_iterations=3)
        e.solve(eo3)                                     # the accepted parameters end in the second buffer
    T0 = e.get_internal()[0].copy()
    status, _ = e.triangulate_points(max_residual_px=np.inf)
    assert (status == TRI_TRIANGULATED).mean() > 0.9
    T, X = (a.copy() for a in e.get_internal())
    np.testing.assert_array_equal(_bits(T), _bits(T0))
    f = load_engine(sc, identical_internal=(T, X))
    assert e.cost() == f.cost()
    if follow == "solve":
        _, eo = options_pair(max_num_iterations=12, threshold_cost_change=1e-9, threshold_step_size=1e-9)
        se, sf = Summary(), Summary()
        e.solve(eo, se)
        f.solve(eo, sf)
        assert len(se.optimization_info_list) >= 2
        assert _iter_rows(se) == _iter_rows(sf)
    else:
        _, ro = options_pair(max_num_iterations=20)
        re_, rf = e.refine_points(ro), f.refine_points(ro)
        for a, b in zip(re_, rf):
            np.testing.assert_array_equal(a, b)
    Te, Xe = e.get_internal()
    Tf, Xf = f.get_internal()
    np.testing.assert_array_equal(_bits(Te), _bits(Tf))
    np.testing.assert_array_equal(_bits(Xe), _bits(Xf))


def test_two_solvers_give_bit_identical_outputs(engine_lib):
    sc = _nan_points(_true_poses(scenes.scene_c3(seed=3, pixel_sigma=0.5, scale=0.1)))
    out = []
    for _ in range(2):
        e = load_engine(sc)
        rc, status, counts = _call(e, deg=1.0, px=3.0)
        assert rc == 0
        out.append((status, counts, _bits(e.get_internal()[1])))
    for a, b in zip(*out):
        np.testing.assert_array_equal(a, b)


def test_solve_never_launches_the_triangulation_kernel(engine_lib):
    sc = _true_poses(scenes.scene_test_ba(seed=1, pixel_sigma=0.5))
    e = load_engine(sc)
    _, eo = options_pair(max_num_iterations=4)
    assert launched_kernels(lambda: e.solve(eo), ["k_triangulate_points"]) == set()
    assert launched_kernels(lambda: e.triangulate_points(), ["k_triangulate_points"]) == {"k_triangulate_points"}


def test_invalid_thresholds(engine_lib):
    sc = _true_poses(scenes.scene_test_ba(seed=2, pixel_sigma=0.5))
    e = load_engine(sc)
    X0 = e.get_internal()[1].copy()
    for rad, res in ((0.0, 0.01), (-0.1, 0.01), (math.nan, 0.01), (math.pi * (1 + 1e-15), 0.01), (4.0, 0.01),
                     (0.1, -1e-3), (0.1, math.nan), (0.1, -math.inf)):
        assert e.L.ba_triangulate_points(e.h, None, rad, res, None, None) == BA_ERR_INVALID, (rad, res)
    np.testing.assert_array_equal(_bits(e.get_internal()[1]), _bits(X0))
    for rad, res in ((math.pi, 0.0), (1e-6, math.inf)):          # the ends of the ranges are valid
        assert e.L.ba_triangulate_points(e.h, None, rad, res, None, None) == 0, (rad, res)


# ------------------------------------------------------------------------------------------------ 6. workflow
# Seeded result of the triangulate-then-solve workflow (scene_c3 seed 0, 0.5 px, scale 0.2, from poses_init, options
# below), measured on one B200: the final cost of the solve from the triangulated landmarks (24 iterations) and of the
# solve from points_init (21 iterations).  initial_lambda is 1e-3 because the triangulated start is already close: with
# the default 100 the first damped step (|step| 6.4e-6) is below threshold_step_size and the reference's loop stops
# after one iteration (cost 9496 against 1214.5 from points_init, which starts 56367 and takes 22 iterations).
WORKFLOW_OPTIONS = dict(max_num_iterations=100, initial_lambda=1e-3)
WORKFLOW_FINAL_COST = {"triangulated": 1214.0931119881636, "points_init": 1225.1648608682854}


def test_triangulate_then_solve(engine_lib):
    sc = scenes.scene_c3(seed=0, pixel_sigma=0.5, scale=0.2)
    e = load_engine(_nan_points(sc))
    status, counts = e.triangulate_points()
    assert (status == TRI_TRIANGULATED).all(), counts          # a NaN left behind would poison the cost
    _, eo = options_pair(**WORKFLOW_OPTIONS)
    se, sf = Summary(), Summary()
    e.solve(eo, se)
    f = load_engine(sc)
    f.solve(eo, sf)
    assert se.convergence_status and sf.convergence_status
    ce, cf = e.cost(), f.cost()
    print(f"WORKFLOW triangulated {ce!r} ({len(se.optimization_info_list)} iterations)  "
          f"points_init {cf!r} ({len(sf.optimization_info_list)} iterations)")
    assert abs(ce - cf) <= 0.01 * cf, (ce, cf)
    assert ce == pytest.approx(WORKFLOW_FINAL_COST["triangulated"], rel=1e-6)
    assert cf == pytest.approx(WORKFLOW_FINAL_COST["points_init"], rel=1e-6)


# ------------------------------------------------------------------------------------------------ 7. C++ drop-in
def test_cpp_dropin_matches_the_mirror(tmp_path, engine_lib):
    """tests/cpp/test_triangulate_points_dropin.cpp: the test_ba scene registered with every landmark at the origin,
    TriangulatePoints, Solve; statuses, points (caller's units and internal) and the solve that follows match the Python
    mirror from the same internal parameters."""
    sc = scenes.scene_test_ba(seed=9, pixel_sigma=0.5)
    sc.points_init = np.zeros_like(sc.points_init)
    iters = 8
    e = load_engine(sc)
    e.finalize_parameters()
    deg, px = R.clear_thresholds(R.problem_from_scene(sc, *e.get_internal()), 1.0, 10.0)
    exe = _compile("test_triangulate_points_dropin.cpp", tmp_path / "triangulate")
    _write_scene(sc, tmp_path / "scene.bin")
    out = subprocess.run([exe, str(tmp_path / "scene.bin"), str(tmp_path / "res.bin"), str(iters), repr(deg), repr(px)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "TRIANGULATE_DROPIN_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
    raw = open(tmp_path / "res.bin", "rb").read()
    N, M = len(sc.poses_init), len(sc.points_init)
    at = 0

    def take(dtype, n):
        nonlocal at
        a = np.frombuffer(raw, dtype, n, at)
        at += a.nbytes
        return a

    T0, X0 = take("<f8", 12 * N).reshape(N, 12), take("<f8", 3 * M).reshape(M, 3)
    triangulated = take("<i4", 1)[0]
    st = take("<i4", M)
    P = take("<f8", 3 * M).reshape(M, 3)
    X1 = take("<f8", 3 * M).reshape(M, 3)
    T2, X2 = take("<f8", 12 * N).reshape(N, 12), take("<f8", 3 * M).reshape(M, 3)
    assert at == len(raw)

    g = load_engine(sc, identical_internal=(T0.copy(), X0.copy()))
    status, _ = g.triangulate_points(min_parallax_deg=deg, max_residual_px=px)
    np.testing.assert_array_equal(st, status)
    assert triangulated == int((status == TRI_TRIANGULATED).sum()) > 0
    assert (status == TRI_LARGE_RESIDUAL).any() and (status == TRI_LOW_PARALLAX).any()
    np.testing.assert_array_equal(X1, g.get_internal()[1])
    np.testing.assert_array_equal(P, g.get_points())
    _, eo = options_pair(max_num_iterations=iters, threshold_cost_change=1e-6, threshold_step_size=1e-6)
    g.solve(eo)
    T, X = g.get_internal()
    np.testing.assert_allclose(T2, T, rtol=0, atol=1e-12)
    np.testing.assert_allclose(X2, X, rtol=0, atol=1e-12 * np.abs(X).max())
