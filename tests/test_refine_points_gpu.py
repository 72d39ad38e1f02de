"""Structure-only bundle adjustment on the device (ba_refine_points, k_refine_points): every selected free landmark runs
the LM loop of Solve (full_bundle_adjustment_solver.cpp:707-1008) alone, with every pose fixed and over all of its
observations, with its own lambda and verdict.

The reference for landmark i is the CPU oracle loaded with every pose (all fixed), landmark i alone and its
observations, started from bit-identical internal parameters.  Selection, untouched data, the solver's state after the
call (a solve after a refinement against a fresh solver given the refined parameters), determinism and the C++ drop-in
are checked directly."""
import copy
import ctypes as C
import subprocess

import numpy as np
import pytest

import oracle
from bundle_adjustment_solver_b200 import scenes
from bundle_adjustment_solver_b200.capi import (POINT_CONVERGED, POINT_MAX_ITERATIONS, POINT_NONFINITE, POINT_SKIPPED,
                                                POINT_UNOBSERVED, ptr)
from bundle_adjustment_solver_b200.solver import BaError, Summary
from helpers import launched_kernels, load_engine, load_oracle, options_pair
from test_cpp_dropin import _compile, _write_scene

pytestmark = pytest.mark.gpu

POINT_RTOL = 1e-9
# A landmark whose depth its views barely constrain amplifies the rounding of C and b: with initial_lambda = 1e-10,
# landmark 52 of test_ba seed 1 (same status and iteration count on both sides) ends 7.5e-9 apart (3.4e-8 relative).
# Points are compared to POINT_RTOL relative or to this share of threshold_step_size, whichever is larger.
POINT_ATOL_OF_STEP = 1e-3
COST_RTOL = 1e-12
# A landmark whose observations it fits exactly (two views of one stereo pose, say) ends with residuals at the rounding
# level of its position, and its final cost is rounding noise on both sides (seen: landmark 52 of test_ba seed 0 / 1,
# 1.1797443532440911e-06 against 1.179744353080828e-06, and 3.5e-13 against the oracle's 3.4e-14; landmark 184 of seed 1
# with initial_lambda = 1e-10, 1.775e-09 against 1.758e-09).  Costs are compared to COST_RTOL relative or COST_ATOL
# absolute (internal units: 1e-8 px summed over the landmark's observations), whichever is larger.
COST_ATOL = 1e-10


# ------------------------------------------------------------------------------------------------ scenes
def _true_poses(sc):
    sc = copy.deepcopy(sc)
    sc.poses_init = sc.poses_true.copy()
    return sc


def _test_ba_scene(seed=0):
    """The test_ba.cpp scene at its true poses (stereo rig, five fixed poses) with 0.5 px pixel noise."""
    return _true_poses(scenes.scene_test_ba(seed=seed, pixel_sigma=0.5))


def _c3_shaped(scale=0.2, seed=0):
    return _true_poses(scenes.scene_c3(seed=seed, pixel_sigma=0.5, scale=scale))


def _long_track_scene(seed=4):
    """One camera; landmark 0 is seen more than 256 times (its track repeated with fresh pixel noise), so the
    engine's by-point path would split it."""
    sc = _true_poses(scenes.scene_trajectory(40, 600, 8, stereo=False, seed=seed, pixel_sigma=0.5))
    rng = np.random.default_rng(seed)
    rows = np.flatnonzero(sc.obs_point == 0)
    rep = np.tile(rows, 300 // len(rows) + 1)
    sc.obs_cam = np.concatenate([sc.obs_cam, sc.obs_cam[rep]]).astype(np.int32)
    sc.obs_pose = np.concatenate([sc.obs_pose, sc.obs_pose[rep]]).astype(np.int32)
    sc.obs_point = np.concatenate([sc.obs_point, sc.obs_point[rep]]).astype(np.int32)
    sc.obs_uv = np.concatenate([sc.obs_uv, sc.obs_uv[rep] + rng.normal(0.0, 0.5, (len(rep), 2))])
    return sc


# ------------------------------------------------------------------------------------------------ reference
def _oracle_for_point(sc, i, rows, opts):
    """Landmark i alone, every pose fixed, its observation rows: (infos, converged, initial cost, final cost, X)."""
    o = oracle.FullBAOracle()
    for k, cid in enumerate(sc.cam_ids):
        o.add_camera(cid, *sc.cam_intr[k], sc.cam_T[k])
    o.add_poses(sc.poses_init)
    o.add_points(sc.points_init[i:i + 1])
    for j in range(len(sc.poses_init)):
        o.make_pose_fixed(j)
    o.add_observations(sc.obs_cam[rows], sc.obs_pose[rows], np.zeros(len(rows), dtype=np.int32), sc.obs_uv[rows])
    infos, conv = o.solve(opts)
    return infos, conv, o.initial_cost(), o.cost(), o.get_internal()[1][0]


def _engine(sc):
    """The engine on the whole scene, started from the oracle's internal parameters (bit-identical start)."""
    return load_engine(sc, identical_internal=load_oracle(sc).get_internal())


def _check_parity(sc, points, **kw):
    """Engine vs oracle on the landmarks `points`; returns the oracle's iteration tables."""
    oo, eo = options_pair(**kw)
    e = _engine(sc)
    X0 = e.get_internal()[1].copy()
    status, iters, costs = e.refine_points(eo)
    X = e.get_internal()[1]
    order = np.argsort(sc.obs_point, kind="stable")
    starts = np.searchsorted(sc.obs_point[order], np.arange(len(sc.points_init) + 1))
    tables = {}
    for i in points:
        rows = np.sort(order[starts[i]:starts[i + 1]])
        assert len(rows) > 0
        infos, conv, c0, c1, Xo = _oracle_for_point(sc, i, rows, oo)
        tables[i] = infos
        assert status[i] == (POINT_CONVERGED if conv else POINT_MAX_ITERATIONS), (i, status[i], conv)
        assert iters[i] == len(infos), (i, iters[i], len(infos))
        assert abs(costs[i, 0] - c0) <= max(COST_RTOL * abs(c0), COST_ATOL), (i, costs[i, 0], c0)
        assert abs(costs[i, 1] - c1) <= max(COST_RTOL * abs(c1), COST_ATOL), (i, costs[i, 1], c1)
        tol = max(POINT_RTOL * np.linalg.norm(Xo), POINT_ATOL_OF_STEP * eo.threshold_step_size)
        assert np.linalg.norm(X[i] - Xo) <= tol, (i, X[i], Xo, X0[i])
    return e, status, iters, costs, tables


def _observed(sc):
    return np.flatnonzero(np.bincount(sc.obs_point, minlength=len(sc.points_init)) > 0)


# ------------------------------------------------------------------------------------------------ 1. parity
def test_every_landmark_of_test_ba_matches_the_oracle(engine_lib):
    sc = _test_ba_scene()
    pts = _observed(sc)
    _, status, iters, _, _ = _check_parity(sc, pts, max_num_iterations=50)
    assert (status[pts] == POINT_CONVERGED).mean() > 0.9
    assert np.median(iters[pts]) >= 5


def test_sampled_landmarks_of_a_c3_shaped_scene_match_the_oracle(engine_lib):
    sc = _c3_shaped()
    pts = np.sort(np.random.default_rng(1).choice(_observed(sc), 300, replace=False))
    _check_parity(sc, pts, max_num_iterations=50)


def test_landmark_with_more_than_256_observations(engine_lib):
    sc = _long_track_scene()
    counts = np.bincount(sc.obs_point, minlength=len(sc.points_init))
    assert counts[0] > 256
    _check_parity(sc, [0] + list(range(1, 40)), max_num_iterations=50)


def test_max_iterations_is_reported(engine_lib):
    sc = _test_ba_scene(seed=2)
    pts = _observed(sc)
    _, status, iters, _, _ = _check_parity(sc, pts, max_num_iterations=3)
    assert (status[pts] == POINT_MAX_ITERATIONS).any()
    assert iters[pts].max() == 3


def test_small_initial_lambda_takes_rejected_steps(engine_lib):
    sc = _test_ba_scene(seed=1)
    pts = _observed(sc)
    _, _, _, _, tables = _check_parity(sc, pts, max_num_iterations=50, initial_lambda=1e-10)
    assert any(info.iteration_status == 2 for t in tables.values() for info in t)


# ------------------------------------------------------------------------------------------------ 2. selection
def _camera_centre_scene():
    """test_ba plus one pose with an identity rotation at (1, 2, 0.5) and a landmark exactly at its camera-0 centre,
    seen from it and from pose 10: its initial cost is not finite."""
    sc = _test_ba_scene(seed=5)
    T = np.eye(4)
    T[:3, 3] = [1.0, 2.0, 0.5]
    sc.poses_true = np.concatenate([sc.poses_true, T[None]])
    sc.poses_init = np.concatenate([sc.poses_init, T[None]])
    sc.points_true = np.concatenate([sc.points_true, [[1.0, 2.0, 0.5]]])
    sc.points_init = np.concatenate([sc.points_init, [[1.0, 2.0, 0.5]]])
    j, i = len(sc.poses_init) - 1, len(sc.points_init) - 1
    sc.obs_cam = np.concatenate([sc.obs_cam, [0, 0]]).astype(np.int32)
    sc.obs_pose = np.concatenate([sc.obs_pose, [j, 10]]).astype(np.int32)
    sc.obs_point = np.concatenate([sc.obs_point, [i, i]]).astype(np.int32)
    sc.obs_uv = np.concatenate([sc.obs_uv, [[320.0, 240.0], [300.0, 200.0]]])
    sc.fixed_points = _observed(sc)[[3, 50, 51, 300]]
    return sc, i


def test_selection_and_untouched_landmarks(engine_lib):
    sc, centre = _camera_centre_scene()
    M = len(sc.points_init)
    observed = np.bincount(sc.obs_point, minlength=M) > 0
    assert observed[sc.fixed_points].all()
    select = np.random.default_rng(3).random(M) < 0.5
    select[centre] = True
    select[sc.fixed_points] = True          # selected but fixed: still skipped
    unobs = np.flatnonzero(~observed)
    select[unobs[:5]] = True
    e = _engine(sc)
    T0, X0 = (a.copy() for a in e.get_internal())
    _, eo = options_pair(max_num_iterations=50)
    sel = np.ascontiguousarray(select.astype(np.uint8))
    costs = np.zeros((M, 2))
    iters = np.full(M, -1, dtype=np.int32)
    status = np.zeros(M, dtype=np.uint8)
    counts = np.zeros(5, dtype=np.int64)
    assert e.L.ba_refine_points(e.h, C.byref(eo), ptr(sel), ptr(costs), ptr(iters), ptr(status), ptr(counts)) == 0
    T, X = e.get_internal()
    np.testing.assert_array_equal(T, T0)
    fixed = np.zeros(M, dtype=bool)
    fixed[sc.fixed_points] = True
    skipped = fixed | ~select
    assert (status[skipped] == POINT_SKIPPED).all()
    untouched = skipped | (status >= POINT_SKIPPED)
    np.testing.assert_array_equal(X[untouched], X0[untouched])
    assert (iters[untouched] == 0).all()
    assert (status[unobs[:5]] == POINT_UNOBSERVED).all()
    assert status[centre] == POINT_NONFINITE and not np.isfinite(costs[centre, 0])
    refined = select & ~fixed & observed
    refined[centre] = False
    assert (status[refined] <= POINT_MAX_ITERATIONS).all() and (iters[refined] >= 1).all()
    assert (np.abs(X[refined] - X0[refined]).max(axis=1) > 0).all()
    np.testing.assert_array_equal(counts, np.bincount(status, minlength=5))
    # costs: skipped observed landmarks report their cost twice, unobserved ones zero
    sk = skipped & observed
    np.testing.assert_array_equal(costs[sk, 0], costs[sk, 1])
    assert (costs[sk, 0] > 0).all() and (costs[~observed] == 0).all()


def test_mirror_writes_back_refined_landmarks_only(engine_lib):
    sc = _test_ba_scene(seed=6)
    sc.fixed_points = np.array([7, 8])
    e = load_engine(sc)
    P0 = e.get_points().copy()
    status, _, _ = e.refine_points()
    refined = status <= POINT_MAX_ITERATIONS
    np.testing.assert_array_equal(e.get_points()[~refined], P0[~refined])
    np.testing.assert_array_equal(e.get_points()[refined], e.get_internal()[1][refined] * e.inverse_scaler)
    assert (status[[7, 8]] == POINT_SKIPPED).all()


def test_options_and_state_are_validated(engine_lib):
    sc = _test_ba_scene()
    e = load_engine(sc)
    for kw in (dict(method=1), dict(method=2), dict(max_num_iterations=0)):   # Gauss-Newton, gradient descent
        _, eo = options_pair(**kw)
        with pytest.raises(BaError):
            e.refine_points(eo)
    with pytest.raises(ValueError):
        e.refine_points(select=np.ones(3, dtype=bool))


# ------------------------------------------------------------------------------------------------ 3. state after
def _iter_rows(summ):
    return [(i.cost, i.cost_change, i.average_reprojection_error, i.abs_step, i.damping_term, i.iteration_status)
            for i in summ.optimization_info_list]


@pytest.mark.parametrize("solve_first", [False, True])
def test_solve_after_refine_equals_a_fresh_solver(engine_lib, solve_first):
    # noisy poses, so the later solve has work to do; tracks of 6 to 10 poses: tile landmarks only, whose solves are
    # bit-reproducible (the FP64 reductions of the by-point Schur paths are not)
    sc = scenes.scene_trajectory(100, 4000, 8, stereo=True, seed=7, n_fixed=2, pixel_sigma=0.5)
    _, eo = options_pair(max_num_iterations=12, threshold_cost_change=1e-9, threshold_step_size=1e-9)
    e = _engine(sc)
    if solve_first:
        _, eo3 = options_pair(max_num_iterations=3)
        e.solve(eo3)                                     # the accepted parameters end in the second buffer
    _, ro = options_pair(max_num_iterations=50)
    status, _, costs = e.refine_points(ro)
    T, X = (a.copy() for a in e.get_internal())
    f = load_engine(sc, identical_internal=(T, X))
    assert e.cost() == pytest.approx(costs[:, 1].sum(), rel=1e-12, abs=0)
    assert e.cost() == f.cost()
    r_e, s_e, _ = e.observation_residuals(2.0)
    r_f, s_f, _ = f.observation_residuals(2.0)
    np.testing.assert_array_equal(r_e, r_f)
    np.testing.assert_array_equal(s_e, s_f)
    se, sf = Summary(), Summary()
    e.solve(eo, se)
    f.solve(eo, sf)
    assert len(se.optimization_info_list) >= 2
    assert _iter_rows(se) == _iter_rows(sf)
    Te, Xe = e.get_internal()
    Tf, Xf = f.get_internal()
    np.testing.assert_array_equal(Te, Tf)
    np.testing.assert_array_equal(Xe, Xf)


def test_remove_observations_after_refine_starts_from_the_refined_points(engine_lib):
    sc = _test_ba_scene(seed=8)
    e = _engine(sc)
    e.refine_points()
    X = e.get_internal()[1].copy()
    keep = np.ones(sc.n_obs, dtype=bool)
    keep[::50] = False
    e.remove_observations(keep)
    e.finalize_parameters()   # uploads the kept rows
    np.testing.assert_array_equal(e.get_internal()[1], X)


def test_solve_never_launches_the_refine_kernel(engine_lib):
    sc = _test_ba_scene()
    e = load_engine(sc)
    _, eo = options_pair(max_num_iterations=4)
    assert launched_kernels(lambda: e.solve(eo), ["k_refine_points"]) == set()
    assert launched_kernels(lambda: e.refine_points(), ["k_refine_points"]) == {"k_refine_points"}


# ------------------------------------------------------------------------------------------------ 4. determinism
def test_refinement_is_bit_reproducible(engine_lib):
    sc = _c3_shaped(scale=0.1, seed=3)
    out = []
    for _ in range(2):
        e = load_engine(sc)
        st, it, c = e.refine_points()
        out.append((st, it, c, e.get_internal()[1]))
    for a, b in zip(*out):
        np.testing.assert_array_equal(a, b)


# ------------------------------------------------------------------------------------------------ 5. C++ drop-in
def test_cpp_dropin_matches_the_mirror(tmp_path, engine_lib):
    """tests/cpp/test_refine_points_dropin.cpp: registration, RefinePoints, Solve; the refined points (caller's units
    and internal) and the solve that follows match the Python mirror from the same internal parameters."""
    sc = scenes.scene_test_ba(seed=9, pixel_sigma=0.5)
    iters = 8
    exe = _compile("test_refine_points_dropin.cpp", tmp_path / "refine")
    _write_scene(sc, tmp_path / "scene.bin")
    out = subprocess.run([exe, str(tmp_path / "scene.bin"), str(tmp_path / "res.bin"), str(iters)],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode == 0 and "REFINE_DROPIN_OK" in out.stdout, out.stdout[-2000:] + out.stderr[-2000:]
    raw = open(tmp_path / "res.bin", "rb").read()
    N, M = len(sc.poses_init), len(sc.points_init)
    at = 0

    def take(dtype, n):
        nonlocal at
        a = np.frombuffer(raw, dtype, n, at)
        at += a.nbytes
        return a

    T0, X0 = take("<f8", 12 * N).reshape(N, 12), take("<f8", 3 * M).reshape(M, 3)
    refined = take("<i4", 1)[0]
    st = take("<i4", M)
    P = take("<f8", 3 * M).reshape(M, 3)
    X1 = take("<f8", 3 * M).reshape(M, 3)
    T2, X2 = take("<f8", 12 * N).reshape(N, 12), take("<f8", 3 * M).reshape(M, 3)
    assert at == len(raw)

    e = load_engine(sc, identical_internal=(T0.copy(), X0.copy()))
    status, _, _ = e.refine_points()
    np.testing.assert_array_equal(st, status)
    assert refined == int((status <= POINT_MAX_ITERATIONS).sum()) > 0
    np.testing.assert_array_equal(X1, e.get_internal()[1])
    np.testing.assert_array_equal(P, e.get_points())
    _, eo = options_pair(max_num_iterations=iters, threshold_cost_change=1e-6, threshold_step_size=1e-6)
    e.solve(eo)
    T, X = e.get_internal()
    np.testing.assert_allclose(T2, T, rtol=0, atol=1e-12)
    np.testing.assert_allclose(X2, X, rtol=0, atol=1e-12 * np.abs(X).max())
