"""GPU parity tests of the full-BA device path against the CPU oracle, through the C-ABI.

Tolerances (BASELINE.json north_star): Hessian/Schur blocks 1e-9 relative (FP64, reduction-order
differences only), final cost 1e-6 relative, same convergence verdict, iterations within +-1.
"""
import numpy as np
import pytest

from bundle_adjustment_solver_b200 import scenes
from helpers import (BLOCK_TOL, blockwise_rel_err, compare_blocks, launched_kernels, load_engine, load_oracle,
                     options_pair, solve_info)

pytestmark = pytest.mark.gpu

@pytest.mark.parametrize("seed", [0, 1])
@pytest.mark.parametrize("accum", [0, 1])
def test_blocks_match_oracle_c1(seed, accum, oracle_mod, engine_lib):
    sc = scenes.scene_test_ba(seed=seed)
    o = load_oracle(sc)
    o.build_only(thres_huber=1.0, lam=100.0, b_accumulate=accum, do_solve=True)
    e = load_engine(sc, identical_internal=o.get_internal())
    e.set_debug(True)
    oo, eo = options_pair(b_accumulate=accum)
    e.build_only(eo, 100.0, do_solve=True)
    assert e.sizes() == o.sizes()
    # same pair set, same order (sorted by point, pose)
    assert all(np.array_equal(x, y) for x, y in zip(e.pairs(), o.pairs()))
    compare_blocks(o, e, o.sizes())
    # reduced solve and back-substitution: x, y  (conditioning of S enters -> looser, stated)
    assert blockwise_rel_err(e.dump("x"), o.dump("x"), 6) < 1e-6
    assert blockwise_rel_err(e.dump("y"), o.dump("y"), 3) < 1e-6


def test_initial_cost_matches(oracle_mod, engine_lib):
    sc = scenes.scene_test_ba(seed=3)
    o = load_oracle(sc)
    o.sizes()
    e = load_engine(sc, identical_internal=o.get_internal())
    assert abs(e.cost() - o.cost()) <= 1e-12 * abs(o.cost())


@pytest.mark.parametrize("seed,accum", [(0, 0), (1, 0), (2, 0), (0, 1)])
def test_solve_c1_matches_oracle(seed, accum, oracle_mod, engine_lib):
    sc = scenes.scene_test_ba(seed=seed)
    kw = dict(max_num_iterations=300, threshold_cost_change=1e-6, threshold_step_size=1e-6, b_accumulate=accum)
    oo, eo = options_pair(**kw)
    o = load_oracle(sc)
    infos_o, conv_o = o.solve(oo)
    e = load_engine(sc, identical_internal=None)
    from bundle_adjustment_solver_b200.solver import Summary
    summ = Summary()
    e.solve(eo, summ)
    infos_e = summ.optimization_info_list
    assert summ.convergence_status == conv_o
    assert abs(len(infos_e) - len(infos_o)) <= 1, (len(infos_e), len(infos_o))
    fo, fe = infos_o[-1].cost, infos_e[-1].cost
    assert abs(fe - fo) <= 1e-6 * abs(fo), (fe, fo)
    # the first iterations must agree tightly (same trajectory)
    for k in range(min(5, len(infos_o), len(infos_e))):
        assert abs(infos_e[k].cost - infos_o[k].cost) <= 1e-9 * abs(infos_o[k].cost)
        assert infos_e[k].iteration_status == infos_o[k].iteration_status
        assert abs(infos_e[k].damping_term - infos_o[k].damping_term) <= 1e-12 * infos_o[k].damping_term
    # poses / points: stated tolerance 1e-6 m (user units), free parameters written back
    Po, Xo = o.get_poses(), o.get_points()
    Pe, Xe = e.get_poses(), e.get_points()
    assert np.abs(Pe - Po).max() < 1e-6
    assert np.abs(Xe - Xo).max() < 1e-6
    # fixed poses untouched
    assert np.array_equal(Pe[:5], sc.poses_init[:5])
    print(summ.brief_report()[-600:])


def test_rejected_steps_match_oracle(oracle_mod, engine_lib):
    """Reject branch on the device (the decision of k_cost_linearize_by_pose + the double-buffer flip that replaces Reserve / Revert,
    full_bundle_adjustment_solver.cpp:457-482, 939-953, 995-1005): the test_ba.cpp scene started undamped
    (tests/test_oracle_cpu.py::test_rejected_step_reporting) rejects 11 of its first 25 steps.  Every status and every
    lambda of the iteration table must match exactly.  Tolerance of the costs: 1e-5 -- with lambda = 1e-10 the
    system is undamped, weakly observed landmarks are fixed only up to the rounding of the reduced solve (unpivoted
    LL^T here, pivoted LDL^T in the reference), measured drift 4e-6 after 25 iterations (profiles/debug_reject_rows.py);
    landmark coordinates are therefore compared through the cost they give, poses directly."""
    sc = scenes.scene_test_ba(seed=0)
    kw = dict(max_num_iterations=25, threshold_cost_change=1e-9, threshold_step_size=1e-9, initial_lambda=1e-10)
    oo, eo = options_pair(**kw)
    o = load_oracle(sc)
    infos_o, conv_o = o.solve(oo)
    st_o = [i.iteration_status for i in infos_o]
    assert st_o.count(2) >= 8 and st_o.count(0) >= 2          # the scene does what it is for
    o_fresh = load_oracle(sc); o_fresh.sizes()
    e = load_engine(sc, identical_internal=o_fresh.get_internal())
    from bundle_adjustment_solver_b200.solver import Summary
    summ = Summary()
    e.solve(eo, summ)
    infos_e = summ.optimization_info_list
    assert len(infos_e) == len(infos_o) == 25 and summ.convergence_status == conv_o
    # rows 0..12 (four accepted steps, seven rejected in a row, two accepted) are compared strictly; behind them the
    # undamped iteration has amplified the rounding differences of the two reduced solves (and of the FP64 reds of
    # the tile flush, whose order varies from run to run) beyond any fixed tolerance, so only sanity is checked
    K_STRICT = 13
    assert [i.iteration_status for i in infos_e[:K_STRICT]] == st_o[:K_STRICT] and st_o[:K_STRICT].count(2) == 7
    n_obs = o.sizes()["n_obs"]
    for k, (ie, io) in enumerate(zip(infos_e, infos_o)):
        if k < K_STRICT:
            # measured drift: 3e-7 over rows 0..11, 1.4e-6 at row 12 in one run (profiles/debug_reject_rows.py), 2.1e-6 at
            # row 3 in another: the dense-GEMM Schur path of this scene flushes with FP64 reds, so the last bits vary
            # from run to run and the undamped iteration amplifies them.  1e-4 still separates a wrong reject branch
            # (a kept trial cost or a missed revert moves these costs by percents)
            tol = 1e-4
            assert abs(ie.cost - io.cost) <= tol * abs(io.cost), (k, ie.cost, io.cost)
            assert abs(ie.damping_term - io.damping_term) <= 1e-12 * io.damping_term, k
            assert abs(ie.average_reprojection_error - io.average_reprojection_error) <= tol * io.average_reprojection_error
        assert ie.iteration_status in (0, 1, 2) and 1e-10 <= ie.damping_term <= 100.0
        if ie.iteration_status == 2:
            assert ie.cost_change == 0.0
            assert abs(ie.average_reprojection_error - np.sqrt(ie.cost / n_obs)) <= 1e-12
    assert e.cost() < 0.02 * infos_e[0].cost + 60.0
    # stop right after the first rejected step: the parameters are the reserved ones, lambda is raised, and the
    # device kept the REJECTED trial cost as previous cost (:1005)
    k = st_o.index(2)
    kw2 = dict(kw); kw2["max_num_iterations"] = k + 1
    oo2, eo2 = options_pair(**kw2)
    o2 = load_oracle(sc); o2.solve(oo2)
    e2 = load_engine(sc, identical_internal=o_fresh.get_internal())
    e2.set_debug(True)
    e2.solve(eo2, Summary())
    T_e, X_e = e2.get_internal()
    T_o, X_o = o2.get_internal()
    assert np.abs(T_e - T_o).max() < 1e-6
    assert abs(e2.cost() - infos_o[k - 1].cost) <= 1e-4 * infos_o[k - 1].cost          # reverted: the accepted cost
    assert abs(e2.cost() - infos_e[k - 1].cost) <= 1e-4 * infos_e[k - 1].cost          # ... and the first device run's
    so, se = o2.dump("scalars"), e2.dump("scalars")
    assert abs(se[1] - so[1]) <= 1e-4 * abs(so[1]) and se[1] > infos_e[k - 1].cost      # trial cost of the rejected step
    assert so[3] <= 0.25 and se[3] <= 0.25                                              # rho of the rejected step


@pytest.mark.parametrize("scene", ["c1", "trajectory"])
@pytest.mark.parametrize("method,iters", [(1, 40), (2, 25)])
def test_refactor_methods_match_oracle(scene, method, iters, oracle_mod, engine_lib):
    """ba_options.method: the Gauss-Newton branch of FullBundleAdjustmentSolverRefactor::Solve
    (full_bundle_adjustment_solver_refactor.cpp:976-982) and SolveByGradientDescent (:1075-1367) against the
    oracle's restatement: every iteration kept (status UPDATE), lambda untouched, same cost trajectory."""
    sc = scenes.scene_test_ba(seed=4) if scene == "c1" else scenes.scene_trajectory(60, 3000, 8, stereo=True, seed=9, n_fixed=2)
    kw = dict(max_num_iterations=iters, threshold_cost_change=1e-9, threshold_step_size=1e-9, method=method)
    oo, eo = options_pair(**kw)
    o = load_oracle(sc)
    infos_o, conv_o = o.solve(oo)
    e = load_engine(sc, identical_internal=o_internal(sc))
    from bundle_adjustment_solver_b200.solver import Summary
    summ = Summary()
    e.solve(eo, summ)
    infos_e = summ.optimization_info_list
    assert summ.convergence_status == conv_o and len(infos_e) == len(infos_o)
    for ie, io in zip(infos_e, infos_o):
        assert ie.iteration_status == 0 and io.iteration_status == 0
        assert ie.damping_term == io.damping_term == 100.0
        assert abs(ie.cost - io.cost) <= 1e-8 * abs(io.cost), (ie.cost, io.cost)
        assert abs(ie.abs_step - io.abs_step) <= 1e-8 * abs(io.abs_step)
    if method == 2:   # clipped gradient steps: each block moves by at most 0.001 (scaled units) per iteration
        assert infos_e[-1].abs_step <= 0.001 + 0.02 / (sum(1 for _ in sc.points_init) + 1)
    assert np.abs(e.get_poses() - o.get_poses()).max() < 1e-6
    assert np.abs(e.get_points() - o.get_points()).max() < 1e-6


def o_internal(sc):
    o = load_oracle(sc)
    o.sizes()
    return o.get_internal()


def test_fixed_points_and_split_point(oracle_mod, engine_lib):
    """Edge cases: fixed landmarks, landmarks seen only by fixed poses, and one landmark with more
    observations than a 256-observation chunk (split path with atomics)."""
    sc = scenes.scene_trajectory(160, 400, 10, stereo=True, seed=5, n_fixed=3)
    # a landmark seen by every pose in both cameras: 320 observations
    rng = np.random.default_rng(0)
    Xbig = np.array([16.0, 0.2, 30.0])
    M = len(sc.points_true)
    sc.points_true = np.vstack([sc.points_true, Xbig])
    sc.points_init = np.vstack([sc.points_init, Xbig + 0.2])
    T_cw = scenes.inv_T(sc.poses_true)
    cams, poses, pts, uvs = [], [], [], []
    for j in range(len(sc.poses_true)):
        for c in range(2):
            Xb = T_cw[j, :3, :3] @ Xbig + T_cw[j, :3, 3]
            Xc = sc.cam_T[c][:3, :3] @ Xb + sc.cam_T[c][:3, 3]
            uvs.append([sc.cam_intr[c, 0] * Xc[0] / Xc[2] + sc.cam_intr[c, 2],
                        sc.cam_intr[c, 1] * Xc[1] / Xc[2] + sc.cam_intr[c, 3]])
            cams.append(c); poses.append(j); pts.append(M)
    sc.obs_cam = np.concatenate([sc.obs_cam, np.array(cams, dtype=np.int32)])
    sc.obs_pose = np.concatenate([sc.obs_pose, np.array(poses, dtype=np.int32)])
    sc.obs_point = np.concatenate([sc.obs_point, np.array(pts, dtype=np.int32)])
    sc.obs_uv = np.vstack([sc.obs_uv, np.array(uvs)])
    sc.fixed_points = np.array([1, 7, 50])
    for accum in (0, 1):
        o = load_oracle(sc)
        o.build_only(thres_huber=1.0, lam=3.0, b_accumulate=accum, do_solve=True)
        e = load_engine(sc, identical_internal=o.get_internal())
        e.set_debug(True)
        oo, eo = options_pair(b_accumulate=accum)
        e.build_only(eo, 3.0, do_solve=True)
        assert e.sizes() == o.sizes()
        compare_blocks(o, e, o.sizes())
        assert blockwise_rel_err(e.dump("y"), o.dump("y"), 3) < 1e-6
    # and a short solve agrees
    oo, eo = options_pair(max_num_iterations=6)
    o = load_oracle(sc)
    infos_o, _ = o.solve(oo)
    e = load_engine(sc)
    from bundle_adjustment_solver_b200.solver import Summary
    summ = Summary()
    e.solve(eo, summ)
    assert len(summ.optimization_info_list) == len(infos_o)
    assert abs(summ.optimization_info_list[-1].cost - infos_o[-1].cost) <= 1e-6 * abs(infos_o[-1].cost)


def test_graph_and_plain_launch_agree(oracle_mod, engine_lib):
    sc = scenes.scene_test_ba(seed=4)
    from bundle_adjustment_solver_b200.solver import Summary
    outs = []
    for use_graph in (1, 0):
        _, eo = options_pair(max_num_iterations=12, use_graph=use_graph, check_every=5)
        e = load_engine(sc)
        summ = Summary()
        e.solve(eo, summ)
        outs.append([i.cost for i in summ.optimization_info_list])
    assert len(outs[0]) == len(outs[1]) == 12
    np.testing.assert_allclose(outs[0], outs[1], rtol=1e-10)


_REJECT_KW = dict(max_num_iterations=12, initial_lambda=1e-10, threshold_cost_change=1e-9, threshold_step_size=1e-9)


@pytest.mark.parametrize("scene,kw,n_strict", [
    ("trajectory", dict(max_num_iterations=12), 12),
    ("trajectory_rejects", _REJECT_KW, 5),
    ("c1", dict(max_num_iterations=15), 5),
])
def test_speculative_pose_side_and_storing_reduce_match_oracle(scene, kw, n_strict, monkeypatch, oracle_mod, engine_lib):
    """The trial-cost pass also linearises the pose side at the trial parameters (k_cost_linearize_by_pose); the next
    iteration starts from those sums, either through k_pose_diag after the clear of S and the adding k_tile_reduce, or
    through the storing k_tile_reduce on banded plans (BA_B200_REDUCE_STORES=0 / 1).  The oracle re-linearises at every
    iteration, so it is the reference of the speculative form: the first n_strict rows of the iteration table have the
    same statuses, lambda within 1e-12 and cost within 1e-9.  The two reduce forms run the same arithmetic in the same
    order: bit-identical tables and parameters on the banded trajectory scenes, where the storing form launches fewer
    kernels; the test_ba.cpp scene (c1) is not banded, both forms launch the same kernels there.
    trajectory_rejects: a mono trajectory with noisy pixels started undamped accepts three steps and then rejects
    (row 3: the trial cost is 1.1e-4 above the accepted one; behind row 4 the cost differences are at rounding level, so
    the oracle is compared up to row 4) -- the storing reduce must read the sums of the KEPT parameter buffer."""
    from bundle_adjustment_solver_b200.solver import Summary
    if scene == "trajectory":
        sc = scenes.scene_trajectory(60, 3000, 10, stereo=True, seed=3, name="spec_traj")
    elif scene == "trajectory_rejects":
        sc = scenes.scene_trajectory(60, 3000, 10, stereo=False, seed=3, pixel_sigma=2.0)
    else:
        sc = scenes.scene_test_ba(seed=0)
    oo, eo = options_pair(**kw)
    o = load_oracle(sc)
    infos_o, _ = o.solve(oo)
    o_fresh = load_oracle(sc); o_fresh.sizes()
    if scene == "trajectory_rejects":
        assert [i.iteration_status for i in infos_o[:5]] == [1, 1, 1, 2, 2]     # the scene does what it is for
    runs = []
    for stores in ("0", "1"):
        monkeypatch.setenv("BA_B200_REDUCE_STORES", stores)
        _, eo = options_pair(**kw)
        e = load_engine(sc, identical_internal=o_fresh.get_internal())
        summ = Summary()
        e.solve(eo, summ)
        infos_e = summ.optimization_info_list
        assert len(infos_e) >= n_strict
        for a, b in zip(infos_e[:n_strict], infos_o[:n_strict]):
            assert a.iteration_status == b.iteration_status
            assert abs(a.damping_term - b.damping_term) <= 1e-12 * b.damping_term
            assert abs(a.cost - b.cost) <= 1e-9 * abs(b.cost), (a.cost, b.cost)
        T, X = e.get_internal()
        if scene == "trajectory":
            assert len(infos_e) == len(infos_o) == kw["max_num_iterations"]
            T_o, X_o = o.get_internal()
            assert np.abs(T - T_o).max() < 1e-8 and np.abs(X - X_o).max() < 1e-8
        runs.append((infos_e, T.copy(), X.copy(), e.last_result.kernel_launches))
    (i0, T0, X0, l0), (i1, T1, X1, l1) = runs
    if scene == "c1":
        # the dense-GEMM Schur path of this scene flushes with FP64 reds: the two runs differ in the last bits
        assert l1 == l0 and len(i0) == len(i1) == kw["max_num_iterations"]
        assert [i.iteration_status for i in i0] == [i.iteration_status for i in i1]
        for a, b in zip(i0, i1):
            assert abs(a.cost - b.cost) <= 1e-8 * abs(a.cost)
            assert abs(a.damping_term - b.damping_term) <= 1e-12 * a.damping_term
        assert np.abs(T0 - T1).max() <= 1e-9 and np.abs(X0 - X1).max() <= 1e-9
    else:
        # the storing reduce drops k_pose_diag (and the clear kernel of a large band): the plan is banded
        assert l1 < l0
        assert [(i.iteration_status, i.cost, i.damping_term) for i in i0] == \
            [(i.iteration_status, i.cost, i.damping_term) for i in i1]
        assert np.array_equal(T0, T1) and np.array_equal(X0, X1)


def test_problem_without_observations_solves(engine_lib):
    """ba_set_observations accepts an empty set: cameras, poses and landmarks but nothing observed.  The cost is 0; the
    reduced system is zero, so the quadratic model predicts no decrease and the step is not taken (status 2, lambda
    kept: rho is not a number), and the solve ends there -- the cost change is 0, below any threshold."""
    from bundle_adjustment_solver_b200.solver import Summary
    sc = scenes.scene_trajectory(12, 200, 4, stereo=True, seed=2, n_fixed=2)
    sc.obs_cam = sc.obs_cam[:0]
    sc.obs_pose = sc.obs_pose[:0]
    sc.obs_point = sc.obs_point[:0]
    sc.obs_uv = sc.obs_uv[:0]
    e = load_engine(sc)
    assert e.sizes()["n_obs"] == 0
    assert e.cost() == 0.0
    summ = Summary()
    _, eo = options_pair(max_num_iterations=10, initial_lambda=100.0)
    e.solve(eo, summ)
    infos = summ.optimization_info_list
    assert summ.convergence_status and len(infos) == 1
    assert (infos[0].iteration_status, infos[0].cost, infos[0].cost_change, infos[0].damping_term) == (2, 0.0, 0.0, 100.0)
    assert summ.result.initial_cost == summ.result.final_cost == 0.0


def test_c3_scaled_blocks_and_iterations(oracle_mod, engine_lib):
    """Config C3 shape at 1/5 scale (40 poses x 10k landmarks would change the structure; keep 200
    poses, 10k landmarks): block parity + 3 LM iterations."""
    sc = scenes.scene_trajectory(200, 10_000, 10, stereo=True, seed=0, name="C3_fifth")
    o = load_oracle(sc)
    o.build_only(thres_huber=1.0, lam=100.0, b_accumulate=0, do_solve=True)
    e = load_engine(sc, identical_internal=o.get_internal())
    e.set_debug(True)
    oo, eo = options_pair()
    e.build_only(eo, 100.0, do_solve=True)
    compare_blocks(o, e, o.sizes())
    assert blockwise_rel_err(e.dump("x"), o.dump("x"), 6) < 1e-6
    oo, eo = options_pair(max_num_iterations=3)
    o = load_oracle(sc)
    infos_o, _ = o.solve(oo)
    e = load_engine(sc)
    from bundle_adjustment_solver_b200.solver import Summary
    summ = Summary()
    e.solve(eo, summ)
    for a, b in zip(summ.optimization_info_list, infos_o):
        assert abs(a.cost - b.cost) <= 1e-8 * abs(b.cost)
        assert a.iteration_status == b.iteration_status


def _solve_vs_numpy(sc, monkeypatch=None, chol_mode=None, band_mode=None, nd_depth=None, nd_chunk=None):
    """Build S, rhs on the device, solve with the engine's reduced solver, compare with numpy."""
    import os
    env = (("BA_B200_CHOL_MODE", chol_mode), ("BA_B200_BAND_MODE", band_mode), ("BA_B200_ND_DEPTH", nd_depth),
           ("BA_B200_ND_CHUNK", nd_chunk))
    for k, v in env:
        if v is None:
            os.environ.pop(k, None)
        else:
            os.environ[k] = str(v)
    try:
        e = load_engine(sc)
        e.set_debug(True)
        _, eo = options_pair()
        e.build_only(eo, 100.0, do_solve=True)
        n = 6 * e.sizes()["N"]
        Sm = e.dump("S").reshape(n, n)
        rhs = e.dump("rhs")
        x = e.dump("x")
    finally:
        for k, _ in env:
            os.environ.pop(k, None)
    xr = np.linalg.solve(Sm, rhs)
    return float(np.abs(x - xr).max() / np.abs(xr).max()), n


@pytest.mark.parametrize("n_poses,track,band_mode,depth,chunk", [
    (120, 10, 5, None, None), (120, 10, 6, None, None),      # C3-like band, level launches / persistent launch
    (100, 6, 6, None, None), (150, 13, 6, None, None),       # narrow and wide boundaries (TPW 8 / 24)
    (200, 4, 6, 3, 5), (200, 4, 5, 3, 5),                    # leaves cut into chains of chunks
    (400, 4, 6, None, None),                                 # C4-like: deep tree
    (61, 5, 6, 1, None),                                     # a single separator
])
def test_partitioned_banded_solve_matches_numpy(n_poses, track, band_mode, depth, chunk, engine_lib):
    """K5 partitioned (nested-dissection) banded solve, csrc/ba_cholesky_nd.cuh: x against numpy.linalg.solve of the
    device-built S, rhs (replaces ldlt().solve, full...cpp:890-908).  Tolerance 1e-9 relative (north_star)."""
    sc = scenes.scene_trajectory(n_poses, 40 * n_poses, track, stereo=True, seed=4, n_fixed=2)
    err, n = _solve_vs_numpy(sc, band_mode=band_mode, nd_depth=depth, nd_chunk=chunk)
    assert err < 1e-9, (err, n)


@pytest.mark.parametrize("n_poses,track,band_mode", [(100, 6, 4), (120, 10, 4), (150, 14, 4), (37, 10, 4)])
def test_banded_reduced_solve_matches_numpy(n_poses, track, band_mode, engine_lib):
    """K5 serial banded kernel (shared-memory DMMA window; the fallback of the partitioned solve and its yardstick) on
    sequential trajectories of three bandwidths; x against numpy.linalg.solve of the device-built S, rhs."""
    sc = scenes.scene_trajectory(n_poses, 40 * n_poses, track, stereo=True, seed=1, n_fixed=2)
    err, n = _solve_vs_numpy(sc, band_mode=band_mode)
    assert err < 1e-9, (err, n)


@pytest.mark.parametrize("chol_mode", [0, 1])
def test_multikernel_and_cluster_reduced_solve_match_numpy(chol_mode, engine_lib):
    sc = scenes.scene_trajectory(120, 4800, 10, stereo=True, seed=2, n_fixed=2)
    err, n = _solve_vs_numpy(sc, chol_mode=chol_mode)
    assert err < 1e-9, (err, n)


SOLVE_KERNELS = ("k_nd_persistent", "k_nd_forward_level", "k_chol_banded_smem", "k_chol_cluster", "k_chol_diag")


def test_reported_solve_is_the_launched_solve(monkeypatch, engine_lib):
    """Every solver runs the reduced solve its own switches select, whatever the other solvers of the process use, and
    ba_debug_solve_info (bench.py's roofline and byte accounting) names that solve: for BA_B200_BAND_MODE 6 / 5 / 4
    and BA_B200_CHOL_MODE unset / 0 / 1 on one banded trajectory, the reported name starts with the one solve kernel
    the build launches.  A switch changed after a solver exists does not change that solver's solve."""
    sc = scenes.scene_trajectory(160, 4800, 6, stereo=True, seed=4, n_fixed=2)
    _, eo = options_pair()
    by_band_mode = {6: "k_nd_persistent", 5: "k_nd_forward_level", 4: "k_chol_banded_smem"}
    for chol_mode in (None, 0, 1):
        for band_mode in (6, 5, 4):
            monkeypatch.setenv("BA_B200_BAND_MODE", str(band_mode))
            if chol_mode is None:
                monkeypatch.delenv("BA_B200_CHOL_MODE", raising=False)
            else:
                monkeypatch.setenv("BA_B200_CHOL_MODE", str(chol_mode))
            e = load_engine(sc)
            launched = launched_kernels(lambda: e.build_only(eo, 100.0, do_solve=True), SOLVE_KERNELS)
            name = solve_info(e)[0]
            want = {None: by_band_mode[band_mode], 0: "k_chol_diag", 1: "k_chol_cluster"}[chol_mode]
            assert launched == {want} and name.startswith(want), (band_mode, chol_mode, launched, name)
    monkeypatch.delenv("BA_B200_CHOL_MODE", raising=False)
    monkeypatch.setenv("BA_B200_BAND_MODE", "6")
    e = load_engine(sc)
    monkeypatch.setenv("BA_B200_BAND_MODE", "4")
    launched = launched_kernels(lambda: e.build_only(eo, 100.0, do_solve=True), SOLVE_KERNELS)
    assert launched == {"k_nd_persistent"} and solve_info(e)[0].startswith("k_nd_persistent"), launched


def test_dense_reduced_system_dmma_two_level(engine_lib):
    """Loop closures make S dense: n = 2388 > 2048 takes the two-level blocked Cholesky with DMMA TRSM/SYRK
    tiles and the multi-CTA backward sweep."""
    sc = scenes.scene_trajectory(400, 40_000, 5, stereo=False, seed=3, heavy_tail=True, loop_fraction=0.05)
    err, n = _solve_vs_numpy(sc)
    assert n > 2048
    assert err < 1e-8, (err, n)


def test_tile_build_with_fixed_poses_points_and_wide_tracks(oracle_mod, engine_lib):
    """Fused tile build next to the by-point path: fixed poses inside the tracks (C-only incidences), fixed
    landmarks (A-only observations), heavy-tailed tracks (some exceed the 16-pose window) and loop closures."""
    sc = scenes.scene_trajectory(120, 6000, 6, stereo=True, seed=5, n_fixed=3, heavy_tail=True, loop_fraction=0.03)
    sc.fixed_poses = np.array([0, 1, 2, 40, 41, 77])
    sc.fixed_points = np.arange(0, 6000, 97)
    for accum in (0, 1):
        o = load_oracle(sc)
        o.build_only(thres_huber=1.0, lam=100.0, b_accumulate=accum, do_solve=True)
        e = load_engine(sc, identical_internal=o.get_internal())
        e.set_debug(True)
        oo, eo = options_pair(b_accumulate=accum)
        e.build_only(eo, 100.0, do_solve=True)
        assert e.sizes() == o.sizes()
        compare_blocks(o, e, o.sizes())
        assert blockwise_rel_err(e.dump("y"), o.dump("y"), 3) < 1e-6


def test_c3_full_size_normal_equations_and_convergence(engine_lib):
    """BASELINE config C3 at full size (200 poses / 50k landmarks / 1.0 M observations), where the oracle is too slow to
    be the checker: size-independent properties of one linearisation + solve -- the reduced system is symmetric and
    solved, every block row of the damped normal equations [A B; B^T C][x; y] = [a; b] holds for the dumped blocks, C^-1
    inverts C -- and the LM loop converges to a lower cost."""
    sc = scenes.scene_c3(seed=100, pose_noise_seed=7)
    e = load_engine(sc)
    e.set_debug(True)
    _, eo = options_pair()
    e.build_only(eo, 100.0, do_solve=True)
    sz = e.sizes()
    N, M, P = sz["N"], sz["M"], sz["P"]
    assert sz["n_obs"] > 900_000 and M == 50_000 and N >= 190
    n = 6 * N
    Sm = e.dump("S").reshape(n, n)
    rhs, x = e.dump("rhs"), e.dump("x").reshape(N, 6)
    assert np.abs(Sm - Sm.T).max() <= 1e-12 * np.abs(Sm).max()
    assert np.linalg.norm(Sm @ x.reshape(-1) - rhs) <= 1e-9 * np.linalg.norm(Sm, 2) * np.linalg.norm(x)
    A, a = e.dump("A").reshape(N, 6, 6), e.dump("a").reshape(N, 6)
    Cd, b = e.dump("C").reshape(M, 3, 3), e.dump("b").reshape(M, 3)
    Ci = e.dump("Cinv").reshape(M, 3, 3)
    B = e.dump("B").reshape(P, 6, 3)
    y = e.dump("y").reshape(-1, 3)[:M]
    pj, pi = e.pairs()                                   # original ids; free poses / points numbered in id order
    free_pose = np.setdiff1d(np.arange(sz["N_total"]), np.asarray(sc.fixed_poses))
    j_of = np.full(sz["N_total"], -1)
    j_of[free_pose] = np.arange(N)
    pjo = j_of[pj]
    assert pjo.min() >= 0 and M == sz["M_total"]
    # C^-1 C = I
    assert np.abs(np.einsum("mij,mjk->mik", Ci, Cd) - np.eye(3)).max() < 1e-9
    # landmark rows: C_i y_i + sum_j B_ji^T x_j = b_i
    r_pt = np.einsum("mij,mj->mi", Cd, y) - b
    np.add.at(r_pt, pi, np.einsum("pkc,pk->pc", B, x[pjo]))
    assert np.abs(r_pt).max() <= 1e-9 * max(np.abs(b).max(), 1e-30)
    # pose rows: A_j x_j + sum_i B_ji y_i = a_j
    r_ps = np.einsum("jkl,jl->jk", A, x) - a
    np.add.at(r_ps, pjo, np.einsum("pkc,pc->pk", B, y[pi]))
    assert np.abs(r_ps).max() <= 1e-8 * np.abs(a).max()
    # the LM loop from the same start: converges, cost goes down, every recorded iteration is consistent
    from bundle_adjustment_solver_b200.solver import Summary
    e2 = load_engine(sc)
    summ = Summary()
    _, eo = options_pair(max_num_iterations=300, threshold_cost_change=1e-6, threshold_step_size=1e-6)
    c0 = e2.cost()
    e2.solve(eo, summ)
    infos = summ.optimization_info_list
    assert summ.convergence_status and 5 < len(infos) < 300
    assert infos[-1].cost < 0.05 * c0
    assert all(i.iteration_status in (0, 1, 2) and 1e-10 <= i.damping_term <= 100.0 for i in infos)


def test_c3_full_size_solve_matches_oracle(oracle_mod, engine_lib):
    """BASELINE config C3 at full size against the oracle run to convergence (about 40 s of CPU): same verdict,
    iteration count within 1, final cost within 1e-6, the first iterations on the same trajectory, poses and points
    within 1e-6 user units (BASELINE.json north_star: the parity bar, at the size the metric is quoted on)."""
    from bundle_adjustment_solver_b200.solver import Summary
    sc = scenes.scene_c3(seed=100, pose_noise_seed=7)
    kw = dict(max_num_iterations=300, threshold_cost_change=1e-6, threshold_step_size=1e-6)
    oo, eo = options_pair(**kw)
    o = load_oracle(sc)
    infos_o, conv_o = o.solve(oo)
    e = load_engine(sc)
    summ = Summary()
    e.solve(eo, summ)
    infos_e = summ.optimization_info_list
    assert conv_o and summ.convergence_status == conv_o
    assert abs(len(infos_e) - len(infos_o)) <= 1, (len(infos_e), len(infos_o))
    fo, fe = infos_o[-1].cost, infos_e[-1].cost
    assert abs(fe - fo) <= 1e-6 * abs(fo), (fe, fo)
    for k in range(10):
        assert abs(infos_e[k].cost - infos_o[k].cost) <= 1e-9 * abs(infos_o[k].cost), k
        assert infos_e[k].iteration_status == infos_o[k].iteration_status
        assert abs(infos_e[k].damping_term - infos_o[k].damping_term) <= 1e-12 * infos_o[k].damping_term
    assert np.abs(e.get_poses() - o.get_poses()).max() < 1e-6
    assert np.abs(e.get_points() - o.get_points()).max() < 1e-6
    assert np.array_equal(e.get_poses()[np.asarray(sc.fixed_poses)], sc.poses_init[np.asarray(sc.fixed_poses)])


def _S_blockwise_rel_err_chunked(Se, So, N, rows=120):
    """blockwise_rel_err of two (6N)^2 reduced systems without the block-view copies (C4: 1.15 GB each)."""
    n = 6 * N
    Se = np.asarray(Se).reshape(n, n)
    So = np.asarray(So).reshape(n, n)
    ref, err = [], []
    for j0 in range(0, N, rows):
        j1 = min(N, j0 + rows)
        a = So[6 * j0:6 * j1].reshape(j1 - j0, 6, N, 6)
        d = Se[6 * j0:6 * j1].reshape(j1 - j0, 6, N, 6) - a
        ref.append(np.sqrt(np.einsum("aibj,aibj->ab", a, a)))
        err.append(np.sqrt(np.einsum("aibj,aibj->ab", d, d)))
    ref, err = np.concatenate(ref), np.concatenate(err)
    return float((err / (np.maximum(ref, 1e-13 * ref.max()) + 1e-300)).max())


@pytest.mark.parametrize("workload", ["c4", "c5"])
def test_c4_c5_full_size_blocks_match_oracle(workload, oracle_mod, engine_lib):
    """BASELINE configs C4 / C5 at full size: one linearisation + Schur complement (the dense LDLT of the oracle is
    what does not scale, the build is seconds) -- every Hessian / Schur block within 1e-9 of the oracle."""
    sc = scenes.scene_c4(seed=100) if workload == "c4" else scenes.scene_c5(seed=100)
    o = load_oracle(sc)
    o.build_only(thres_huber=1.0, lam=100.0, b_accumulate=0, do_solve=False)
    e = load_engine(sc, identical_internal=o.get_internal())
    e.set_debug(True)
    _, eo = options_pair()
    e.build_only(eo, 100.0, do_solve=False)
    sz = o.sizes()
    assert e.sizes() == sz and sz["n_obs"] > 4_500_000
    assert all(np.array_equal(x, y) for x, y in zip(e.pairs(), o.pairs()))
    compare_blocks(o, e, sz, check_S=False)
    assert blockwise_rel_err(e.dump("rhs"), o.dump("rhs"), 6) <= BLOCK_TOL
    assert _S_blockwise_rel_err_chunked(e.dump("S"), o.dump("S"), sz["N"]) <= BLOCK_TOL


@pytest.mark.parametrize("workload,n_win", [("c4", 250), ("c5", 160)])
def test_c4_c5_pose_window_iterations_match_oracle(workload, n_win, oracle_mod, engine_lib):
    """A window of consecutive poses of the C4 / C5 scene (same tracks, same band) small enough for the oracle's dense
    LDLT: three LM iterations, every row of the iteration table and the parameters."""
    from bundle_adjustment_solver_b200.solver import Summary
    full = scenes.scene_c4(seed=100) if workload == "c4" else scenes.scene_c5(seed=100)
    sc = scenes.restrict_poses(full, 0, n_win)
    assert len(sc.fixed_poses) >= 1 and sc.n_obs > 300_000
    oo, eo = options_pair(max_num_iterations=3, threshold_cost_change=0.0, threshold_step_size=0.0)
    o = load_oracle(sc)
    infos_o, _ = o.solve(oo)
    o_fresh = load_oracle(sc); o_fresh.sizes()
    e = load_engine(sc, identical_internal=o_fresh.get_internal())
    summ = Summary()
    e.solve(eo, summ)
    infos_e = summ.optimization_info_list
    assert len(infos_e) == len(infos_o) == 3
    for a, b in zip(infos_e, infos_o):
        assert abs(a.cost - b.cost) <= 1e-9 * abs(b.cost)
        assert a.iteration_status == b.iteration_status
        assert abs(a.damping_term - b.damping_term) <= 1e-12 * b.damping_term
    T_e, X_e = e.get_internal()
    T_o, X_o = o.get_internal()
    assert np.abs(T_e - T_o).max() < 1e-8 and np.abs(X_e - X_o).max() < 1e-8


def test_update_parameters_with_one_set_keeps_the_other(engine_lib):
    """ba_update_parameters(T, NULL) / (NULL, X) after a solve: the set that is not supplied keeps its ACCEPTED values
    (they may live in parameter buffer 1), it must not fall back to whatever buffer 0 holds."""
    from bundle_adjustment_solver_b200.solver import Summary
    from bundle_adjustment_solver_b200.capi import ptr
    sc = scenes.scene_trajectory(30, 800, 6, stereo=True, seed=4, n_fixed=2)
    for iters in (3, 4):          # an odd and an even number of accepted steps: `cur` ends on either buffer
        e = load_engine(sc)
        _, eo = options_pair(max_num_iterations=iters, threshold_cost_change=0.0, threshold_step_size=0.0)
        e.solve(eo, Summary())
        T, X = e.get_internal()
        c_ref = e.cost()
        L = e.L
        assert L.ba_update_parameters(e.h, ptr(np.ascontiguousarray(T)), None) == 0
        T1, X1 = e.get_internal()
        assert np.array_equal(T1, T) and np.array_equal(X1, X)
        assert abs(e.cost() - c_ref) <= 1e-13 * c_ref
        assert L.ba_update_parameters(e.h, None, ptr(np.ascontiguousarray(X))) == 0
        T2, X2 = e.get_internal()
        assert np.array_equal(T2, T) and np.array_equal(X2, X)
        assert abs(e.cost() - c_ref) <= 1e-13 * c_ref


def test_tile_build_is_bit_reproducible(engine_lib):
    """north_star (2): no global atomics in the common path.  The fused tile build flushes every CTA's Schur products
    into a private staging window and k_tile_reduce adds the windows into S in CTA order, so two runs of the same
    problem give bit-identical S, rhs, x and LM trajectories (landmarks outside every window still go through the
    by-point path with its FP64 reds: none in this scene)."""
    from bundle_adjustment_solver_b200.solver import Summary
    sc = scenes.scene_trajectory(120, 20_000, 8, stereo=True, seed=31, n_fixed=2)
    _, eo = options_pair()
    runs = []
    for _ in range(3):
        e = load_engine(sc)
        e.set_debug(True)
        e.build_only(eo, 100.0, do_solve=True)
        runs.append((e.dump("S").copy(), e.dump("rhs").copy(), e.dump("x").copy()))
    for S1, r1, x1 in runs[1:]:
        assert np.array_equal(S1, runs[0][0]) and np.array_equal(r1, runs[0][1]) and np.array_equal(x1, runs[0][2])
    costs = []
    for _ in range(2):
        e = load_engine(sc)
        summ = Summary()
        _, eo2 = options_pair(max_num_iterations=12, threshold_cost_change=0.0, threshold_step_size=0.0)
        e.solve(eo2, summ)
        costs.append([i.cost for i in summ.optimization_info_list])
    assert costs[0] == costs[1]


def test_band_only_clearing_of_the_reduced_system_is_equivalent(monkeypatch, engine_lib):
    """Large banded systems (C4: 1.15 GB dense) clear only the band of S per iteration; forced on a small banded
    problem the LM trajectory must be the one of the full clear (same kernels, same inputs)."""
    from bundle_adjustment_solver_b200 import capi
    from bundle_adjustment_solver_b200 import solver as S
    sc = scenes.scene_trajectory(150, 6000, 8, stereo=True, seed=12, n_fixed=2)
    outs = []
    for mb in ("0", "100000"):
        monkeypatch.setenv("BA_B200_BAND_CLEAR_MIN_MB", mb)
        e = S.load_scene(S.FullBundleAdjustmentSolver(device=0), sc)
        summ = S.Summary()
        e.solve(capi.default_options(max_num_iterations=25, threshold_cost_change=1e-9, threshold_step_size=1e-9), summ)
        assert solve_info(e)[1][6] == (1.0 if mb == "0" else 0.0)     # band-only clearing reported as set
        outs.append({"COSTS": np.array([i.cost for i in summ.optimization_info_list]),
                     "POSES": np.array([float(np.abs(e.get_poses()).sum())])})
    assert len(outs[0]["COSTS"]) == len(outs[1]["COSTS"]) == 25
    np.testing.assert_allclose(outs[0]["COSTS"], outs[1]["COSTS"], rtol=1e-10)
    np.testing.assert_allclose(outs[0]["POSES"], outs[1]["POSES"], rtol=1e-10)


@pytest.mark.parametrize("workload", ["c4", "c5"])
def test_c4_c5_full_size_properties(workload, engine_lib):
    """BASELINE configs C4 (2000 poses / 1 M landmarks / 8.0 M observations, banded) and C5 (1778 / 1 M / 5.0 M, mono,
    dense reduced system) at full size, where the oracle cannot be the checker: the cost is additive over a split
    of the landmarks (two engines holding one half each), and the first LM iterations behave -- valid statuses,
    lambda inside its bounds, every accepted step lowers the cost, parameters stay finite."""
    from bundle_adjustment_solver_b200 import sharding
    from bundle_adjustment_solver_b200.solver import Summary
    sc = scenes.scene_c4(seed=100) if workload == "c4" else scenes.scene_c5(seed=100)
    assert sc.n_obs > 4_500_000
    e = load_engine(sc)
    c_full = e.cost()
    halves = [load_engine(sharding.shard_scene(sc, r, 2)).cost() for r in range(2)]
    assert abs(c_full - sum(halves)) <= 1e-11 * c_full
    summ = Summary()
    _, eo = options_pair(max_num_iterations=4, threshold_cost_change=0.0, threshold_step_size=0.0)
    e.solve(eo, summ)
    infos = summ.optimization_info_list
    assert len(infos) == 4 and not summ.convergence_status      # the last allowed iteration never reports convergence
    prev = c_full
    for i in infos:
        assert i.iteration_status in (0, 1, 2) and 1e-10 <= i.damping_term <= 100.0
        if i.iteration_status != 2:
            assert i.cost < prev
            prev = i.cost
    assert infos[-1].cost < 0.9 * c_full
    assert np.isfinite(e.get_poses()).all() and np.isfinite(e.get_points()).all()


def test_bal_file_round_trip_solves_on_the_device(tmp_path, oracle_mod, engine_lib):
    """bal.py end to end: a mono trajectory scene written in the 'Bundle Adjustment in the Large' layout, read back and
    solved on the device follows the oracle's LM trajectory on the same file."""
    from bundle_adjustment_solver_b200 import bal
    from bundle_adjustment_solver_b200.solver import Summary
    sc = scenes.scene_trajectory(40, 1500, 6, stereo=False, seed=13, n_fixed=2)
    sc.cam_intr[0, 2:] = 0.0                               # the format has no principal point
    T_cw = scenes.inv_T(sc.poses_true)
    Xc = np.einsum("nij,nj->ni", T_cw[sc.obs_pose, :3, :3], sc.points_true[sc.obs_point]) + T_cw[sc.obs_pose, :3, 3]
    f0 = sc.cam_intr[0, 0]
    sc.obs_uv = np.stack([f0 * Xc[:, 0] / Xc[:, 2], f0 * Xc[:, 1] / Xc[:, 2]], axis=1)
    path = tmp_path / "problem.txt"
    bal.save_bal(sc, path)
    back = bal.load_bal(path, n_fixed=2)
    oo, eo = options_pair(max_num_iterations=8, threshold_cost_change=0.0, threshold_step_size=0.0)
    o = load_oracle(back)
    infos_o, _ = o.solve(oo)
    e = load_engine(back)
    summ = Summary()
    e.solve(eo, summ)
    infos_e = summ.optimization_info_list
    assert len(infos_e) == len(infos_o) == 8
    for a, b in zip(infos_e, infos_o):
        assert abs(a.cost - b.cost) <= 1e-8 * abs(b.cost) and a.iteration_status == b.iteration_status
    assert infos_e[-1].cost < 0.2 * infos_e[0].cost
