"""Observation structures the trajectory and test_ba.cpp scenes never produce, against the CPU oracle.

Those scenes have a rig with camera slots 0 and 1, at most one observation per (pose, landmark, camera), the left list
of a frame inserted right before its right list, an observation on every free pose, and tracks well inside the tile
limits.  The scenes here are mutations of them that reach the other branches of the kernels:

  A  a 4-camera rig (ids neither contiguous nor sorted): incidences of 1..4 observations, camera slots 2 and 3;
  B  repeated observations (same camera, pixels moved by about 1 px) and a shuffled insertion order: the last-writer
     rule of the reference mode (B = the block of the last INSERTED observation of the pair);
  C  camera ids outside [0, 4096) and rows with an unknown camera, pose or landmark: the slow path of
     ba_set_observations_scaled and its drop rules;
  D  the tile classification limits: free-pose span 16 / 17, 20 / 21 incidences, runs of fewer than 6 landmarks;
  E  the dense-GEMM threshold of the by-point Schur product, 6 N + 1 <= 769: N = 128 / 129;
  F  free poses without observations (zero 6 x 6 pivots in every reduced solve) and a landmark without observations.

Every case asserts the path it was built for (kernel names from torch.profiler, or the reduced solve's name), so a
change of the classification heuristics fails here instead of silently dropping the coverage."""
import copy

import numpy as np
import pytest

from bundle_adjustment_solver_b200 import scenes
from bundle_adjustment_solver_b200.solver import Summary
from helpers import blockwise_rel_err, compare_blocks, launched_kernels, load_engine, load_oracle, options_pair, solve_info

pytestmark = pytest.mark.gpu

TILE, BT_TILE, BT_PAIRS = "k_build_tiles", "k_backsub_tiles", "k_backsub_pairs"
DENSE, PAIRS_LIST = "k_schur_dense_gemm", "k_schur_pairs_list"
TILE_ONLY = {TILE, BT_TILE}


# ------------------------------------------------------------------------------------------------ scene mutations
def _project(sc, pose, point, slot, rng=None, sigma=0.0):
    """Pixels of landmarks `point` seen from poses `pose` through rig slots `slot` (true parameters, the projection of
    scenes.scene_trajectory), with Gaussian noise of sigma px."""
    T_cw = scenes.inv_T(sc.poses_true[pose])
    Xb = np.einsum("nij,nj->ni", T_cw[:, :3, :3], sc.points_true[point]) + T_cw[:, :3, 3]
    Xc = np.einsum("nij,nj->ni", sc.cam_T[slot, :3, :3], Xb) + sc.cam_T[slot, :3, 3]
    f = sc.cam_intr[slot]
    uv = np.stack([f[:, 0] * Xc[:, 0] / Xc[:, 2] + f[:, 2], f[:, 1] * Xc[:, 1] / Xc[:, 2] + f[:, 3]], axis=1)
    return uv + rng.normal(0.0, sigma, uv.shape) if sigma > 0 else uv


def _with_obs(sc, cam, pose, point, uv):
    out = copy.deepcopy(sc)
    out.obs_cam = np.asarray(cam, dtype=np.int32)
    out.obs_pose = np.asarray(pose, dtype=np.int32)
    out.obs_point = np.asarray(point, dtype=np.int32)
    out.obs_uv = np.asarray(uv, dtype=np.float64).reshape(-1, 2)
    return out


RIG_IDS = [7, 2, 31, 0]


def _rig4(mono, seed):
    """Case A: every (pose, landmark) incidence of a mono scene seen by a random non-empty subset of a 4-camera rig with
    its own extrinsic and intrinsics per camera; per frame, camera list after camera list (slot order)."""
    rng = np.random.default_rng(seed)
    sc = copy.deepcopy(mono)
    sc.cam_ids = list(RIG_IDS)
    sc.cam_intr = np.array([[525.0, 525.0, 320.0, 240.0], [480.0, 470.0, 300.0, 250.0],
                            [610.0, 600.0, 330.0, 235.0], [550.0, 545.0, 310.0, 245.0]])
    sc.cam_T = np.stack([np.eye(4),
                         scenes.make_T(scenes.rot_y(0.04) @ scenes.rot_x(-0.02), [-0.12, 0.0, 0.0]),
                         scenes.make_T(scenes.rot_y(-0.05), [0.10, -0.05, 0.02]),
                         scenes.make_T(scenes.rot_x(0.03) @ scenes.rot_z(0.02), [0.0, 0.08, -0.03])])
    subset = rng.integers(1, 16, mono.n_obs)                      # non-empty subsets of the 4 cameras
    seen = (subset[:, None] >> np.arange(4)) & 1
    k, slot = np.nonzero(seen)
    pose, point = mono.obs_pose[k], mono.obs_point[k]
    o = np.lexsort((point, slot, pose))
    k, slot, pose, point = k[o], slot[o], pose[o], point[o]
    uv = _project(sc, pose, point, slot, rng, 0.5)
    return _with_obs(sc, np.asarray(RIG_IDS)[slot], pose, point, uv)


def _repeat_and_shuffle(sc, seed, frac=0.1):
    """Case B: about frac of the observations repeated (same camera, pixels moved by up to 1 px, so the last writer and
    the sum of a pair differ), each repeat inserted at a random later position; then one fixed random permutation of the
    whole insertion order."""
    rng = np.random.default_rng(seed)
    n = sc.n_obs
    dup = np.sort(rng.choice(n, int(frac * n), replace=False))
    later = rng.integers(dup + 1, n + 1)                          # the repeat goes in front of row `later`
    key = np.concatenate([2 * np.arange(n), 2 * later - 1])
    src = np.concatenate([np.arange(n), dup])
    uv = np.concatenate([sc.obs_uv, sc.obs_uv[dup] + rng.uniform(-1.0, 1.0, (len(dup), 2))])
    o = np.argsort(key, kind="stable")
    o = o[rng.permutation(len(o))]
    return _with_obs(sc, sc.obs_cam[src[o]], sc.obs_pose[src[o]], sc.obs_point[src[o]], uv[o])


def _foreign_ids_and_bad_rows(sc, seed, frac=0.05):
    """Case C: the camera ids of a stereo scene become -5 and 4100 (outside the [0, 4096) table of the fast path), and
    rows with an unregistered camera, pose -1 / N_total or landmark -1 / M_total are mixed into the insertion order."""
    rng = np.random.default_rng(seed)
    ids = np.array([-5, 4100])
    out = copy.deepcopy(sc)
    out.cam_ids = list(ids)
    n, Nt, Mt = sc.n_obs, len(sc.poses_init), len(sc.points_init)
    cam, pose, point, uv = ids[sc.obs_cam], sc.obs_pose.copy(), sc.obs_point.copy(), sc.obs_uv.copy()
    nb = int(frac * n)
    src = rng.integers(0, n, nb)
    bcam, bpose, bpoint = cam[src].copy(), pose[src].copy(), point[src].copy()
    kind = np.arange(nb) % 6
    bcam[kind == 0] = rng.choice([0, 1, 4096, -1], (kind == 0).sum())
    bpose[kind == 1] = -1
    bpose[kind == 2] = Nt
    bpoint[kind == 3] = -1
    bpoint[kind == 4] = Mt
    bcam[kind == 5] = 4099
    bpose[kind == 5] = Nt + 7                                     # several defects in one row
    o = rng.permutation(n + nb)
    cat = lambda a, b: np.concatenate([a, b])[o]
    return _with_obs(out, cat(cam, bcam), cat(pose, bpose), cat(point, bpoint), cat(uv, sc.obs_uv[src])), n


def _drop_landmarks(sc, drop):
    """Remove landmarks (mask) and their observations; the others keep their order."""
    keep = ~drop
    remap = np.full(len(keep), -1)
    remap[keep] = np.arange(keep.sum())
    out = copy.deepcopy(sc)
    out.points_true, out.points_init = sc.points_true[keep], sc.points_init[keep]
    ko = keep[sc.obs_point]
    out = _with_obs(out, sc.obs_cam[ko], sc.obs_pose[ko], remap[sc.obs_point[ko]], sc.obs_uv[ko])
    return out


def _add_landmarks(sc, tracks, rng):
    """Append one stereo landmark per track (array of pose ids), in front of the track's middle, observed by both
    cameras of every pose of the track (rows appended after the existing ones)."""
    out = copy.deepcopy(sc)
    M = len(sc.points_true)
    Xt = np.array([[0.2 * np.mean(t) + rng.uniform(-0.5, 0.5), rng.uniform(-1.0, 1.0), rng.uniform(6.0, 10.0)]
                   for t in tracks])
    out.points_true = np.vstack([sc.points_true, Xt])
    out.points_init = np.vstack([sc.points_init, Xt + rng.uniform(-0.5, 0.5, Xt.shape)])
    pose = np.concatenate([np.repeat(np.asarray(t), 2) for t in tracks])
    slot = np.concatenate([np.tile([0, 1], len(t)) for t in tracks])
    point = np.concatenate([np.full(2 * len(t), M + k) for k, t in enumerate(tracks)])
    uv = _project(out, pose, point, slot, rng, 0.5)
    return _with_obs(out, np.concatenate([sc.obs_cam, slot]), np.concatenate([sc.obs_pose, pose]),
                     np.concatenate([sc.obs_point, point]), np.vstack([sc.obs_uv, uv]))


def _drop_pose_observations(sc, poses):
    keep = ~np.isin(sc.obs_pose, poses)
    return _with_obs(sc, sc.obs_cam[keep], sc.obs_pose[keep], sc.obs_point[keep], sc.obs_uv[keep])


def _add_unobserved_landmark(sc):
    out = copy.deepcopy(sc)
    X = np.array([[3.0, 0.5, 8.0]])
    out.points_true = np.vstack([sc.points_true, X])
    out.points_init = np.vstack([sc.points_init, X + 0.3])
    return out


# ------------------------------------------------------------------------------------------------ checks
def _launched(run):
    """Schur and back-substitution kernels that run() launches."""
    return launched_kernels(run, (TILE, BT_TILE, BT_PAIRS, DENSE, PAIRS_LIST))


def _landmark_step_error(sc, e):
    """max over landmarks with pairs of |y_i - C_i^-1 (b_i - sum_j B_ji^T x_j)| relative to the size of the terms,
    recomputed from the dumped blocks (as test_backsub_tiles_gpu.test_landmark_steps_match_dumped_blocks)."""
    sz = e.sizes()
    N, M, P = sz["N"], sz["M"], sz["P"]
    Cd = e.dump("C").reshape(M, 3, 3)
    b = e.dump("b").reshape(M, 3)
    B = e.dump("B").reshape(P, 6, 3)
    x = e.dump("x").reshape(N, 6)
    y = e.dump("y").reshape(-1, 3)[:M]
    pj, pi = e.pairs()
    j_of = np.full(sz["N_total"], -1)
    j_of[np.setdiff1d(np.arange(sz["N_total"]), np.asarray(sc.fixed_poses))] = np.arange(N)
    i_of = np.full(sz["M_total"], -1)
    i_of[np.setdiff1d(np.arange(sz["M_total"]), np.asarray(sc.fixed_points))] = np.arange(M)
    assert j_of[pj].min() >= 0 and i_of[pi].min() >= 0 and P > 0
    Btx = np.zeros((M, 3))
    np.add.at(Btx, i_of[pi], np.einsum("pkc,pk->pc", B, x[j_of[pj]]))
    has_pairs = np.zeros(M, dtype=bool)
    has_pairs[i_of[pi]] = True
    Cd, b, Btx, y = Cd[has_pairs], b[has_pairs], Btx[has_pairs], y[has_pairs]
    y_ref = np.linalg.solve(Cd, (b - Btx)[:, :, None])[:, :, 0]
    scale = np.linalg.norm(np.linalg.inv(Cd), ord=2, axis=(1, 2)) * (np.linalg.norm(b, axis=1) + np.linalg.norm(Btx, axis=1))
    return float((np.linalg.norm(y - y_ref, axis=1) / scale).max())


def _check_blocks(sc, accum, lam=100.0):
    """One linearisation + Schur complement + reduced solve + back-substitution against the oracle's, from bit-identical
    parameters.  Returns the kernels it launched and the engine."""
    o = load_oracle(sc)
    o.build_only(thres_huber=1.0, lam=lam, b_accumulate=accum, do_solve=True)
    e = load_engine(sc, identical_internal=o.get_internal())
    e.set_debug(True)
    _, eo = options_pair(b_accumulate=accum)
    launched = _launched(lambda: e.build_only(eo, lam, do_solve=True))
    sz = o.sizes()
    assert e.sizes() == sz
    assert all(np.array_equal(a, b) for a, b in zip(e.pairs(), o.pairs()))
    compare_blocks(o, e, sz)           # S checks the B of the Schur producers (tile operands, Bsoa of the pairs)
    # reduced solve and back-substitution (the conditioning of S enters; same bound as the block tests of
    # test_full_ba_gpu); y checks the B that k_backsub_tiles forms again
    assert blockwise_rel_err(e.dump("x"), o.dump("x"), 6) < 1e-6
    assert blockwise_rel_err(e.dump("y"), o.dump("y"), 3) < 1e-6
    err = _landmark_step_error(sc, e)
    assert err <= 1e-12, err
    return launched, e, o


def _check_lm(sc, accum, iters=8):
    """iters LM iterations from the oracle's internal parameters: statuses equal, lambda within 1e-12, costs within
    1e-9, final internal parameters within 1e-8.  Returns (start, engine result, oracle result)."""
    oo, eo = options_pair(max_num_iterations=iters, threshold_cost_change=0.0, threshold_step_size=0.0,
                          b_accumulate=accum)
    o = load_oracle(sc)
    infos_o, _ = o.solve(oo)
    o0 = load_oracle(sc)
    o0.sizes()
    start = tuple(a.copy() for a in o0.get_internal())
    e = load_engine(sc, identical_internal=start)
    summ = Summary()
    e.solve(eo, summ)
    infos_e = summ.optimization_info_list
    assert len(infos_e) == len(infos_o) == iters
    for k, (a, b) in enumerate(zip(infos_e, infos_o)):
        assert a.iteration_status == b.iteration_status, k
        assert abs(a.damping_term - b.damping_term) <= 1e-12 * b.damping_term, k
        assert abs(a.cost - b.cost) <= 1e-9 * abs(b.cost), (k, a.cost, b.cost)
    T_e, X_e = e.get_internal()
    T_o, X_o = o.get_internal()
    assert np.abs(T_e - T_o).max() < 1e-8 and np.abs(X_e - X_o).max() < 1e-8
    return start, (T_e, X_e), (T_o, X_o)


# ------------------------------------------------------------------------------------------------ A: 4-camera rig
def _scene_rig(kind):
    if kind == "banded":      # N = 148 > 128: tile path, banded plan (storing reduce)
        mono = scenes.scene_trajectory(150, 3000, 8, stereo=False, seed=41, n_fixed=2)
    else:                     # N = 98: heavy tails and loop closures, by-point landmarks, dense-GEMM Schur product
        mono = scenes.scene_trajectory(100, 2500, 6, stereo=False, seed=42, n_fixed=2, heavy_tail=True, loop_fraction=0.05)
    return _rig4(mono, seed=43)


@pytest.mark.parametrize("accum", [0, 1])
@pytest.mark.parametrize("kind", ["banded", "loops"])
def test_four_camera_rig_matches_oracle(kind, accum, oracle_mod, engine_lib):
    sc = _scene_rig(kind)
    per_inc = np.bincount(np.unique(np.stack([sc.obs_pose, sc.obs_point], 1), axis=0, return_counts=True)[1])
    assert per_inc[3] > 0 and per_inc[4] > 0                      # incidences of 3 and 4 observations
    launched, e, _ = _check_blocks(sc, accum)
    if kind == "banded":
        assert launched == TILE_ONLY, launched
        assert solve_info(e)[0].startswith("k_nd_persistent")    # banded plan: the storing reduce of the tile flush
    else:
        assert {DENSE, BT_PAIRS} <= launched and PAIRS_LIST not in launched, launched
    _check_lm(sc, accum)


# ------------------------------------------------------------------------------------------------ B: repeats, order
def _scene_repeats(kind):
    if kind == "tiles":       # stereo trajectory, every landmark a tile landmark
        base = scenes.scene_trajectory(120, 3000, 8, stereo=True, seed=51, n_fixed=2, pixel_sigma=0.5)
    else:                     # test_ba.cpp scene: dense co-visibility, by-point path
        base = scenes.scene_test_ba(seed=1, pixel_sigma=0.5)
    return _repeat_and_shuffle(base, seed=52)


@pytest.mark.parametrize("accum", [0, 1])
@pytest.mark.parametrize("kind", ["tiles", "by_point"])
def test_repeated_and_reordered_observations_match_oracle(kind, accum, oracle_mod, engine_lib):
    """Reference mode is the sharp check: a pair's B is the block of its last INSERTED observation, which is a repeat
    of the same camera, or the left camera's, as often as not."""
    sc = _scene_repeats(kind)
    key = np.stack([sc.obs_pose, sc.obs_point, sc.obs_cam], 1)
    assert len(np.unique(key, axis=0)) < len(key)                 # same camera twice on one pair
    launched, _, _ = _check_blocks(sc, accum)
    if kind == "tiles":
        assert launched == TILE_ONLY, launched
    else:
        assert {DENSE, BT_PAIRS} <= launched, launched
    _check_lm(sc, accum)


# ------------------------------------------------------------------------------------------------ C: ids, bad rows
@pytest.mark.parametrize("accum", [0, 1])
def test_camera_ids_outside_the_table_and_dropped_rows_match_oracle(accum, oracle_mod, engine_lib):
    base = scenes.scene_trajectory(120, 3000, 6, stereo=True, seed=61, n_fixed=3, pixel_sigma=0.5, heavy_tail=True,
                                   loop_fraction=0.03)
    sc, n_valid = _foreign_ids_and_bad_rows(base, seed=62)
    assert min(sc.cam_ids) < 0 and max(sc.cam_ids) >= 4096 and sc.n_obs > n_valid
    o = load_oracle(sc)
    e = load_engine(sc)
    assert e.num_total_observations == o.sizes()["n_obs"] == n_valid
    launched, _, _ = _check_blocks(sc, accum)
    assert {TILE, BT_TILE, DENSE, BT_PAIRS} <= launched, launched
    _check_lm(sc, accum)


# ------------------------------------------------------------------------------------------------ D: tile limits
# fixed poses inside the tracks of the incidence-limit landmarks: 100..119 holds 4 of them (16 free poses, 20
# incidences), 140..160 holds 5 (16 free poses, 21 incidences)
D_FIXED = np.array([0, 1, 102, 105, 108, 111, 142, 145, 148, 151, 154])


def _scene_tile_limits(variant):
    base = scenes.scene_trajectory(170, 2500, 5, stereo=True, seed=74, n_fixed=2, pixel_sigma=0.5)
    base.fixed_poses = D_FIXED
    rng = np.random.default_rng(72)
    if variant == "at_limits":      # span 16 (no fixed pose inside), 20 incidences with span 16: tile landmarks
        tracks = [np.arange(40, 56)] * 8 + [np.arange(100, 120)] * 8
    elif variant == "span_17":      # 17 free poses
        tracks = [np.arange(40, 57)] * 8
    elif variant == "incidences_21":
        tracks = [np.arange(140, 161)] * 8
    else:                           # "short_runs": a staircase of span-16 windows, 3 landmarks each, no other landmark
        # starts in it -- a run holds one step (the next one widens the window to 17): fewer than 6 landmarks
        first = np.full(len(base.points_true), len(base.poses_init))
        np.minimum.at(first, base.obs_point, base.obs_pose)
        base = _drop_landmarks(base, (first >= 60) & (first < 76))
        tracks = [np.arange(60 + s, 76 + s) for s in range(5) for _ in range(3)]
    return _add_landmarks(base, tracks, rng)


@pytest.mark.parametrize("variant", ["at_limits", "span_17", "incidences_21", "short_runs"])
def test_tile_classification_limits_match_oracle(variant, oracle_mod, engine_lib):
    """A landmark is a tile landmark when its free poses span at most kTileW = 16 and it has at most kTileMaxInc = 20
    incidences (fixed poses included), and its window run holds at least kMinPts = 6 landmarks.  The base scene has only
    short tracks, so the by-point kernels run exactly when one of the added landmarks misses a limit.  N = 159 > 128:
    the small-system rule that sends every landmark to the by-point path does not apply, and the by-point Schur product
    is the pair list.  LM in reference mode."""
    sc = _scene_tile_limits(variant)
    for accum in (0, 1):
        launched, _, _ = _check_blocks(sc, accum)
        if variant == "at_limits":
            assert launched == TILE_ONLY, launched
        else:
            assert launched == TILE_ONLY | {BT_PAIRS, PAIRS_LIST}, launched
    _check_lm(sc, 0, iters=6)


# ------------------------------------------------------------------------------------------------ E: dense threshold
@pytest.mark.parametrize("n_free", [128, 129])
def test_dense_gemm_threshold_matches_oracle(n_free, oracle_mod, engine_lib):
    """k_schur_dense_gemm takes the by-point landmarks while 6 N + 1 <= 769, k_schur_pairs_list beyond."""
    sc = scenes.scene_trajectory(n_free + 2, 3000, 6, stereo=False, seed=81, n_fixed=2, pixel_sigma=0.5,
                                 heavy_tail=True, loop_fraction=0.05)
    for accum in (0, 1):
        launched, e, _ = _check_blocks(sc, accum)
        assert e.sizes()["N"] == n_free
        assert (DENSE in launched) == (n_free == 128) and (PAIRS_LIST in launched) == (n_free == 129), launched
    _check_lm(sc, 0, iters=6)


# ------------------------------------------------------------------------------------------------ F: zero pivots
def _f_base():
    return _add_unobserved_landmark(scenes.scene_trajectory(160, 4800, 6, stereo=True, seed=4, n_fixed=2,
                                                            pixel_sigma=0.5))


def _f_poses():
    """Free poses (ids) to strip of their observations, taken from the partition plan the engine uses for this scene:
    the first free pose, one inside the own block of a leaf, one inside a separator, the last free pose."""
    from test_nd_plan_cpu import nd_plan
    sc = _f_base()
    e = load_engine(sc)
    _, vals = solve_info(e)
    N, bw = e.sizes()["N"], int(vals[3])
    meta, nodes = nd_plan(N, (bw - 5) // 6)
    assert meta["valid"] and meta["depth"] >= 1, meta
    mid = lambda nd: nd["own0"] // 6 + nd["k"] // 12
    leaf = next(nd for nd in nodes if nd["child1"] < 0 and nd["own0"] > 0 and nd["own0"] + nd["k"] < 6 * N)
    sep = next(nd for nd in nodes if nd["child1"] >= 0)
    free = np.setdiff1d(np.arange(len(sc.poses_init)), sc.fixed_poses)
    kinds = {"first": 0, "leaf": mid(leaf), "separator": mid(sep), "last": N - 1}
    return {k: int(free[j]) for k, j in kinds.items()}, (N, bw)


def _check_zero_pivot_solve(S, rhs, x, free_idx, tol):
    rows = (6 * np.asarray(free_idx)[:, None] + np.arange(6)).ravel()
    assert np.all(S[rows] == 0.0) and np.all(rhs[rows] == 0.0)   # the scene does what it is for
    assert np.isfinite(x).all()
    assert np.all(x[rows] == 0.0), x[rows]
    keep = np.setdiff1d(np.arange(len(rhs)), rows)
    xr = np.linalg.solve(S[np.ix_(keep, keep)], rhs[keep])
    err = float(np.abs(x[keep] - xr).max() / np.abs(xr).max())
    assert err < tol, err


@pytest.mark.parametrize("band_mode,chol_mode,solve_name", [
    (6, None, "k_nd_persistent"), (5, None, "k_nd_forward_level"), (4, None, "k_chol_banded_smem"),
    (None, 0, "k_chol_diag+k_chol_trsm"), (None, 1, "k_chol_cluster")])
def test_free_poses_without_observations_solve(band_mode, chol_mode, solve_name, monkeypatch, engine_lib):
    """An unobserved free pose has an exactly zero 6 x 6 block and rhs in S; every reduced solve emulates Eigen LDLT's
    D^+ = 0 there: x is exactly 0 for that pose and the rest solves the system without its rows and columns (1e-9
    relative against numpy).  The poses sit at the first and last free index, inside a leaf's own block and inside a
    separator of the partitioned solve.  The switches select the solve of the solver created after they are set."""
    poses, (N, bw) = _f_poses()
    for k, v in (("BA_B200_BAND_MODE", band_mode), ("BA_B200_CHOL_MODE", chol_mode)):
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, str(v))
    e = load_engine(_drop_pose_observations(_f_base(), list(poses.values())))
    e.set_debug(True)
    e.build_only(options_pair()[1], 100.0, do_solve=True)
    n = 6 * e.sizes()["N"]
    name, vals = solve_info(e)
    assert name.startswith(solve_name), name
    assert int(vals[3]) == bw                                     # same band, so the same partition as chosen from
    fixed = _f_base().fixed_poses
    free_idx = [int(np.sum(~np.isin(np.arange(p), fixed))) for p in poses.values()]
    _check_zero_pivot_solve(e.dump("S").reshape(n, n), e.dump("rhs"), e.dump("x"), free_idx, 1e-9)


def test_free_poses_without_observations_dense_two_level(engine_lib):
    """The loop-closure shape of test_full_ba_gpu.test_dense_reduced_system_dmma_two_level (n > 2048: the two-level
    blocked Cholesky) with three unobserved free poses.  1e-8: the bound that test states for this shape."""
    sc = scenes.scene_trajectory(400, 40_000, 5, stereo=False, seed=3, heavy_tail=True, loop_fraction=0.05)
    free = np.setdiff1d(np.arange(400), sc.fixed_poses)
    idx = [0, 200, len(free) - 1]
    sc = _drop_pose_observations(sc, free[idx])
    e = load_engine(sc)
    e.set_debug(True)
    e.build_only(options_pair()[1], 100.0, do_solve=True)
    n = 6 * e.sizes()["N"]
    assert n > 2048
    assert solve_info(e)[0].startswith("k_chol_diag+k_chol_trsm")
    _check_zero_pivot_solve(e.dump("S").reshape(n, n), e.dump("rhs"), e.dump("x"), idx, 1e-8)


@pytest.mark.parametrize("accum", [0, 1])
def test_unobserved_poses_and_landmark_match_oracle(accum, oracle_mod, engine_lib):
    """The same scene against the oracle (pivoted LDLT): blocks, x, y and 8 LM iterations.  The unobserved poses and the
    unobserved landmark come back bit-identical to their input; the landmark's step is exactly 0."""
    poses, _ = _f_poses()
    sc = _drop_pose_observations(_f_base(), list(poses.values()))
    launched, e, _ = _check_blocks(sc, accum)
    assert launched == TILE_ONLY, launched                        # windows with an uncovered slot in their middle
    M = e.sizes()["M"]
    assert np.all(e.dump("y").reshape(-1, 3)[M - 1] == 0.0)      # the last landmark is free and unobserved
    start, (T_e, X_e), (T_o, X_o) = _check_lm(sc, accum)
    p = list(poses.values())
    assert np.array_equal(T_e[p], start[0][p]) and np.array_equal(T_o[p], start[0][p])
    assert np.array_equal(X_e[-1], start[1][-1]) and np.array_equal(X_o[-1], start[1][-1])
