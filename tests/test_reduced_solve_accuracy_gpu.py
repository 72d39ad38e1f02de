"""Accuracy of every reduced solve on undamped systems, against a solution refined beyond double precision.

The LM loop spends most of its iterations at small damping (lambda is divided on every accepted step, down to 1e-10),
where S is far from diagonal: kappa_2(S) reaches 1e9 on mono trajectories.  There numpy.linalg.solve is itself off by
up to 1e-9, so "x against numpy" cannot judge a solve, and every reduced solve multiplies by explicit inverses of the
factor's diagonal blocks, whose error grows with kappa(L_kk) <= sqrt(kappa_2(S)) (Du Croz & Higham 1992).  So the
reference here is refined_solve (a Cholesky solve plus iterative refinement with an accurately summed residual), and
the engine's x must meet

    backward error  eta(x) = ||r - S x||_inf / (||S||_inf ||x||_inf + ||r||_inf) <= u (4 n + 64 sqrt(kappa_2(S)))
    forward error   ||x - x*||_inf / ||x*||_inf <= 2 sqrt(n) kappa_2(S) (the bound above)

with u = 2^-53: 4 n for the growth of Cholesky, 64 sqrt(kappa) for what the explicit inverses may add.  A wrong tile,
a missed update or FP32 anywhere in the chain puts eta orders of magnitude above it.  Every case asserts the path it
was built for (kernel name, half-bandwidth, cluster size), so a change of the plan heuristics fails here instead of
dropping the coverage; each prints n, lambda, kappa_2 and the engine's and LAPACK's backward and forward errors.

The shapes are the edges of each path: the partition shapes of the partitioned solve, the widest window of the serial
banded kernel (bw + 8 <= kBandMaxW), the dense path's rhs row alone in its tile row (n % 64 == 0), the last one-level
size (n = 2046) and the first two-level sizes, the cluster sizes 1 / 4 / 8 / 16 and the max_rows <= 12 limit of the
cluster path, and a single free pose."""
import copy
import fractions
import math

import numpy as np
import pytest
import scipy.linalg

from bundle_adjustment_solver_b200 import scenes
from bundle_adjustment_solver_b200.solver import Summary
from helpers import load_engine, load_oracle, options_pair, solve_info

U = 2.0 ** -53
LAMBDAS = [100.0, 1e-10]


# ------------------------------------------------------------------------------------------------ reference
def _need_extended():
    if np.finfo(np.longdouble).eps > 1e-18:
        pytest.skip("np.longdouble is not an extended type on this platform")


def _split(a):
    """Veltkamp split: a = hi + lo exactly, both with at most 26 significant bits."""
    c = 134217729.0 * a
    hi = c - (c - a)
    return hi, a - hi


def _residual(S, r, xh, xl, rows=256):
    """r - S (xh + xl) rounded once to double: every product S_ij xh_j as an exact sum of two doubles (Dekker), each
    row summed exactly by math.fsum; S xl enters as a plain sum (its terms are 2^-53 of the others)."""
    Sh, Sl = _split(S)
    xhh, xhl = _split(xh)
    lo_part = S @ xl
    out = np.empty_like(r)
    for i0 in range(0, len(r), rows):
        sl = slice(i0, i0 + rows)
        P = S[sl] * xh
        E = ((Sh[sl] * xhh - P) + Sh[sl] * xhl + Sl[sl] * xhh) + Sl[sl] * xhl
        T = np.concatenate([r[sl, None], -lo_part[sl, None], -P, -E], axis=1)
        out[sl] = [math.fsum(row) for row in T.tolist()]
    return out


def refined_solve(S, r, max_rounds=5, tol=1e-18):
    """x* of S x = r for SPD S with kappa_2(S) 2^-53 < 1: a Cholesky solve in double, then corrections from the
    residual until one is below tol of x (asserted within max_rounds); x is kept as a pair of doubles and returned as
    np.longdouble.  The residual is summed exactly: one rounded in long double stalls near kappa_2 2^-64 (1e-13 of x
    at kappa_2 = 1e9) instead of converging."""
    _need_extended()
    cf = scipy.linalg.cho_factor(S, lower=True)
    xh = scipy.linalg.cho_solve(cf, r)
    xl = np.zeros_like(xh)
    for _ in range(max_rounds):
        d = scipy.linalg.cho_solve(cf, _residual(S, r, xh, xl))
        s = xh + d                                    # (xh, xl) += d, renormalised
        bb = s - xh
        e = (xh - (s - bb)) + (d - bb) + xl
        xh = s + e
        xl = e - (xh - s)
        if np.abs(d).max() <= tol * np.abs(xh).max():
            return xh.astype(np.longdouble) + xl.astype(np.longdouble)
    raise AssertionError(f"iterative refinement did not converge in {max_rounds} rounds")


def backward_error(S, r, x):
    SL, rL, xL = (np.asarray(a).astype(np.longdouble) for a in (S, r, x))
    res = np.abs(rL - SL @ xL).max()
    return float(res / (np.abs(SL).sum(axis=1).max() * np.abs(xL).max() + np.abs(rL).max()))


def forward_error(x, x_ref):
    xL = np.asarray(x).astype(np.longdouble)
    return float(np.abs(xL - x_ref).max() / np.abs(x_ref).max())


def kappa2(S):
    ev = np.linalg.eigvalsh(S)
    assert ev[0] > 0.0, ev[0]
    return float(ev[-1] / ev[0])


def eta_bound(n, kappa):
    return U * (4 * n + 64 * math.sqrt(kappa))


def _fraction_solve(A, b):
    """Exact solution of A x = b (integers) by Gaussian elimination over the rationals."""
    n = len(b)
    M = [[fractions.Fraction(int(v)) for v in row] + [fractions.Fraction(int(bi))] for row, bi in zip(A, b)]
    for k in range(n):
        p = next(i for i in range(k, n) if M[i][k] != 0)
        M[k], M[p] = M[p], M[k]
        for i in range(k + 1, n):
            f = M[i][k] / M[k][k]
            if f:
                for j in range(k, n + 1):
                    M[i][j] -= f * M[k][j]
    x = [fractions.Fraction(0)] * n
    for i in reversed(range(n)):
        x[i] = (M[i][n] - sum(M[i][j] * x[j] for j in range(i + 1, n))) / M[i][i]
    return x


def test_refined_solve_is_exact_on_an_integer_system():
    """24 x 24 diagonally dominant integer SPD matrix, integer right-hand side: refined_solve against the exact
    rational solution, to 1e-17 relative."""
    _need_extended()
    rng = np.random.default_rng(7)
    B = rng.integers(-9, 10, (24, 24))
    A = B + B.T
    A += np.diag(np.abs(A).sum(axis=1) + rng.integers(1, 20, 24))
    b = rng.integers(-1000, 1001, 24)
    x_exact = _fraction_solve(A, b)
    x = refined_solve(A.astype(np.float64), b.astype(np.float64))
    scale = max(abs(v) for v in x_exact)
    # the comparison is exact: each long double converts to a Fraction without rounding
    err = max(abs(fractions.Fraction(float(xi)) + fractions.Fraction(float(xi - np.longdouble(float(xi)))) - xe)
              for xi, xe in zip(x, x_exact)) / scale
    assert err <= 1e-17, float(err)


def test_refined_solve_converges_on_an_undamped_reduced_system(oracle_mod):
    """S of a mono trajectory at lambda = 1e-10 (kappa_2 ~ 1e9), built by the CPU oracle: the refinement converges,
    and LAPACK's Cholesky solve lands within 10 u kappa_2 of it (the first-order bound of a backward-stable solve)."""
    sc = scenes.scene_trajectory(120, 4800, 6, stereo=False, seed=2)
    o = load_oracle(sc)
    o.build_only(lam=1e-10, do_solve=True)
    n = 6 * o.sizes()["N"]
    S, r = o.dump("S").reshape(n, n), o.dump("rhs")
    x_ref = refined_solve(S, r)
    kappa = kappa2(S)
    assert kappa > 1e8                                            # the scene does what it is for
    x_lapack = scipy.linalg.cho_solve(scipy.linalg.cho_factor(S, lower=True), r)
    fwd = forward_error(x_lapack, x_ref)
    eta = backward_error(S, r, x_lapack)
    print(f"n {n} kappa2 {kappa:.2e} eta_lapack {eta:.2e} fwd_lapack {fwd:.2e}")
    assert fwd <= 10 * U * kappa, (fwd, kappa)
    assert eta <= U * 4 * n, eta
    assert backward_error(S, r, x_ref) < 1e-18


# ------------------------------------------------------------------------------------------------ scenes
def _add_landmarks(sc, tracks, rng, depth=(6.0, 10.0)):
    """Append one landmark per track (array of pose ids), seen by every camera of the rig from every pose of the
    track (rows appended after the existing ones), with exact pixels."""
    out = copy.deepcopy(sc)
    M, n_cam = len(sc.points_true), len(sc.cam_ids)
    Xt = np.array([[0.2 * np.mean(t) + rng.uniform(-0.5, 0.5), rng.uniform(-1.0, 1.0), rng.uniform(*depth)]
                   for t in tracks])
    out.points_true = np.vstack([sc.points_true, Xt])
    out.points_init = np.vstack([sc.points_init, Xt + rng.uniform(-0.5, 0.5, Xt.shape)])
    pose = np.concatenate([np.repeat(np.asarray(t), n_cam) for t in tracks])
    slot = np.concatenate([np.tile(np.arange(n_cam), len(t)) for t in tracks])
    point = np.concatenate([np.full(n_cam * len(t), M + k) for k, t in enumerate(tracks)])
    T_cw = scenes.inv_T(out.poses_true[pose])
    Xb = np.einsum("nij,nj->ni", T_cw[:, :3, :3], out.points_true[point]) + T_cw[:, :3, 3]
    Xc = np.einsum("nij,nj->ni", out.cam_T[slot, :3, :3], Xb) + out.cam_T[slot, :3, 3]
    f = out.cam_intr[slot]
    uv = np.stack([f[:, 0] * Xc[:, 0] / Xc[:, 2] + f[:, 2], f[:, 1] * Xc[:, 1] / Xc[:, 2] + f[:, 3]], axis=1)
    out.obs_cam = np.concatenate([sc.obs_cam, slot]).astype(np.int32)
    out.obs_pose = np.concatenate([sc.obs_pose, pose]).astype(np.int32)
    out.obs_point = np.concatenate([sc.obs_point, point]).astype(np.int32)
    out.obs_uv = np.vstack([sc.obs_uv, uv])
    return out


def _band(sc):
    """Half-bandwidth of S, 6 max_j (j - first co-visible free pose of j) + 5, from the scene's observations."""
    Nt = len(sc.poses_init)
    free = np.ones(Nt, dtype=bool)
    free[np.asarray(sc.fixed_poses, dtype=int)] = False
    j_of = np.cumsum(free) - 1
    fp, pt = sc.obs_pose[free[sc.obs_pose]], sc.obs_point[free[sc.obs_pose]]
    first = np.full(len(sc.points_true), Nt)
    np.minimum.at(first, pt, j_of[fp])
    return 6 * int((j_of[fp] - first[pt]).max()) + 5


def _partitioned_scene(n_poses, track):
    return scenes.scene_trajectory(n_poses, 40 * n_poses, track, stereo=False, seed=4, n_fixed=2)


def _window_scene(span):
    """Mono trajectory of short tracks (4 +- 2 poses) and eight landmarks on 1 + span consecutive free poses."""
    sc = scenes.scene_trajectory(122, 3000, 4, stereo=False, seed=12, n_fixed=2)
    return _add_landmarks(sc, [np.arange(40, 41 + span)] * 8, np.random.default_rng(13))


def _covisible_scene(n_free):
    """Mono trajectory with one more landmark seen by every pose: every free pose is co-visible with the first, so
    the envelope of S is full and max_rows = T - 1 (T tile rows over n + 1 rows)."""
    sc = scenes.scene_trajectory(n_free + 2, max(60, 40 * n_free), 6, stereo=False, seed=20 + n_free, n_fixed=2)
    return _add_landmarks(sc, [np.arange(n_free + 2)], np.random.default_rng(n_free), depth=(30.0, 30.0))


def _loop_scene(n_free):
    return scenes.scene_trajectory(n_free + 2, 30 * (n_free + 2), 5, stereo=False, seed=3, n_fixed=2, heavy_tail=True,
                                   loop_fraction=0.05)


# ------------------------------------------------------------------------------------------------ device cases
def _set_switches(monkeypatch, band_mode=None, chol_mode=None, nd_depth=None, nd_chunk=None):
    for k, v in (("BA_B200_BAND_MODE", band_mode), ("BA_B200_CHOL_MODE", chol_mode), ("BA_B200_ND_DEPTH", nd_depth),
                 ("BA_B200_ND_CHUNK", nd_chunk)):
        if v is None:
            monkeypatch.delenv(k, raising=False)
        else:
            monkeypatch.setenv(k, str(v))


def _engine_solve(sc, lam):
    """S, rhs and x of one build + reduced solve on the device (debug on), and the solve the plan selected."""
    e = load_engine(sc)
    e.set_debug(True)
    e.build_only(options_pair()[1], lam, do_solve=True)
    n = 6 * e.sizes()["N"]
    name, vals = solve_info(e)
    return e.dump("S").reshape(n, n), e.dump("rhs"), e.dump("x"), name, vals


def _check_accuracy(S, r, x, lam, label):
    """The acceptance rule of the module docstring; prints the per-case row."""
    n = len(r)
    assert np.isfinite(x).all()
    kappa = kappa2(S)
    x_ref = refined_solve(S, r)
    x_lapack = scipy.linalg.cho_solve(scipy.linalg.cho_factor(S, lower=True), r)
    eta, eta_l = backward_error(S, r, x), backward_error(S, r, x_lapack)
    fwd, fwd_l = forward_error(x, x_ref), forward_error(x_lapack, x_ref)
    bound = eta_bound(n, kappa)
    print(f"\nACCURACY {label} n {n} lam {lam:.0e} kappa2 {kappa:.2e} eta_engine {eta:.2e} eta_lapack {eta_l:.2e} "
          f"fwd_engine {fwd:.2e} fwd_lapack {fwd_l:.2e} eta_bound {bound:.2e}")
    assert eta <= bound, (eta, bound)
    assert fwd <= 2 * math.sqrt(n) * kappa * bound, (fwd, kappa, bound)


def _run_case(monkeypatch, sc, lam, label, want, switches=None, n=None, bw=None, cluster=None):
    _set_switches(monkeypatch, **(switches or {}))
    S, r, x, name, vals = _engine_solve(sc, lam)
    if n is not None:
        assert len(r) == n, (len(r), n)
    assert name.startswith(want), name
    if bw is not None:
        assert int(vals[3]) == bw, (vals[3], bw)
    if cluster is not None:
        assert int(vals[4]) == cluster, (vals[4], cluster)
    _check_accuracy(S, r, x, lam, label)
    return name, vals


ND_NAME = {6: "k_nd_persistent", 5: "k_nd_forward_level"}


@pytest.mark.gpu
@pytest.mark.parametrize("n_poses,track,band_mode,depth,chunk", [
    (200, 10, 5, None, None), (200, 10, 6, None, None),      # C3 band, level launches / persistent launch
    (100, 6, 6, None, None), (300, 13, 6, None, None),       # narrow and wide boundaries
    (200, 4, 6, 3, 6), (200, 4, 5, 3, 6),                    # leaves cut into chains of chunks (39 fronts)
    (400, 4, 6, None, None),                                 # deep tree
    (61, 5, 6, 1, None),                                     # a single separator
])
def test_partitioned_solve_accuracy_undamped(n_poses, track, band_mode, depth, chunk, monkeypatch, engine_lib):
    """The partitioned banded solve (ba_cholesky_nd.cuh), mono and undamped, on the partition shapes of
    test_full_ba_gpu.test_partitioned_banded_solve_matches_numpy -- with more poses where that test's scene is too
    short for a partition to halve the serial kernel's chain (the planner then takes k_chol_banded_smem: N = 118 with
    track 10, N = 148 with track 13), and chunks of 6 poses where chunks of 5 overflow the leaves of 21 poses."""
    sc = _partitioned_scene(n_poses, track)
    _run_case(monkeypatch, sc, 1e-10, f"partitioned{band_mode} N={n_poses - 2} track={track}", ND_NAME[band_mode],
              dict(band_mode=band_mode, nd_depth=depth, nd_chunk=chunk), bw=_band(sc))


@pytest.mark.gpu
@pytest.mark.parametrize("lam", LAMBDAS)
@pytest.mark.parametrize("span", [16, 17])
def test_serial_banded_solve_accuracy_at_the_window_limit(span, lam, monkeypatch, engine_lib):
    """k_chol_banded_smem takes S while bw + 8 <= kBandMaxW = 112: tracks over 17 free poses (span 16, bw = 101) are
    the widest it accepts; with span 17 (bw = 107) the plan must take another solve."""
    sc = _window_scene(span)
    bw = _band(sc)
    assert bw == 6 * span + 5
    if span == 16:
        _run_case(monkeypatch, sc, lam, "banded bw=101", "k_chol_banded_smem", dict(band_mode=4), bw=bw)
    else:
        _set_switches(monkeypatch, band_mode=4)
        S, r, x, name, vals = _engine_solve(sc, lam)
        assert not name.startswith("k_chol_banded_smem") and int(vals[3]) == bw, name
        _check_accuracy(S, r, x, lam, f"{name.split()[0]} bw=107")


DENSE = "k_chol_diag+k_chol_trsm"


@pytest.mark.gpu
@pytest.mark.parametrize("lam", LAMBDAS)
@pytest.mark.parametrize("n_free,kind", [
    (128, "forced"),    # n = 768: the rhs row alone in tile row 12 (first_tile[n / 64] = 0)
    (130, "forced"),    # n = 780
    (341, "natural"),   # n = 2046: last one-level size, 62-wide last diagonal block sharing its tile with the rhs row
    (342, "natural"),   # n = 2052: first two-level size, last group of one 4-wide panel
    (352, "natural"),   # n = 2112: two-level, n % 64 == 0, multi-CTA backward sweep
    (352, "forced"),
])
def test_dense_solve_accuracy_at_tile_edges(n_free, kind, lam, monkeypatch, engine_lib):
    """The multi-kernel blocked Cholesky (k_chol_diag, k_chol_trsm(_tail), k_syrk_update, backward sweeps): natural on
    loop-closure scenes, forced with BA_B200_CHOL_MODE=0 on banded ones, where TRSM, SYRK and the backward sweep skip
    the tiles left of the envelope."""
    if kind == "natural":
        sc, switches = _loop_scene(n_free), None
    else:
        sc, switches = _partitioned_scene(n_free + 2, 6), dict(chol_mode=0)
    _run_case(monkeypatch, sc, lam, f"dense-{kind} N={n_free}", DENSE, switches, n=6 * n_free)


@pytest.mark.gpu
@pytest.mark.parametrize("lam", LAMBDAS)
@pytest.mark.parametrize("n_free,cluster", [
    (1, 1), (10, 1), (11, 1),     # one tile row / two tile rows
    (22, 4), (32, 8), (43, 16),   # max_rows 2 / 3 / 4
    (138, 16),                    # 13 tile rows: max_rows 12, the largest the cluster path takes
    (139, None),                  # 14 tile rows: the dense path
])
def test_cluster_solve_accuracy_by_size(n_free, cluster, lam, monkeypatch, engine_lib):
    """k_chol_cluster on fully co-visible scenes (natural path): the cluster sizes 1 / 4 / 8 / 16 and the max_rows <= 12
    limit, beyond which the plan takes the multi-kernel path."""
    sc = _covisible_scene(n_free)
    if cluster is None:
        _run_case(monkeypatch, sc, lam, f"cluster-limit N={n_free}", DENSE, n=6 * n_free)
    else:
        _run_case(monkeypatch, sc, lam, f"cluster{cluster} N={n_free}", "k_chol_cluster", n=6 * n_free, cluster=cluster)


@pytest.mark.gpu
@pytest.mark.parametrize("lam", LAMBDAS)
@pytest.mark.parametrize("scene", ["test_ba", "banded"])
def test_cluster_solve_accuracy_natural_and_forced(scene, lam, monkeypatch, engine_lib):
    """The test_ba.cpp scene (natural cluster path, dense co-visibility) and a banded mono trajectory forced onto the
    cluster path with BA_B200_CHOL_MODE=1 (envelope skipping inside the cluster kernel)."""
    if scene == "test_ba":
        _run_case(monkeypatch, scenes.scene_test_ba(seed=0), lam, "cluster test_ba", "k_chol_cluster")
    else:
        sc = scenes.scene_trajectory(120, 4800, 6, stereo=False, seed=2)
        _run_case(monkeypatch, sc, lam, "cluster-forced N=118", "k_chol_cluster", dict(chol_mode=1))


# ------------------------------------------------------------------------------------------------ LM rows
@pytest.mark.gpu
@pytest.mark.parametrize("chol_mode", [None, 0, 1])
@pytest.mark.parametrize("scene", ["trajectory", "test_ba"])
def test_lm_iteration_rows_at_low_damping_match_oracle(scene, chol_mode, monkeypatch, oracle_mod, engine_lib):
    """Six LM iterations from lambda = 1e-4 through each reduced solve: every field of the iteration table against the
    oracle (pivoted LDLT), from bit-identical internal parameters -- status, lambda within 1e-12, cost within 1e-9,
    abs_step (the mean step norm that the convergence test reads) within 1e-8, cost_change within 1e-9 of the cost,
    average_reprojection_error within 1e-9."""
    if scene == "trajectory":
        sc = scenes.scene_trajectory(200, 8000, 10, stereo=True, seed=2, n_fixed=2)
        want = {None: "k_nd_persistent", 0: DENSE, 1: "k_chol_cluster"}[chol_mode]
    else:
        sc = scenes.scene_test_ba(seed=0)
        want = {None: "k_chol_cluster", 0: DENSE, 1: "k_chol_cluster"}[chol_mode]
    kw = dict(max_num_iterations=6, initial_lambda=1e-4, threshold_cost_change=0.0, threshold_step_size=0.0)
    oo, eo = options_pair(**kw)
    o = load_oracle(sc)
    infos_o, _ = o.solve(oo)
    o0 = load_oracle(sc)
    o0.sizes()
    _set_switches(monkeypatch, chol_mode=chol_mode)
    e = load_engine(sc, identical_internal=o0.get_internal())
    summ = Summary()
    e.solve(eo, summ)
    assert solve_info(e)[0].startswith(want)
    infos_e = summ.optimization_info_list
    assert len(infos_e) == len(infos_o) == 6
    for k, (a, b) in enumerate(zip(infos_e, infos_o)):
        print(f"\nROW {scene} chol_mode={chol_mode} k={k} status {a.iteration_status}/{b.iteration_status} "
              f"cost {abs(a.cost - b.cost) / abs(b.cost):.1e} abs_step {abs(a.abs_step - b.abs_step) / b.abs_step:.1e} "
              f"cost_change {abs(a.cost_change - b.cost_change) / abs(b.cost):.1e} "
              f"are {abs(a.average_reprojection_error - b.average_reprojection_error) / b.average_reprojection_error:.1e}")
    for k, (a, b) in enumerate(zip(infos_e, infos_o)):
        assert a.iteration_status == b.iteration_status, k
        assert abs(a.damping_term - b.damping_term) <= 1e-12 * b.damping_term, k
        assert abs(a.cost - b.cost) <= 1e-9 * abs(b.cost), (k, a.cost, b.cost)
        assert abs(a.abs_step - b.abs_step) <= 1e-8 * abs(b.abs_step), (k, a.abs_step, b.abs_step)
        assert abs(a.cost_change - b.cost_change) <= 1e-9 * abs(b.cost), (k, a.cost_change, b.cost_change)
        assert abs(a.average_reprojection_error - b.average_reprojection_error) <= \
            1e-9 * b.average_reprojection_error, (k, a.average_reprojection_error, b.average_reprojection_error)
