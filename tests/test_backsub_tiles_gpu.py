"""Back-substitution of the tile landmarks (k_backsub_tiles): the fused tile build keeps its B blocks on chip, the
back-substitution forms them again from the landmarks' observations, and every pair's B is written to global memory
only when the blocks are kept for ba_debug_dump.

The block-parity tests compare the dumped B, which the debug-only k_pair_blocks fill writes, with the oracle; the B the
tile producers feed into the Schur GEMM is checked through S and the B formed by k_backsub_tiles through y (below).
All three come from the same device helpers, linearize_obs and add_B."""
import numpy as np
import pytest

from bundle_adjustment_solver_b200 import scenes
from bundle_adjustment_solver_b200.solver import Summary
from helpers import launched_kernels, load_engine, options_pair

pytestmark = pytest.mark.gpu


def _tile_only_scene():
    # every landmark fits a 16-pose window: tile path only, no FP64 reds anywhere in the iteration
    return scenes.scene_trajectory(120, 20_000, 8, stereo=True, seed=31, n_fixed=2)


def _mixed_scene():
    # tile landmarks next to by-point landmarks (tracks wider than the window, loop closures), fixed poses inside the
    # tracks and fixed landmarks
    sc = scenes.scene_trajectory(120, 6000, 6, stereo=True, seed=5, n_fixed=3, heavy_tail=True, loop_fraction=0.03)
    sc.fixed_poses = np.array([0, 1, 2, 40, 41, 77])
    sc.fixed_points = np.arange(0, 6000, 97)
    return sc


def _backsub_kernels(run):
    """Names of the back-substitution kernels that run() launches."""
    return launched_kernels(run, ("k_backsub_tiles", "k_backsub_pairs"))


def _check_paths(sc, scene):
    """The scenes cover what the tests rely on: the tile-only scene has no by-point landmark (so no FP64 reds), the
    mixed scene has both kinds."""
    e = load_engine(sc)
    _, eo = options_pair()
    launched = _backsub_kernels(lambda: e.build_only(eo, 100.0, do_solve=True))
    expected = {"k_backsub_tiles"} if scene == "tile_only" else {"k_backsub_tiles", "k_backsub_pairs"}
    assert launched == expected, launched


def _solve(sc, debug):
    e = load_engine(sc)
    e.set_debug(debug)
    summ = Summary()
    _, eo = options_pair(max_num_iterations=12, threshold_cost_change=0.0, threshold_step_size=0.0)
    e.solve(eo, summ)
    T, X = e.get_internal()
    return [i.cost for i in summ.optimization_info_list], T.copy(), X.copy()


@pytest.mark.parametrize("scene", ["tile_only", "mixed"])
def test_debug_block_fill_does_not_change_the_solve(scene, engine_lib):
    """With debug on, the build also stores every pair's B (k_pair_blocks over all pairs) for ba_debug_dump; nothing
    the iteration computes may change.  The tile-only scene has no FP64 reds, so the two solves are bit-identical.
    The by-point landmarks of the mixed scene go through the dense-GEMM Schur path, which adds its split-K partials
    into S with FP64 reds in a run-dependent order; there the two solves agree to rounding."""
    sc = _tile_only_scene() if scene == "tile_only" else _mixed_scene()
    _check_paths(sc, scene)
    c0, T0, X0 = _solve(sc, False)
    c1, T1, X1 = _solve(sc, True)
    assert len(c0) == len(c1) == 12
    if scene == "tile_only":
        assert c0 == c1
        assert np.array_equal(T0, T1) and np.array_equal(X0, X1)
    else:
        np.testing.assert_allclose(c1, c0, rtol=1e-10)
        assert np.abs(T1 - T0).max() <= 1e-9 and np.abs(X1 - X0).max() <= 1e-9


@pytest.mark.parametrize("accum", [0, 1])
def test_landmark_steps_match_dumped_blocks(accum, engine_lib):
    """y_i = C_i^-1 (b_i - sum_j B_ji^T x_j) for every free landmark, recomputed in NumPy from the dumped damped C, b,
    B and x.  The tile landmarks' B is formed again in the back-substitution, the dumped one by k_pair_blocks: the same
    helper at the same parameters, so the only differences are summation orders.  Error per landmark relative to the
    size of the terms, ||C_i^-1|| (||b_i|| + ||sum_j B_ji^T x_j||)."""
    sc = _mixed_scene()
    e = load_engine(sc)
    e.set_debug(True)
    _, eo = options_pair(b_accumulate=accum)
    launched = _backsub_kernels(lambda: e.build_only(eo, 100.0, do_solve=True))
    assert launched == {"k_backsub_tiles", "k_backsub_pairs"}, launched      # both kinds of landmark are covered
    sz = e.sizes()
    N, M, P = sz["N"], sz["M"], sz["P"]
    Cd = e.dump("C").reshape(M, 3, 3)
    b = e.dump("b").reshape(M, 3)
    B = e.dump("B").reshape(P, 6, 3)
    x = e.dump("x").reshape(N, 6)
    y = e.dump("y").reshape(-1, 3)[:M]
    pj, pi = e.pairs()                                   # original ids; free poses / points numbered in id order
    j_of = np.full(sz["N_total"], -1)
    j_of[np.setdiff1d(np.arange(sz["N_total"]), np.asarray(sc.fixed_poses))] = np.arange(N)
    i_of = np.full(sz["M_total"], -1)
    i_of[np.setdiff1d(np.arange(sz["M_total"]), np.asarray(sc.fixed_points))] = np.arange(M)
    assert j_of[pj].min() >= 0 and i_of[pi].min() >= 0 and P > 0
    Btx = np.zeros((M, 3))
    np.add.at(Btx, i_of[pi], np.einsum("pkc,pk->pc", B, x[j_of[pj]]))
    y_ref = np.linalg.solve(Cd, (b - Btx)[:, :, None])[:, :, 0]
    Ci_norm = np.linalg.norm(np.linalg.inv(Cd), ord=2, axis=(1, 2))
    scale = Ci_norm * (np.linalg.norm(b, axis=1) + np.linalg.norm(Btx, axis=1))
    has_pairs = np.zeros(M, dtype=bool)
    has_pairs[i_of[pi]] = True
    assert has_pairs.sum() > 0.9 * M
    err = np.linalg.norm(y - y_ref, axis=1) / scale
    assert err[has_pairs].max() <= 1e-12, float(err[has_pairs].max())
