"""bench.py's command line: --steps sets the number of timed LM iterations, and --dump-outputs writes what the last
timed step computed (the same result as a direct solve of that many iterations)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH = os.path.join(ROOT, "bench.py")


def test_steps_below_one_is_rejected():
    r = subprocess.run([sys.executable, BENCH, "--steps", "0"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr, r.stderr[-2000:]


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(tmp_path, engine_lib):
    from bundle_adjustment_solver_b200 import capi, scenes
    from bundle_adjustment_solver_b200 import solver as S
    steps = 3
    r = subprocess.run([sys.executable, BENCH, "--gpus", "1", "--steps", str(steps), "--warmup", "3", "--workload", "c1",
                        "--quick", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["quick"]
    out = {n: np.load(tmp_path / f"{n}.npy") for n in ("poses", "points", "cost")}
    assert all(a.dtype == np.float64 for a in out.values())

    sc = scenes.scene_test_ba(seed=0)               # bench.py's c1 workload on rank 0
    e = S.load_scene(S.FullBundleAdjustmentSolver(device=0), sc)
    summ = S.Summary()
    e.solve(capi.default_options(max_num_iterations=steps, threshold_cost_change=0.0, threshold_step_size=0.0,
                                 check_every=steps), summ)
    assert len(summ.optimization_info_list) == steps
    T, X = e.get_internal()
    assert out["poses"].shape == T.shape and out["points"].shape == X.shape
    np.testing.assert_allclose(out["cost"], [e.last_result.initial_cost, e.last_result.final_cost], rtol=1e-8)
    np.testing.assert_allclose(out["poses"], T, rtol=0, atol=1e-7)
    np.testing.assert_allclose(out["points"], X, rtol=0, atol=1e-7)
