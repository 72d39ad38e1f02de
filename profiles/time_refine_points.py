"""Time of ba_refine_points (structure-only bundle adjustment, k_refine_points) on the bench.py scenes at their true
poses, from points_init, beside what a caller does without it: a solver with every pose fixed and ba_solve.

  python profiles/time_refine_points.py [--workloads c3,c4] [--reps 10] [--out results/refine_points.json]

Refinement: the host clock around the C-ABI call (it ends in a stream synchronise; it includes the copy of the
refined points to the host), the kernel alone from the CUDA activities of torch.profiler in a separate pass, and the
histogram of iterations per landmark; once with the default thresholds (1e-5) and once with 1e-10.  Every repetition
starts from the same points: ba_update_parameters re-uploads them between calls.  All-fixed baseline (in a child process): the host ba_finalize of a solver whose poses are all
fixed, its ba_solve time and iteration count, and its final total cost against the sum of the per-landmark final
costs of the refinement.  The card name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (make_scene())

os.dup2(bench._REAL_STDOUT.fileno(), 1)   # bench.py sends fd 1 to stderr for its one-JSON-line protocol; undo that here
from bundle_adjustment_solver_b200 import solver as S  # noqa: E402
from bundle_adjustment_solver_b200.capi import default_options, ptr  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi unavailable"


def scene(w):
    sc = bench.make_scene(w, 0, 1.0)
    sc.poses_init = sc.poses_true.copy()
    return sc


def refine(w, reps, thr):
    import torch
    from torch.profiler import ProfilerActivity, profile
    sc = scene(w)
    e = S.load_scene(S.FullBundleAdjustmentSolver(device=0), sc)
    e._upload()
    T0, X0 = (np.ascontiguousarray(a) for a in e.get_internal())
    M = len(X0)
    opt = default_options(threshold_step_size=thr, threshold_cost_change=thr)
    st = np.zeros(M, dtype=np.uint8)
    it = np.zeros(M, dtype=np.int32)
    costs = np.zeros((M, 2))
    counts = np.zeros(5, dtype=np.int64)

    def call():
        rc = e.L.ba_refine_points(e.h, opt, None, ptr(costs), ptr(it), ptr(st), ptr(counts))
        if rc != 0:
            raise RuntimeError(e.L.ba_last_error(e.h).decode())

    t0 = time.perf_counter()
    call()   # the first call after a finalize uploads the landmark -> observation ranges
    first_ms = 1e3 * (time.perf_counter() - t0)
    ts = []
    for _ in range(reps):
        e.update_parameters_internal(T0, X0)
        t0 = time.perf_counter()
        call()
        ts.append(1e3 * (time.perf_counter() - t0))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            e.update_parameters_internal(T0, X0)
            call()
        torch.cuda.synchronize()
    ks = [ev.device_time_total for ev in prof.events()
          if ev.device_type == torch.autograd.DeviceType.CUDA and "k_refine_points" in ev.name]
    if not ks:
        raise RuntimeError("no k_refine_points activity in the profile")
    hist = np.bincount(it[st <= 1], minlength=51)
    return dict(M=M, n_obs=sc.n_obs, first_call_ms=first_ms, call_ms_median=float(np.median(ts)),
                call_ms_min=float(np.min(ts)), kernel_us_median=float(np.median(ks)), kernel_samples=len(ks),
                counts=counts.tolist(), iterations_hist={int(k): int(v) for k, v in enumerate(hist) if v},
                cost_initial=float(costs[:, 0].sum()), cost_final=float(costs[:, 1].sum()))


def all_fixed(w):
    """What a caller does today: every pose fixed, one host finalize, ba_solve."""
    sc = scene(w)
    sc.fixed_poses = np.arange(len(sc.poses_init))
    e = S.load_scene(S.FullBundleAdjustmentSolver(device=0), sc)
    t0 = time.perf_counter()
    e._upload()
    fin_ms = 1e3 * (time.perf_counter() - t0)
    summ = S.Summary()
    t0 = time.perf_counter()
    e.solve(default_options(), summ)
    solve_ms = 1e3 * (time.perf_counter() - t0)
    return dict(finalize_ms=fin_ms, solve_ms=solve_ms, iterations=len(summ.optimization_info_list),
                converged=bool(summ.convergence_status), final_cost=e.cost())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c4")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--all-fixed-child", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.all_fixed_child:
        print("ALLFIXED " + json.dumps(all_fixed(a.all_fixed_child)))
        return
    import torch
    torch.cuda.init()
    torch.zeros(1, device="cuda")
    info = dict(card=card(), rows={})
    print(f"card: {info['card']}")
    for w in a.workloads.split(","):
        r = refine(w, a.reps, 1e-5)
        # the thresholds are absolute and each landmark has a small cost of its own: the default 1e-5 stops a landmark
        # long before the all-fixed solve stops the whole problem; a second row with tight thresholds
        r["tight_1e-10"] = t = refine(w, a.reps, 1e-10)
        print(f"{w}: M {r['M']}  obs {r['n_obs']}  call {r['call_ms_median']:.2f} ms (min {r['call_ms_min']:.2f}, first "
              f"{r['first_call_ms']:.2f})  kernel {r['kernel_us_median']:.0f} us  counts {r['counts']}")
        print(f"    iterations per refined landmark: {r['iterations_hist']}")
        print(f"    thresholds 1e-10: call {t['call_ms_median']:.2f} ms  kernel {t['kernel_us_median']:.0f} us  "
              f"counts {t['counts']}  sum of final costs {t['cost_final']:.6e}  iterations {t['iterations_hist']}")
        q = subprocess.run([sys.executable, __file__, "--all-fixed-child", w], capture_output=True, text=True)
        line = [ln for ln in q.stdout.splitlines() if ln.startswith("ALLFIXED ")]
        if q.returncode == 0 and line:
            b = json.loads(line[0][9:])
            b["final_cost_over_refined_sum"] = b["final_cost"] / r["cost_final"]
            print(f"    every pose fixed + ba_solve: finalize {b['finalize_ms']:.1f} ms  solve {b['solve_ms']:.1f} ms  "
                  f"{b['iterations']} iterations (converged {b['converged']})  final cost {b['final_cost']:.6e} vs "
                  f"sum of per-landmark final costs {r['cost_final']:.6e} (thresholds 1e-10: {t['cost_final']:.6e})")
        else:
            b = dict(error=(q.stderr or q.stdout)[-1500:], returncode=q.returncode)
            print(f"    every pose fixed + ba_solve: failed (rc {q.returncode}): {b['error'][-400:]}")
        r["all_fixed"] = b
        info["rows"][w] = r
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
