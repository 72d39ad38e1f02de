"""Time of ba_triangulate_points (k_triangulate_points) on the bench.py scenes at their true poses, every landmark
registered without a position (NaN).

  python profiles/time_triangulate_points.py [--workloads c3,c4] [--reps 20] [--out results/triangulate_points.json]

The solver runs on torch's current stream, so CUDA events recorded there bracket the device work of one call; the host
clock around the call is reported too (it ends in a stream synchronise and includes the copy of the statuses and of the
points to the host).  The kernel alone comes from the CUDA activities of torch.profiler, in a separate pass.  The first
call after a finalize also uploads the landmark -> observation ranges and is reported apart.  The triangulation does not
read the landmarks' positions, so the repetitions do the same work.  The card name and power limit are read in the
same run."""
import argparse
import json
import math
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
from bundle_adjustment_solver_b200.capi import ptr  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi unavailable"


def triangulate(w, reps, min_parallax_deg=1.0, max_residual_px=2.0):
    import torch
    from torch.profiler import ProfilerActivity, profile
    sc = bench.make_scene(w, 0, 1.0)
    sc.poses_init = sc.poses_true.copy()
    sc.points_init = np.full_like(sc.points_init, np.nan)
    e = S.load_scene(S.FullBundleAdjustmentSolver(device=0, stream=torch.cuda.current_stream().cuda_stream), sc)
    e._upload()
    M = len(sc.points_init)
    st = np.zeros(M, dtype=np.uint8)
    counts = np.zeros(6, dtype=np.int64)
    rad, res = math.radians(min_parallax_deg), max_residual_px * e.scaler

    def call():
        rc = e.L.ba_triangulate_points(e.h, None, rad, res, ptr(st), ptr(counts))
        if rc != 0:
            raise RuntimeError(e.L.ba_last_error(e.h).decode())

    t0 = time.perf_counter()
    call()   # the first call after a finalize uploads the landmark -> observation ranges
    first_ms = 1e3 * (time.perf_counter() - t0)
    host, dev = [], []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        t0 = time.perf_counter()
        call()
        host.append(1e3 * (time.perf_counter() - t0))
        b.record()
        b.synchronize()
        dev.append(a.elapsed_time(b))
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            call()
        torch.cuda.synchronize()
    ks = [ev.device_time_total for ev in prof.events()
          if ev.device_type == torch.autograd.DeviceType.CUDA and "k_triangulate_points" in ev.name]
    if not ks:
        raise RuntimeError("no k_triangulate_points activity in the profile")
    return dict(M=M, n_obs=sc.n_obs, min_parallax_deg=min_parallax_deg, max_residual_px=max_residual_px,
                first_call_ms=first_ms, call_ms_median=float(np.median(host)), call_ms_min=float(np.min(host)),
                call_event_ms_median=float(np.median(dev)), kernel_us_median=float(np.median(ks)),
                kernel_us_min=float(np.min(ks)), kernel_samples=len(ks), counts=counts.tolist())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c4")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    torch.cuda.init()
    torch.zeros(1, device="cuda")
    info = dict(card=card(), rows={})
    print(f"card: {info['card']}")
    for w in a.workloads.split(","):
        r = triangulate(w, a.reps)
        print(f"{w}: M {r['M']}  obs {r['n_obs']}  call {r['call_ms_median']:.2f} ms (min {r['call_ms_min']:.2f}, events "
              f"{r['call_event_ms_median']:.2f}, first {r['first_call_ms']:.2f})  kernel {r['kernel_us_median']:.1f} us "
              f"(min {r['kernel_us_min']:.1f})  counts {r['counts']}")
        info["rows"][w] = r
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(info, f, indent=1)


if __name__ == "__main__":
    main()
