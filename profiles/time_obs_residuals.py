"""Time of ba_observation_residuals (per-observation residuals + status, k_obs_residuals) on the bench.py scenes.

  python profiles/time_obs_residuals.py [--workloads c3,c4] [--reps 30] [--out results/obs_residuals.json]

Host clock around the C-ABI call (it ends in a stream synchronise): the first call after a finalize (it uploads the
row map), then residuals + status + counts, then status only.  The kernel alone comes from the CUDA activities of
torch.profiler, in a separate pass.  Bytes model per row: 28 B read (pixel 16, pose / point / camera-flags indices 12)
+ 4 B row map + the outputs written (16 B residual + 1 B status, or 1 B status only); pose and point gathers are not
counted (they hit L2).  The HBM rate is bench.peaks() (measured when MEASURED_PEAKS.json is present).  The C3 working
set (~1M rows, ~49 MB) fits the 126 MB L2, so its repeated calls read from L2; C4 (~8M rows, ~390 MB) does not."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (peaks(), make_scene())

os.dup2(bench._REAL_STDOUT.fileno(), 1)   # bench.py sends fd 1 to stderr for its one-JSON-line protocol; undo that here
from bundle_adjustment_solver_b200 import solver as S  # noqa: E402
from bundle_adjustment_solver_b200.capi import ptr  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip() or "nvidia-smi unavailable"


def call(e, n, thr, res, st, cnt):
    rc = e.L.ba_observation_residuals(e.h, thr, ptr(res), ptr(st), ptr(cnt))
    if rc != 0:
        raise RuntimeError(e.L.ba_last_error(e.h).decode())


def host_ms(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(1e3 * (time.perf_counter() - t0))
    return float(np.median(ts)), float(np.min(ts))


def kernel_us(fn, reps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    ts = [ev.device_time_total for ev in prof.events()
          if ev.device_type == torch.autograd.DeviceType.CUDA and "k_obs_residuals" in ev.name]
    if not ts:
        raise RuntimeError("no k_obs_residuals activity in the profile")
    return float(np.median(ts)), len(ts)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="c3,c4")
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    torch.cuda.init()
    torch.zeros(1, device="cuda")
    hbm_gbs, hbm_src = bench.peaks()
    info = dict(card=card(), hbm_gbs=hbm_gbs, hbm_source=hbm_src, rows={})
    print(f"card: {info['card']}   HBM rate {hbm_gbs:.0f} GB/s ({hbm_src})")
    for w in a.workloads.split(","):
        sc = bench.make_scene(w, 0, 1.0)
        e = S.load_scene(S.FullBundleAdjustmentSolver(device=0), sc)
        e._upload()
        n = e._num_rows()
        res, st, cnt = np.zeros((n, 2)), np.zeros(n, dtype=np.uint8), np.zeros(4, dtype=np.int64)
        t0 = time.perf_counter()
        call(e, n, np.inf, res, st, cnt)
        first = 1e3 * (time.perf_counter() - t0)
        full = lambda: call(e, n, 0.05, res, st, cnt)
        status = lambda: call(e, n, 0.05, None, st, None)
        full(); status()   # warm-up of both shapes
        full_ms = host_ms(full, a.reps)
        status_ms = host_ms(status, a.reps)
        k_full, nk = kernel_us(full, a.reps)
        k_status, _ = kernel_us(status, a.reps)
        b_full, b_status = n * (28 + 4 + 17), n * (28 + 4 + 1)
        row = dict(n_rows=n, first_call_ms=first, call_ms_median_min=full_ms, status_only_ms_median_min=status_ms,
                   kernel_us=k_full, kernel_status_only_us=k_status, kernels_profiled=nk,
                   bytes=b_full, bytes_status_only=b_status,
                   kernel_gbs=b_full / (k_full * 1e3), kernel_status_only_gbs=b_status / (k_status * 1e3),
                   share_of_hbm=b_full / (k_full * 1e3) / hbm_gbs,
                   share_of_hbm_status_only=b_status / (k_status * 1e3) / hbm_gbs, counts=cnt.tolist())
        info["rows"][w] = row
        print(f"{w}: {n} rows | first call {first:.2f} ms (row-map upload) | call: residuals+status {full_ms[0]:.3f} ms "
              f"(min {full_ms[1]:.3f}), status only {status_ms[0]:.3f} ms (min {status_ms[1]:.3f}) | kernel "
              f"{k_full:.1f} us ({row['kernel_gbs']:.0f} GB/s, {100 * row['share_of_hbm']:.0f}% of HBM), status only "
              f"{k_status:.1f} us ({row['kernel_status_only_gbs']:.0f} GB/s)")
        del e
    print(f"card: {info['card']}")
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        json.dump(info, open(a.out, "w"), indent=1)


if __name__ == "__main__":
    main()
