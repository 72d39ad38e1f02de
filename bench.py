#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 bundle-adjustment engine.

Metric (BASELINE.json): LM iters/s & Schur-build obs/s at 1/2/4/8 B200; time-to-converge vs CPU.  One "step" = one
full Levenberg-Marquardt iteration (linearise, Schur complement, reduced solve, back-substitution, trial cost,
accept / lambda) over the workload's observations.  `value` = observations x LM iterations per second (whole job,
all ranks), device-resident; `lm_iters_per_s` and `schur_build_obs_per_s` are reported beside it.

Workload
  N = 1 : config C3 "stereo full BA, 200 poses / 50k landmarks / ~1M observations on 1 B200" (the configuration the
          metric is quoted on).
  N > 1 : config C4 "2000 poses / 1M landmarks / ~8M observations landmark-sharded over the GPUs with S all-reduce":
          ONE problem, every rank keeps a contiguous landmark range (strong scaling).  The same line carries
          `strong_scaling` (the same problem on rank 0 alone), `mgpu_parity` (the first sharded LM iterations
          against that single-GPU solve), `weak_c3` (every rank its own 50k landmarks on the same 200 poses) and the
          frame-sharded pose-only batch C2.

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --impl reference ...                     # the reference's algorithm on host cores (oracle)
  python bench.py ... --dump-outputs DIR                   # also save what the last timed step computed, as .npy
"""
import argparse
import glob
import json
import os
import re
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the checkout may be read-only and is left as it is: no bytecode caches next to the sources
sys.dont_write_bytecode = True

# stdout carries exactly ONE JSON line: library chatter written to fd 1 (e.g. NCCL's version banner) is sent
# to stderr for the whole run and the result goes to the saved descriptor
_REAL_STDOUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(line):
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


METRIC = "LM-iteration observation throughput (observations x LM iters/s; full iteration: linearise, Schur, solve, back-substitute, cost/accept)"
UNIT = "obs/s"
FP64_TENSOR_PEAK = 37.1   # TFLOP/s, measured on this pool's B200 (profiles/micro/dmma_peak.cu -> profiles/micro/dmma_peak.txt)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def make_scene(workload, rank, scale):
    from bundle_adjustment_solver_b200 import scenes
    if workload == "c3":
        return scenes.scene_c3(seed=100 + rank, scale=scale, pose_noise_seed=7)
    if workload == "c1":
        return scenes.scene_test_ba(seed=rank)
    if workload == "c4":
        return scenes.scene_c4(seed=100 + rank, scale=scale)
    if workload == "c5":
        return scenes.scene_c5(seed=100 + rank, scale=scale)
    raise SystemExit(f"unknown workload {workload}")


WORKLOAD_NAMES = {
    "c1": "C1 test_ba.cpp stereo full BA (60 poses / 660 landmarks / 34,019 observations)",
    "c3": "C3 stereo full BA, 200 poses / 50k landmarks / ~1M observations",
    "c4": "C4 stereo full BA, 2000 poses / 1M landmarks / ~8M observations",
    "c5": "C5 BAL-Venice-shaped mono full BA (1778 poses / ~1M points / ~5M observations)",
}


# BA_B200_SPEC_LIN=0 selects the separate pose-side pass (k_linearize_by_pose) + point-order cost pass (engine default:
# one pass in pose order for the trial cost and the next iteration's pose side, k_cost_linearize_by_pose)
SPEC_LIN = os.environ.get("BA_B200_SPEC_LIN", "1") != "0"


def algorithmic_bytes(sz, n_obs_free_pose, solve_info):
    """Algorithmic bytes per LM iteration of the implemented design (DESIGN.md 'Kernels').
    pose side  (k_linearize_by_pose): 28 B/obs in pose order, A / a and the S diagonal; clearing S costs
               8 (6N+1)^2 bytes when the whole buffer is cleared and 8 (6N)(bw+2) when only the band is
    point side (k_build_tiles, fused K1+K3+K4): 20 B/obs (pixel, camera) + 24 B per (pose, landmark) incidence,
               pose / point gathers, B written once (144 B/pair), per-landmark blocks (144 B), S tile flush
    back-substitution: B read once (144 B/pair) + per-landmark blocks;   cost: 28 B/obs."""
    O, Nt, Mt, N, M, P = sz["n_obs"], sz["N_total"], sz["M_total"], sz["N"], sz["M"], sz["P"]
    n = 6 * N
    clear = 8 * n * (int(solve_info["bw"]) + 2) if solve_info["band_clear"] else 8 * (n + 1) * (n + 1)
    b = {}
    b["linearize"] = 28 * n_obs_free_pose + 96 * Nt + 24 * Mt + 2 * 336 * N + clear
    banded = "k_nd" in solve_info["kernel"] or "banded" in solve_info["kernel"]
    stores = SPEC_LIN and banded and os.environ.get("BA_B200_REDUCE_STORES", "1") != "0"
    if SPEC_LIN:
        # speculative pose side: the pass over the observations in pose order is the trial-cost pass (update_cost);
        # the linearize phase only clears S and damps / stores the per-pose sums (216 B read, 336 B + 336 B written) --
        # and is empty on banded plans, where the storing form of k_tile_reduce does both (charged to schur)
        b["linearize"] = 0 if stores else (216 + 2 * 336) * N + clear
    b["schur"] = 20 * O + 24 * P + 96 * Nt + 24 * Mt + 144 * P + 144 * M + int(solve_info["alg_bytes"])
    if stores:
        b["schur"] += (216 + 2 * 336) * N
    b["backsub"] = 144 * P + 8 * P + 48 * N + 24 * M + (144 + 24 + 24 + 24 + 24) * Mt
    b["update_cost"] = 28 * O + 96 * Nt * 2 + 24 * Mt + (216 * N if SPEC_LIN else 0)
    b["schur_flops"] = 330.0 * O
    return b


def solve_info(L, s):
    import ctypes as C
    name = C.create_string_buffer(512)
    vals = np.zeros(8)
    rc = L.ba_debug_solve_info(s.h, name, 512, vals.ctypes.data_as(C.c_void_p))
    if rc != 0:
        raise SystemExit("ba_debug_solve_info failed")
    return {"kernel": name.value.decode(), "alg_flops": float(vals[0]), "exec_flops": float(vals[1]),
            "dense_flops": float(vals[2]), "bw": int(vals[3]), "ctas": int(vals[4]), "chain_steps": float(vals[5]),
            "band_clear": bool(vals[6]), "alg_bytes": float(vals[7])}


DUMP_BYTES = 64_000_000   # --dump-outputs: all files together, .npy headers included


def dump_outputs(out_dir, s, res):
    """What ba_solve hands its caller after the last timed step, as float64 .npy files, so that two builds can be
    compared output for output: poses.npy (N_total x 12, world-to-camera R row-major | t) and points.npy (M_total x 3),
    both in the engine's internal units as ba_get_poses / ba_get_points return them, and cost.npy (initial, final cost
    of the timed solve).  Points beyond the size budget are a seeded sample of rows, the same rows for the same
    arguments."""
    T, X = s.get_internal()
    cost = np.array([res.initial_cost, res.final_cost], dtype=np.float64)
    rows = (DUMP_BYTES - 3 * 4096 - T.nbytes - cost.nbytes) // (3 * 8)
    if len(X) > rows:
        X = X[np.sort(np.random.default_rng(0).choice(len(X), rows, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in (("poses", T), ("points", X), ("cost", cost)):
        np.save(os.path.join(out_dir, name + ".npy"), a)


def ncu_traffic_table():
    """DRAM traffic per launch (dram__bytes_read.sum + dram__bytes_write.sum, MB) of each kernel from the newest
    committed `ncu --set full` summary of the default C3 workload (profiles/rNN_ncu_full_c3_summary.md)."""
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_ncu_full_c3_summary.md")))
    if not files:
        return None, None
    tab = {}
    hdr = None
    for ln in open(files[-1]):
        cells = [c.strip() for c in ln.strip().strip("|").split("|")]
        if ln.startswith("| kernel"):
            hdr = [re.sub(r"\s*\[.*\]", "", c) for c in cells]
            continue
        if hdr is None or not ln.startswith("|") or ln.startswith("|---"):
            continue
        try:
            row = dict(zip(hdr, cells))
            tab[row["kernel"]] = (float(row["dram_rd"]) + float(row["dram_wr"])) * 1e6
        except (KeyError, ValueError):
            continue
    return tab, os.path.relpath(files[-1], ROOT)


PHASE_KERNELS = {   # kernel-name prefixes of the ncu summary per phase
    "linearize": ("k_linearize_by_pose", "k_finish_poses", "k_clear_band", "k_pose_diag"),
    "schur": ("k_build_tiles", "k_tile_reduce", "k_linearize_by_point", "k_pair_blocks", "k_finish_points", "k_schur"),
    "solve": ("k_nd_", "k_chol_"),
    "backsub": ("k_backsub_pairs", "k_backsub_points"),
    "update_cost": ("k_cost", "k_update_poses", "k_reduce_decide"),
}


def phase_traffic(tab, phase):
    if not tab:
        return None
    v = [b for k, b in tab.items() if k.startswith(PHASE_KERNELS[phase])]
    return float(sum(v)) if v else None


# ------------------------------------------------------------------------------------------------------------
# config C2: batched pose-only BA
# ------------------------------------------------------------------------------------------------------------
def poseonly_c2(device, stream, rank, world, dist, dev, frames=4096, points=300, reps=5, cpu_legs=True):
    """Config C2: batched 6-DoF stereo pose-only BA, `frames` independent frames x `points` observations, frames split
    evenly over the ranks with no communication.  Device-resident timing (ba_poseonly_upload / ba_poseonly_run, CUDA
    events on the launching stream), end to end through ba_poseonly_solve_batched from host buffers, and the float
    oracle on 1 and on all host cores (rank 0, N = 1)."""
    import ctypes as C
    import torch
    from bundle_adjustment_solver_b200 import capi, scenes, sharding
    from bundle_adjustment_solver_b200 import solver as S
    L = capi.lib()
    full = scenes.scene_poseonly_batch(n_frames=frames, n_points=points, seed=1)
    pb = sharding.shard_poseonly_batch(full, rank, world) if world > 1 else full
    f32 = lambda a: None if a is None else np.ascontiguousarray(a, dtype=np.float32)
    off = np.ascontiguousarray(pb.offsets, dtype=np.int32)
    arrs = [f32(pb.points), f32(pb.px_left), f32(pb.px_right), f32(pb.intr_left), f32(pb.intr_right),
            f32(pb.left_to_right), None, None, f32(pb.poses_init)]
    h = C.c_void_p()
    rc = L.ba_poseonly_upload(C.byref(h), device, pb.kind, pb.n_frames, capi.ptr(off), *[capi.ptr(a) for a in arrs])
    if rc != 0:
        raise SystemExit("ba_poseonly_upload failed")
    opt = capi.PoseOnlyOptions(1e-6, 1e-6, 1.5, 2.5, 100)
    for _ in range(3):
        L.ba_poseonly_run(h, C.byref(opt), C.c_void_p(stream.cuda_stream))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        L.ba_poseonly_run(h, C.byref(opt), C.c_void_p(stream.cuda_stream))
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    res = (capi.PoseOnlyResult * max(1, pb.n_frames))()
    poses = np.zeros((pb.n_frames, 12), dtype=np.float32)
    L.ba_poseonly_download(h, capi.ptr(poses), None, None, res)
    L.ba_poseonly_free(h)
    iters_sum = float(np.sum([res[k].n_iterations for k in range(pb.n_frames)]))
    n_pts = int(off[-1])
    # end to end from host buffers through the reference-facing batched entry point (H2D + solve + D2H inside)
    po = S.PoseOnlyBundleAdjustmentSolver(device=device)
    run = lambda: po.solve_batched(pb.kind, pb.offsets, pb.points, pb.px_left, pb.px_right, pb.intr_left, pb.intr_right,
                                   pb.poses_init, opt, left_to_right=pb.left_to_right)
    run()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    out = run()
    e2e_s = time.perf_counter() - t0
    agg = torch.tensor([ms, e2e_s], dtype=torch.float64, device=dev)
    tot = torch.tensor([iters_sum, float(n_pts), float(np.abs(poses - pb.poses_true).max()) if pb.n_frames else 0.0],
                       dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(agg, op=dist.ReduceOp.MAX)
        err = tot[2:].clone()
        dist.all_reduce(tot)
        dist.all_reduce(err, op=dist.ReduceOp.MAX)
        tot[2] = err[0]
    ms, e2e_s = float(agg[0]), float(agg[1])
    iters = float(tot[0]) / frames
    all_pts = float(tot[1])
    # 240 FP32 flop per stereo point per GN iteration (SURVEY 8d); FP32 ALU peak = SMs x 128 lanes x 2 x clock
    prop = torch.cuda.get_device_properties(device)
    fp32_peak = prop.multi_processor_count * 128 * 2 * 1.965e9 / 1e12 * world
    fp32_tf = 240.0 * all_pts * iters / (ms * 1e-3) / 1e12
    r = {"workload": f"C2 batched 6-DoF stereo pose-only BA, {frames} frames x {points} points (FP32)",
         "n_gpus": world, "frames_per_gpu": pb.n_frames, "sharding": "frames split evenly over the ranks, no communication",
         "ms_per_batch": ms, "frames_per_s": frames / (ms * 1e-3),
         "point_iterations_per_s": all_pts * iters / (ms * 1e-3), "mean_gn_iterations": iters,
         "max_pose_err_vs_truth": float(tot[2]),
         "roofline": {"bound": "fp32 alu / latency (34 MB working set is L2-resident; not HBM)", "achieved_tflops": fp32_tf,
                      "peak_tflops": fp32_peak, "frac": fp32_tf / fp32_peak,
                      "peak_source": "SMs x 128 FMA lanes x 2 x 1.965 GHz (nominal FP32 ALU rate, no measured figure in MEASURED_PEAKS.json)",
                      "hbm_frac_if_streamed_once": 28.0 * all_pts / (ms * 1e-3) / 1e9 / (peaks()[0] * world)},
         "e2e": {"frames_per_s": frames / e2e_s, "wall_ms": 1e3 * e2e_s,
                 "h2d_bytes": int(28 * n_pts + 48 * pb.n_frames + 4 * len(off)), "d2h_bytes": int(48 * pb.n_frames + 2 * n_pts + 24 * pb.n_frames),
                 "through": "ba_poseonly_solve_batched (host buffers in, poses / masks / results out)"},
         "note": "one warp per frame, persistent over the GN iterations"}
    del out
    if cpu_legs and rank == 0 and world == 1:
        import oracle
        from concurrent.futures import ThreadPoolExecutor
        oopt = oracle.PoseOnlyOptions(1e-6, 1e-6, 1.5, 2.5, 100)
        solve = lambda b, native=True: oracle.poseonly_solve_batched(b.kind, b.offsets, b.points, b.px_left, b.px_right, b.intr_left,
                                                                    b.intr_right, b.poses_init, oopt, left_to_right=b.left_to_right,
                                                                    native=native)
        solve(sharding.shard_poseonly_batch(full, 0, 64))          # builds / loads the native library
        t0 = time.perf_counter()
        solve(full)
        t1 = time.perf_counter() - t0
        cores = os.cpu_count() or 1
        parts = [sharding.shard_poseonly_batch(full, q, cores) for q in range(cores)]
        with ThreadPoolExecutor(cores) as ex:                      # ctypes releases the GIL during the call
            t0 = time.perf_counter()
            list(ex.map(solve, parts))
            tn = time.perf_counter() - t0
        r["cpu_baseline"] = {"kind": "port", "unit": "frames/s", "one_core": {"value": frames / t1, "cores": 1, "wall_s": t1},
                             "all_cores": {"value": frames / tn, "cores": cores, "wall_s": tn},
                             "sample": f"all {frames} frames, float oracle built -O2 -march=native (the reference's flags)"}
    return r


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, loaded = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
                loaded.append(float(f[7]) > 0)
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        under = [s for s, l in zip(sm, loaded) if l] or sm
        return {"sm_mhz": float(np.median(under)) if under else None,
                "sm_max_mhz": float(max(mx)) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "samples_under_load": int(sum(loaded))}


# ------------------------------------------------------------------------------------------------------------
# CPU legs (the oracle is the checker / the reported baseline, never the product path)
# ------------------------------------------------------------------------------------------------------------
def cpu_sample(sc, workload):
    """The CPU leg runs on a BOUNDED sample of the workload: C1 / C3 as they are; C4 / C5 on a window of consecutive
    poses (same tracks, same band) -- the oracle's dense unblocked LDLT of the full 12 k reduced system alone takes
    ten minutes per iteration.  Throughput is quoted per observation; the sample favours the CPU (the cubic term of
    the reduced solve is 500x smaller per observation than on the full problem)."""
    from bundle_adjustment_solver_b200 import scenes
    if workload == "c4":
        return scenes.restrict_poses(sc, 0, 250), "poses 0..249 of the scene (about 1.0 M observations, 6N = 1,488)"
    if workload == "c5":
        return scenes.restrict_poses(sc, 0, 160), "poses 0..159 of the scene (about 0.44 M observations, 6N = 948)"
    return sc, "the whole workload"


def cpu_iterations(sc, iters, native):
    import oracle
    from bundle_adjustment_solver_b200 import solver as S
    o = S.load_scene(oracle.FullBAOracle(native=native), sc)
    o.sizes()
    oo = oracle.default_full_options(max_num_iterations=iters, threshold_cost_change=0.0, threshold_step_size=0.0)
    t0 = time.perf_counter()
    infos, _ = o.solve(oo)
    return time.perf_counter() - t0, len(infos)


def cpu_to_convergence(sc, native=True, max_iters=300):
    import oracle
    from bundle_adjustment_solver_b200 import solver as S
    t0 = time.perf_counter()
    o = S.load_scene(oracle.FullBAOracle(native=native), sc)
    oo = oracle.default_full_options(max_num_iterations=max_iters, threshold_cost_change=1e-6, threshold_step_size=1e-6)
    infos, conv = o.solve(oo)
    return {"wall_s": time.perf_counter() - t0, "lm_iterations": len(infos), "converged": bool(conv),
            "final_cost": infos[-1].cost if infos else None}


def gpu_to_convergence(sc, device, stream, max_iters=300):
    """Registration, FinalizeParameters (sorts, H2D), LM loop to convergence, D2H write-back: wall time from host buffers."""
    import torch
    from bundle_adjustment_solver_b200 import capi
    from bundle_adjustment_solver_b200 import solver as S
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    s = S.FullBundleAdjustmentSolver(device=device, stream=stream)
    S.load_scene(s, sc)
    summ = S.Summary()
    s.solve(capi.default_options(max_num_iterations=max_iters, threshold_cost_change=1e-6, threshold_step_size=1e-6), summ)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    it = len(summ.optimization_info_list)
    return {"wall_s": dt, "lm_iterations": it, "converged": bool(summ.convergence_status),
            "final_cost": summ.optimization_info_list[-1].cost if it else None}


def run_reference(args, rank, world):
    """--impl reference: the reference's own algorithm on the host cores.  The reference cannot be compiled here (no
    Eigen / Ceres / OpenCV), so this is the oracle port (kind 'port') built with the reference's flags
    (CMakeLists.txt:6: -O2 -march=native), single thread like the reference (it has no threads), on a bounded number
    of LM iterations of the same workload."""
    if rank != 0:
        return
    workload = args.workload or ("c3" if world == 1 else "c4")
    sc, sample = cpu_sample(make_scene(workload, 0, args.scale), workload)
    warm = 1 if args.warmup > 0 else 0
    if warm:
        cpu_iterations(sc, 1, True)
    dt, n = cpu_iterations(sc, args.steps, True)
    dt_p, n_p = cpu_iterations(sc, args.steps, False)
    value = sc.n_obs * n / dt
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": n,
        "warmup": warm, "ms_per_step": 1e3 * dt / n, "higher_is_better": True, "scaling": "weak" if world == 1 else "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD_NAMES[workload], "n_obs": sc.n_obs, "scale": args.scale},
        "lm_iters_per_s": n / dt,
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": 1, "kind": "port",
                         "sample": f"{n} LM iterations on {sample}, oracle/ba_oracle.cpp built -O2 -march=native "
                                   f"(the reference's CMake flags), host has {os.cpu_count()} cores; the reference is single-threaded",
                         "portable_build_value": sc.n_obs * n_p / dt_p,
                         "caveat": "a port of the reference's algorithm with sparse B storage and a scalar unblocked LDLT; the "
                                   "reference itself (Eigen) cannot be built in this image, so a GPU / CPU ratio taken from "
                                   "this line is an upper bound on what the Eigen build would give"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default=None, choices=list(WORKLOAD_NAMES),
                    help="default: c3 on one GPU, c4 (one problem sharded over the GPUs) on several")
    ap.add_argument("--scale", type=float, default=1.0)
    ap.add_argument("--weak", action="store_true", help="N > 1: every rank its own scene of the workload (weak scaling) as the headline")
    ap.add_argument("--cpu-iters", type=int, default=4, help="LM iterations of the CPU baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-poseonly", action="store_true", help="skip the C2 pose-only sub-benchmark")
    ap.add_argument("--no-extras", action="store_true", help="N > 1: skip strong_scaling / mgpu_parity / weak_c3")
    ap.add_argument("--no-converge", action="store_true", help="skip the time-to-converge legs (C1 and C3, GPU and CPU)")
    ap.add_argument("--e2e-max-iters", type=int, default=300,
                    help="iteration cap of the end-to-end solve (SURVEY 8d: thresholds 1e-6f, max 300 iterations)")
    ap.add_argument("--quick", action="store_true", help="profiling run: no clock-settling loop, phases, e2e or CPU baseline")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the poses, points and cost of the last timed step to DIR/<name>.npy (--impl b200; on "
                         "several GPUs rank 0 writes, with its share of the landmarks)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(3, args.warmup)
    workload = args.workload or ("c3" if world == 1 else "c4")

    import ctypes as C

    import torch
    import torch.distributed as dist

    from bundle_adjustment_solver_b200 import capi, sharding
    from bundle_adjustment_solver_b200 import solver as S

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(device=dev)
    L = capi.lib()

    # N > 1: ONE problem, every rank generates the same scene and keeps its contiguous landmark range (strong scaling);
    # --weak: every rank brings its own landmarks seen from the SAME poses (pose_noise_seed fixed)
    strong = world > 1 and not args.weak
    full_sc = make_scene(workload, 0, args.scale) if strong else None
    sc = sharding.shard_scene(full_sc, rank, world) if strong else make_scene(workload, rank, args.scale)

    comm_ready = [False]

    def join_comm(s, sz):
        """First call: create the process's communicator (NCCL set-up, ~0.4 s); later solvers attach to it."""
        if world == 1:
            return
        tot = torch.tensor([sz["M"], sz["n_obs"]], dtype=torch.int64, device=dev)
        dist.all_reduce(tot)
        if comm_ready[0]:
            rc = L.ba_comm_attach(s.h, int(tot[0]), int(tot[1]))
        else:
            idbuf = torch.zeros(128, dtype=torch.uint8)
            if rank == 0:
                raw = (C.c_ubyte * 128)()
                assert L.ba_comm_get_unique_id(raw) == 0
                idbuf = torch.tensor(list(raw), dtype=torch.uint8)
            idbuf = idbuf.to(dev)
            dist.broadcast(idbuf, 0)
            raw = (C.c_ubyte * 128)(*idbuf.cpu().tolist())
            rc = L.ba_comm_init(s.h, raw, rank, world, int(tot[0]), int(tot[1]))
            comm_ready[0] = True
        if rc != 0:
            raise SystemExit(f"ba_comm_init / attach failed: {L.ba_last_error(s.h)}")

    def new_solver(scene, comm=True):
        s = S.FullBundleAdjustmentSolver(device=local_rank, stream=stream.cuda_stream)
        S.load_scene(s, scene)
        s._upload()
        if comm:
            join_comm(s, s.sizes())
        return s

    def solve_n(s, n_it, check_every=None, profile=False):
        s.set_profile(profile)
        opt = capi.default_options(max_num_iterations=n_it, threshold_cost_change=0.0, threshold_step_size=0.0,
                                   check_every=check_every or n_it)
        res = capi.Result()
        rc = L.ba_solve(s.h, C.byref(opt), None, 0, C.byref(res))
        if rc != 0:
            raise SystemExit(f"ba_solve failed: {L.ba_last_error(s.h)}")
        assert res.n_iterations == n_it, (res.n_iterations, n_it)
        return res

    def timed_steps(s, steps, warmup, settle=True, collective=True):
        """W warm-up steps, then exactly `steps` LM iterations from the initial guess between CUDA events on the
        launching stream; max over ranks."""
        T0, X0 = s.internal_parameters()
        solve_n(s, warmup)
        t_w = time.perf_counter()
        while settle and time.perf_counter() - t_w < 1.0:
            solve_n(s, steps)
        s.update_parameters_internal(T0, X0)
        torch.cuda.synchronize()
        if world > 1 and collective:
            dist.barrier()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        res = solve_n(s, steps)
        ev1.record(stream)
        torch.cuda.synchronize()
        if world > 1 and collective:
            dist.barrier()
        ms = ev0.elapsed_time(ev1)
        if world > 1 and collective:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms, res

    with torch.cuda.stream(stream):
        s = new_solver(sc)
        sz = s.sizes()
        sinfo = solve_info(L, s)
        T12_0, X_0 = s.internal_parameters()
        n_obs_free_pose = int(np.count_nonzero(~np.isin(sc.obs_pose, sc.fixed_poses)))

        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        ms, res = timed_steps(s, args.steps, args.warmup, settle=not args.quick)
        launches = int(res.kernel_launches)
        clocks = sampler.stop() if rank == 0 else None
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, s, res)
        nobs_all = torch.tensor([sz["n_obs"]], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(nobs_all)
        total_obs = float(nobs_all[0])
        value = total_obs * args.steps / (ms * 1e-3)

        if args.quick:
            if rank == 0:
                emit({"quick": True, "ms_per_step": ms / args.steps, "value": value, "gpu_launches": launches})
            if world > 1:
                dist.destroy_process_group()
            return
        # ---- per-phase device times (CUDA events on the launching stream, plain launches)
        s.update_parameters_internal(T12_0, X_0)
        solve_n(s, args.warmup, profile=True)
        s.update_parameters_internal(T12_0, X_0)
        resp = solve_n(s, args.steps, profile=True)
        s.set_profile(False)
        ph = {"linearize": resp.t_linearize_ms / args.steps, "schur": resp.t_schur_ms / args.steps,
              "solve": resp.t_solve_ms / args.steps, "backsub": resp.t_backsub_ms / args.steps,
              "update_cost": resp.t_update_cost_ms / args.steps}

        # ---- N > 1: the first sharded LM iterations against the same problem solved on rank 0 alone, and the time of
        #      that single-GPU solve (strong-scaling reference measured in the same job)
        extras = {}
        if strong and not args.no_extras:
            K = 3
            s.update_parameters_internal(T12_0, X_0)
            summ = S.Summary()
            s.solve(capi.default_options(max_num_iterations=K, threshold_cost_change=0.0, threshold_step_size=0.0), summ)
            rows = [(i.cost, i.damping_term, i.iteration_status) for i in summ.optimization_info_list]
            if rank == 0:
                s1 = new_solver(full_sc, comm=False)
                summ1 = S.Summary()
                s1.solve(capi.default_options(max_num_iterations=K, threshold_cost_change=0.0, threshold_step_size=0.0), summ1)
                rows1 = [(i.cost, i.damping_term, i.iteration_status) for i in summ1.optimization_info_list]
                ok = len(rows) == len(rows1) == K and all(
                    abs(a[0] - b[0]) <= 1e-9 * abs(b[0]) and abs(a[1] - b[1]) <= 1e-12 * b[1] and a[2] == b[2]
                    for a, b in zip(rows, rows1))
                extras["mgpu_parity"] = bool(ok)
                extras["mgpu_parity_detail"] = {
                    "iterations": K, "tolerance": "cost 1e-9 relative, lambda 1e-12, identical status",
                    "max_rel_cost_diff": float(max(abs(a[0] - b[0]) / abs(b[0]) for a, b in zip(rows, rows1))) if rows1 else None}
                s1.update_parameters_internal(*s1.internal_parameters())
                ms1, _ = timed_steps(s1, args.steps, args.warmup, settle=False, collective=False)
                extras["strong_scaling"] = {"single_gpu_ms_per_step": ms1 / args.steps, "ms_per_step": ms / args.steps,
                                            "speedup": ms1 / ms, "efficiency": ms1 / ms / world,
                                            "single_gpu_solve_kernel": solve_info(L, s1)["kernel"]}
                del s1
            dist.barrier()

        # ---- end to end through the C-ABI from host buffers: register + finalize (H2D pack) + solve to convergence
        #      + read back.  Per-step bytes = totals / LM iterations.  N > 1: the communicator of this process is
        #      already up (a process joins once and then solves problem after problem); the solver attaches to it.
        e2e = None
        if not args.no_e2e:
            # the timed solver above is done: release it, so that the end-to-end solve runs in the steady state of a
            # process that solves one problem after another (device buffers come back from the stream-ordered pool
            # instead of growing it next to a live problem -- that growth alone varied between 10 and 150 ms)
            del s
            torch.cuda.synchronize()
            s2 = S.FullBundleAdjustmentSolver(device=local_rank, stream=stream.cuda_stream)
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            S.load_scene(s2, sc)
            t_reg = time.perf_counter()
            s2._upload()
            join_comm(s2, sz)
            t_fin = time.perf_counter()
            opt = capi.default_options(max_num_iterations=args.e2e_max_iters, threshold_cost_change=1e-6,
                                       threshold_step_size=1e-6)
            summ = S.Summary()
            s2.solve(opt, summ)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            stages = {"register_ms": 1e3 * (t_reg - t0), "finalize_h2d_ms": 1e3 * (t_fin - t_reg),
                      "solve_writeback_ms": 1e3 * (t0 + dt - t_fin)}
            it = len(summ.optimization_info_list)
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt[0])
            h2d = sc.n_obs * (16 + 16 + 12 + 12) + sz["N_total"] * 96 * 2 + sz["M_total"] * 24 * 2 + sz["P"] * 12
            d2h = sz["N_total"] * 96 + sz["M_total"] * 24 + it * 64
            e2e = {"value": total_obs * it / dt, "unit": UNIT, "h2d_bytes_per_step": int(h2d / max(it, 1)),
                   "d2h_bytes_per_step": int(d2h / max(it, 1)), "lm_iterations": it, "converged": bool(summ.convergence_status),
                   "wall_s": dt, "stages_ms": stages, "final_cost": summ.optimization_info_list[-1].cost if it else None,
                   "includes": "host registration, FinalizeParameters (sorts, H2D pack), LM loop to convergence, D2H write-back"
                               + ("; the process's NCCL communicator already exists (ba_comm_attach)" if world > 1 else "")}
            del s2

        # ---- N > 1: weak scaling of C3 (every rank its own 50k landmarks on the same 200 poses) beside the headline
        if strong and not args.no_extras:
            w_sc = make_scene("c3", rank, 1.0)
            sw = new_solver(w_sc)
            ms_w, _ = timed_steps(sw, args.steps, args.warmup, settle=False)
            nw = torch.tensor([float(w_sc.n_obs)], dtype=torch.float64, device=dev)
            dist.all_reduce(nw)
            del sw
            weak = {"workload": WORKLOAD_NAMES["c3"] + " per GPU (own landmarks, same poses)", "ms_per_step": ms_w / args.steps,
                    "value": float(nw[0]) * args.steps / (ms_w * 1e-3), "unit": UNIT, "scaling": "weak"}
            if rank == 0:
                s1 = new_solver(w_sc, comm=False)
                ms1, _ = timed_steps(s1, args.steps, args.warmup, settle=False, collective=False)
                weak["single_gpu_ms_per_step"] = ms1 / args.steps
                weak["efficiency"] = ms1 / ms_w
                del s1
            dist.barrier()
            extras["weak_c3"] = weak

        po2 = None
        if not args.no_poseonly:
            po2 = poseonly_c2(local_rank, stream, rank, world, dist, dev, cpu_legs=not args.no_cpu_baseline)

        # ---- time to converge (third BASELINE metric): GPU from host buffers (N = 1) vs the CPU port, C1 and C3
        converge = None
        if world == 1 and not args.no_converge and not args.no_cpu_baseline:
            converge = {}
            for wl in ("c1", "c3"):
                wsc = make_scene(wl, 0, 1.0)
                gpu_to_convergence(wsc, local_rank, stream.cuda_stream)             # warm pool / code
                g = gpu_to_convergence(wsc, local_rank, stream.cuda_stream)
                c = cpu_to_convergence(wsc, native=True)
                converge[wl] = {"workload": WORKLOAD_NAMES[wl], "gpu": g, "cpu": dict(c, cores=1, kind="port", build="-O2 -march=native"),
                                "speedup": c["wall_s"] / g["wall_s"],
                                "same_verdict": g["converged"] == c["converged"],
                                "iterations_within_1": abs(g["lm_iterations"] - c["lm_iterations"]) <= 1,
                                "final_cost_rel_diff": abs(g["final_cost"] - c["final_cost"]) / abs(c["final_cost"])}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm_peak, peak_src = peaks()
    ab = algorithmic_bytes(sz, n_obs_free_pose, sinfo)
    tab, tab_src = ncu_traffic_table() if (workload == "c3" and args.scale == 1.0 and world == 1) else (None, None)
    phases = {}
    for k in ("linearize", "schur", "backsub", "update_cost"):
        gbs = ab[k] / (ph[k] * 1e-3) / 1e9 if ph[k] > 0 else 0.0
        phases[k] = {"ms": ph[k], "algorithmic_bytes": ab[k], "achieved_gbs": gbs, "frac_hbm": gbs / hbm_peak,
                     "traffic": phase_traffic(tab, k)}
    t_solve = ph["solve"] * 1e-3
    tf = lambda fl: fl / t_solve / 1e12 if t_solve > 0 else 0.0
    phases["solve"] = {"ms": ph["solve"], "kernel": sinfo["kernel"], "algorithmic_flops": sinfo["alg_flops"],
                       "achieved_tflops": tf(sinfo["alg_flops"]), "executed_flops": sinfo["exec_flops"],
                       "executed_tflops": tf(sinfo["exec_flops"]), "dense_equivalent_flops": sinfo["dense_flops"],
                       "dense_equivalent_tflops": tf(sinfo["dense_flops"]), "half_bandwidth": sinfo["bw"],
                       "ctas": sinfo["ctas"], "dependent_panel_steps": sinfo["chain_steps"], "traffic": phase_traffic(tab, "solve")}
    # Jacobian / Schur build time: with the speculative pose side the pose-side Jacobians are formed in the trial-cost
    # pass, so that pass is charged to the build as well (conservative: it also evaluates the cost)
    t_build = ph["linearize"] + ph["schur"] + (ph["update_cost"] if SPEC_LIN else 0.0)
    banded = "k_nd" in sinfo["kernel"] or "banded" in sinfo["kernel"]
    stores = SPEC_LIN and banded and os.environ.get("BA_B200_REDUCE_STORES", "1") != "0"
    kernels = {"linearize": ("(none: the storing form of k_tile_reduce writes the damped pose-side blocks, S is not cleared)" if stores
                             else "k_pose_diag (damps and stores the per-pose sums of the accepted parameters)") if SPEC_LIN
               else "k_linearize_by_pose (ordered per-pose finish in the last chunk)",
               "schur": "k_build_tiles (linearise + C^-1 + Schur DMMA GEMM) + k_tile_reduce",
               "backsub": "k_backsub_pairs+k_backsub_points_update_poses",
               "update_cost": "k_cost_linearize_by_pose (trial cost + pose-side sums at the trial parameters + decision)" if SPEC_LIN
               else "k_cost_decide",
               "solve": sinfo["kernel"]}
    # the dominant kernel of the step by device time
    dom = max(ph, key=lambda k: ph[k])
    if dom == "solve":
        roofline = {"bound": "tensor", "kernel": kernels[dom], "achieved": phases["solve"]["achieved_tflops"],
                    "peak": FP64_TENSOR_PEAK, "unit": "TFLOP/s", "frac": phases["solve"]["achieved_tflops"] / FP64_TENSOR_PEAK,
                    "traffic": phases["solve"]["traffic"],
                    "executed_frac": phases["solve"]["executed_tflops"] / FP64_TENSOR_PEAK,
                    "peak_source": "measured FP64 DMMA throughput (profiles/micro/dmma_peak.cu; MEASURED_PEAKS.json has no FP64 figure)",
                    "note": "achieved = ALGORITHMIC flops of the reduced solve (Cholesky inside the envelope of S + the two triangular "
                            "solves) / solve time; executed_frac counts the flops the partitioned kernel really issues (fill of the "
                            "fronts, padding).  The solve is bound by its chain of dependent 8-column panel steps "
                            f"({sinfo['chain_steps']:.0f} on the critical path) on {sinfo['ctas']} of 148 SMs, not by FP64 throughput; "
                            "the dense-equivalent n^3/3 figure is kept under phases.solve only"}
    else:
        roofline = {"bound": "hbm", "kernel": kernels[dom], "achieved": phases[dom]["achieved_gbs"], "peak": hbm_peak,
                    "unit": "GB/s", "frac": phases[dom]["frac_hbm"], "traffic": phases[dom]["traffic"], "peak_source": peak_src}
    # the Jacobian / Schur build (BASELINE metric "Schur-build obs/s"): both build phases together
    build_bytes = ab["linearize"] + ab["schur"] + (ab["update_cost"] if SPEC_LIN else 0)
    build_gbs = build_bytes / (t_build * 1e-3) / 1e9 if t_build > 0 else 0.0
    tl, ts = phase_traffic(tab, "linearize"), phase_traffic(tab, "schur")
    if SPEC_LIN and tab:
        # the pose-side Jacobians are formed in the trial-cost pass; no kernel of its own is left in the linearize phase
        # when the storing reduce is active
        tu = phase_traffic(tab, "update_cost")
        tl = (tl or 0.0) + (tu or 0.0)
    roofline_build = {"bound": "hbm", "kernel": " ; ".join([kernels["linearize"], kernels["schur"]] + ([kernels["update_cost"]] if SPEC_LIN else [])),
                      "achieved": build_gbs,
                      "peak": hbm_peak, "unit": "GB/s", "frac": build_gbs / hbm_peak, "algorithmic_bytes": build_bytes,
                      "traffic": (tl + ts) if (tl is not None and ts is not None) else None, "traffic_source": tab_src,
                      "peak_source": peak_src,
                      "fp64_tflops": (ab["schur_flops"] / (t_build * 1e-3) / 1e12) if t_build > 0 else 0.0}
    for name, fr in [("roofline", roofline["frac"]), ("roofline_build", roofline_build["frac"])] + [
            (k, v["frac_hbm"]) for k, v in phases.items() if "frac_hbm" in v]:
        assert fr <= 1.2, f"{name}: fraction {fr:.2f} of peak is not a roofline point -- the accounting is wrong"

    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        it_cpu = max(1, args.cpu_iters)
        csc, sample = cpu_sample(sc, workload)
        dtc, n_c = cpu_iterations(csc, it_cpu, True)
        dtp, n_p = cpu_iterations(csc, it_cpu, False)
        cpu = {"value": csc.n_obs * n_c / dtc, "unit": UNIT, "cores": 1, "kind": "port",
               "sample": f"{n_c} LM iterations on {sample} on 1 of {os.cpu_count()} host cores "
                         f"(oracle/ba_oracle.cpp built -O2 -march=native like the reference's CMakeLists.txt:6; the reference is "
                         f"single-threaded), {dtc:.1f} s",
               "ms_per_step": 1e3 * dtc / n_c,
               "portable_build": {"value": csc.n_obs * n_p / dtp, "ms_per_step": 1e3 * dtp / n_p, "flags": "-O2 -ffp-contract=off (the parity checker)"},
               "caveat": "port with sparse B storage and a scalar unblocked LDLT; the Eigen reference cannot be built in this image"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD_NAMES[workload], "per_gpu": {k: sz[k] for k in ("N", "M", "P", "n_obs")},
                   "scale": args.scale,
                   "parallelism": (f"one problem, landmarks sharded x{world}, band of S all-reduced (NCCL), LM scalars exchanged through "
                                   f"peer memory" if strong else f"landmark-sharded x{world}, S all-reduce") if world > 1 else "single GPU",
                   "l2": "no flush: per-iteration working set %.0f MB exceeds the 126 MB L2" % (
                       (ab["linearize"] + ab["schur"] + ab["backsub"] + ab["update_cost"]) / 1e6),
                   "cuda_graph": True},
        "lm_iters_per_s": args.steps / (ms * 1e-3),
        "schur_build_obs_per_s": total_obs / (t_build * 1e-3) if t_build > 0 else None,
        "phases": phases, "roofline": roofline, "roofline_build": roofline_build, "poseonly_c2": po2, "cpu_baseline": cpu,
        "time_to_converge": converge, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
    }
    line.update(extras)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
