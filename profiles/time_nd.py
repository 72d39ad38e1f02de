"""Reduced solve K5 on banded systems: serial window kernel (BA_B200_BAND_MODE=4) against the partitioned solve
(5: one launch per tree level, 6: one persistent launch).  Warm, graph-replayed timing through ba_debug_time_solve and
the agreement of x between the modes (and with numpy for C3)."""
import ctypes as C
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bundle_adjustment_solver_b200 import capi, scenes
from bundle_adjustment_solver_b200 import solver as S

wl = sys.argv[1] if len(sys.argv) > 1 else "c3"
scale = float(sys.argv[2]) if len(sys.argv) > 2 else 1.0
modes = [int(m) for m in sys.argv[3].split(",")] if len(sys.argv) > 3 else [4, 5, 6]
sc = scenes.scene_c3(seed=100, pose_noise_seed=7, scale=scale) if wl == "c3" else scenes.scene_c4(seed=100, scale=scale)
opt = capi.default_options()
L = capi.lib()


def engine(mode):
    """A solver under BA_B200_BAND_MODE=mode: the engine reads its switches when a solver is created."""
    os.environ["BA_B200_BAND_MODE"] = str(mode)
    e = S.load_scene(S.FullBundleAdjustmentSolver(device=0), sc)
    e._upload()
    if wl == "c3":
        e.set_debug(True)
    return e


engines = {mode: engine(mode) for mode in modes}
xs = {}
for mode in modes:
    e = engines[mode]
    e.build_only(opt, 100.0, do_solve=True)
    xs[mode] = e.dump("x").copy()
    if wl == "c3" and mode == modes[0]:
        n = 6 * e.sizes()["N"]
        Sm = e.dump("S").reshape(n, n)
        rhs = e.dump("rhs")
        xr = np.linalg.solve(Sm, rhs)
    if wl == "c3":
        print(f"{wl} mode {mode}: max |x - numpy| / max |x| = {np.abs(xs[mode] - xr).max() / np.abs(xr).max():.3e}", flush=True)
for mode in modes[1:]:
    d = np.abs(xs[mode] - xs[modes[0]]).max() / np.abs(xs[modes[0]]).max()
    print(f"{wl} mode {mode} vs mode {modes[0]}: max rel diff of x = {d:.3e}", flush=True)
for mode in modes:
    e = engines[mode]
    ms = C.c_float(0)
    e.build_only(opt, 100.0, do_solve=False)
    rc = L.ba_debug_time_solve(e.h, 15, 20, C.byref(ms))
    print(f"{wl} scale {scale} band mode {mode}: reduced solve {ms.value * 1000:9.1f} us  rc={rc}", flush=True)
