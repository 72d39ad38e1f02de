"""Per-kernel device time of the C3 LM iteration with torch.profiler (CUDA activities), plain launches (no CUDA graph):
20 iterations from the initial guess after 5 warm-up iterations, averaged per iteration.

    python profiles/time_kernels.py [TREE]      # TREE: a checkout with a built library (default: this repository)
"""
import collections
import ctypes as C
import os
import sys

ROOT = os.path.abspath(sys.argv[1]) if len(sys.argv) > 1 else os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
from torch.profiler import ProfilerActivity, profile  # noqa: E402

from bundle_adjustment_solver_b200 import capi, scenes  # noqa: E402
from bundle_adjustment_solver_b200 import solver as S  # noqa: E402

K = 20
sc = scenes.scene_c3(seed=100, pose_noise_seed=7)
s = S.FullBundleAdjustmentSolver(device=0)
S.load_scene(s, sc)
s._upload()
T0, X0 = s.internal_parameters()
L = capi.lib()


def run(n):
    s.update_parameters_internal(T0, X0)
    opt = capi.default_options(max_num_iterations=n, threshold_cost_change=0.0, threshold_step_size=0.0,
                               check_every=n, use_graph=0)
    res = capi.Result()
    rc = L.ba_solve(s.h, C.byref(opt), None, 0, C.byref(res))
    assert rc == 0, L.ba_last_error(s.h)
    torch.cuda.synchronize()
    assert res.n_iterations == n, res.n_iterations


run(5)
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    run(K)
tot, cnt = collections.defaultdict(float), collections.Counter()
for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA:
        name = e.name.split("<")[0].split("(")[0].replace("void ", "").replace("ba::", "")
        tot[name] += e.device_time_total
        cnt[name] += 1
for name, t in sorted(tot.items(), key=lambda kv: -kv[1]):
    print(f"KERN {name:40s} {t / K:9.2f} us/iter  launches/iter {cnt[name] / K:.2f}")
