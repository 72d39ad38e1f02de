"""Shared helpers for the parity tests (oracle = checker, engine = product path through the C-ABI)."""
import numpy as np

import oracle
from bundle_adjustment_solver_b200 import solver as S

# Hessian / Schur blocks against the oracle: FP64, reduction-order differences only (BASELINE.json north_star)
BLOCK_TOL = 1e-9


def load_oracle(sc):
    return S.load_scene(oracle.FullBAOracle(), sc)


def load_engine(sc, device=0, identical_internal=None):
    """identical_internal: (T12, X) taken from the oracle so both sides start from bit-identical
    internal parameters (removes the 1-ulp freedom of the host-side pose inversion)."""
    e = S.load_scene(S.FullBundleAdjustmentSolver(device=device), sc)
    e._upload(internal_override=identical_internal)
    return e


def blockwise_rel_err(got, ref, block):
    """max over blocks of ||got-ref||_F / ||ref||_F, with blocks whose reference norm is below
    1e-13 of the largest block norm compared absolutely against that scale."""
    got = np.asarray(got).reshape(-1, block)
    ref = np.asarray(ref).reshape(-1, block)
    assert got.shape == ref.shape, (got.shape, ref.shape)
    if ref.size == 0:
        return 0.0
    nr = np.linalg.norm(ref, axis=1)
    scale = nr.max() if nr.size else 0.0
    den = np.maximum(nr, 1e-13 * scale) + 1e-300
    return float((np.linalg.norm(got - ref, axis=1) / den).max())


def options_pair(**kw):
    """Same options for oracle and engine."""
    from bundle_adjustment_solver_b200.capi import default_options
    eo = default_options(**kw)
    okw = {k: v for k, v in kw.items() if k not in ("inverse_scaler", "check_every", "use_graph")}
    oo = oracle.default_full_options(**okw)
    return oo, eo


def S_block_view(Sflat, N):
    """(n*n,) column-major symmetric -> (N*N, 36) array of 6x6 blocks (row-major inside a block)."""
    n = 6 * N
    Sm = np.asarray(Sflat).reshape(n, n).T  # symmetric anyway
    return Sm.reshape(N, 6, N, 6).transpose(0, 2, 1, 3).reshape(N * N, 36)


def compare_blocks(o, e, sizes, tol=BLOCK_TOL, check_S=True):
    """Every dumped block of the engine (debug on) against the oracle after the same build: A, a, C, b, Cinv, B and,
    with check_S, the reduced system S and its rhs.  Returns the errors, fails on any above tol."""
    N = sizes["N"]
    errs = {}
    for name, blk in (("A", 36), ("a", 6), ("C", 9), ("b", 3), ("Cinv", 9), ("B", 18)):
        errs[name] = blockwise_rel_err(e.dump(name), o.dump(name), blk)
    if check_S:
        errs["S"] = blockwise_rel_err(S_block_view(e.dump("S"), N), S_block_view(o.dump("S"), N), 36)
        errs["rhs"] = blockwise_rel_err(e.dump("rhs"), o.dump("rhs"), 6)
    bad = {k: v for k, v in errs.items() if not v <= tol}
    assert not bad, f"block parity failed: {bad} (all: {errs})"
    return errs


def launched_kernels(run, names):
    """Which of `names` appear among the kernels that run() launches (CUDA activities of torch.profiler).

    The profiler keeps only the device activities whose timestamps, mapped onto the host clock, fall inside its capture
    window, and late in a long test session that mapping lags: the first tens of milliseconds of a window lose their
    kernels (seen in the full GPU suite, where the first kernels of a build went missing while the later ones were
    reported).  So run() starts after a pause, behind a marker kernel (torch.cuda._sleep); only a profile that reports
    the marker -- and with it everything launched after it -- is used.  Without the marker the profile is taken again
    with a pause twice as long."""
    import time

    import torch
    from torch.profiler import ProfilerActivity, profile
    pause = 0.05
    for _ in range(8):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            time.sleep(pause)
            torch.cuda._sleep(100_000)
            run()
            torch.cuda.synchronize()
            time.sleep(0.05)
        seen = {e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
        if any("spin_kernel" in n for n in seen):
            return {k for k in names if any(k in n for n in seen)}
        pause *= 2
    raise AssertionError(f"no profile kept its marker kernel (last pause {pause / 2} s): {sorted(seen)}")


def solve_info(e):
    """(name, vals) of the reduced solve the engine's plan selected (ba_debug_solve_info)."""
    import ctypes as C
    from bundle_adjustment_solver_b200.capi import ptr
    name = C.create_string_buffer(512)
    vals = np.zeros(8)
    assert e.L.ba_debug_solve_info(e.h, name, 512, ptr(vals)) == 0
    return name.value.decode(), vals
