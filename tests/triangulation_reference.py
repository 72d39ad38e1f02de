"""Float64 numpy restatement of ba_triangulate_points (include/ba_b200.h): the rays, the multi-view midpoint and the
status rules, in the engine's internal units.  The tests compare the engine with it.

Observation k of landmark i, in point order (lowest pose index first, then insertion order): the observing camera is
R_k = R_c R_jw, t_k = R_c t_jw + t_c; its centre c_k = -R_k^T t_k and its unit ray d_k = R_k^T m_k / |m_k| with
m_k = ((u - cx) / fx, (v - cy) / fy, 1); f is the first observation.  Rules, first match wins:
  1. fixed or not selected: SKIPPED;  2. fewer than two observations: TOO_FEW_OBSERVATIONS;
  3. min_k d_f . d_k > cos(min_parallax): LOW_PARALLAX;
  4. X = c_f + A^-1 g, A = sum_k (I - d_k d_k^T), g = sum_k (I - d_k d_k^T)(c_k - c_f); X not finite: LOW_PARALLAX;
  5. depth <= 0 (or a non-finite residual) in some observing camera: BEHIND_CAMERA;
  6. |r_u| + |r_v| > max_residual on some observation: LARGE_RESIDUAL;
  7. TRIANGULATED."""
from dataclasses import dataclass

import numpy as np

from bundle_adjustment_solver_b200.capi import (TRI_BEHIND_CAMERA, TRI_LARGE_RESIDUAL, TRI_LOW_PARALLAX, TRI_SKIPPED,
                                                TRI_TOO_FEW_OBSERVATIONS, TRI_TRIANGULATED)

SCALER = 0.01


@dataclass
class Problem:
    """A registered problem in internal units: cameras (fx fy cx cy | R_c 9 | t_c 3), poses T_jw (R 9 | t 3), points,
    point_free, and the observation rows in insertion order (camera slot, pose, point, scaled pixel)."""
    cams: np.ndarray        # (n_cam, 16)
    poses: np.ndarray       # (N, 12)
    points: np.ndarray      # (M, 3)
    point_free: np.ndarray  # (M,) bool
    obs_cam: np.ndarray
    obs_pose: np.ndarray
    obs_point: np.ndarray
    obs_uv: np.ndarray      # (n, 2)


def problem_from_scene(sc, poses12=None, points=None):
    """The internal problem the Python mirror registers for scene `sc` (cameras and pixels scaled by 0.01 as it does);
    poses12 / points: the engine's internal parameters (get_internal()), so both sides start from the same values."""
    cams = np.zeros((len(sc.cam_ids), 16))
    cams[:, :4] = np.asarray(sc.cam_intr, dtype=np.float64) * SCALER
    cT = np.asarray(sc.cam_T, dtype=np.float64).reshape(-1, 4, 4)
    cams[:, 4:13] = cT[:, :3, :3].reshape(-1, 9)
    cams[:, 13:16] = cT[:, :3, 3] * SCALER
    slot = {cid: k for k, cid in enumerate(sc.cam_ids)}
    free = np.ones(len(sc.points_init), dtype=bool)
    free[np.asarray(sc.fixed_points, dtype=np.int64)] = False
    return Problem(cams=cams, poses=np.asarray(poses12, dtype=np.float64), points=np.asarray(points, dtype=np.float64),
                   point_free=free, obs_cam=np.array([slot[c] for c in sc.obs_cam], dtype=np.int64),
                   obs_pose=np.asarray(sc.obs_pose, dtype=np.int64), obs_point=np.asarray(sc.obs_point, dtype=np.int64),
                   obs_uv=np.asarray(sc.obs_uv, dtype=np.float64) * SCALER)


def rays(pb, rows):
    """(centres, unit rays) of observation rows `rows`, world frame."""
    cam = pb.cams[pb.obs_cam[rows]]
    T = pb.poses[pb.obs_pose[rows]]
    Rc = cam[:, 4:13].reshape(-1, 3, 3)
    Rjw = T[:, :9].reshape(-1, 3, 3)
    Rk = Rc @ Rjw
    tk = np.einsum("nij,nj->ni", Rc, T[:, 9:12]) + cam[:, 13:16]
    c = -np.einsum("nji,nj->ni", Rk, tk)
    uv = pb.obs_uv[rows]
    m = np.stack([(uv[:, 0] - cam[:, 2]) / cam[:, 0], (uv[:, 1] - cam[:, 3]) / cam[:, 1], np.ones(len(rows))], axis=1)
    d = np.einsum("nji,nj->ni", Rk, m) / np.linalg.norm(m, axis=1)[:, None]
    return c, d


def project(pb, rows, X):
    """(depth, r_u, r_v) of observation rows `rows` at landmark positions X (one per row), as project() forms them."""
    cam = pb.cams[pb.obs_cam[rows]]
    T = pb.poses[pb.obs_pose[rows]]
    Xb = np.einsum("nij,nj->ni", T[:, :9].reshape(-1, 3, 3), X) + T[:, 9:12]
    Xc = np.einsum("nij,nj->ni", cam[:, 4:13].reshape(-1, 3, 3), Xb) + cam[:, 13:16]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        invz = 1.0 / Xc[:, 2]
        ru = cam[:, 0] * (Xc[:, 0] * invz) + cam[:, 2] - pb.obs_uv[rows, 0]
        rv = cam[:, 1] * (Xc[:, 1] * invz) + cam[:, 3] - pb.obs_uv[rows, 1]
    return Xc[:, 2], ru, rv


@dataclass
class Result:
    status: np.ndarray     # (M,) uint8, TRI_*
    points: np.ndarray     # (M, 3): the triangulated position where TRIANGULATED, the input otherwise
    min_dot: np.ndarray    # (M,) min_k d_f . d_k (NaN below two observations)
    X: np.ndarray          # (M, 3) the midpoint wherever it was formed (NaN elsewhere)
    min_depth: np.ndarray  # (M,) smallest depth at X over the observations (NaN where X was not formed)
    max_res: np.ndarray    # (M,) largest |r_u| + |r_v| at X (NaN where X was not formed)


def triangulate(pb, select=None, min_parallax=np.radians(1.0), max_residual=np.inf):
    """The rules above on every landmark; min_parallax in radians, max_residual in internal units."""
    M = len(pb.points)
    n = len(pb.obs_point)
    order = np.lexsort((np.arange(n), pb.obs_pose, pb.obs_point))   # point order: (point, pose, insertion)
    starts = np.searchsorted(pb.obs_point[order], np.arange(M + 1))
    cnt = np.diff(starts)
    sel = pb.point_free.copy()
    if select is not None:
        sel &= np.asarray(select, dtype=bool)
    status = np.full(M, TRI_SKIPPED, dtype=np.uint8)
    status[sel & (cnt < 2)] = TRI_TOO_FEW_OBSERVATIONS
    cand = np.flatnonzero(sel & (cnt >= 2))
    out = Result(status=status, points=pb.points.copy(), min_dot=np.full(M, np.nan), X=np.full((M, 3), np.nan),
                 min_depth=np.full(M, np.nan), max_res=np.full(M, np.nan))
    if len(cand) == 0:
        return out
    rows = np.concatenate([order[starts[i]:starts[i + 1]] for i in cand])
    owner = np.repeat(np.arange(len(cand)), cnt[cand])           # index into cand of every row
    seg = np.concatenate([[0], np.cumsum(cnt[cand])[:-1]])
    c, d = rays(pb, rows)
    cf, df = c[seg][owner], d[seg][owner]
    dot = np.einsum("ni,ni->n", df, d)
    min_dot = np.fmin.reduceat(dot, seg)
    out.min_dot[cand] = min_dot
    with np.errstate(invalid="ignore"):
        low = min_dot > np.cos(min_parallax)
    P = np.eye(3)[None] - d[:, :, None] * d[:, None, :]
    A = np.add.reduceat(P, seg, axis=0)
    g = np.add.reduceat(np.einsum("nij,nj->ni", P, c - cf), seg, axis=0)
    X = np.full((len(cand), 3), np.nan)
    solve = ~low
    for k in np.flatnonzero(solve):
        try:
            X[k] = cf[seg[k]] + np.linalg.solve(A[k], g[k])
        except np.linalg.LinAlgError:
            pass
    low |= solve & ~np.isfinite(X).all(axis=1)
    formed = ~low
    out.X[cand[formed]] = X[formed]
    status[cand[low]] = TRI_LOW_PARALLAX
    depth, ru, rv = project(pb, rows, X[owner])
    with np.errstate(invalid="ignore"):
        behind_row = ~(depth > 0) | ~np.isfinite(ru) | ~np.isfinite(rv)
        res = np.abs(ru) + np.abs(rv)
        large_row = res > max_residual
    behind = np.logical_or.reduceat(behind_row, seg)
    large = np.logical_or.reduceat(large_row, seg)
    out.min_depth[cand[formed]] = np.fmin.reduceat(depth, seg)[formed]
    out.max_res[cand[formed]] = np.fmax.reduceat(res, seg)[formed]
    b = formed & behind
    lr = formed & ~behind & large
    ok = formed & ~behind & ~large
    status[cand[b]] = TRI_BEHIND_CAMERA
    status[cand[lr]] = TRI_LARGE_RESIDUAL
    status[cand[ok]] = TRI_TRIANGULATED
    out.points[cand[ok]] = X[ok]
    return out


def clear_thresholds(pb, min_parallax_deg, max_residual_px, select=None, rel=1e-6):
    """Thresholds near the requested ones (degrees, caller's pixels) such that no landmark of the reference lies within
    `rel` relative of either: min d_f . d_k against cos(min_parallax), the largest residual at X against max_residual
    (landmarks that pass the parallax and depth rules).  Ties are excluded by construction.  Returns (degrees, pixels)."""
    deg = float(min_parallax_deg)
    for _ in range(200):
        r = triangulate(pb, select, np.radians(deg), np.inf)
        cm = np.cos(np.radians(deg))
        md = r.min_dot[np.isfinite(r.min_dot)]
        if not (np.abs(md - cm) <= rel * abs(cm)).any():
            break
        deg *= 1.001
    else:
        raise AssertionError("no clear parallax threshold")
    px = float(max_residual_px)
    if np.isfinite(px):
        front = r.max_res[(r.min_depth > 0) & np.isfinite(r.max_res)]
        for _ in range(200):
            t = px * SCALER
            if not (np.abs(front - t) <= rel * t).any():
                break
            px *= 1.001
        else:
            raise AssertionError("no clear residual threshold")
    return deg, px
