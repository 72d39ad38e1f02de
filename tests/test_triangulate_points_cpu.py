"""CPU checks of the triangulation interface and of its float64 reference: the reference (triangulation_reference.py)
on hand-made two- and four-view cases with known answers, the C-ABI declaration and the BA_TRI_* states against the
ctypes binding, and the C++ driver of TriangulatePoints (plain and refactor front-end) compiling against the library."""
import ctypes as C
import os
import re

import numpy as np

from bundle_adjustment_solver_b200 import capi
from test_cpp_dropin import _compile
import triangulation_reference as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


# ------------------------------------------------------------------------------------------------ hand cases
def _problem(centres, X, pixel_offsets=None):
    """One pinhole camera (fx = fy = 525 px, principal point (320, 240), internal units), identity rotations, camera
    centres `centres` (internal units); landmark 0 observed once from every pose at its exact projection of X (which
    may lie behind the cameras), plus per-row pixel offsets in pixels."""
    cams = np.zeros((1, 16))
    cams[0, :4] = np.array([525.0, 525.0, 320.0, 240.0]) * R.SCALER
    cams[0, 4:13] = np.eye(3).ravel()
    n = len(centres)
    poses = np.zeros((n, 12))
    poses[:, :9] = np.eye(3).ravel()
    poses[:, 9:] = -np.asarray(centres, dtype=np.float64)          # t = -R c
    Xc = np.asarray(X, dtype=np.float64)[None] - np.asarray(centres)
    uv = np.stack([cams[0, 0] * Xc[:, 0] / Xc[:, 2] + cams[0, 2], cams[0, 1] * Xc[:, 1] / Xc[:, 2] + cams[0, 3]], axis=1)
    if pixel_offsets is not None:
        uv = uv + np.asarray(pixel_offsets, dtype=np.float64) * R.SCALER
    return R.Problem(cams=cams, poses=poses, points=np.full((1, 3), np.nan), point_free=np.ones(1, dtype=bool),
                     obs_cam=np.zeros(n, dtype=np.int64), obs_pose=np.arange(n), obs_point=np.zeros(n, dtype=np.int64),
                     obs_uv=uv)


def test_two_rays_meet_at_the_point():
    X = np.array([0.013, -0.021, 0.085])
    r = R.triangulate(_problem([[0.0, 0.0, 0.0], [0.01, 0.002, -0.001]], X))
    assert r.status[0] == capi.TRI_TRIANGULATED
    np.testing.assert_allclose(r.points[0], X, rtol=1e-12, atol=0)
    assert r.max_res[0] < 1e-12 and r.min_depth[0] > 0


def test_parallel_rays_are_low_parallax():
    # the same pixel from two centres a baseline apart: parallel rays, the point is at infinity
    pb = _problem([[0.0, 0.0, 0.0], [0.01, 0.0, 0.0]], [0.0, 0.0, 0.1])
    pb.obs_uv[1] = pb.obs_uv[0]
    r = R.triangulate(pb, min_parallax=np.radians(0.01))
    assert r.status[0] == capi.TRI_LOW_PARALLAX and np.isnan(r.points[0]).all()
    # a real baseline passes a small threshold and fails one larger than its parallax (about 5.7 degrees here)
    pb = _problem([[0.0, 0.0, 0.0], [0.01, 0.0, 0.0]], [0.0, 0.0, 0.1])
    assert R.triangulate(pb, min_parallax=np.radians(5.0)).status[0] == capi.TRI_TRIANGULATED
    assert R.triangulate(pb, min_parallax=np.radians(6.0)).status[0] == capi.TRI_LOW_PARALLAX


def test_point_behind_the_cameras():
    X = np.array([0.01, 0.02, -0.08])
    r = R.triangulate(_problem([[0.0, 0.0, 0.0], [0.012, -0.003, 0.0], [0.02, 0.004, 0.001]], X))
    assert r.status[0] == capi.TRI_BEHIND_CAMERA
    np.testing.assert_allclose(r.X[0], X, rtol=1e-12, atol=0)     # the lines meet there, behind every camera
    assert np.isnan(r.points[0]).all()                              # not written


def test_one_outlier_pixel():
    centres = [[0.0, 0.0, 0.0], [0.01, 0.0, 0.0], [0.02, 0.001, 0.0], [0.03, -0.001, 0.001]]
    off = np.zeros((4, 2))
    off[2, 0] = 5.0                                                 # 5 px on one row
    pb = _problem(centres, [0.015, 0.01, 0.09], off)
    assert R.triangulate(pb, max_residual=2.0 * R.SCALER).status[0] == capi.TRI_LARGE_RESIDUAL
    r = R.triangulate(pb, max_residual=np.inf)
    assert r.status[0] == capi.TRI_TRIANGULATED and r.max_res[0] > 2.0 * R.SCALER


def test_too_few_skipped_and_selected():
    pb = _problem([[0.0, 0.0, 0.0], [0.01, 0.0, 0.0]], [0.0, 0.0, 0.1])
    keep = np.array([True, False])                                  # one observation left
    one = R.Problem(cams=pb.cams, poses=pb.poses, points=pb.points, point_free=pb.point_free, obs_cam=pb.obs_cam[keep],
                    obs_pose=pb.obs_pose[keep], obs_point=pb.obs_point[keep], obs_uv=pb.obs_uv[keep])
    assert R.triangulate(one).status[0] == capi.TRI_TOO_FEW_OBSERVATIONS
    assert R.triangulate(pb, select=[False]).status[0] == capi.TRI_SKIPPED
    pb.point_free[0] = False
    assert R.triangulate(pb).status[0] == capi.TRI_SKIPPED


# ------------------------------------------------------------------------------------------------ interface
def test_header_declares_the_entry_point_and_states():
    hdr = open(os.path.join(ROOT, "include", "ba_b200.h")).read()
    assert re.search(r"int ba_triangulate_points\(ba_solver \*s, const uint8_t \*select, double min_parallax, "
                     r"double max_residual,\s+uint8_t \*status, long long \*counts\);", hdr)
    states = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define BA_TRI_([A-Z_]+) (\d+)", hdr)}
    assert states == {"TRIANGULATED": capi.TRI_TRIANGULATED, "SKIPPED": capi.TRI_SKIPPED,
                      "TOO_FEW_OBSERVATIONS": capi.TRI_TOO_FEW_OBSERVATIONS, "LOW_PARALLAX": capi.TRI_LOW_PARALLAX,
                      "BEHIND_CAMERA": capi.TRI_BEHIND_CAMERA, "LARGE_RESIDUAL": capi.TRI_LARGE_RESIDUAL}
    assert "ba_triangulate_points" in capi.SYMBOLS


def test_binding_argtypes(engine_lib):
    assert engine_lib.ba_triangulate_points.argtypes == [C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                                         C.c_void_p, C.c_void_p]


def test_triangulate_points_dropin_compiles(tmp_path, engine_lib):
    exe = _compile("test_triangulate_points_dropin.cpp", tmp_path / "triangulate")
    assert os.path.exists(exe)
