"""ctypes binding of the C-ABI declared in include/ba_b200.h (libba_b200.so).

This is the only Python path into the engine; there is no CPU fallback: if the shared library
is missing or no CUDA device is present, calls raise.
"""
import ctypes as C
import os

import numpy as np

from . import _build


class BaError(RuntimeError):
    pass


class Options(C.Structure):
    """ba_options; mirrors Options (core/solver_option_and_summary.h:47-72)."""
    _fields_ = [
        ("solver_type", C.c_int),
        ("threshold_step_size", C.c_float),
        ("threshold_cost_change", C.c_float),
        ("threshold_huber_loss", C.c_float),
        ("threshold_outlier_rejection", C.c_float),
        ("max_num_iterations", C.c_int),
        ("initial_lambda", C.c_float),
        ("decrease_ratio_lambda", C.c_float),
        ("increase_ratio_lambda", C.c_float),
        ("b_accumulate", C.c_int),
        ("inverse_scaler", C.c_double),
        ("check_every", C.c_int),
        ("use_graph", C.c_int),
        ("method", C.c_int),   # BA_METHOD_*: 0 LM, 1 Gauss-Newton (refactor class), 2 gradient descent
    ]


def default_options(**kw):
    o = Options(1, 1e-5, 1e-5, 1.0, 2.0, 50, 100.0, 0.33, 3.0, 0, 100.0, 0, 1, 0)
    for k, v in kw.items():
        setattr(o, k, v)
    return o


class IterInfo(C.Structure):
    _fields_ = [
        ("cost", C.c_double), ("cost_change", C.c_double), ("average_reprojection_error", C.c_double),
        ("abs_gradient", C.c_double), ("abs_step", C.c_double), ("damping_term", C.c_double),
        ("iter_time", C.c_double), ("iteration_status", C.c_int), ("_pad", C.c_int),
    ]


class Result(C.Structure):
    _fields_ = [
        ("n_iterations", C.c_int), ("converged", C.c_int), ("initial_cost", C.c_double),
        ("final_cost", C.c_double), ("total_time_ms", C.c_double), ("device_time_ms", C.c_double),
        ("t_linearize_ms", C.c_double), ("t_schur_ms", C.c_double), ("t_solve_ms", C.c_double),
        ("t_backsub_ms", C.c_double), ("t_update_cost_ms", C.c_double), ("kernel_launches", C.c_longlong),
    ]


class PoseOnlyOptions(C.Structure):
    _fields_ = [
        ("threshold_step_size", C.c_float), ("threshold_cost_change", C.c_float),
        ("threshold_huber_loss", C.c_float), ("threshold_outlier_rejection", C.c_float),
        ("max_num_iterations", C.c_int),
    ]


class PoseOnlyResult(C.Structure):
    _fields_ = [
        ("n_iterations", C.c_int), ("converged", C.c_int), ("success", C.c_int), ("n_summary", C.c_int),
        ("final_error", C.c_float), ("final_step", C.c_float),
    ]


# row status of ba_observation_residuals (BA_OBS_*)
OBS_INLIER, OBS_OUTLIER, OBS_BEHIND_CAMERA, OBS_DROPPED = 0, 1, 2, 3
# landmark status of ba_refine_points (BA_POINT_*)
POINT_CONVERGED, POINT_MAX_ITERATIONS, POINT_SKIPPED, POINT_UNOBSERVED, POINT_NONFINITE = 0, 1, 2, 3, 4
# landmark status of ba_triangulate_points (BA_TRI_*)
(TRI_TRIANGULATED, TRI_SKIPPED, TRI_TOO_FEW_OBSERVATIONS, TRI_LOW_PARALLAX, TRI_BEHIND_CAMERA,
 TRI_LARGE_RESIDUAL) = 0, 1, 2, 3, 4, 5

# every symbol include/ba_b200.h declares
SYMBOLS = [
    "ba_create", "ba_destroy", "ba_reset", "ba_last_error", "ba_set_stream", "ba_set_profile", "ba_set_debug",
    "ba_set_cameras", "ba_set_poses", "ba_set_points", "ba_set_observations", "ba_set_observations_scaled", "ba_finalize",
    "ba_update_parameters", "ba_solve", "ba_build_only", "ba_cost", "ba_observation_residuals", "ba_refine_points", "ba_triangulate_points", "ba_get_poses", "ba_get_points",
    "ba_get_sizes", "ba_debug_dump", "ba_debug_pairs", "ba_debug_time_solve", "ba_debug_nd_plan", "ba_debug_solve_info", "ba_comm_get_unique_id", "ba_comm_init",
    "ba_comm_destroy", "ba_comm_attach", "ba_comm_shutdown", "ba_geometry_batched", "ba_geometry_batched_f", "ba_poseonly_solve_batched", "ba_poseonly_upload", "ba_poseonly_run",
    "ba_poseonly_download", "ba_poseonly_free", "ba_version",
]

_lib = None


def lib_path():
    return _build.LIB


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_build.LIB):
            raise BaError("libba_b200.so is not built (run __graft_entry__.build()); there is no CPU fallback")
        L = C.CDLL(_build.LIB)
        vp, i, ll = C.c_void_p, C.c_int, C.c_longlong
        L.ba_create.argtypes = [C.POINTER(vp), i]
        L.ba_destroy.argtypes = [vp]
        L.ba_destroy.restype = None
        L.ba_reset.argtypes = [vp]
        L.ba_last_error.argtypes = [vp]
        L.ba_last_error.restype = C.c_char_p
        L.ba_set_stream.argtypes = [vp, vp]
        L.ba_set_profile.argtypes = [vp, i]
        L.ba_set_debug.argtypes = [vp, i]
        L.ba_set_cameras.argtypes = [vp, i, vp, vp, vp]
        L.ba_set_poses.argtypes = [vp, i, vp, vp]
        L.ba_set_points.argtypes = [vp, i, vp, vp]
        L.ba_set_observations.argtypes = [vp, ll, vp, vp, vp, vp, C.POINTER(ll)]
        L.ba_set_observations_scaled.argtypes = [vp, ll, vp, vp, vp, vp, C.c_double, C.POINTER(ll)]
        L.ba_finalize.argtypes = [vp]
        L.ba_update_parameters.argtypes = [vp, vp, vp]
        L.ba_solve.argtypes = [vp, C.POINTER(Options), vp, i, C.POINTER(Result)]
        L.ba_build_only.argtypes = [vp, C.POINTER(Options), C.c_double, i]
        L.ba_cost.argtypes = [vp, C.POINTER(C.c_double)]
        L.ba_observation_residuals.argtypes = [vp, C.c_double, vp, vp, vp]
        L.ba_refine_points.argtypes = [vp, C.POINTER(Options), vp, vp, vp, vp, vp]
        L.ba_triangulate_points.argtypes = [vp, vp, C.c_double, C.c_double, vp, vp]
        L.ba_get_poses.argtypes = [vp, vp]
        L.ba_get_points.argtypes = [vp, vp]
        L.ba_get_sizes.argtypes = [vp, vp]
        L.ba_debug_dump.argtypes = [vp, i, vp]
        L.ba_debug_dump.restype = ll
        L.ba_debug_pairs.argtypes = [vp, vp, vp]
        L.ba_debug_time_solve.argtypes = [vp, i, i, C.POINTER(C.c_float)]
        L.ba_debug_nd_plan.argtypes = [i, i, i, i, i, vp, vp, i]
        L.ba_debug_solve_info.argtypes = [vp, C.c_char_p, i, vp]
        L.ba_comm_get_unique_id.argtypes = [vp]
        L.ba_comm_init.argtypes = [vp, vp, i, i, ll, ll]
        L.ba_comm_destroy.argtypes = [vp]
        L.ba_comm_attach.argtypes = [vp, ll, ll]
        L.ba_comm_shutdown.argtypes = [i]
        L.ba_geometry_batched.argtypes = [i, i, ll, vp, vp, vp]
        L.ba_geometry_batched_f.argtypes = [i, i, ll, vp, vp, vp]
        L.ba_poseonly_solve_batched.argtypes = [i, i, i] + [vp] * 12 + [C.POINTER(PoseOnlyOptions)] + [vp] * 4
        L.ba_poseonly_upload.argtypes = [C.POINTER(vp), i, i, i] + [vp] * 10
        L.ba_poseonly_run.argtypes = [vp, C.POINTER(PoseOnlyOptions), vp]
        L.ba_poseonly_download.argtypes = [vp, vp, vp, vp, vp]
        L.ba_poseonly_free.argtypes = [vp]
        L.ba_poseonly_free.restype = None
        L.ba_version.restype = C.c_char_p
        _lib = L
    return _lib


def ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)
