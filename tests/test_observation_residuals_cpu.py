"""CPU checks of the per-observation residual interface: the C-ABI declares ba_observation_residuals and the BA_OBS_*
row states, the ctypes binding mirrors both, and the drop-in C++ driver of the outlier extensions (on the plain and the
refactor front-end) compiles against the shims and the library."""
import os
import re

from bundle_adjustment_solver_b200 import capi
from test_cpp_dropin import _compile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_declares_the_entry_point_and_row_states():
    hdr = open(os.path.join(ROOT, "include", "ba_b200.h")).read()
    assert re.search(r"int ba_observation_residuals\(ba_solver \*s, double threshold, double \*residuals, "
                     r"uint8_t \*status, long long \*counts\);", hdr)
    states = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define BA_OBS_([A-Z_]+) (\d+)", hdr)}
    assert states == {"INLIER": capi.OBS_INLIER, "OUTLIER": capi.OBS_OUTLIER,
                      "BEHIND_CAMERA": capi.OBS_BEHIND_CAMERA, "DROPPED": capi.OBS_DROPPED}
    assert "ba_observation_residuals" in capi.SYMBOLS


def test_binding_argtypes(engine_lib):
    import ctypes as C
    assert engine_lib.ba_observation_residuals.argtypes == [C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]


def test_outliers_dropin_compiles(tmp_path, engine_lib):
    exe = _compile("test_ba_outliers_dropin.cpp", tmp_path / "outliers")
    assert os.path.exists(exe)
