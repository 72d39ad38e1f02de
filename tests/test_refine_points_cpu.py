"""CPU checks of the structure-only refinement interface: the C-ABI declares ba_refine_points and the BA_POINT_*
landmark states, the ctypes binding mirrors both, and the drop-in C++ driver of RefinePoints (on the plain and the
refactor front-end) compiles against the shims and the library."""
import ctypes as C
import os
import re

from bundle_adjustment_solver_b200 import capi
from test_cpp_dropin import _compile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_header_declares_the_entry_point_and_landmark_states():
    hdr = open(os.path.join(ROOT, "include", "ba_b200.h")).read()
    assert re.search(r"int ba_refine_points\(ba_solver \*s, const ba_options \*opt, const uint8_t \*select, "
                     r"double \*costs, int \*iterations,\s+uint8_t \*status, long long \*counts\);", hdr)
    states = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define BA_POINT_([A-Z_]+) (\d+)", hdr)}
    assert states == {"CONVERGED": capi.POINT_CONVERGED, "MAX_ITERATIONS": capi.POINT_MAX_ITERATIONS,
                      "SKIPPED": capi.POINT_SKIPPED, "UNOBSERVED": capi.POINT_UNOBSERVED,
                      "NONFINITE": capi.POINT_NONFINITE}
    assert "ba_refine_points" in capi.SYMBOLS


def test_binding_argtypes(engine_lib):
    assert engine_lib.ba_refine_points.argtypes == [C.c_void_p, C.POINTER(capi.Options)] + [C.c_void_p] * 5


def test_refine_points_dropin_compiles(tmp_path, engine_lib):
    exe = _compile("test_refine_points_dropin.cpp", tmp_path / "refine")
    assert os.path.exists(exe)
