"""ctypes binding of the sketch-program tangent exports of the host mirror (gcs_host_program_run_tangents,
gcs_host_program_desc in 2d_geometry_constraint_solver_b200/host/src/capi_host.cpp): program_lib's
Program with SketchProgram::runTangents and the program's C-ABI descriptor."""
import ctypes as C
import importlib

import numpy as np

import program_lib
from host_lib import _dp, load
from program_lib import sketch_values  # noqa: F401  (re-exported for the tangent tests)

capi = importlib.import_module("2d_geometry_constraint_solver_b200").capi


def _tangent_api(lib):
    if getattr(lib, "_tangent_api", False):
        return lib
    vp, dp = C.c_void_p, C.POINTER(C.c_double)
    lib.gcs_host_program_run_tangents.argtypes = [vp, C.c_int64, dp, C.c_int, dp, dp, dp, C.POINTER(C.c_uint32), C.c_int,
                                                  C.POINTER(C.c_int64)]
    lib.gcs_host_program_desc.argtypes = [vp, C.POINTER(capi.CProgramDesc)]
    lib._tangent_api = True
    return lib


class Program(program_lib.Program):
    """program_lib.Program plus run_tangents() and desc()."""

    def run_tangents(self, values, dvalues, n_devices=1):
        """values [K][n_values] (radians for angles), dvalues [K][n_values][T] (the same units).  Returns
        (rc, positions [K][n_slots][4], dpositions [K][n_slots][4][T], nonconverged [K], stats)."""
        values = np.ascontiguousarray(np.atleast_2d(values), dtype=np.float64)
        dvalues = np.ascontiguousarray(dvalues, dtype=np.float64)
        K = values.shape[0]
        T = dvalues.shape[2] if dvalues.ndim == 3 else 0
        slots = self.describe()["slots"]
        pos = np.zeros((K, slots, 4))
        dpos = np.zeros((K, slots, 4, max(T, 1)))
        nc = np.zeros(K, dtype=np.uint32)
        stats = np.zeros(7, dtype=np.int64)
        rc = _tangent_api(load()).gcs_host_program_run_tangents(self.handle, K, _dp(values), T, _dp(dvalues), _dp(pos), _dp(dpos),
                                                                nc.ctypes.data_as(C.POINTER(C.c_uint32)), n_devices,
                                                                stats.ctypes.data_as(C.POINTER(C.c_int64)))
        keys = ("launches", "compile_us", "upload_us", "device_us", "download_us", "run_us", "devices")
        return rc, pos, dpos, nc, dict(zip(keys, (int(v) for v in stats)))

    def desc(self):
        """The program's gcs_b200_program_desc (capi.CProgramDesc); its pointers stay valid while this object lives."""
        d = capi.CProgramDesc()
        _tangent_api(load()).gcs_host_program_desc(self.handle, C.byref(d))
        d._owner = self
        return d
