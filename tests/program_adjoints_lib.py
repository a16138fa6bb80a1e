"""ctypes binding of the sketch-program adjoint exports of the host mirror (gcs_host_program_run_recorded,
gcs_host_program_adjoints in 2d_geometry_constraint_solver_b200/host/src/capi_host.cpp):
program_tangents_lib's Program with SketchProgram::record and SketchProgram::adjoints."""
import ctypes as C

import numpy as np

import program_tangents_lib
from host_lib import _dp, load
from program_lib import sketch_values  # noqa: F401  (re-exported for the adjoint tests)

_KEYS = ("launches", "compile_us", "upload_us", "device_us", "download_us", "run_us", "devices")


def _adjoint_api(lib):
    if getattr(lib, "_adjoint_api", False):
        return lib
    vp, dp, lp = C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int64)
    lib.gcs_host_program_run_recorded.argtypes = [vp, C.c_int64, dp, dp, C.POINTER(C.c_uint32), C.c_int, lp]
    lib.gcs_host_program_adjoints.argtypes = [vp, C.c_int, dp, dp, lp]
    lib._adjoint_api = True
    return lib


class Program(program_tangents_lib.Program):
    """program_tangents_lib.Program plus record() and adjoints()."""

    def record(self, values, n_devices=1):
        """values [K][n_values] (radians for angles).  Returns (rc, positions [K][n_slots][4], nonconverged [K], stats)."""
        values = np.ascontiguousarray(np.atleast_2d(values), dtype=np.float64)
        K = values.shape[0]
        slots = self.describe()["slots"]
        pos = np.zeros((K, slots, 4))
        nc = np.zeros(K, dtype=np.uint32)
        stats = np.zeros(7, dtype=np.int64)
        rc = _adjoint_api(load()).gcs_host_program_run_recorded(self.handle, K, _dp(values), _dp(pos), nc.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                                n_devices, stats.ctypes.data_as(C.POINTER(C.c_int64)))
        self._recorded_k = K
        return rc, pos, nc, dict(zip(_KEYS, (int(v) for v in stats)))

    def adjoints(self, adj_positions, K=None):
        """adj_positions [K][n_slots][4][T] for the last record() (K: its instance count, or given).  Returns
        (rc, adj_values [K][n_values][T] in radians for angles, stats)."""
        adj = np.ascontiguousarray(adj_positions, dtype=np.float64)
        K = adj.shape[0] if K is None else K
        T = adj.shape[3] if adj.ndim == 4 else 0
        values = self.describe()["values"]
        out = np.zeros((K, values, max(T, 1)))
        stats = np.zeros(7, dtype=np.int64)
        rc = _adjoint_api(load()).gcs_host_program_adjoints(self.handle, T, _dp(adj), _dp(out), stats.ctypes.data_as(C.POINTER(C.c_int64)))
        return rc, out, dict(zip(_KEYS, (int(v) for v in stats)))
