"""ctypes binding of the sketch-program exports of the host mirror (gcs_host_program_* in
2d_geometry_constraint_solver_b200/host/src/capi_host.cpp; gcs/b200/sketch_program.hpp)."""
import ctypes as C

import numpy as np

from host_lib import Edge, Element, _dp, from_c, last_error, load, to_c


def _program_api(lib):
    if getattr(lib, "_program_api", False):
        return lib
    vp, ip, lp = C.c_void_p, C.POINTER(C.c_int32), C.POINTER(C.c_int64)
    lib.gcs_host_program_create.argtypes = [C.c_int, C.POINTER(Element), C.c_int, C.POINTER(Edge), C.POINTER(vp)]
    lib.gcs_host_program_create_leaves.argtypes = [C.c_int, C.POINTER(Element), C.c_int, ip, ip, C.POINTER(Edge), C.POINTER(vp)]
    lib.gcs_host_program_describe.argtypes = [vp, lp, lp, ip, lp, ip, ip, C.POINTER(C.c_uint8), C.POINTER(C.c_uint8), ip, ip]
    lib.gcs_host_program_run.argtypes = [vp, C.c_int64, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.c_int, lp]
    lib.gcs_host_program_solve.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(Element)]
    lib.gcs_host_program_destroy.argtypes = [vp]
    lib._program_api = True
    return lib


class Program:
    """A compiled sketch program (SketchProgram through the plain-C exports).  Values are indexed by
    the order of the real (non-virtual) edges of the sketch, or of the leaf list."""

    def __init__(self, elements, edges=None, leaves=None):
        lib = _program_api(load())
        self.elements = elements
        self.handle = C.c_void_p()
        if leaves is None:
            els, eds = to_c(elements, edges)
            self.rc = lib.gcs_host_program_create(len(elements), els, len(edges), eds, C.byref(self.handle))
        else:
            els, _ = to_c(elements, [])
            flat, offs = [], [0]
            for lf in leaves:
                flat += lf["edges"]
                offs.append(len(flat))
            _, eds = to_c([], flat)
            n = len(leaves)
            le = (C.c_int32 * max(3 * n, 1))(*[i for lf in leaves for i in lf["elems"]])
            eo = (C.c_int32 * (n + 1))(*offs)
            self.rc = lib.gcs_host_program_create_leaves(len(elements), els, n, le, eo, eds, C.byref(self.handle))
        self.error = last_error() if self.rc != 0 else ""

    def __del__(self):
        if getattr(self, "handle", None) and self.handle.value:
            _program_api(load()).gcs_host_program_destroy(self.handle)
            self.handle = C.c_void_p()

    def describe(self):
        """dict(waves, rows, slots, values, leaves, unsupported, offsets, row_solver, row_leaf, row_elems, row_values, row_code,
        solved_after, leaf_solver, leaf_level) as numpy arrays."""
        lib = _program_api(load())
        counts = np.zeros(6, dtype=np.int64)
        lib.gcs_host_program_describe(self.handle, counts.ctypes.data_as(C.POINTER(C.c_int64)), None, None, None, None, None, None, None, None,
                                      None)
        waves, rows, slots, values, leaves, unsupported = (int(v) for v in counts)
        d = {"waves": waves, "rows": rows, "slots": slots, "values": values, "leaves": leaves, "unsupported": unsupported,
             "offsets": np.zeros(waves * 5 + 1, dtype=np.int64), "row_solver": np.zeros(rows, dtype=np.int32),
             "row_leaf": np.zeros(rows, dtype=np.int64), "row_elems": np.zeros((rows, 3), dtype=np.int32),
             "row_values": np.zeros((rows, 3), dtype=np.int32), "row_code": np.zeros(rows, dtype=np.uint8), "solved_after": np.zeros(slots, dtype=np.uint8),
             "leaf_solver": np.zeros(leaves, dtype=np.int32), "leaf_level": np.zeros(leaves, dtype=np.int32)}
        ip, lp = C.POINTER(C.c_int32), C.POINTER(C.c_int64)
        lib.gcs_host_program_describe(self.handle, None, d["offsets"].ctypes.data_as(lp), d["row_solver"].ctypes.data_as(ip),
                                      d["row_leaf"].ctypes.data_as(lp), d["row_elems"].ctypes.data_as(ip), d["row_values"].ctypes.data_as(ip),
                                      d["row_code"].ctypes.data_as(C.POINTER(C.c_uint8)), d["solved_after"].ctypes.data_as(C.POINTER(C.c_uint8)), d["leaf_solver"].ctypes.data_as(ip),
                                      d["leaf_level"].ctypes.data_as(ip))
        return d

    def run(self, values, n_devices=1):
        """values [K][n_values] (radians for angles).  Returns (rc, positions [K][n_slots][4], nonconverged [K], stats)."""
        values = np.ascontiguousarray(np.atleast_2d(values), dtype=np.float64)
        K = values.shape[0]
        slots = self.describe()["slots"]
        pos = np.zeros((K, slots, 4))
        nc = np.zeros(K, dtype=np.uint32)
        stats = np.zeros(7, dtype=np.int64)
        rc = _program_api(load()).gcs_host_program_run(self.handle, K, _dp(values), _dp(pos), nc.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                      n_devices, stats.ctypes.data_as(C.POINTER(C.c_int64)))
        keys = ("launches", "compile_us", "upload_us", "device_us", "download_us", "run_us", "devices")
        return rc, pos, nc, dict(zip(keys, (int(v) for v in stats)))

    def solve(self, values=None):
        """SketchProgram::solve() after setting the constraints' values (None: keep them).  Returns (rc, elements)."""
        els, _ = to_c(self.elements, [])
        v = None if values is None else np.ascontiguousarray(values, dtype=np.float64)
        rc = _program_api(load()).gcs_host_program_solve(self.handle, None if v is None else _dp(v), els)
        return rc, from_c(self.elements, els)


def sketch_values(edges):
    """The value table of a sketch's own constraints: one value per real edge, in edge order."""
    return np.array([e.get("value", 0.0) for e in edges if e["type"] != 2], dtype=np.float64)
