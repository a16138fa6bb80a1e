"""ctypes binding of the C ABI in include/gcs_b200.h.

This is plumbing for bench.py and the tests: the product is the CUDA library
(`libgcs_b200.so`, built from csrc/) and the C++ host mirror (host/).  There is no CPU
fallback here: if the library is missing, `load()` raises; if no CUDA device is present every
compute entry point returns GCS_E_NO_DEVICE and `check()` raises.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass, field

import numpy as np

MAX_IN_COLS = 13
MAX_OUT_COLS = 4
MAX_SEEDS = 8

KIND_PP, KIND_SDD, KIND_PPL, KIND_PLL, KIND_ANG = 1, 2, 3, 4, 5
KIND_NAMES = {1: "K1_PP", 2: "K2_SDD", 3: "K3_PPL", 4: "K4_PLL", 5: "K5_ANG"}
IN_COLS = {1: 6, 2: 9, 3: 10, 4: 12, 5: 13}
OUT_COLS = {1: 2, 2: 4, 3: 2, 4: 2, 5: 4}
IN_COL_NAMES = {
    1: ["ax", "ay", "ra", "bx", "by", "rb"],
    2: ["p1x", "p1y", "p2x", "p2y", "s1", "s2", "gnx", "gny", "canvas_len"],
    3: ["px", "py", "r", "xa", "ya", "xb", "yb", "s", "cfx", "cfy"],
    4: ["xa1", "ya1", "xb1", "yb1", "s1", "xa2", "ya2", "xb2", "yb2", "s2", "cfx", "cfy"],
    5: ["fdx", "fdy", "cosA", "gnx", "gny", "cfdx", "cfdy", "px", "py", "s", "r2x", "r2y",
        "canvas_len"],
}

MEM_HOST, MEM_DEVICE = 0, 1
VARIANT_DEFAULT, VARIANT_STATIC, VARIANT_REFILL, VARIANT_SORTED, VARIANT_PAIR = 0, 1, 2, 3, 4
# tolerance-class arithmetic (discrete outputs identical, coordinates to 1e-9): auto / static / sorted
VARIANT_CONTRACTED, VARIANT_CONTRACTED_STATIC, VARIANT_CONTRACTED_SORTED = 5, 6, 7
VARIANT_CONTRACTED_SEQ, VARIANT_SEQ = 8, 9  # one lane per sub-system, seeds in sequence: contracted / bit-identical
VARIANT_CONTRACTED_LINEAR = 10  # K4 in the contracted class: closed form, decisions certified (other kinds: as VARIANT_CONTRACTED)

CODE_COLLINEAR = 0x10
CODE_CANVAS_PARALLEL = 0x20

GCS_OK, GCS_E_INVALID, GCS_E_NO_DEVICE, GCS_E_CUDA, GCS_E_NOT_INIT, GCS_E_NOMEM = 0, -1, -2, -3, -4, -5

CONVERGENCE_THRESHOLD = 0.00001
MAXIMUM_ITERATIONS = 1000


def make_code(sign0, sign1=0, flags=0):
    """GCS_MAKE_CODE of gcs_b200.h, vectorised."""
    s0 = (np.asarray(sign0).astype(np.int64) + 1) & 3
    s1 = (np.asarray(sign1).astype(np.int64) + 1) & 3
    return (s0 | (s1 << 2) | np.asarray(flags).astype(np.int64)).astype(np.uint8)


class CBatch(C.Structure):
    _fields_ = [
        ("kind", C.c_int32),
        ("n_seeds", C.c_int32),
        ("n", C.c_int64),
        ("mem", C.c_int32),
        ("variant", C.c_int32),
        ("in_", C.c_void_p * MAX_IN_COLS),
        ("code", C.c_void_p),
        ("guesses", C.c_void_p),
        ("out", C.c_void_p * MAX_OUT_COLS),
        ("cand", C.c_void_p),
        ("iters", C.c_void_p),
        ("converged", C.c_void_p),
        ("root_index", C.c_void_p),
    ]


class CProgramRow(C.Structure):
    """gcs_b200_program_row: one leaf of a sketch program."""
    _fields_ = [
        ("solver", C.c_int32),
        ("elem", C.c_int32 * 3),
        ("value", C.c_int32 * 3),
        ("code", C.c_int32),
        ("sign", C.c_double * 3),
        ("canvas", C.c_double * 9),
    ]


class CProgramDesc(C.Structure):
    """gcs_b200_program_desc."""
    _fields_ = [
        ("n_waves", C.c_int32),
        ("n_slots", C.c_int32),
        ("n_values", C.c_int32),
        ("reserved", C.c_int32),
        ("n_rows", C.c_int64),
        ("rows", C.POINTER(CProgramRow)),
        ("offsets", C.POINTER(C.c_int64)),
        ("slot_is_line", C.POINTER(C.c_uint8)),
        ("initial", C.POINTER(C.c_double)),
        ("value_is_angle", C.POINTER(C.c_uint8)),
    ]


class CFitDesc(C.Structure):
    """gcs_b200_fit_desc."""
    _fields_ = [
        ("n_free", C.c_int32),
        ("n_obs", C.c_int32),
        ("free_values", C.POINTER(C.c_int32)),
        ("lower", C.POINTER(C.c_double)),
        ("upper", C.POINTER(C.c_double)),
        ("obs_slots", C.POINTER(C.c_int32)),
        ("obs_coords", C.POINTER(C.c_int32)),
        ("weights", C.POINTER(C.c_double)),
        ("max_iterations", C.c_int32),
        ("reserved", C.c_int32),
        ("lambda0", C.c_double),
        ("cost_tol", C.c_double),
        ("ftol", C.c_double),
        ("xtol", C.c_double),
        ("gtol", C.c_double),
    ]


class CFitResult(C.Structure):
    """gcs_b200_fit_result."""
    _fields_ = [
        ("status", C.c_int32),
        ("iterations", C.c_int32),
        ("cost", C.c_double),
        ("grad_inf", C.c_double),
        ("lambda_", C.c_double),
    ]


# gcs_b200_fit_result.status
FIT_RUNNING, FIT_COST, FIT_GTOL, FIT_FTOL, FIT_XTOL, FIT_STALLED, FIT_START_FAILED = range(7)


_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# GCS_B200_LIB: developer override to A/B an experimental build of the same library
LIB_PATH = os.environ.get("GCS_B200_LIB") or os.path.join(_PKG_DIR, "libgcs_b200.so")
_lib = None

EXPORTS = [
    "gcs_b200_kind_in_cols", "gcs_b200_kind_out_cols", "gcs_b200_device_count", "gcs_b200_init",
    "gcs_b200_shutdown", "gcs_b200_last_error", "gcs_b200_version", "gcs_b200_solve",
    "gcs_b200_solve_host", "gcs_b200_solve_host_async", "gcs_b200_wait", "gcs_b200_solve_sharded", "gcs_b200_launch_count", "gcs_b200_kernel_name", "gcs_b200_default_variant",
    "gcs_b200_fp64_probe", "gcs_b200_synth_pp", "gcs_b200_selftest", "gcs_b200_host_alloc", "gcs_b200_host_free",
    "gcs_b200_contracted_stats", "gcs_b200_contracted_stats_ex", "gcs_b200_column_may_be_null", "gcs_b200_host_alloc_ex",
    "gcs_b200_solve_host_range_async", "gcs_b200_pcie_probe", "gcs_b200_solve_many",
    "gcs_b200_debug_path_buffer", "gcs_b200_resolve_variant",
    "gcs_b200_program_create", "gcs_b200_program_run", "gcs_b200_program_run_host", "gcs_b200_program_destroy",
    "gcs_b200_program_run_tangents", "gcs_b200_program_run_tangents_host",
    "gcs_b200_program_run_recorded", "gcs_b200_program_run_recorded_host", "gcs_b200_program_adjoints",
    "gcs_b200_program_adjoints_host", "gcs_b200_program_fit", "gcs_b200_program_fit_host", "gcs_b200_fit_check",
    "gcs_b200_program_run_fused", "gcs_b200_program_run_fused_host",
]


def load():
    """Load libgcs_b200.so (built in-tree by __graft_entry__.build()).  Raises if absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing: the CUDA extension was not built "
            "(run `python -c 'import __graft_entry__ as g; g.build()'`). There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.gcs_b200_kind_in_cols.argtypes = [C.c_int]
    lib.gcs_b200_kind_out_cols.argtypes = [C.c_int]
    lib.gcs_b200_init.argtypes = [C.c_int, C.POINTER(C.c_int)]
    lib.gcs_b200_last_error.restype = C.c_char_p
    lib.gcs_b200_version.restype = C.c_char_p
    lib.gcs_b200_solve.argtypes = [C.POINTER(CBatch), C.c_int, C.c_void_p]
    lib.gcs_b200_solve_many.argtypes = [C.POINTER(C.POINTER(CBatch)), C.c_int, C.c_int, C.c_void_p]
    lib.gcs_b200_solve_host.argtypes = [C.POINTER(CBatch), C.c_int]
    lib.gcs_b200_solve_sharded.argtypes = [C.POINTER(CBatch), C.c_int]
    lib.gcs_b200_solve_host_async.argtypes = [C.POINTER(CBatch), C.c_int]
    lib.gcs_b200_wait.argtypes = [C.c_int]
    lib.gcs_b200_solve_host_range_async.argtypes = [C.POINTER(CBatch), C.c_int, C.c_int64, C.c_int64]
    lib.gcs_b200_launch_count.restype = C.c_int64
    lib.gcs_b200_kernel_name.argtypes = [C.c_int, C.c_int, C.c_int]
    lib.gcs_b200_kernel_name.restype = C.c_char_p
    lib.gcs_b200_default_variant.argtypes = [C.c_int64, C.c_int]
    lib.gcs_b200_resolve_variant.argtypes = [C.c_int, C.c_int, C.c_int64, C.c_int]
    lib.gcs_b200_contracted_stats.argtypes = [C.c_int, C.POINTER(C.c_uint64), C.c_int]
    lib.gcs_b200_contracted_stats_ex.argtypes = [C.c_int, C.POINTER(C.c_uint64), C.c_int]
    lib.gcs_b200_column_may_be_null.argtypes = [C.c_int, C.c_int]
    lib.gcs_b200_host_alloc.argtypes = [C.c_size_t]
    lib.gcs_b200_host_alloc.restype = C.c_void_p
    lib.gcs_b200_host_alloc_ex.argtypes = [C.c_size_t, C.c_int]
    lib.gcs_b200_host_alloc_ex.restype = C.c_void_p
    lib.gcs_b200_host_free.argtypes = [C.c_void_p]
    lib.gcs_b200_pcie_probe.argtypes = [C.c_int, C.c_size_t, C.c_size_t, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_double)]
    lib.gcs_b200_debug_path_buffer.argtypes = [C.c_int, C.c_void_p, C.c_int64]
    lib.gcs_b200_fp64_probe.argtypes = [C.c_int, C.c_int]
    lib.gcs_b200_fp64_probe.restype = C.c_double
    lib.gcs_b200_selftest.argtypes = [C.c_int, C.c_uint64, C.c_int64, C.POINTER(C.c_uint64)]
    lib.gcs_b200_synth_pp.argtypes = [C.c_int, C.c_void_p, C.c_uint64, C.c_int64, C.c_int64,
                                      C.c_int, C.POINTER(C.c_void_p), C.c_void_p]
    lib.gcs_b200_program_create.argtypes = [C.POINTER(CProgramDesc), C.c_int, C.POINTER(C.c_void_p)]
    lib.gcs_b200_program_run.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.gcs_b200_program_run_host.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                              C.POINTER(C.c_float)]
    lib.gcs_b200_program_run_tangents.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                                  C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.gcs_b200_program_run_tangents_host.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                                       C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_float)]
    lib.gcs_b200_program_run_recorded.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    lib.gcs_b200_program_run_recorded_host.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int,
                                                       C.POINTER(C.c_float)]
    lib.gcs_b200_program_run_fused.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                               C.c_void_p, C.c_void_p]
    lib.gcs_b200_program_run_fused_host.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                                    C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
    lib.gcs_b200_program_adjoints.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.gcs_b200_program_adjoints_host.argtypes = [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
    lib.gcs_b200_program_fit.argtypes = [C.c_void_p, C.POINTER(CFitDesc), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_void_p, C.c_int, C.c_void_p]
    lib.gcs_b200_program_fit_host.argtypes = [C.c_void_p, C.POINTER(CFitDesc), C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_float)]
    lib.gcs_b200_fit_check.argtypes = [C.POINTER(CProgramDesc), C.POINTER(CFitDesc)]
    lib.gcs_b200_program_destroy.argtypes = [C.c_void_p]
    _lib = lib
    return lib


def pcie_probe(device, bytes_up, bytes_down, pieces=1, write_combined=False, reps=5):
    """gcs_b200_pcie_probe -> dict(h2d_gbs, d2h_gbs, both_ms_best, both_ms_median)."""
    out = (C.c_double * 4)()
    check(load().gcs_b200_pcie_probe(device, bytes_up, bytes_down, pieces, 1 if write_combined else 0, reps, out), "gcs_b200_pcie_probe")
    return {"h2d_gbs": out[0], "d2h_gbs": out[1], "both_ms_best": out[2], "both_ms_median": out[3]}


class PinnedArray:
    """numpy view of page-locked memory from gcs_b200_host_alloc[_ex] (freed with the object)."""

    def __init__(self, shape, dtype=np.float64, write_combined=False):
        self.shape = tuple(int(v) for v in (shape if isinstance(shape, (tuple, list)) else (shape,)))
        self.nbytes = int(np.prod(self.shape)) * np.dtype(dtype).itemsize
        self.ptr = load().gcs_b200_host_alloc_ex(max(self.nbytes, 1), 1 if write_combined else 0)
        if not self.ptr:
            raise GcsError("gcs_b200_host_alloc_ex failed (no CUDA device?)")
        buf = (C.c_char * max(self.nbytes, 1)).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(self.shape))).reshape(self.shape)

    def __del__(self):
        try:
            if self.ptr:
                load().gcs_b200_host_free(self.ptr)
                self.ptr = None
        except Exception:
            pass


class GcsError(RuntimeError):
    pass


def check(rc: int, what: str = "gcs_b200"):
    if rc != 0:
        msg = load().gcs_b200_last_error()
        raise GcsError(f"{what} failed with code {rc}: {msg.decode() if msg else ''}")


def init(devices=None):
    lib = load()
    if devices is None:
        check(lib.gcs_b200_init(0, None), "gcs_b200_init")
    else:
        arr = (C.c_int * len(devices))(*devices)
        check(lib.gcs_b200_init(len(devices), arr), "gcs_b200_init")


@dataclass
class HostBatch:
    """A batch whose columns are numpy arrays (GCS_MEM_HOST).  Keeps the arrays alive."""
    kind: int
    n_seeds: int
    cols: list                      # kind-specific input columns, float64[n]; None = an anchor column of zeros (passed as NULL)
    code: np.ndarray                # uint8[n]
    guesses: np.ndarray | None = None   # float64[n_seeds, 2, n]
    variant: int = VARIANT_DEFAULT
    want_cand: bool = True
    out: list = field(default_factory=list)
    cand: np.ndarray | None = None
    iters: np.ndarray | None = None
    converged: np.ndarray | None = None
    root_index: np.ndarray | None = None

    @property
    def n(self):
        return int(self.code.shape[0])

    def alloc_outputs(self):
        n = self.n
        self.out = [np.full(n, np.nan) for _ in range(OUT_COLS[self.kind])]
        self.cand = np.full((self.n_seeds, 2, n), np.nan) if self.want_cand else None
        self.iters = np.full((self.n_seeds, n), -1, dtype=np.int16)
        self.converged = np.full((self.n_seeds, n), 255, dtype=np.uint8)
        self.root_index = np.full(n, 255, dtype=np.uint8)
        return self

    def slice(self, lo, hi):
        """Contiguous index range [lo, hi) as a new HostBatch (inputs are views)."""
        g = None if self.guesses is None else np.ascontiguousarray(self.guesses[:, :, lo:hi])
        return HostBatch(self.kind, self.n_seeds, [None if c is None else c[lo:hi] for c in self.cols], self.code[lo:hi],
                         g, self.variant, self.want_cand)

    def take(self, index):
        """The rows `index` (bool mask or index array) as a new HostBatch (inputs are copies)."""
        g = None if self.guesses is None else np.ascontiguousarray(self.guesses[:, :, index])
        return HostBatch(self.kind, self.n_seeds, [None if c is None else np.ascontiguousarray(c[index]) for c in self.cols],
                         np.ascontiguousarray(self.code[index]), g, self.variant, self.want_cand)

    def anchored(self):
        """The same batch with every anchor column that is identically +0.0 replaced by None (NULL at
        the ABI: not stored, not copied).  Raises if a column the shape needs to be zero is not."""
        cols = list(self.cols)
        lib = load()
        for c, col in enumerate(cols):
            if col is not None and lib.gcs_b200_column_may_be_null(self.kind, c) and not col.view(np.uint64).any():
                cols[c] = None
        return HostBatch(self.kind, self.n_seeds, cols, self.code, self.guesses, self.variant, self.want_cand)

    def dense_cols(self):
        """Input columns with the NULL ones materialised as zeros (for checkers that take no NULLs)."""
        n = self.n
        return [np.zeros(n) if c is None else c for c in self.cols]

    def input_bytes(self):
        """Bytes of input a host-buffer call uploads: present columns + the code column (+ guesses)."""
        n = self.n
        b = sum(8 * n for c in self.cols if c is not None) + n
        return b + (0 if self.guesses is None else self.guesses.nbytes)

    def cbatch(self, dense=False) -> CBatch:
        assert len(self.cols) == IN_COLS[self.kind], (len(self.cols), self.kind)
        b = CBatch()
        b.kind, b.n_seeds, b.n, b.mem, b.variant = self.kind, self.n_seeds, self.n, MEM_HOST, self.variant
        n = self.n
        cols = self.cols
        if dense:
            cols = self._dense = self.dense_cols()  # kept alive with the batch
        for i, c in enumerate(cols):
            if c is None:
                b.in_[i] = None
                continue
            assert c.dtype == np.float64 and c.flags["C_CONTIGUOUS"] and c.shape == (n,)
            b.in_[i] = c.ctypes.data
        assert self.code.dtype == np.uint8 and self.code.flags["C_CONTIGUOUS"]
        b.code = self.code.ctypes.data
        if self.guesses is not None:
            assert self.guesses.dtype == np.float64 and self.guesses.flags["C_CONTIGUOUS"]
            assert self.guesses.shape == (self.n_seeds, 2, n)
            b.guesses = self.guesses.ctypes.data
        for i, o in enumerate(self.out):
            b.out[i] = o.ctypes.data
        b.cand = self.cand.ctypes.data if self.cand is not None else None
        b.iters = self.iters.ctypes.data if self.iters is not None else None
        b.converged = self.converged.ctypes.data if self.converged is not None else None
        b.root_index = self.root_index.ctypes.data if self.root_index is not None else None
        return b


def solve_host(batch: HostBatch, device: int = 0) -> HostBatch:
    """gcs_b200_solve_host: H2D, kernel, D2H, synchronised."""
    if not batch.out:
        batch.alloc_outputs()
    cb = batch.cbatch()
    check(load().gcs_b200_solve_host(C.byref(cb), device), "gcs_b200_solve_host")
    return batch


def solve_host_async(batch: HostBatch, device: int = 0) -> HostBatch:
    """gcs_b200_solve_host_async: enqueue only; results are valid after wait(device)."""
    if not batch.out:
        batch.alloc_outputs()
    cb = batch.cbatch()
    check(load().gcs_b200_solve_host_async(C.byref(cb), device), "gcs_b200_solve_host_async")
    return batch


def solve_host_range_async(batch: HostBatch, device: int, first: int, count: int) -> HostBatch:
    """gcs_b200_solve_host_range_async: rows [first, first+count) only; valid after wait(device)."""
    if not batch.out:
        batch.alloc_outputs()
    cb = batch.cbatch()
    check(load().gcs_b200_solve_host_range_async(C.byref(cb), device, first, count), "gcs_b200_solve_host_range_async")
    return batch


def wait(device: int = 0):
    check(load().gcs_b200_wait(device), "gcs_b200_wait")


def solve_sharded(batch: HostBatch, n_dev: int) -> HostBatch:
    if not batch.out:
        batch.alloc_outputs()
    cb = batch.cbatch()
    check(load().gcs_b200_solve_sharded(C.byref(cb), n_dev), "gcs_b200_solve_sharded")
    return batch


def solve_many(device_batches, stream=None):
    """gcs_b200_solve_many over DeviceBatch objects of one device, on `stream` (default: torch's current)."""
    first = device_batches[0]
    torch = first.torch
    s = torch.cuda.current_stream(first.device) if stream is None else stream
    idx = first.device.index if first.device.index is not None else torch.cuda.current_device()
    arr = (C.POINTER(CBatch) * len(device_batches))(*[C.pointer(b._cb) for b in device_batches])
    check(load().gcs_b200_solve_many(arr, len(device_batches), idx, C.c_void_p(s.cuda_stream)), "gcs_b200_solve_many")


class DeviceBatch:
    """A batch resident in HBM as torch tensors (torch is only the allocator / stream owner)."""

    def __init__(self, host: HostBatch, device, want_cand=False, variant=None):
        import torch
        self.torch = torch
        self.device = torch.device(device)
        self.kind, self.n_seeds = host.kind, host.n_seeds
        self.variant = host.variant if variant is None else variant
        self.n = host.n
        dev = self.device
        self.cols = [None if c is None else torch.from_numpy(c).to(dev) for c in host.cols]
        self.code = torch.from_numpy(host.code).to(dev)
        self.guesses = None if host.guesses is None else torch.from_numpy(host.guesses).to(dev)
        n = self.n
        self.out = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(OUT_COLS[self.kind])]
        self.cand = torch.empty((self.n_seeds, 2, n), dtype=torch.float64, device=dev) if want_cand else None
        self.iters = torch.empty((self.n_seeds, n), dtype=torch.int16, device=dev)
        self.converged = torch.empty((self.n_seeds, n), dtype=torch.uint8, device=dev)
        self.root_index = torch.empty(n, dtype=torch.uint8, device=dev)
        self._cb = self._make_cbatch()

    @classmethod
    def empty(cls, kind, n_seeds, n, device, variant=VARIANT_DEFAULT, want_cand=False):
        """Uninitialised device-resident batch (columns to be filled on the device)."""
        import torch
        self = cls.__new__(cls)
        self.torch = torch
        self.device = torch.device(device)
        self.kind, self.n_seeds, self.variant, self.n = kind, n_seeds, variant, n
        dev = self.device
        self.cols = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(IN_COLS[kind])]
        self.code = torch.empty(n, dtype=torch.uint8, device=dev)
        self.guesses = None
        self.out = [torch.empty(n, dtype=torch.float64, device=dev) for _ in range(OUT_COLS[kind])]
        self.cand = torch.empty((n_seeds, 2, n), dtype=torch.float64, device=dev) if want_cand else None
        self.iters = torch.empty((n_seeds, n), dtype=torch.int16, device=dev)
        self.converged = torch.empty((n_seeds, n), dtype=torch.uint8, device=dev)
        self.root_index = torch.empty(n, dtype=torch.uint8, device=dev)
        self._cb = self._make_cbatch()
        return self

    def _make_cbatch(self):
        b = CBatch()
        b.kind, b.n_seeds, b.n, b.mem, b.variant = self.kind, self.n_seeds, self.n, MEM_DEVICE, self.variant
        for i, c in enumerate(self.cols):
            b.in_[i] = None if c is None else c.data_ptr()
        b.code = self.code.data_ptr()
        b.guesses = self.guesses.data_ptr() if self.guesses is not None else None
        for i, o in enumerate(self.out):
            b.out[i] = o.data_ptr()
        b.cand = self.cand.data_ptr() if self.cand is not None else None
        b.iters = self.iters.data_ptr()
        b.converged = self.converged.data_ptr()
        b.root_index = self.root_index.data_ptr()
        return b

    def set_variant(self, variant):
        self.variant = variant
        self._cb.variant = variant

    def solve(self, stream=None):
        """Enqueue gcs_b200_solve on `stream` (default: torch's current stream)."""
        torch = self.torch
        s = torch.cuda.current_stream(self.device) if stream is None else stream
        idx = self.device.index if self.device.index is not None else torch.cuda.current_device()
        check(load().gcs_b200_solve(C.byref(self._cb), idx, C.c_void_p(s.cuda_stream)), "gcs_b200_solve")

    def to_host(self, host: HostBatch) -> HostBatch:
        host.out = [o.cpu().numpy() for o in self.out]
        host.cand = self.cand.cpu().numpy() if self.cand is not None else None
        host.iters = self.iters.cpu().numpy()
        host.converged = self.converged.cpu().numpy()
        host.root_index = self.root_index.cpu().numpy()
        return host

    def algorithmic_bytes(self):
        """Minimum HBM traffic of one launch: inputs + code + outputs + per-seed flags."""
        n, ns = self.n, self.n_seeds
        b = sum(8 for c in self.cols if c is not None) + 1 + OUT_COLS[self.kind] * 8 + ns * 3 + 1
        if self.cand is not None:
            b += ns * 16
        if self.guesses is not None:
            b += ns * 16
        return n * b
