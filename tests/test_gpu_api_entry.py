"""The C ABI's entry points on the GPU: the kernel each (kind, seed count, variant) launches and how
launches are counted, the exact failure of every device-taking entry point for a device that is not
present and for malformed arguments, and that no entry point changes its caller's current device."""
import ctypes as C
import importlib
import os
import re
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
gcs = importlib.import_module("2d_geometry_constraint_solver_b200")
capi, synth = gcs.capi, gcs.synth

PP, SDD, PPL, PLL, ANG = capi.KIND_PP, capi.KIND_SDD, capi.KIND_PPL, capi.KIND_PLL, capi.KIND_ANG
VARIANTS = list(range(capi.VARIANT_CONTRACTED_LINEAR + 1))  # DEFAULT and every explicit variant
SEEDS = {PP: (2, 8), SDD: (2,), PPL: (2, 8), PLL: (2, 8), ANG: (2,)}  # K2 / K5 take 2 seeds only
N = 300  # small enough that DEFAULT picks the static kernel for every kind

# The kernel gcs_b200_solve launches for N sub-systems, by variant: {k} the kind, {s} the seed
# count, {t} the sorted kernel's tile (two runs per lane of 128).
KERNEL = {
    capi.VARIANT_DEFAULT: "newton_static_kernel<{k}, {s}, false>",
    capi.VARIANT_STATIC: "newton_static_kernel<{k}, {s}, false>",
    capi.VARIANT_REFILL: "newton_refill_kernel<{k}, {s}, 64, 4>",
    capi.VARIANT_SORTED: "newton_sorted_kernel<{k}, {s}, {t}, 128, false>",
    capi.VARIANT_PAIR: "newton_pair_kernel<{k}>",
    capi.VARIANT_CONTRACTED: "newton_static_kernel<{k}, {s}, true>",
    capi.VARIANT_CONTRACTED_STATIC: "newton_static_kernel<{k}, {s}, true>",
    capi.VARIANT_CONTRACTED_SORTED: "newton_sorted_kernel<{k}, {s}, {t}, 128, true>",
    capi.VARIANT_CONTRACTED_SEQ: "newton_seq_kernel<{k}, {s}, true>",
    capi.VARIANT_SEQ: "newton_seq_kernel<{k}, {s}, false>",
    capi.VARIANT_CONTRACTED_LINEAR: "newton_static_kernel<{k}, {s}, true>",
}
# where a kind or seed count launches another kernel: the pair kernel exists for 2 seeds only, the
# contracted K4 is the linear kernel, the contracted 8-seed K1 the seq kernel
KERNEL_EXCEPT = {
    (PP, 8, capi.VARIANT_PAIR): "newton_static_kernel<1, 8, false>",
    (PPL, 8, capi.VARIANT_PAIR): "newton_static_kernel<3, 8, false>",
    (PLL, 8, capi.VARIANT_PAIR): "newton_static_kernel<4, 8, false>",
    (PP, 8, capi.VARIANT_CONTRACTED): "newton_seq_kernel<1, 8, true>",
    (PP, 8, capi.VARIANT_CONTRACTED_LINEAR): "newton_seq_kernel<1, 8, true>",
    (PLL, 2, capi.VARIANT_CONTRACTED): "newton_linear_kernel<2>",
    (PLL, 8, capi.VARIANT_CONTRACTED): "newton_linear_kernel<8>",
    (PLL, 2, capi.VARIANT_CONTRACTED_LINEAR): "newton_linear_kernel<2>",
    (PLL, 8, capi.VARIANT_CONTRACTED_LINEAR): "newton_linear_kernel<8>",
}


def _expected_kernel(kind, seeds, variant):
    return KERNEL_EXCEPT.get((kind, seeds, variant)) or KERNEL[variant].format(k=kind, s=seeds, t=256 // seeds)


@pytest.fixture(scope="module")
def lib(gpu):
    return gpu.load()


def _host_batch(kind, n, seeds=2):
    return synth.make(kind, n, **({"n_seeds": seeds} if seeds != 2 else {})).alloc_outputs()


@pytest.mark.parametrize("kind", sorted(SEEDS))
def test_each_variant_launches_its_one_kernel(lib, kind):
    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    cases = [(s, v) for s in SEEDS[kind] for v in VARIANTS]
    batches = {s: capi.DeviceBatch(_host_batch(kind, N, s), "cuda:0") for s in SEEDS[kind]}
    stream = torch.cuda.current_stream(0)
    torch.cuda.synchronize()
    counted = []
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for s, v in cases:
            batches[s].set_variant(v)
            before = lib.gcs_b200_launch_count()
            batches[s].solve(stream)
            counted.append(lib.gcs_b200_launch_count() - before)
        torch.cuda.synchronize()
    kernels = [e.name for e in sorted(prof.events(), key=lambda e: e.time_range.start)
               if e.device_type == DeviceType.CUDA and not e.name.startswith(("Memcpy", "Memset"))]
    launched = [m.group(0) if (m := re.search(r"newton_\w+_kernel<[^>]*>", name)) else name for name in kernels]
    assert counted == [1] * len(cases)
    assert launched == [_expected_kernel(kind, s, v) for s, v in cases]


def test_launch_count_of_an_empty_batch_the_selftest_and_the_generator(lib):
    import torch

    empty = _empty_batch(capi.MEM_DEVICE)
    before = lib.gcs_b200_launch_count()
    assert lib.gcs_b200_solve(C.byref(empty), 0, None) == 0, lib.gcs_b200_last_error()
    assert lib.gcs_b200_launch_count() == before

    counts = (C.c_uint64 * 8)()
    before = lib.gcs_b200_launch_count()
    assert lib.gcs_b200_selftest(0, 1, 1 << 12, counts) == 0, lib.gcs_b200_last_error()
    assert lib.gcs_b200_launch_count() == before + 1

    db = capi.DeviceBatch.empty(PP, 2, 4096, "cuda:0")
    cols = (C.c_void_p * 6)(*[c.data_ptr() for c in db.cols])
    stream = torch.cuda.current_stream(0)
    before = lib.gcs_b200_launch_count()
    rc = lib.gcs_b200_synth_pp(0, C.c_void_p(stream.cuda_stream), synth.BASE_SEED, 0, 4096, 0, cols, C.c_void_p(db.code.data_ptr()))
    assert rc == 0, lib.gcs_b200_last_error()
    assert lib.gcs_b200_launch_count() == before + 1
    torch.cuda.synchronize()


# ---- argument errors -------------------------------------------------------------------------

def _empty_batch(mem):
    b = capi.CBatch()
    b.kind, b.n_seeds, b.n, b.mem = PP, 2, 0, mem
    return b


def _tiny_program():
    """One wave with one K1 row (solver 1, the zero-fixed triangle) over point slots 0 .. 2 and
    length values 0 .. 2.  Returns (descriptor, the arrays it points into)."""
    row = capi.CProgramRow()
    row.solver, row.code = 1, 6
    row.elem[:] = [0, 1, 2]
    row.value[:] = [0, 1, 2]
    row.sign[:] = [1.0, 1.0, 1.0]
    keep = [(capi.CProgramRow * 1)(row), (C.c_int64 * 6)(0, 1, 1, 1, 1, 1), (C.c_uint8 * 3)(), (C.c_double * 12)(),
            (C.c_uint8 * 3)()]
    d = capi.CProgramDesc()
    d.n_waves, d.n_slots, d.n_values, d.n_rows = 1, 3, 3, 1
    d.rows = C.cast(keep[0], C.POINTER(capi.CProgramRow))
    d.offsets = C.cast(keep[1], C.POINTER(C.c_int64))
    d.slot_is_line = C.cast(keep[2], C.POINTER(C.c_uint8))
    d.initial = C.cast(keep[3], C.POINTER(C.c_double))
    d.value_is_angle = C.cast(keep[4], C.POINTER(C.c_uint8))
    return d, keep


class _Args:
    """What the argument-error cases call with."""

    def __init__(self, lib):
        self.lib = lib
        self.absent = lib.gcs_b200_device_count()  # the first ordinal that is not present
        self.dev0 = _empty_batch(capi.MEM_DEVICE)
        self.host0 = _empty_batch(capi.MEM_HOST)
        self.hb = _host_batch(PP, 10)
        self.host10 = self.hb.cbatch()
        self.desc, self._keep = _tiny_program()
        self.prog = C.c_void_p()
        self.values = (C.c_double * 3)(3.0, 4.0, 5.0)
        self.positions = (C.c_double * 12)()
        self.cols = (C.c_void_p * 6)(*[1] * 6)  # never dereferenced: every case fails before
        self.out4 = (C.c_double * 4)()
        self.counts = (C.c_uint64 * 8)()

    def with_fields(self, b, **fields):
        c = capi.CBatch.from_buffer_copy(b)
        for k, v in fields.items():
            setattr(c, k, v)
        return c

    def without_column(self, b, col):
        c = capi.CBatch.from_buffer_copy(b)
        c.in_[col] = None
        return c

    def pair(self, b):
        return (C.POINTER(capi.CBatch) * 2)(C.pointer(b), C.pointer(b))


ABSENT = "device {absent} not present"
OUT_OF_RANGE = "device {absent} out of range ({absent} present)"
E_INVALID, E_NO_DEVICE = capi.GCS_E_INVALID, capi.GCS_E_NO_DEVICE

# (id, call, code, gcs_b200_last_error())
ERRORS = [
    ("init-absent", lambda a: a.lib.gcs_b200_init(1, (C.c_int * 1)(a.absent)), E_NO_DEVICE, OUT_OF_RANGE),
    ("init-twice", lambda a: a.lib.gcs_b200_init(2, (C.c_int * 2)(0, 0)), E_INVALID, "device 0 listed twice"),
    ("solve-absent", lambda a: a.lib.gcs_b200_solve(C.byref(a.dev0), a.absent, None), E_NO_DEVICE, ABSENT),
    ("solve-null", lambda a: a.lib.gcs_b200_solve(None, 0, None), E_INVALID, "null batch"),
    ("solve-host-memory", lambda a: a.lib.gcs_b200_solve(C.byref(a.host0), 0, None), E_INVALID,
     "gcs_b200_solve needs device pointers (mem=GCS_MEM_DEVICE)"),
    ("solve-kind", lambda a: a.lib.gcs_b200_solve(C.byref(a.with_fields(a.dev0, kind=9)), 0, None), E_INVALID, "unknown kind 9"),
    ("solve-n", lambda a: a.lib.gcs_b200_solve(C.byref(a.with_fields(a.dev0, n=-1)), 0, None), E_INVALID, "negative n"),
    ("solve-variant", lambda a: a.lib.gcs_b200_solve(C.byref(a.with_fields(a.dev0, variant=11)), 0, None), E_INVALID,
     "unknown variant 11"),
    ("solve-guess-seeds", lambda a: a.lib.gcs_b200_solve(C.byref(a.with_fields(a.dev0, kind=SDD, n_seeds=8)), 0, None), E_INVALID,
     "kind 2 takes exactly 2 seeds"),
    ("solve-seeds", lambda a: a.lib.gcs_b200_solve(C.byref(a.with_fields(a.dev0, n_seeds=3)), 0, None), E_INVALID,
     "n_seeds must be 2 or 8 (got 3)"),
    ("solve-column", lambda a: a.lib.gcs_b200_solve(C.byref(a.without_column(a.host10, 2)), 0, None), E_INVALID,
     "input column 2 of kind 1 is null (only the anchor columns may be)"),
    ("solve-code", lambda a: a.lib.gcs_b200_solve(C.byref(a.with_fields(a.host10, code=None)), 0, None), E_INVALID,
     "code column is null"),
    ("solve_many-absent", lambda a: a.lib.gcs_b200_solve_many(a.pair(a.dev0), 2, a.absent, None), E_NO_DEVICE, ABSENT),
    ("solve_many-list", lambda a: a.lib.gcs_b200_solve_many(None, 2, 0, None), E_INVALID, "bad batch list"),
    ("solve_many-host-memory", lambda a: a.lib.gcs_b200_solve_many(a.pair(a.host0), 2, 0, None), E_INVALID,
     "gcs_b200_solve_many needs device pointers (batch 0)"),
    ("solve_host-absent", lambda a: a.lib.gcs_b200_solve_host(C.byref(a.host0), a.absent), E_NO_DEVICE, ABSENT),
    ("solve_host-device-memory", lambda a: a.lib.gcs_b200_solve_host(C.byref(a.dev0), 0), E_INVALID,
     "this entry point needs host pointers (mem=GCS_MEM_HOST)"),
    ("solve_host_async-absent", lambda a: a.lib.gcs_b200_solve_host_async(C.byref(a.host0), a.absent), E_NO_DEVICE, ABSENT),
    ("solve_host_async-null", lambda a: a.lib.gcs_b200_solve_host_async(None, 0), E_INVALID, "null batch"),
    ("solve_host_range_async-absent", lambda a: a.lib.gcs_b200_solve_host_range_async(C.byref(a.host0), a.absent, 0, 0), E_NO_DEVICE,
     ABSENT),
    ("solve_host_range_async-range", lambda a: a.lib.gcs_b200_solve_host_range_async(C.byref(a.host10), 0, 5, 20), E_INVALID,
     "index range [5, 25) outside the batch of 10"),
    ("wait-absent", lambda a: a.lib.gcs_b200_wait(a.absent), E_NO_DEVICE, ABSENT),
    ("solve_sharded-device-memory", lambda a: a.lib.gcs_b200_solve_sharded(C.byref(a.dev0), 1), E_INVALID,
     "gcs_b200_solve_sharded needs host pointers"),
    ("contracted_stats-absent", lambda a: a.lib.gcs_b200_contracted_stats(a.absent, None, 0), E_NO_DEVICE, ABSENT),
    ("contracted_stats_ex-absent", lambda a: a.lib.gcs_b200_contracted_stats_ex(a.absent, None, 0), E_NO_DEVICE, ABSENT),
    ("debug_path_buffer-absent", lambda a: a.lib.gcs_b200_debug_path_buffer(a.absent, None, 0), E_NO_DEVICE, ABSENT),
    ("debug_path_buffer-capacity", lambda a: a.lib.gcs_b200_debug_path_buffer(0, None, -1), E_INVALID, "negative capacity"),
    ("fp64_probe-absent", lambda a: a.lib.gcs_b200_fp64_probe(a.absent, 2), E_NO_DEVICE, ABSENT),
    ("fp64_probe-warps", lambda a: a.lib.gcs_b200_fp64_probe(0, 1100), E_INVALID, "probe: warps per SM must be 1..32"),
    ("pcie_probe-absent", lambda a: a.lib.gcs_b200_pcie_probe(a.absent, 4096, 4096, 1, 0, 1, a.out4), E_NO_DEVICE, ABSENT),
    ("pcie_probe-arguments", lambda a: a.lib.gcs_b200_pcie_probe(0, 0, 4096, 1, 0, 1, a.out4), E_INVALID, "bad probe arguments"),
    ("selftest-absent", lambda a: a.lib.gcs_b200_selftest(a.absent, 1, 16, a.counts), E_NO_DEVICE, ABSENT),
    ("selftest-arguments", lambda a: a.lib.gcs_b200_selftest(0, 1, -1, a.counts), E_INVALID, "bad selftest arguments"),
    ("synth_pp-absent", lambda a: a.lib.gcs_b200_synth_pp(a.absent, None, 1, 0, 16, 0, a.cols, C.c_void_p(1)), E_NO_DEVICE, ABSENT),
    ("synth_pp-arguments", lambda a: a.lib.gcs_b200_synth_pp(0, None, 1, 0, -1, 0, a.cols, C.c_void_p(1)), E_INVALID,
     "bad synth arguments"),
    ("synth_pp-column", lambda a: a.lib.gcs_b200_synth_pp(0, None, 1, 0, 16, 0, (C.c_void_p * 6)(1, 1, 1, None, 1, 1), C.c_void_p(1)),
     E_INVALID, "synth column 3 is null"),
    ("program_create-absent", lambda a: a.lib.gcs_b200_program_create(C.byref(a.desc), a.absent, C.byref(a.prog)), E_NO_DEVICE,
     OUT_OF_RANGE),
    ("program_create-null", lambda a: a.lib.gcs_b200_program_create(None, 0, C.byref(a.prog)), E_INVALID, "null program descriptor"),
    ("program_create-handle", lambda a: a.lib.gcs_b200_program_create(C.byref(a.desc), 0, None), E_INVALID, "null output handle"),
    ("program_run-null", lambda a: a.lib.gcs_b200_program_run(None, 1, a.values, a.positions, None, 0, None), E_INVALID,
     "null program"),
    ("program_run_host-null", lambda a: a.lib.gcs_b200_program_run_host(None, 1, a.values, a.positions, None, 0, None), E_INVALID,
     "null program"),
    ("program_run_tangents-directions", lambda a: a.lib.gcs_b200_program_run_tangents(None, 1, a.values, a.positions, None, 0, None,
                                                                                       None, 0, None), E_INVALID,
     "n_tangents must be >= 1 (got 0)"),
    ("program_run_tangents_host-variant", lambda a: a.lib.gcs_b200_program_run_tangents_host(None, 1, a.values, a.positions, None, 1,
                                                                                             a.values, a.positions, 11, None),
     E_INVALID, "unknown variant 11"),
    ("program_run_recorded-null", lambda a: a.lib.gcs_b200_program_run_recorded(None, 1, a.values, a.positions, None, 0, None),
     E_INVALID, "null program"),
    ("program_run_recorded_host-null", lambda a: a.lib.gcs_b200_program_run_recorded_host(None, 1, a.values, a.positions, None, 0,
                                                                                           None), E_INVALID, "null program"),
    ("program_adjoints-cotangents", lambda a: a.lib.gcs_b200_program_adjoints(None, 0, a.positions, a.values, None), E_INVALID,
     "n_cotangents must be >= 1 (got 0)"),
    ("program_adjoints_host-null", lambda a: a.lib.gcs_b200_program_adjoints_host(None, 1, a.positions, a.values, None), E_INVALID,
     "null program"),
]


@pytest.mark.parametrize("call,code,text", [e[1:] for e in ERRORS], ids=[e[0] for e in ERRORS])
def test_argument_errors(lib, call, code, text):
    a = _Args(lib)
    assert call(a) == code
    assert lib.gcs_b200_last_error().decode() == text.format(absent=a.absent)


def test_argument_errors_of_a_program(lib):
    a = _Args(lib)
    assert lib.gcs_b200_program_create(C.byref(a.desc), 0, C.byref(a.prog)) == 0, lib.gcs_b200_last_error()
    try:
        cases = [
            (lambda: lib.gcs_b200_program_run(a.prog, 0, a.values, a.positions, None, 0, None), "n_instances must be >= 1 (got 0)"),
            (lambda: lib.gcs_b200_program_run_host(a.prog, 1, None, a.positions, None, 0, None), "null value or position table"),
            (lambda: lib.gcs_b200_program_run_recorded(a.prog, 1, a.values, a.positions, None, 11, None), "unknown variant 11"),
            (lambda: lib.gcs_b200_program_run_tangents(a.prog, 1, a.values, a.positions, None, 1, None, a.positions, 0, None),
             "null tangent table (dvalues or dpositions)"),
            (lambda: lib.gcs_b200_program_adjoints(a.prog, 1, a.positions, a.values, None),
             "no recorded run: call gcs_b200_program_run_recorded first"),
            (lambda: lib.gcs_b200_program_adjoints_host(a.prog, 1, None, a.values, None), "null adjoint table (adj_positions or adj_values)"),
        ]
        for call, text in cases:
            assert call() == E_INVALID
            assert lib.gcs_b200_last_error().decode() == text
    finally:
        lib.gcs_b200_program_destroy(a.prog)


# ---- the caller's device ------------------------------------------------------------------------
# Each case runs in a fresh process, so that every device is used for the first time by the case's
# first call.  Device 0 is current throughout; the calls work on device 1.

def _runtime():
    rt = C.CDLL("libcudart.so.12")  # the runtime libgcs_b200.so loaded
    rt.cudaMalloc.argtypes = [C.POINTER(C.c_void_p), C.c_size_t]
    rt.cudaMemcpy.argtypes = [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int]
    return rt


def _device_alloc(rt, device, nbytes, src=None):
    """cudaMalloc on `device` (filled from host address `src`), device 0 current again afterwards."""
    assert rt.cudaSetDevice(device) == 0
    d = C.c_void_p()
    assert rt.cudaMalloc(C.byref(d), nbytes) == 0
    if src:
        assert rt.cudaMemcpy(d, src, nbytes, 1) == 0
    assert rt.cudaSetDevice(0) == 0
    return d.value


def _device_batch(rt, device, kind, n):
    hb = _host_batch(kind, n)
    cb = hb.cbatch()
    for c in range(capi.IN_COLS[kind]):
        cb.in_[c] = _device_alloc(rt, device, 8 * n, cb.in_[c])
    cb.code = _device_alloc(rt, device, n, cb.code)
    for c in range(capi.OUT_COLS[kind]):
        cb.out[c] = _device_alloc(rt, device, 8 * n)
    cb.cand = None
    cb.iters, cb.converged = _device_alloc(rt, device, 2 * 2 * n), _device_alloc(rt, device, 2 * n)
    cb.root_index = _device_alloc(rt, device, n)
    cb.mem = capi.MEM_DEVICE
    return cb


def _synchronize(rt, device):
    assert rt.cudaSetDevice(device) == 0
    assert rt.cudaDeviceSynchronize() == 0
    assert rt.cudaSetDevice(0) == 0


def _case_init_1_0(lib, rt):
    yield "gcs_b200_init([1, 0])", lib.gcs_b200_init(2, (C.c_int * 2)(1, 0))


def _case_init_0_1(lib, rt):
    yield "gcs_b200_init([0, 1])", lib.gcs_b200_init(2, (C.c_int * 2)(0, 1))


def _case_solve(lib, rt):
    a, b = _device_batch(rt, 1, PP, 4096), _device_batch(rt, 1, PPL, 4096)
    yield "gcs_b200_solve", lib.gcs_b200_solve(C.byref(a), 1, None)
    yield "gcs_b200_solve_many", lib.gcs_b200_solve_many((C.POINTER(capi.CBatch) * 2)(C.pointer(a), C.pointer(b)), 2, 1, None)
    _synchronize(rt, 1)


def _case_host(lib, rt):
    hb = _host_batch(PP, 4096)
    cb = hb.cbatch()
    yield "gcs_b200_solve_host", lib.gcs_b200_solve_host(C.byref(cb), 1)
    yield "gcs_b200_solve_host_async", lib.gcs_b200_solve_host_async(C.byref(cb), 1)
    yield "gcs_b200_wait", lib.gcs_b200_wait(1)
    yield "gcs_b200_solve_host_range_async", lib.gcs_b200_solve_host_range_async(C.byref(cb), 1, 0, 2048)
    yield "gcs_b200_wait", lib.gcs_b200_wait(1)
    yield "gcs_b200_pcie_probe", lib.gcs_b200_pcie_probe(1, 1 << 20, 1 << 20, 1, 0, 1, (C.c_double * 4)())


def _case_selftest(lib, rt):
    yield "gcs_b200_selftest", lib.gcs_b200_selftest(1, 1, 1 << 12, (C.c_uint64 * 8)())


def _case_fp64_probe(lib, rt):
    cycles = lib.gcs_b200_fp64_probe(1, 2)
    yield "gcs_b200_fp64_probe", 0 if cycles > 0 else cycles


def _case_contracted_stats_ex(lib, rt):
    yield "gcs_b200_contracted_stats_ex", lib.gcs_b200_contracted_stats_ex(1, (C.c_uint64 * 8)(), 0)


def _case_synth_pp(lib, rt):
    cols = (C.c_void_p * 6)(*[_device_alloc(rt, 1, 8 * 4096) for _ in range(6)])
    yield "gcs_b200_synth_pp", lib.gcs_b200_synth_pp(1, None, 1, 0, 4096, 0, cols, _device_alloc(rt, 1, 4096))
    _synchronize(rt, 1)


def _case_program(lib, rt):
    desc, keep = _tiny_program()
    prog = C.c_void_p()
    values, positions, nonconverged = (C.c_double * 3)(3.0, 4.0, 5.0), (C.c_double * 12)(), (C.c_uint32 * 1)()
    yield "gcs_b200_program_create", lib.gcs_b200_program_create(C.byref(desc), 1, C.byref(prog))
    yield "gcs_b200_program_run_host", lib.gcs_b200_program_run_host(prog, 1, values, positions, nonconverged, 0, None)
    lib.gcs_b200_program_destroy(prog)
    yield "gcs_b200_program_destroy", 0


def _case_shutdown(lib, rt):
    hb = _host_batch(PP, 4096)
    yield "gcs_b200_init([0, 1])", lib.gcs_b200_init(2, (C.c_int * 2)(0, 1))
    yield "gcs_b200_solve_host", lib.gcs_b200_solve_host(C.byref(hb.cbatch()), 1)
    lib.gcs_b200_shutdown()
    yield "gcs_b200_shutdown", 0


CASES = {name[len("_case_"):]: f for name, f in globals().items() if name.startswith("_case_")}


def run_case(name):
    """The body of one case's process: every call must succeed and leave device 0 current."""
    lib = capi.load()
    rt = _runtime()
    current = C.c_int(-1)
    assert rt.cudaSetDevice(0) == 0
    for what, rc in CASES[name](lib, rt):
        assert rc == 0, f"{what}: {rc} {lib.gcs_b200_last_error().decode()}"
        assert rt.cudaGetDevice(C.byref(current)) == 0
        assert current.value == 0, f"{what} left device {current.value} current"


@pytest.mark.parametrize("case", sorted(CASES))
def test_entry_points_leave_the_callers_device_current(lib, case):
    if lib.gcs_b200_device_count() < 2:
        pytest.skip("needs two visible CUDA devices")
    child = (f"import sys; sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, 'tests')!r}]; "
             "import test_gpu_api_entry as T; T.run_case(sys.argv[1])")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", child, case], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                       timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stdout[-4000:]
