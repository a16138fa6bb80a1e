"""Fused sketch-program runs on the GPU (gcs_b200_program_run_fused[_host], SketchProgram::runFused):
every wave in one cooperative launch.  Every comparison is against the wave-by-wave run
(gcs_b200_program_run / _run_tangents with GCS_VARIANT_DEFAULT), bit for bit, NaN with NaN, with the
nonconverged counts equal."""
import ctypes as C

import numpy as np
import pytest

import host_lib as H
import program_restate as R
import program_tangents_lib as PT
import sketch_gen as S
from host_lib import _dp
from test_gpu_host import WHOLE_SKETCHES
from test_gpu_sketch_program_abi import Prog, _directions, _same, _values

pytestmark = pytest.mark.gpu

SEEDS = [s for s, _, _ in WHOLE_SKETCHES]
GCS_E_INVALID = -1


@pytest.fixture(scope="module")
def lib(gpu, built):
    built.build_host()
    return gpu.load()


@pytest.fixture(scope="module")
def golden(lib):
    """{seed: (Arrays of the leaf-list program of a golden sketch, its values in radians)}"""
    out = {}
    for seed, first, n in WHOLE_SKETCHES:
        el, lv = S.make_sketch(n, seed=seed, first_shape=first)
        prog = PT.Program(el, leaves=lv)
        assert prog.rc == 0, prog.error
        out[seed] = (R.Arrays.from_desc(prog.desc()), np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT]))
    return out


@pytest.fixture(scope="module")
def linkages(lib):
    """{name: (Arrays, values in radians)} of the 20 k linkage and the 100 k one (configs[3])"""
    out = {}
    for name, n, seed in (("linkage20k", 20000, 6), ("linkage100k", 100000, 4)):
        el, edges = S.make_linkage(n, seed=seed)
        prog = PT.Program(el, edges)
        assert prog.rc == 0, prog.error
        out[name] = (R.Arrays.from_desc(prog.desc()), PT.sketch_values(edges))
    return out


class FProg(Prog):
    """Prog plus the fused entry points."""

    def run_fused_host(self, vals, dvals=None, counts=True):
        """gcs_b200_program_run_fused_host: (positions, tangents or None, nonconverged or None, launches)"""
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        K = vals.shape[0]
        T = 0 if dvals is None else dvals.shape[2]
        pos = np.zeros((K, self.arrays.n_slots, 4))
        dpos = np.zeros((K, self.arrays.n_slots, 4, T)) if T else None
        dv = np.ascontiguousarray(dvals, dtype=np.float64) if T else None
        nc = np.zeros(K, dtype=np.uint32) if counts else None
        before = self.lib.gcs_b200_launch_count()
        rc = self.lib.gcs_b200_program_run_fused_host(self.h, K, vals.ctypes.data, pos.ctypes.data, nc.ctypes.data if counts else None, T,
                                                      dv.ctypes.data if T else None, dpos.ctypes.data if T else None, None)
        assert rc == 0, self.lib.gcs_b200_last_error()
        return pos, dpos, nc, self.lib.gcs_b200_launch_count() - before

    def run_fused(self, vals, pos, nc=None, dvals=None, dpos=None, stream=None):
        """gcs_b200_program_run_fused on torch tensors, enqueued on `stream` (None: the NULL stream); no synchronisation."""
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        T = 0 if dvals is None else dvals.shape[2]
        rc = self.lib.gcs_b200_program_run_fused(self.h, vals.shape[0], ptr(vals), ptr(pos), ptr(nc), T, ptr(dvals), ptr(dpos),
                                                 None if stream is None else stream.cuda_stream)
        assert rc == 0, self.lib.gcs_b200_last_error()


def _check(lib, p, vals, dvals=None, what=""):
    """fused against the wave run: positions, counts and tangents; returns the wave run's.  The two runs
    use two programs made from the same arrays, so the fused run's _host tables never already hold the
    wave run's answer: a fused run that wrote nothing could not pass."""
    with FProg(lib, p) as waves, FProg(lib, p) as fused:
        want, dwant, wnc, _ = waves.run_host(vals, dvals)
        got, dgot, nc, launches = fused.run_fused_host(vals, dvals)
    assert launches == 1, what
    assert _same(got, want) and np.array_equal(nc, wnc), what
    assert dvals is None or _same(dgot, dwant), what
    return want, dwant, wnc


# ---- 1. plain runs ----

@pytest.mark.parametrize("unrealisable", [0.0, 0.25])
@pytest.mark.parametrize("K", [1, 33])
@pytest.mark.parametrize("seed", SEEDS)
def test_fused_equals_the_wave_run_on_the_golden_sketches(lib, golden, seed, K, unrealisable):
    p, base = golden[seed]
    vals, bad = _values(p, base, K, seed=seed + K, unrealisable=unrealisable)
    _, _, nc = _check(lib, p, vals)
    assert len(bad) == 0 or nc[bad].min() > 0  # the unrealisable sets leave rows unsolved


@pytest.mark.parametrize("seed", SEEDS)
def test_fused_equals_the_wave_run_on_every_wave_layout(lib, golden, seed):
    """R.transforms (per-kind waves, one row per wave, empty waves, reversed segments) and programs
    without rows, plain and with T = 3"""
    p, base = golden[seed]
    K = 33
    vals, _ = _values(p, base, K, seed=seed + 5, unrealisable=0.1)
    dvals = _directions(p, K, 3, seed=seed + 6)
    layouts = list(R.transforms(p)) + [("no_rows_0", R.without_rows(p, 0)), ("no_rows_3", R.without_rows(p, 3))]
    for name, q in layouts:
        _check(lib, q, vals, what=name)
        _check(lib, q, vals, dvals, what=name)


@pytest.mark.parametrize("e", [-40, 40])
@pytest.mark.parametrize("seed", SEEDS)
def test_fused_equals_the_wave_run_at_scale(lib, golden, seed, e):
    """every length value and initial position x 2^e"""
    p0, base = golden[seed]
    angle = p0.value_is_angle.astype(bool)
    p = R.Arrays(p0.rows, p0.offsets, p0.slot_is_line, np.ldexp(p0.initial, e), p0.value_is_angle)
    vals, _ = _values(p, base, 4, seed=seed)
    vals = np.where(angle[None, :], vals, np.ldexp(vals, e))
    _check(lib, p, vals, what=f"2^{e}")
    _check(lib, p, vals, _directions(p, 4, 2, seed=seed + 1), what=f"2^{e}")


@pytest.mark.parametrize("case", [("linkage20k", 1), ("linkage20k", 16), ("linkage20k", 257), ("linkage100k", 1)])
def test_fused_equals_the_wave_run_on_the_linkages(lib, linkages, case):
    name, K = case
    p, base = linkages[name]
    vals, _ = _values(p, base, K, seed=K)
    _check(lib, p, vals, what=name)


# ---- 2. waves larger than the grid ----

def test_waves_larger_than_the_grid_are_grid_strided(lib, golden):
    """K such that the largest wave has at least 4x the threads the device can hold at all (2048 per
    SM), so at least 4x the fused grid's threads: plain and T = 1"""
    import torch
    p, base = golden[31]
    widest = max(int(p.offsets[R.KINDS * (w + 1)] - p.offsets[R.KINDS * w]) for w in range(p.n_waves))
    K = -(-4 * torch.cuda.get_device_properties(0).multi_processor_count * 2048 // widest)
    vals, _ = _values(p, base, K, seed=7, unrealisable=0.01)
    print(f"largest wave {widest} rows, K = {K}: {widest * K} sub-systems")
    _check(lib, p, vals)
    _check(lib, p, vals, _directions(p, K, 1, seed=8))


# ---- 3. tangent runs ----

@pytest.mark.parametrize("T", [1, 8, 32])
@pytest.mark.parametrize("K", [1, 33])
@pytest.mark.parametrize("seed", SEEDS)
def test_fused_tangents_equal_the_wave_run(lib, golden, seed, K, T):
    """at K = 33 a quarter of the value sets is unrealisable: NaN tangents downstream of unsolved rows"""
    p, base = golden[seed]
    vals, bad = _values(p, base, K, seed=seed + T, unrealisable=0.25 if K > 1 else 0.0)
    dvals = _directions(p, K, T, seed=seed + 2 * T)
    _, dwant, _ = _check(lib, p, vals, dvals)
    assert len(bad) == 0 or np.isnan(dwant[bad]).any()


# ---- 4. instances are independent ----

def test_each_instance_equals_a_one_instance_fused_run(lib, golden):
    p, base = golden[32]
    K = 9
    vals, _ = _values(p, base, K, seed=3, unrealisable=0.25)
    dvals = _directions(p, K, 2, seed=4)
    with FProg(lib, p) as many, FProg(lib, p) as single:
        pos, dpos, nc, _ = many.run_fused_host(vals, dvals)
        for k in range(K):
            one, done, onc, _ = single.run_fused_host(vals[k:k + 1], dvals[k:k + 1])
            assert _same(one[0], pos[k]) and _same(done[0], dpos[k]) and onc[0] == nc[k], k


# ---- 5. one launch, no copies ----

def profile_fused_runs():
    """The body of test_a_fused_run_is_one_launch_and_no_copy's process.  Prints one JSON line: the
    launch-count increase of every device and _host fused run, and the device activity of a
    torch.profiler session over the device runs, in start order."""
    import json

    import torch
    from torch.autograd import DeviceType
    from torch.profiler import ProfilerActivity, profile

    import importlib
    capi = importlib.import_module("2d_geometry_constraint_solver_b200").capi
    capi.init([0])
    lib = capi.load()
    seed, first, n = [c for c in WHOLE_SKETCHES if c[0] == 33][0]
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    prog_h = PT.Program(el, leaves=lv)
    p = R.Arrays.from_desc(prog_h.desc())
    base = np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])
    dev = torch.device("cuda", 0)
    out = {"device": [], "host": [], "events": []}
    with FProg(lib, p) as prog:
        cases = []
        for K in (1, 33, 4096):
            for T in (0, 2):
                vals, _ = _values(p, base, K, seed=K)
                dvals = _directions(p, K, T, seed=T) if T else None
                tables = (torch.from_numpy(vals).to(dev), torch.empty((K, p.n_slots, 4), dtype=torch.float64, device=dev),
                          torch.empty(K, dtype=torch.int32, device=dev), torch.from_numpy(dvals).to(dev) if T else None,
                          torch.empty((K, p.n_slots, 4, T), dtype=torch.float64, device=dev) if T else None)
                prog.run_fused(*tables)  # warm-up, on the NULL stream
                torch.cuda.synchronize()  # runs of one program must not overlap: the _host run uses the program's stream
                before = lib.gcs_b200_launch_count()
                prog.run_fused_host(vals, dvals)
                out["host"].append(lib.gcs_b200_launch_count() - before)
                cases.append(tables)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for tables in cases:
                before = lib.gcs_b200_launch_count()
                prog.run_fused(*tables)
                out["device"].append(lib.gcs_b200_launch_count() - before)
                torch.cuda.synchronize()  # one run after the other, each alone on the device
    events = sorted((e for e in prof.events() if e.device_type == DeviceType.CUDA), key=lambda e: e.time_range.start)
    out["events"] = [e.name for e in events]
    print(json.dumps(out))


def test_a_fused_run_is_one_launch_and_no_copy(lib):
    """In a process of its own (no earlier profiler session or other test's work shares it), K = 1, 33,
    4096 and T = 0, 2: the launch count rises by exactly 1 per fused run, through the device and the
    _host entry point.  Under torch.profiler, the device entry point's runs show one
    program_fused_kernel each, and no memcpy, memset or other kernel between the first and the last."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    child = (f"import sys; sys.path[:0] = [{root!r}, {os.path.join(root, 'tests')!r}]; "
             "import test_gpu_sketch_program_fused as T; T.profile_fused_runs()")
    flags = ["-s"] if sys.flags.no_user_site else []
    r = subprocess.run([sys.executable, *flags, "-c", child], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600,
                       cwd=root)
    assert r.returncode == 0, (r.stdout[-2000:], r.stderr[-4000:])
    out = json.loads(r.stdout.strip().splitlines()[-1])
    assert out["device"] == [1] * 6 and out["host"] == [1] * 6, out
    fused = [i for i, name in enumerate(out["events"]) if "program_fused_kernel" in name]
    assert len(fused) == 6, out["events"]
    window = out["events"][fused[0]:fused[-1] + 1]
    assert all("program_fused_kernel" in name for name in window), window


# ---- 6. the caller's stream and device ----

@pytest.mark.parametrize("T", [0, 2])
def test_a_fused_run_is_ordered_on_the_callers_stream(lib, golden, T):
    """On a side stream: the values are NaN, then a sleep of about 50 ms, then the real values are
    written, the program runs, and its results are cloned and overwritten with NaN.  The clones equal the
    wave run: the launch started after the values were written and ended before the clones."""
    import torch
    p, base = golden[32]
    K = 33
    vals, _ = _values(p, base, K, seed=5)
    dvals = _directions(p, K, T, seed=6) if T else None
    s = torch.cuda.Stream(device=0)
    dev = torch.device("cuda", 0)
    real = torch.from_numpy(vals).to(dev)
    dv = torch.from_numpy(dvals).to(dev) if T else None
    v = torch.empty_like(real)
    pos = torch.empty((K, p.n_slots, 4), dtype=torch.float64, device=dev)
    dpos = torch.empty((K, p.n_slots, 4, T), dtype=torch.float64, device=dev) if T else None
    nc = torch.empty(K, dtype=torch.int32, device=dev)
    with FProg(lib, p) as prog:
        want, dwant, wnc, _ = prog.run_host(vals, dvals)
        torch.cuda.synchronize()
        with torch.cuda.stream(s):
            v.fill_(float("nan"))
            torch.cuda._sleep(100_000_000)
            v.copy_(real)
            prog.run_fused(v, pos, nc, dv, dpos, stream=s)
            still_running = not s.query()
            got, gnc = pos.clone(), nc.clone()
            dgot = dpos.clone() if T else None
            pos.fill_(float("nan"))
        s.synchronize()
    assert still_running, "the run synchronised its stream"
    assert _same(got.cpu().numpy(), want) and np.array_equal(gnc.cpu().numpy().astype(np.uint32), wnc)
    assert T == 0 or _same(dgot.cpu().numpy(), dwant)
    assert torch.isnan(pos).all()


def test_a_fused_run_on_another_device_keeps_the_callers_device(lib, golden):
    import torch
    if lib.gcs_b200_device_count() < 2:
        pytest.skip("one device visible")
    p, base = golden[33]
    vals, _ = _values(p, base, 9, seed=3)
    dvals = _directions(p, 9, 2, seed=4)
    with FProg(lib, p, device=0) as p0:
        want, dwant, wnc, _ = p0.run_host(vals, dvals)
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 1)
    with FProg(lib, p, device=1) as p1:
        v, dv = torch.from_numpy(vals).to(dev), torch.from_numpy(dvals).to(dev)
        pos = torch.empty((9, p.n_slots, 4), dtype=torch.float64, device=dev)
        dpos = torch.empty((9, p.n_slots, 4, 2), dtype=torch.float64, device=dev)
        nc = torch.empty(9, dtype=torch.int32, device=dev)
        p1.run_fused(v, pos, nc, dv, dpos, stream=torch.cuda.Stream(device=1))
        assert torch.cuda.current_device() == 0
        torch.cuda.synchronize(dev)
        hpos, hdpos, hnc, _ = p1.run_fused_host(vals, dvals)
        assert torch.cuda.current_device() == 0
    assert _same(pos.cpu().numpy(), want) and _same(dpos.cpu().numpy(), dwant)
    assert np.array_equal(nc.cpu().numpy().astype(np.uint32), wnc)
    assert _same(hpos, want) and _same(hdpos, dwant) and np.array_equal(hnc, wnc)


# ---- 7. the tape and the batch buffers are left alone ----

def test_a_fused_run_leaves_a_recorded_run_and_later_wave_runs_alone(lib, golden):
    from test_gpu_sketch_program_adjoints import _adjoints, _record
    p, base = golden[31]
    K = 33
    vals, _ = _values(p, base, K, seed=11, unrealisable=0.1)
    other, _ = _values(p, base, 2 * K, seed=12)
    ob = np.random.default_rng(13).standard_normal((K, p.n_slots, 4, 2))
    with FProg(lib, p) as prog:
        _record(prog, vals)
        want, _ = _adjoints(prog, ob)
        wave, dwave, wnc, _ = prog.run_host(other, _directions(p, 2 * K, 3, seed=14))
        _record(prog, vals)
        prog.run_fused_host(other, _directions(p, 2 * K, 3, seed=14))
        got, _ = _adjoints(prog, ob)
        assert _same(got, want)
        after, dafter, anc, _ = prog.run_host(other, _directions(p, 2 * K, 3, seed=14))
        assert _same(after, wave) and _same(dafter, dwave) and np.array_equal(anc, wnc)


def test_the_fused_entry_points_refuse_what_the_wave_runs_refuse(lib, golden):
    p, _ = golden[31]
    buf = (C.c_double * 8)()
    with FProg(lib, p) as prog:
        cases = [
            ((prog.h, 0, buf, buf, None, 0, None, None), b"n_instances must be >= 1 (got 0)"),
            ((prog.h, 1, buf, buf, None, -1, buf, buf), b"n_tangents must be >= 0 (got -1)"),
            ((prog.h, 1, None, buf, None, 0, None, None), b"null value or position table"),
            ((prog.h, 1, buf, buf, None, 2, None, buf), b"null tangent table (dvalues or dpositions)"),
        ]
        for fn in (lib.gcs_b200_program_run_fused, lib.gcs_b200_program_run_fused_host):
            for args, message in cases:
                before = lib.gcs_b200_launch_count()
                assert fn(*args, None) == GCS_E_INVALID, message
                assert lib.gcs_b200_last_error() == message
                assert lib.gcs_b200_launch_count() == before


# ---- 8. SketchProgram::runFused ----

def _host_fused(prog, vals, dvals, n_devices):
    lib = H.load()
    lib.gcs_host_program_run_fused.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_double),
                                               C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.c_int,
                                               C.POINTER(C.c_int64)]
    vals = np.ascontiguousarray(vals)
    K, T = vals.shape[0], 0 if dvals is None else dvals.shape[2]
    slots = prog.describe()["slots"]
    pos, dpos = np.zeros((K, slots, 4)), np.zeros((K, slots, 4, max(T, 1)))
    nc, stats = np.zeros(K, dtype=np.uint32), np.zeros(7, dtype=np.int64)
    rc = lib.gcs_host_program_run_fused(prog.handle, K, _dp(vals), T, None if dvals is None else _dp(np.ascontiguousarray(dvals)), _dp(pos),
                                        _dp(dpos), nc.ctypes.data_as(C.POINTER(C.c_uint32)), n_devices,
                                        stats.ctypes.data_as(C.POINTER(C.c_int64)))
    assert rc == 0, H.last_error()
    return pos, dpos[..., :T], nc, stats


def test_sketch_program_run_fused_equals_run_and_run_tangents_on_every_device(lib):
    import torch
    el, edges = S.make_linkage(20000, seed=6)
    prog = PT.Program(el, edges)
    assert prog.rc == 0, prog.error
    base = PT.sketch_values(edges)
    K, T = 40, 3
    rng = np.random.default_rng(21)
    vals = base[None, :] * (1.0 + 1e-3 * rng.uniform(-1.0, 1.0, size=(K, len(base))))
    dvals = rng.standard_normal((K, len(base), T))
    rc, want, wnc, _ = prog.run(vals)
    assert rc == 0, H.last_error()
    rc, _, dwant, _, _ = prog.run_tangents(vals, dvals)
    assert rc == 0, H.last_error()
    ndev = torch.cuda.device_count()
    for n in sorted({1, ndev}):
        # each fused run on a program of its own: neither its staging nor its device tables hold the
        # answer of an earlier run
        for d in (None, dvals):
            fresh = PT.Program(el, edges)
            assert fresh.rc == 0, fresh.error
            pos, dpos, nc, stats = _host_fused(fresh, vals, d, n)
            assert _same(pos, want) and np.array_equal(nc, wnc), n
            assert d is None or _same(dpos, dwant), n
            assert stats[0] == min(n, K), n  # one launch per device
