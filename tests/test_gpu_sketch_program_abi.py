"""Sketch programs through the raw C ABI on the GPU (gcs_b200_program_*, descriptors built with
tests/program_restate.py): the device entry points on a caller's stream, every kernel mapping a run
can pick, wave layouts that must not change a result, and buffer growth between runs.  Everything
compares bit for bit, NaN with NaN, unless a test says otherwise."""
import ctypes as C

import numpy as np
import pytest

import program_restate as R
import program_tangents_lib as PT
import sketch_gen as S
from test_gpu_host import WHOLE_SKETCHES
from util import bits, rel_err

pytestmark = pytest.mark.gpu

KERNEL_OF = {1: "static", 2: "refill", 3: "sorted", 4: "pair", 9: "seq"}  # GCS_VARIANT_* -> kernel


def _same(a, b):
    return a.shape == b.shape and bool(((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))).all())


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


def _values(p, base, K, seed, unrealisable=0.0):
    """K value sets as the ABI takes them (angle slots hold cos): distances moved by up to 1e-3 relative,
    angles by up to 1e-2 rad, set 0 unmoved; a share `unrealisable` of the sets gets one distance x 1e4.
    Returns (values [K][n_values], the unrealisable sets)."""
    angle = p.value_is_angle.astype(bool)
    rng = np.random.default_rng(seed)
    u = rng.uniform(-1.0, 1.0, size=(K, len(base)))
    v = np.where(angle, base + 1e-2 * u, base * (1.0 + 1e-3 * u))
    v[0] = base
    bad = np.sort(rng.choice(np.arange(1, K), size=int(round(unrealisable * K)), replace=False)) if unrealisable else np.zeros(0, dtype=int)
    for k in bad:
        d = rng.choice(np.flatnonzero(~angle))
        v[k, d] *= 1e4
    return np.where(angle, np.cos(v), v), bad


def _directions(p, K, T, seed):
    return np.random.default_rng(seed).standard_normal((K, p.n_values, T))


class Prog:
    """A program made by gcs_b200_program_create from Arrays."""

    def __init__(self, lib, arrays, device=0):
        self.lib, self.arrays, self.h = lib, arrays, C.c_void_p()
        assert lib.gcs_b200_program_create(C.byref(arrays.desc()), device, C.byref(self.h)) == 0, lib.gcs_b200_last_error()

    def close(self):
        if self.h.value:
            self.lib.gcs_b200_program_destroy(self.h)
            self.h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def run_host(self, vals, dvals=None, variant=0, counts=True):
        """gcs_b200_program_run[_tangents]_host: (positions, tangents or None, nonconverged or None, launches)"""
        vals = np.ascontiguousarray(vals, dtype=np.float64)
        K = vals.shape[0]
        pos = np.zeros((K, self.arrays.n_slots, 4))
        nc = np.zeros(K, dtype=np.uint32) if counts else None
        ncp = nc.ctypes.data if counts else None
        before = self.lib.gcs_b200_launch_count()
        if dvals is None:
            rc = self.lib.gcs_b200_program_run_host(self.h, K, vals.ctypes.data, pos.ctypes.data, ncp, variant, None)
            dpos = None
        else:
            dvals = np.ascontiguousarray(dvals, dtype=np.float64)
            T = dvals.shape[2]
            dpos = np.zeros((K, self.arrays.n_slots, 4, T))
            rc = self.lib.gcs_b200_program_run_tangents_host(self.h, K, vals.ctypes.data, pos.ctypes.data, ncp, T, dvals.ctypes.data,
                                                             dpos.ctypes.data, variant, None)
        assert rc == 0, self.lib.gcs_b200_last_error()
        return pos, dpos, nc, self.lib.gcs_b200_launch_count() - before

    def run(self, vals, pos, nc=None, dvals=None, dpos=None, variant=0, stream=None):
        """gcs_b200_program_run[_tangents] on torch tensors, enqueued on `stream` (None: the NULL stream); no synchronisation."""
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        sp = None if stream is None else stream.cuda_stream
        K = vals.shape[0]
        if dvals is None:
            rc = self.lib.gcs_b200_program_run(self.h, K, ptr(vals), ptr(pos), ptr(nc), variant, sp)
        else:
            rc = self.lib.gcs_b200_program_run_tangents(self.h, K, ptr(vals), ptr(pos), ptr(nc), dvals.shape[2], ptr(dvals), ptr(dpos),
                                                        variant, sp)
        assert rc == 0, self.lib.gcs_b200_last_error()


def _run_device(prog, vals, dvals=None, stream=None, counts=True, device=0):
    """prog.run on device copies of the tables, synchronised: (positions, tangents or None, nonconverged or None)"""
    import torch
    dev = torch.device("cuda", device)
    K = vals.shape[0]
    v = torch.from_numpy(np.ascontiguousarray(vals)).to(dev)
    pos = torch.empty((K, prog.arrays.n_slots, 4), dtype=torch.float64, device=dev)
    nc = torch.full((K,), 12345, dtype=torch.int32, device=dev) if counts else None
    dv = None if dvals is None else torch.from_numpy(np.ascontiguousarray(dvals)).to(dev)
    dpos = None if dvals is None else torch.empty((K, prog.arrays.n_slots, 4, dvals.shape[2]), dtype=torch.float64, device=dev)
    torch.cuda.synchronize(dev)
    prog.run(v, pos, nc, dv, dpos, stream=stream)
    torch.cuda.synchronize(dev)
    return (pos.cpu().numpy(), None if dpos is None else dpos.cpu().numpy(),
            None if nc is None else nc.cpu().numpy().astype(np.uint32))


# ---- 1. the device entry points on a caller's stream ----

@pytest.mark.parametrize("K", [1, 33])
@pytest.mark.parametrize("where", ["side_stream", "null_stream"])
def test_the_device_entry_points_equal_the_host_ones(lib, golden, K, where):
    import torch
    p, base = golden[31]
    vals, _ = _values(p, base, K, seed=K)
    stream = torch.cuda.Stream(device=0) if where == "side_stream" else None
    with Prog(lib, p) as prog:
        for T in (0, 1, 5):
            dvals = _directions(p, K, T, seed=T) if T else None
            want, dwant, wnc, _ = prog.run_host(vals, dvals)
            got, dgot, nc = _run_device(prog, vals, dvals, stream)
            assert _same(got, want) and np.array_equal(nc, wnc), T
            assert T == 0 or _same(dgot, dwant), T
            got, dgot, _ = _run_device(prog, vals, dvals, stream, counts=False)  # nonconverged = NULL
            assert _same(got, want) and (T == 0 or _same(dgot, dwant)), T


@pytest.mark.parametrize("T", [0, 2])
def test_a_run_is_ordered_on_the_callers_stream(lib, golden, T):
    """On a side stream: the values are NaN, then a sleep of about 50 ms, then the real values are
    written, the program runs, and its results are cloned and overwritten with NaN.  The clones equal a
    host run: no launch of the run (gather, solve_many's side streams, scatter, tangent kernel, the
    counts' memset, the doubling copies) started before the values were written, and every one ended
    before the clones.  The positions stay NaN: nothing of the run wrote after the overwrite."""
    import torch
    p, base = golden[32]
    K = 33
    vals, _ = _values(p, base, K, seed=5)
    dvals = _directions(p, K, T, seed=6) if T else None
    s = torch.cuda.Stream(device=0)
    dev = torch.device("cuda", 0)
    real = torch.from_numpy(vals).to(dev)
    dreal = torch.from_numpy(dvals).to(dev) if T else None
    v = torch.empty_like(real)
    dv = torch.empty_like(dreal) if T else None
    pos = torch.empty((K, p.n_slots, 4), dtype=torch.float64, device=dev)
    dpos = torch.empty((K, p.n_slots, 4, T), dtype=torch.float64, device=dev) if T else None
    nc = torch.empty(K, dtype=torch.int32, device=dev)
    with Prog(lib, p) as prog:
        want, dwant, wnc, _ = prog.run_host(vals, dvals)
        v.copy_(real)
        if T:
            dv.copy_(dreal)
        torch.cuda.synchronize()
        prog.run(v, pos, nc, dv, dpos, stream=s)  # warm-up at the same K: no buffer grows below
        s.synchronize()
        with torch.cuda.stream(s):
            v.fill_(float("nan"))
            if T:
                dv.fill_(float("nan"))
            torch.cuda._sleep(100_000_000)
            v.copy_(real)
            if T:
                dv.copy_(dreal)
            prog.run(v, pos, nc, dv, dpos, stream=s)
            still_running = not s.query()
            got, gnc = pos.clone(), nc.clone()
            dgot = dpos.clone() if T else None
            pos.fill_(float("nan"))
            if T:
                dpos.fill_(float("nan"))
        s.synchronize()
    assert still_running, "the run synchronised its stream"
    assert _same(got.cpu().numpy(), want) and np.array_equal(gnc.cpu().numpy().astype(np.uint32), wnc)
    assert T == 0 or _same(dgot.cpu().numpy(), dwant)
    assert torch.isnan(pos).all() and (T == 0 or torch.isnan(dpos).all())


def test_a_program_on_another_device_runs_while_device_0_is_current(lib, golden):
    import torch
    if lib.gcs_b200_device_count() < 2:
        pytest.skip("one device visible")
    p, base = golden[33]
    vals, _ = _values(p, base, 9, seed=3)
    dvals = _directions(p, 9, 2, seed=4)
    with Prog(lib, p, device=0) as p0:
        want, dwant, wnc = _run_device(p0, vals, dvals)
    torch.cuda.set_device(0)
    with Prog(lib, p, device=1) as p1:
        assert torch.cuda.current_device() == 0
        got, dgot, nc = _run_device(p1, vals, dvals, stream=torch.cuda.Stream(device=1), device=1)
        assert torch.cuda.current_device() == 0
        hpos, hdpos, hnc, _ = p1.run_host(vals, dvals)
        assert torch.cuda.current_device() == 0
    assert _same(got, want) and _same(dgot, dwant) and np.array_equal(nc, wnc)
    assert _same(hpos, want) and _same(hdpos, dwant) and np.array_equal(hnc, wnc)


# ---- 2. every kernel mapping inside a program ----

@pytest.mark.parametrize("seed", [s for s, _, _ in WHOLE_SKETCHES])
def test_default_at_large_k_runs_the_sorted_and_seq_kernels(lib, golden, seed):
    """K = 4096 instances, about 1% with an unrealisable distance (runs that spin to the iteration cap
    inside sorted tiles).  GCS_VARIANT_DEFAULT resolves every kind's largest waves to the sorted kernel
    (K4: the seq kernel) there.  Positions, counts and tangents (T = 2) equal 64 runs of 64 instances
    (static launches only) and, on a sample of instances, the CPU restatement."""
    p, base = golden[seed]
    K, T, chunk = 4096, 2, 64
    vals, bad = _values(p, base, K, seed=seed, unrealisable=0.01)
    dvals = _directions(p, K, T, seed=seed + 1)
    resolved = {}
    for w in range(p.n_waves):
        for k in range(1, R.KINDS + 1):
            lo, hi = p.segment(w, k)
            if hi > lo:
                v = lib.gcs_b200_resolve_variant(0, k, (hi - lo) * K, 2)
                assert lib.gcs_b200_resolve_variant(0, k, (hi - lo) * chunk, 2) == 1  # the K = 64 runs: static
                resolved.setdefault(k, {}).setdefault(KERNEL_OF[v], 0)
                resolved[k][KERNEL_OF[v]] += 1
    print(f"sketch {seed}, K = {K}: waves per kernel and kind {resolved}")
    assert set(resolved) == {1, 2, 3, 4, 5}
    for k, kernels in resolved.items():
        assert kernels.get("seq" if k == 4 else "sorted", 0) > 0, (k, kernels)
    with Prog(lib, p) as prog:
        pos, _, nc, _ = prog.run_host(vals)
        tpos, dpos, tnc, _ = prog.run_host(vals, dvals)
        assert _same(tpos, pos) and np.array_equal(tnc, nc)
        assert nc[bad].min() > 0
        for lo in range(0, K, chunk):
            sl = slice(lo, lo + chunk)
            cpos, _, cnc, _ = prog.run_host(vals[sl])
            assert _same(pos[sl], cpos) and np.array_equal(nc[sl], cnc), lo
            cpos, cdpos, cnc, _ = prog.run_host(vals[sl], dvals[sl])
            assert _same(pos[sl], cpos) and _same(dpos[sl], cdpos) and np.array_equal(nc[sl], cnc), lo
    sample = np.union1d([0, 31, 32, 33, 2047, 4095], bad)
    want, dwant, wnc = R.restate(p, vals[sample], dvals[sample])
    assert _same(pos[sample], want) and _same(dpos[sample], dwant) and np.array_equal(nc[sample], wnc)


@pytest.mark.parametrize("seed", [s for s, _, _ in WHOLE_SKETCHES])
def test_explicit_bit_identical_variants_equal_the_default(lib, golden, seed):
    """GCS_VARIANT_STATIC, _REFILL, _SORTED, _PAIR and _SEQ at K = 64, plain and tangent runs."""
    p, base = golden[seed]
    vals, _ = _values(p, base, 64, seed=seed + 2)
    dvals = _directions(p, 64, 3, seed=seed + 3)
    with Prog(lib, p) as prog:
        want, _, wnc, _ = prog.run_host(vals)
        _, dwant, _, _ = prog.run_host(vals, dvals)
        for variant in (1, 2, 3, 4, 9):
            pos, _, nc, _ = prog.run_host(vals, variant=variant)
            assert _same(pos, want) and np.array_equal(nc, wnc), variant
            pos, dpos, nc, _ = prog.run_host(vals, dvals, variant=variant)
            assert _same(pos, want) and _same(dpos, dwant) and np.array_equal(nc, wnc), variant


def _prefix(p, w):
    """waves [0, w) of the program"""
    hi = int(p.offsets[R.KINDS * w])
    return R.Arrays(p.rows[:hi], p.offsets[:R.KINDS * w + 1], p.slot_is_line, p.initial, p.value_is_angle)


@pytest.mark.parametrize("variant", [5, 6, 7, 8, 10])  # GCS_VARIANT_CONTRACTED, _STATIC, _SORTED, _SEQ, _LINEAR
@pytest.mark.parametrize("seed", [s for s, _, _ in WHOLE_SKETCHES])
def test_contracted_variants_keep_the_contract_row_by_row(lib, golden, seed, variant):
    """Wave by wave, without the chain's amplification: wave w gathered from the state a contracted run
    of waves [0, w) leaves and solved by the CPU oracle, against a contracted run of waves [0, w].  Every
    row's output within 1e-9 relative at the scale of its inputs (util.rel_err), NaN where the oracle
    has NaN; every other slot bit-identical; the increase of the nonconverged count equal to the
    oracle's."""
    p, base = golden[seed]
    K = 4
    vals, _ = _values(p, base, K, seed=seed + 4)
    zero = np.zeros((K, p.n_values, 1))
    with Prog(lib, _prefix(p, 0)) as prog:
        state, _, nc, _ = prog.run_host(vals, variant=variant)
    worst = 0.0
    for w in range(p.n_waves):
        batches, anchors = R.gather_wave(p, w, state, np.zeros(state.shape + (1,)), vals, zero)
        want = state.copy()
        for slot, x, _ in anchors:
            for q in x:
                want[:, slot, q] = x[q]
        with Prog(lib, _prefix(p, w + 1)) as prog:
            got, _, gnc, _ = prog.run_host(vals, variant=variant)
        targets = p.rows["elem"][int(p.offsets[R.KINDS * w]):int(p.offsets[R.KINDS * (w + 1)]), 2]
        rest = np.setdiff1d(np.arange(p.n_slots), targets)
        assert _same(got[:, rest], want[:, rest]), w
        added = np.zeros(K, dtype=np.uint32)
        for k, lo, hi, hb, _ in batches:
            R.O.solve(hb.alloc_outputs())
            added += R.not_converged(hb).reshape(hi - lo, K).sum(axis=0).astype(np.uint32)
            with np.errstate(invalid="ignore"):
                scale = np.max(np.stack([np.where(np.isfinite(c), np.abs(c), 0.0) for c in hb.dense_cols()]), axis=0)
            for q, ref in enumerate(hb.out):
                mine = got[:, p.rows["elem"][lo:hi, 2], q].T.reshape(-1)  # sub-system (row i, instance j) at i * K + j
                assert np.array_equal(np.isnan(mine), np.isnan(ref)), (w, k, q)
                fin = np.isfinite(ref)
                assert np.array_equal(mine[~fin], ref[~fin]) or np.isnan(ref[~fin]).all(), (w, k, q)
                err = rel_err(mine[fin], ref[fin], scale[fin])
                if err.size:
                    worst = max(worst, float(err.max()))
                    assert err.max() <= 1e-9, (w, k, q, err.max())
        assert np.array_equal(gnc - nc, added), w
        state, nc = got, gnc
    print(f"sketch {seed}, variant {variant}: worst row error {worst:.3e}")


# ---- 3. wave layouts that leave every result unchanged ----

LAYOUTS = ["split_by_kind", "split_by_kind_reversed", "one_row_per_wave", "empty_waves", "reversed_segments"]


@pytest.mark.parametrize("layout", LAYOUTS)
@pytest.mark.parametrize("seed", [s for s, _, _ in WHOLE_SKETCHES])
def test_wave_layouts_do_not_change_a_run(lib, golden, seed, layout):
    """The compiled program against the same rows split per kind (in kind order and reversed), one row
    per wave, with empty waves around and between the waves, and with every segment reversed: K = 33,
    T = 3; empty waves add no launch."""
    p, base = golden[seed]
    q = dict(R.transforms(p))[layout]
    K = 33
    vals, _ = _values(p, base, K, seed=seed + 5)
    dvals = _directions(p, K, 3, seed=seed + 6)
    with Prog(lib, p) as a, Prog(lib, q) as b:
        want, dwant, wnc, launches = a.run_host(vals, dvals)
        got, dgot, nc, blaunches = b.run_host(vals, dvals)
        assert _same(got, want) and _same(dgot, dwant) and np.array_equal(nc, wnc)
        if layout == "empty_waves":
            assert blaunches == launches and a.run_host(vals)[3] == b.run_host(vals)[3]


@pytest.mark.parametrize("seed", [s for s, _, _ in WHOLE_SKETCHES])
def test_slot_and_value_labels_do_not_change_a_run(lib, golden, seed):
    """Slots and values permuted, with unused slots (NaN initial positions) and unused NaN values added:
    the same results under the relabelling, the unused slots untouched (NaN, tangent 0)."""
    p, base = golden[seed]
    q, slot_map, value_map = R.relabelled(p, seed=seed)
    K, T = 33, 3
    vals, _ = _values(p, base, K, seed=seed + 7)
    dvals = _directions(p, K, T, seed=seed + 8)
    qvals = np.full((K, q.n_values), np.nan)
    qvals[:, value_map] = vals
    qdvals = np.full((K, q.n_values, T), np.nan)
    qdvals[:, value_map] = dvals
    unused = np.setdiff1d(np.arange(q.n_slots), slot_map)
    with Prog(lib, p) as a, Prog(lib, q) as b:
        want, dwant, wnc, _ = a.run_host(vals, dvals)
        got, dgot, nc, _ = b.run_host(qvals, qdvals)
    assert _same(got[:, slot_map], want) and _same(dgot[:, slot_map], dwant) and np.array_equal(nc, wnc)
    assert np.isnan(got[:, unused]).all() and not dgot[:, unused].any()


@pytest.mark.parametrize("n_waves", [0, 3])
def test_a_program_without_rows_leaves_the_initial_positions(lib, golden, n_waves):
    """Every instance is the initial positions, also at K not a power of two (the doubling copies)."""
    p, base = golden[31]
    q = R.without_rows(p, n_waves)
    with Prog(lib, q) as prog:
        for K in (1, 2, 3, 5, 1000):
            vals, _ = _values(p, base, K, seed=K)
            pos, _, nc, _ = prog.run_host(vals)
            assert _same(pos, np.broadcast_to(p.initial, pos.shape)) and not nc.any(), K
            pos, dpos, nc, _ = prog.run_host(vals, _directions(p, K, 2, seed=K))
            assert _same(pos, np.broadcast_to(p.initial, pos.shape)) and not dpos.any() and not nc.any(), K
            pos, _, nc = _run_device(prog, vals)
            assert _same(pos, np.broadcast_to(p.initial, pos.shape)) and not nc.any(), K


# ---- 4. buffer growth between runs ----

GROWTH = [(1, 0), (300, 0), (2, 0), (300, 3), (300, 0), (5, 40), (400, 1)]  # (K, T); T = 0: a plain run


@pytest.mark.parametrize("entry", ["host", "device"])
def test_a_reused_program_equals_a_fresh_one_while_its_buffers_grow(lib, golden, entry):
    import torch
    p, base = golden[33]
    stream = torch.cuda.Stream(device=0)
    with Prog(lib, p) as prog:
        for i, (K, T) in enumerate(GROWTH):
            vals, _ = _values(p, base, K, seed=100 + i)
            dvals = _directions(p, K, T, seed=200 + i) if T else None
            if entry == "host":
                got, dgot, nc, _ = prog.run_host(vals, dvals)
            else:
                got, dgot, nc = _run_device(prog, vals, dvals, stream)
            with Prog(lib, p) as fresh:
                want, dwant, wnc, _ = fresh.run_host(vals, dvals)
            assert _same(got, want) and np.array_equal(nc, wnc) and (T == 0 or _same(dgot, dwant)), (K, T)
