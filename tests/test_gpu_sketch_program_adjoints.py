"""Sketch-program adjoints on the GPU: a recorded run leaves the results of a plain run untouched, the
device sweep equals the wave-by-wave CPU restatement (tests/program_restate_adjoints.py) bit for bit,
and it is the transpose of the tangent run: full Jacobians agree entrywise on the golden sketches and
dot products agree on the linkages."""
import ctypes as C

import numpy as np
import pytest

import host_lib as H
import program_adjoints_lib as P
import program_restate as R
import sketch_gen as S
from program_restate_adjoints import restate_adjoints
from test_gpu_host import WHOLE_SKETCHES, _ref_loops, _triangle_strip
from test_gpu_sketch_program_abi import Prog, _directions, _values, golden, lib  # noqa: F401  (fixtures)
from util import bits, digest

pytestmark = pytest.mark.gpu


def _same(a, b):
    return a.shape == b.shape and bool(((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))).all())


@pytest.fixture(scope="module")
def host(lib):
    return H.load()


def _record(prog, vals, counts=True, variant=0):
    """gcs_b200_program_run_recorded_host: (positions, nonconverged, launches)"""
    lib = prog.lib
    vals = np.ascontiguousarray(vals, dtype=np.float64)
    K = vals.shape[0]
    pos = np.zeros((K, prog.arrays.n_slots, 4))
    nc = np.zeros(K, dtype=np.uint32)
    before = lib.gcs_b200_launch_count()
    rc = lib.gcs_b200_program_run_recorded_host(prog.h, K, vals.ctypes.data, pos.ctypes.data, nc.ctypes.data if counts else None, variant, None)
    assert rc == 0, lib.gcs_b200_last_error()
    return pos, nc, lib.gcs_b200_launch_count() - before


def _adjoints(prog, ob):
    """gcs_b200_program_adjoints_host: (adj_values [K][n_values][T], launches)"""
    lib = prog.lib
    ob = np.ascontiguousarray(ob, dtype=np.float64)
    K, T = ob.shape[0], ob.shape[3]
    av = np.full((K, prog.arrays.n_values, T), 7.0)
    before = lib.gcs_b200_launch_count()
    rc = lib.gcs_b200_program_adjoints_host(prog.h, T, ob.ctypes.data, av.ctypes.data, None)
    assert rc == 0, lib.gcs_b200_last_error()
    return av, lib.gcs_b200_launch_count() - before


def _cotangents(prog, vals, T, seed):
    """[K][n_slots][4][T] random cotangents.  The golden sketches have rows without a root, and nearly every
    instance has some coordinate downstream of one: cotangent 0 weighs every coordinate (NaN rule), the
    others only those with finite tangents (prog: a Prog whose tangent run tells which)."""
    _, dpos, _, _ = prog.run_host(vals, np.ones((vals.shape[0], prog.arrays.n_values, 1)))
    ob = np.random.default_rng(seed).standard_normal((vals.shape[0], prog.arrays.n_slots, 4, T))
    ob[..., 1 if T > 1 else 0:] *= np.isfinite(dpos)
    return ob


def _non_empty_waves(p):
    return sum(1 for w in range(p.n_waves) if p.segment(w, 1)[0] < p.segment(w, R.KINDS)[1])


# ---- 1. a recorded run is a plain run ----

@pytest.mark.parametrize("seed", [31, 32, 33])
def test_a_recorded_run_leaves_the_results_and_launches_of_a_plain_run(lib, golden, seed):
    p, base = golden[seed]
    vals, _ = _values(p, base, 5, seed=seed, unrealisable=0.2)
    with Prog(lib, p) as prog:
        want, _, wnc, wl = prog.run_host(vals)
        got, nc, launches = _record(prog, vals)
    assert _same(got, want) and np.array_equal(nc, wnc) and launches == wl


def test_a_recorded_run_of_the_100k_linkage_matches_its_reference_digest(host):
    el, edges = S.make_linkage(100000, seed=4)
    prog = P.Program(el, edges)
    vals = P.sketch_values(edges)[None, :]
    rc, pos, nc, st = prog.run(vals)
    rc2, rpos, rnc, rst = prog.record(vals)
    assert rc == rc2 == 0, H.last_error()
    assert _same(pos, rpos) and np.array_equal(nc, rnc) and st["launches"] == rst["launches"]
    assert digest(np.ascontiguousarray(rpos[0, :, :2])) == str(_ref_loops()["config4_xy_sha256"])


# ---- 2. the device sweep equals the CPU restatement ----

@pytest.mark.parametrize("T", [1, 3])
@pytest.mark.parametrize("seed", [31, 32, 33])
def test_device_adjoints_equal_the_cpu_restatement(lib, golden, seed, T):
    """The golden leaf lists, K = 4 with one unrealisable instance, random cotangents (_cotangents): every
    adjoint equal, NaN with NaN."""
    p, base = golden[seed]
    vals, _ = _values(p, base, 4, seed=seed, unrealisable=0.25)
    with Prog(lib, p) as prog:
        ob = _cotangents(prog, vals, T, seed=seed + T)
        _record(prog, vals)
        got, _ = _adjoints(prog, ob)
    want = restate_adjoints(p, vals, ob)
    assert _same(got, want)
    assert np.isfinite(got[..., -1]).all()


def test_the_restated_sketches_hold_every_solver(golden):
    """solvers 1 and 2 (anchor pb.x holds v0) and 3 (pb.y holds sign1 * v1) among them"""
    assert set().union(*(set(int(s) for s in golden[seed][0].rows["solver"]) for seed in golden)) == set(range(1, 9))


# ---- 3. duality with the tangents ----

def _written(p):
    """[(slot, coordinate)] a run writes: every row's target, the zero-fixed rows' anchors"""
    out = set()
    for r in p.rows:
        s, c = int(r["solver"]), int(r["elem"][2])
        out |= {(c, q) for q in range(4 if p.slot_is_line[c] else 2)}
        if s <= 3:
            a, b = int(r["elem"][0]), int(r["elem"][1])
            out |= {(a, q) for q in range(4 if s == 3 else 2)} | {(b, 0), (b, 1)}
    return sorted(out)


@pytest.mark.parametrize("seed", [31, 32, 33])
def test_the_full_jacobians_of_both_modes_agree(lib, golden, seed):
    """K = 1.  Forward: identity directions, T = n_values.  Reverse: one-hot cotangents over every written
    coordinate, in chunks.  Entry by entry within 1e-12 of the largest |entry| of the coordinate's row,
    over the rows finite in forward mode, which are finite in reverse mode too.  A row is all NaN in
    reverse mode only where forward mode has NaN: forward mode spreads the NaN of a row without a root
    even through coefficients that are exactly 0 (NaN * 0), while reverse mode flags only a non-zero
    adjoint reaching that row, so some rows are NaN forward and finite in reverse."""
    p, base = golden[seed]
    vals, _ = _values(p, base, 1, seed=seed)
    nv = p.n_values
    with Prog(lib, p) as prog:
        _, dpos, _, _ = prog.run_host(vals, np.eye(nv)[None])
        _record(prog, vals)
        coords = _written(p)
        rev = np.zeros((len(coords), nv))
        step = 1024
        for lo in range(0, len(coords), step):
            chunk = coords[lo:lo + step]
            ob = np.zeros((1, p.n_slots, 4, len(chunk)))
            for t, (s, q) in enumerate(chunk):
                ob[0, s, q, t] = 1.0
            av, _ = _adjoints(prog, ob)
            rev[lo:lo + len(chunk)] = av[0].T
    fwd = np.stack([dpos[0, s, q] for s, q in coords])
    finite = np.isfinite(fwd).all(axis=1)
    rev_nan = np.isnan(rev).all(axis=1)
    assert not (rev_nan & ~np.isnan(fwd).any(axis=1)).any()
    assert np.isfinite(rev[finite]).all()
    f, r = fwd[finite], rev[finite]
    scale = np.maximum(np.abs(f).max(axis=1, keepdims=True), np.finfo(float).tiny)
    worst = float((np.abs(f - r) / scale).max())
    print(f"seed {seed}: {len(f)} rows of {nv} compared, {int((~finite).sum())} rows not finite forward, "
          f"{int(rev_nan.sum())} NaN in reverse, worst {worst:.2e} of the row scale")
    assert finite.any()
    assert worst <= 1e-12


@pytest.mark.parametrize("case", ["linkage20k", "linkage100k"])
def test_dot_products_of_both_modes_agree_on_the_linkages(host, case):
    """T = 4: <o, J v> (runTangents) = <J^T o, v> (adjoints), within 1e-9 of sum |o_i (J v)_i|, through the
    C++ layer (radians for angles)."""
    el, edges = S.make_linkage(100000, seed=4) if case == "linkage100k" else S.make_linkage(20000, seed=6)
    prog = P.Program(el, edges)
    vals = P.sketch_values(edges)[None, :]
    T = 4
    rng = np.random.default_rng(12)
    dv = rng.standard_normal((1, vals.shape[1], T))
    rc, _, dpos, nc, _ = prog.run_tangents(vals, dv)
    assert rc == 0 and nc[0] == 0, H.last_error()
    ob = rng.standard_normal(dpos.shape)
    rc, _, _, _ = prog.record(vals)
    rc2, av, _ = prog.adjoints(ob)
    assert rc == rc2 == 0, H.last_error()
    terms = (ob * dpos).reshape(-1, T)
    lhs, rhs = terms.sum(axis=0), (av * dv).reshape(-1, T).sum(axis=0)
    rel = np.abs(lhs - rhs) / np.abs(terms).sum(axis=0)
    print(f"{case}: relative gap {rel}")
    assert (rel <= 1e-9).all(), rel


# ---- 4. shared reads and overwrites ----

def _shared_reads(p):
    """A row of solver 4-8 duplicated into its own segment with a new target slot: in that wave two rows
    read the same slots a, b and the same values."""
    r = int(np.flatnonzero(p.rows["solver"] >= 4)[0])
    seg = int(np.searchsorted(p.offsets, r, side="right")) - 1
    row = p.rows[r].copy()
    row["elem"][2] = p.n_slots
    rows = np.insert(p.rows, int(p.offsets[seg + 1]), row)
    offsets = p.offsets.copy()
    offsets[seg + 1:] += 1
    initial = np.vstack([p.initial, p.initial[p.rows[r]["elem"][2]][None]])
    return R.Arrays(rows, offsets, np.append(p.slot_is_line, p.slot_is_line[p.rows[r]["elem"][2]]), initial, p.value_is_angle)


def _twice(p):
    """every wave run twice: the second pass rewrites every slot the first wrote"""
    return p.with_waves(p.waves() + p.waves())


@pytest.mark.parametrize("layout", ["shared_reads", "overwrites"])
def test_shared_reads_and_overwritten_slots_follow_the_restatement(lib, golden, layout):
    p, base = golden[32]
    q = _shared_reads(p) if layout == "shared_reads" else _twice(p)
    vals, _ = _values(p, base, 3, seed=4)
    with Prog(lib, q) as prog:
        ob = _cotangents(prog, vals, 2, seed=5)
        _record(prog, vals)
        first, _ = _adjoints(prog, ob)
        second, _ = _adjoints(prog, ob)
    assert _same(first, second) and np.isfinite(first[..., 1]).all()
    assert _same(first, restate_adjoints(q, vals, ob))


# ---- 5. independence ----

def test_instances_and_cotangents_are_independent(lib, golden):
    p, base = golden[31]
    vals, _ = _values(p, base, 16, seed=9, unrealisable=0.125)
    with Prog(lib, p) as prog:
        ob = _cotangents(prog, vals, 3, seed=10)
        _record(prog, vals)
        full, _ = _adjoints(prog, ob)
        for t in range(3):
            one, _ = _adjoints(prog, np.ascontiguousarray(ob[..., t:t + 1]))
            assert _same(one[..., 0], full[..., t]), t
        for k in range(16):
            _record(prog, vals[k:k + 1])
            one, _ = _adjoints(prog, ob[k:k + 1])
            assert _same(one[0], full[k]), k


# ---- 6. rows without a root ----

def test_the_nan_rule_of_rows_without_a_root(host):
    """The unrealisable instance of the tangent tests (instance 1).  A cotangent on the target of a failed
    row makes adj_values[1][:, t] NaN; one on the coordinates whose tangents are finite gives finite
    adjoints that contract with random directions as the forward run does; instances 0 and 2 equal
    their single-instance sweeps."""
    el, edges = S.make_linkage(3000, seed=11)
    prog = P.Program(el, edges)
    d = prog.describe()
    vals = np.repeat(P.sketch_values(edges)[None, :], 3, axis=0)
    r = d["rows"] // 2
    v1 = int(d["row_values"][r][1])
    vals[1, v1] = 1e4 * vals[1, v1]
    T = 4
    dv = np.random.default_rng(8).standard_normal((3, vals.shape[1], T))
    rc, _, dpos, nc, _ = prog.run_tangents(vals, dv)
    assert rc == 0 and nc[1] > 0 and nc[0] == nc[2] == 0
    nan_slots = np.flatnonzero(np.isnan(dpos[1]).any(axis=(1, 2)))
    finite = np.isfinite(dpos).all(axis=3, keepdims=True)
    rng = np.random.default_rng(3)
    ob = rng.standard_normal(dpos.shape) * finite
    ob[1, nan_slots[0], :2, 0] = 1.0  # t = 0 of instance 1 reaches a row without a root
    rc, _, _, _ = prog.record(vals)
    rc2, av, _ = prog.adjoints(ob)
    assert rc == rc2 == 0, H.last_error()
    assert np.isnan(av[1, :, 0]).all()
    assert np.isfinite(av[1, :, 1:]).all() and np.isfinite(av[0]).all() and np.isfinite(av[2]).all()
    for t in range(1, T):
        terms = (ob[1, ..., t] * np.where(finite[1, ..., 0], dpos[1, ..., t], 0.0)).ravel()
        gap = abs(terms.sum() - (av[1, :, t] * dv[1, :, t]).sum())
        assert gap <= 1e-9 * np.abs(terms).sum(), t
    for k in (0, 2):
        rc, _, _, _ = prog.record(vals[k:k + 1])
        rc2, one, _ = prog.adjoints(ob[k:k + 1])
        assert rc == rc2 == 0 and _same(one[0], av[k]), k


# ---- 7. layouts ----

def test_relabelled_slots_and_values_give_the_same_adjoints(lib, golden):
    p, base = golden[33]
    vals, _ = _values(p, base, 3, seed=2, unrealisable=0.34)
    q, slot_map, value_map = R.relabelled(p, seed=4)
    qv = np.zeros((3, q.n_values))
    qv[:, value_map] = vals
    with Prog(lib, p) as prog:
        ob = _cotangents(prog, vals, 2, seed=3)
        _record(prog, vals)
        want, _ = _adjoints(prog, ob)
    qob = np.zeros((3, q.n_slots, 4, 2))
    qob[:, slot_map] = ob
    with Prog(lib, q) as prog:
        _record(prog, qv)
        got, _ = _adjoints(prog, qob)
    assert _same(got[:, value_map], want)
    unused = np.setdiff1d(np.arange(q.n_values), value_map)
    assert (got[:, unused][np.isfinite(got[:, unused])] == 0.0).all()


@pytest.mark.parametrize("layout", ["split_by_kind", "split_by_kind_reversed", "one_row_per_wave", "empty_waves", "reversed_segments"])
def test_wave_layouts_change_only_the_order_of_the_sums(lib, golden, layout):
    p, base = golden[31]
    q = dict(R.transforms(p))[layout]
    vals, _ = _values(p, base, 3, seed=6, unrealisable=0.34)
    with Prog(lib, p) as prog:
        ob = _cotangents(prog, vals, 2, seed=7)
        _record(prog, vals)
        want, _ = _adjoints(prog, ob)
    with Prog(lib, q) as prog:
        _record(prog, vals)
        got, _ = _adjoints(prog, ob)
    assert np.array_equal(np.isnan(got), np.isnan(want))
    ok = np.isfinite(want)
    scale = np.maximum(np.abs(want).max(axis=1, keepdims=True), 1.0)
    assert (np.abs(got - want)[ok] <= 1e-12 * np.broadcast_to(scale, want.shape)[ok]).all()


# ---- 8. the device entry points and the caller's stream ----

def _adjoints_device(prog, ob, stream):
    import torch
    dev = torch.device("cuda", 0)
    o = torch.from_numpy(np.ascontiguousarray(ob)).to(dev)
    o_before = o.clone()
    av = torch.empty((ob.shape[0], prog.arrays.n_values, ob.shape[3]), dtype=torch.float64, device=dev)
    torch.cuda.synchronize()
    rc = prog.lib.gcs_b200_program_adjoints(prog.h, ob.shape[3], o.data_ptr(), av.data_ptr(), None if stream is None else stream.cuda_stream)
    assert rc == 0, prog.lib.gcs_b200_last_error()
    torch.cuda.synchronize()
    assert torch.equal(o, o_before)  # the caller's cotangents are not consumed
    return av.cpu().numpy()


@pytest.mark.parametrize("where", ["side_stream", "null_stream"])
def test_the_device_entry_points_equal_the_host_ones(lib, golden, where):
    import torch
    p, base = golden[31]
    K = 5
    vals, _ = _values(p, base, K, seed=11, unrealisable=0.2)
    stream = torch.cuda.Stream(device=0) if where == "side_stream" else None
    with Prog(lib, p) as prog:
        ob = _cotangents(prog, vals, 3, seed=12)
        _record(prog, vals)
        want, _ = _adjoints(prog, ob)
        got = _adjoints_device(prog, ob, stream)
        assert _same(got, want)
        # a recorded run on the device entry point, then the device sweep
        v = torch.from_numpy(vals).to("cuda:0")
        pos = torch.empty((K, p.n_slots, 4), dtype=torch.float64, device="cuda:0")
        assert lib.gcs_b200_program_run_recorded(prog.h, K, v.data_ptr(), pos.data_ptr(), None, 0,
                                                 None if stream is None else stream.cuda_stream) == 0
        got = _adjoints_device(prog, ob, stream)
        assert _same(got, want)


def test_a_sweep_is_ordered_on_the_callers_stream(lib, golden):
    """On a side stream: the cotangents are NaN, then a sleep, then the real cotangents are written, the
    sweep runs, and its result is cloned and overwritten with NaN.  The clone equals a host sweep and
    the call returned while the stream was still busy."""
    import torch
    p, base = golden[32]
    K = 9
    vals, _ = _values(p, base, K, seed=13)
    s = torch.cuda.Stream(device=0)
    dev = torch.device("cuda", 0)
    av = torch.empty((K, p.n_values, 2), dtype=torch.float64, device=dev)
    with Prog(lib, p) as prog:
        ob = _cotangents(prog, vals, 2, seed=14)
        real = torch.from_numpy(ob).to(dev)
        o = torch.empty_like(real)
        _record(prog, vals)
        want, _ = _adjoints(prog, ob)
        with torch.cuda.stream(s):
            o.fill_(float("nan"))
            torch.cuda._sleep(100_000_000)
            o.copy_(real)
            assert lib.gcs_b200_program_adjoints(prog.h, 2, o.data_ptr(), av.data_ptr(), s.cuda_stream) == 0
            still_running = not s.query()
            got = av.clone()
            av.fill_(float("nan"))
        s.synchronize()
    assert still_running, "the sweep synchronised its stream"
    assert _same(got.cpu().numpy(), want)
    assert torch.isnan(av).all()


# ---- 9. the tape, 10. launches ----

def test_plain_and_tangent_runs_leave_the_tape_and_a_new_record_replaces_it(lib, golden):
    p, base = golden[33]
    vals, _ = _values(p, base, 6, seed=15, unrealisable=0.17)
    other, _ = _values(p, base, 6, seed=16)
    with Prog(lib, p) as prog:
        ob = _cotangents(prog, vals, 2, seed=17)
        _record(prog, vals)
        want, _ = _adjoints(prog, ob)
        prog.run_host(other)
        prog.run_host(other, _directions(p, 6, 3, seed=1))
        got, _ = _adjoints(prog, ob)
        assert _same(got, want)
        _record(prog, other[:2])
        got, _ = _adjoints(prog, ob[:2])
    assert _same(got, restate_adjoints(p, other[:2], ob[:2]))


def test_a_sweep_adds_at_most_two_launches_per_wave(lib, golden):
    p, base = golden[31]
    waves = _non_empty_waves(p)
    with Prog(lib, p) as prog:
        for K, T in ((1, 1), (7, 4)):
            vals, _ = _values(p, base, K, seed=K)
            ob = _cotangents(prog, vals, T, seed=T)
            _record(prog, vals)
            _, launches = _adjoints(prog, ob)
            assert launches <= 2 * waves + 1, (K, T, launches, waves)


# ---- 11. devices, 12. the contracted class ----

def test_adjoints_do_not_depend_on_the_device_count(host, lib):
    ndev = lib.gcs_b200_device_count()
    if ndev < 2:
        pytest.skip("needs two visible devices")
    el, edges = S.make_linkage(20000, seed=6)
    prog = P.Program(el, edges)
    vals = np.repeat(P.sketch_values(edges)[None, :], 8, axis=0)
    vals *= 1.0 + 1e-4 * np.random.default_rng(9).uniform(-1, 1, size=vals.shape)
    ob = np.random.default_rng(10).standard_normal((8, prog.describe()["slots"], 4, 2))
    rc, _, _, _ = prog.record(vals, n_devices=1)
    rc2, one, _ = prog.adjoints(ob)
    rc3, _, _, _ = prog.record(vals, n_devices=2)
    rc4, two, st = prog.adjoints(ob)
    assert rc == rc2 == rc3 == rc4 == 0 and st["devices"] == 2 and _same(one, two)


def test_the_contracted_class_agrees_on_adjoints(host):
    """The 400-leaf strip, as the contracted tangent test: adjoints within 1e-8 relative of the
    bit-identical class, for GCS_VARIANT_CONTRACTED and its explicit mappings."""
    pts, el, lv = _triangle_strip(402)
    prog = P.Program(el, leaves=lv)
    vals = np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])
    vals = vals * (1.0 + 1e-7 * np.random.default_rng(2).uniform(-1.0, 1.0, size=(4, len(vals))))
    ob = np.random.default_rng(4).standard_normal((4, prog.describe()["slots"], 4, 3))
    rc, _, nc, _ = prog.record(vals)
    rc2, base, _ = prog.adjoints(ob)
    assert rc == rc2 == 0 and not nc.any()
    scale = max(1.0, float(np.abs(base).max()))
    for variant in (5, 6, 7, 8, 10):
        old = host.gcs_host_set_variant(variant)
        try:
            rc, _, nc2, _ = prog.record(vals)
            rc2, fast, _ = prog.adjoints(ob)
        finally:
            host.gcs_host_set_variant(old)
        assert rc == rc2 == 0 and np.array_equal(nc, nc2), variant
        worst = float(np.abs(base - fast).max()) / scale
        print(f"contracted variant {variant}: adjoints within {worst:.3e} relative")
        assert worst <= 1e-8, (variant, worst)
