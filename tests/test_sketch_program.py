"""Sketch programs without a device: what SketchProgram::compile makes of a sketch (waves, solvers,
rows, value slots) against the plan of the wave solver, and the descriptor checks of
gcs_b200_program_create, which run before any device is touched."""
import ctypes as C

import numpy as np
import pytest

import host_lib as H
import program_lib as P
import program_restate as R
import program_tangents_lib as PT
import sketch_gen as S

GOLDEN_SKETCHES = [(31, 1, 3000), (32, 2, 3000), (33, 3, 3000)]
KIND_OF_SOLVER = {1: 1, 2: 2, 3: 5, 4: 1, 5: 2, 6: 3, 7: 4, 8: 5}


@pytest.fixture(scope="module")
def host(built):
    built.build_host()
    return H.load()


def _leaf_values(leaves):
    """Value slots of each leaf in a leaf-list program: its real edges' positions in the flat edge order."""
    out, at = [], 0
    for lf in leaves:
        real = [e for e in lf["edges"] if e["type"] != S.VIRT]
        out.append(set(range(at, at + len(real))))
        at += len(real)
    return out


def _check_against_plan(prog, elements, leaves):
    d = prog.describe()
    plan = H.leaves_solve(elements, leaves, 2)
    assert plan["rc"] == 0
    assert d["waves"] == plan["waves"] and d["leaves"] == len(leaves)
    assert list(d["leaf_solver"]) == plan["solver"] and list(d["leaf_level"]) == plan["level"]
    solved = [i for i, s in enumerate(plan["solver"]) if s != 0]
    # one row per solved leaf, in its wave's segment of its kind
    assert d["rows"] == len(solved) and sorted(d["row_leaf"]) == solved
    for w in range(d["waves"]):
        for k in range(5):
            for r in range(d["offsets"][5 * w + k], d["offsets"][5 * w + k + 1]):
                leaf = int(d["row_leaf"][r])
                assert plan["level"][leaf] == w and KIND_OF_SOLVER[plan["solver"][leaf]] == k + 1
                assert d["row_solver"][r] == plan["solver"][leaf]
    return d


@pytest.mark.parametrize("seed,first,n", GOLDEN_SKETCHES)
def test_program_of_a_leaf_list_follows_the_wave_plan(host, seed, first, n):
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    prog = P.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    d = _check_against_plan(prog, el, lv)
    held = _leaf_values(lv)
    for r in range(d["rows"]):
        leaf = int(d["row_leaf"][r])
        assert set(lv[leaf]["elems"]) == set(d["row_elems"][r])
        used = [int(v) for v in d["row_values"][r] if v >= 0]
        assert used and set(used) <= held[leaf], (r, used, held[leaf])


def test_all_solvers_and_kinds_occur_across_the_golden_sketches(host):
    solvers = set()
    for seed, first, n in GOLDEN_SKETCHES:
        el, lv = S.make_sketch(n, seed=seed, first_shape=first)
        solvers |= set(int(s) for s in P.Program(el, leaves=lv).describe()["row_solver"])
    assert solvers == set(range(1, 9))
    assert {KIND_OF_SOLVER[s] for s in solvers} == {1, 2, 3, 4, 5}


def test_program_of_a_whole_linkage(host):
    """The whole-sketch entry point: check, decomposition and compile of a 20k linkage.  Every leaf
    is solved, every row reads values only of constraints between its own elements, and after a run
    every element is solved."""
    el, edges = S.make_linkage(20000, seed=6)
    prog = P.Program(el, edges)
    assert prog.rc == 0, prog.error
    d = prog.describe()
    assert d["leaves"] == len(el) - 2 and d["rows"] == d["leaves"] and d["unsupported"] == 0
    assert d["values"] == len(edges) and d["slots"] == len(el)
    assert d["solved_after"].all()
    pair = [(e["a"], e["b"]) for e in edges if e["type"] != S.VIRT]
    for r in range(d["rows"]):
        mine = set(int(x) for x in d["row_elems"][r])
        for v in d["row_values"][r]:
            if v >= 0:
                assert set(pair[v]) <= mine
    assert set(d["row_solver"]) == {1, 4}
    assert d["offsets"][-1] == d["rows"] and (np.diff(d["offsets"]) >= 0).all()


def test_a_leaf_the_reference_loop_throws_on_stops_the_compile(host):
    """The leaf list of test_an_exception_mid_list_stops_the_loop_like_the_reference: leaf 30 lacks a
    constraint, so the reference's loop throws at it (getConstraintBetweenNodes).  compile throws the
    same exception; its message is the one the packer raises for that leaf with its two parents solved."""
    el, lv = S.make_sketch(60, seed=9, p_line=0.0)
    bad = {"elems": lv[30]["elems"], "edges": [dict(e) for e in lv[30]["edges"] if e["type"] != 2]}
    real = [e for e in bad["edges"] if e["type"] == 0 and max(e["a"], e["b"]) == max(bad["elems"])]
    bad["edges"].remove(real[0])
    lv2 = lv[:30] + [bad] + lv[31:]
    prog = P.Program(el, leaves=lv2)
    assert prog.rc == -1
    # the same leaf alone, the parents solved as the loop would have them: the packer raises there
    local = {g: i for i, g in enumerate(bad["elems"])}
    new = max(bad["elems"])
    els = [dict(el[g], is_set=g != new, pos=[1.0 + i, 2.0 * i]) for i, g in enumerate(bad["elems"])]
    eds = [dict(e, a=local[e["a"]], b=local[e["b"]]) for e in bad["edges"]]
    sid, *_ = H.component_pack(els, eds)
    assert sid == -1
    assert prog.error == H.last_error() and prog.error


def _descriptor(capi):
    """A valid two-wave program: a ZeroFixedPointsTriangle, then a TwoFixedPointsDistance."""
    rows = (capi.CProgramRow * 2)()
    rows[0].solver, rows[0].code = 1, 2
    rows[0].elem[:] = [0, 1, 2]
    rows[0].value[:] = [0, 1, 2]
    rows[1].solver, rows[1].code = 4, 0
    rows[1].elem[:] = [1, 2, 3]
    rows[1].value[:] = [-1, 3, 4]
    for r in rows:
        r.sign[:] = [1.0, 1.0, 1.0]
    offsets = (C.c_int64 * 11)(0, 1, 1, 1, 1, 1, 2, 2, 2, 2, 2)
    is_line = (C.c_uint8 * 4)(0, 0, 0, 0)
    initial = (C.c_double * 16)()
    angle = (C.c_uint8 * 5)()
    d = capi.CProgramDesc(n_waves=2, n_slots=4, n_values=5, n_rows=2)
    d.rows, d.offsets, d.slot_is_line, d.initial, d.value_is_angle = rows, offsets, is_line, initial, angle
    return d, (rows, offsets, is_line, initial, angle)


@pytest.mark.parametrize("defect,message", [
    ("slot", "element slot"), ("value", "value slot"), ("offsets", "offsets decrease"), ("solver", "unknown solver id"),
    ("kind", "segment"), ("type", "wrong element type"), ("angle", "angle slot"),
])
def test_malformed_descriptors_are_refused_before_any_device_call(gcs, built, defect, message):
    capi = gcs.capi
    lib = capi.load()
    d, keep = _descriptor(capi)
    rows, offsets, is_line, _, angle = keep
    if defect == "slot":
        rows[1].elem[2] = 4
    elif defect == "value":
        rows[1].value[1] = 5
    elif defect == "offsets":
        offsets[1], offsets[2] = 1, 0
    elif defect == "solver":
        rows[1].solver = 9
    elif defect == "kind":  # a K4 row (TwoFixedLinesFreePoint) in the K1 segment
        rows[1].solver = 7
    elif defect == "type":
        is_line[3] = 1
    elif defect == "angle":
        angle[3] = 1
    h = C.c_void_p()
    assert lib.gcs_b200_program_create(C.byref(d), 0, C.byref(h)) == capi.GCS_E_INVALID
    assert message in lib.gcs_b200_last_error().decode()
    assert not h.value


def test_a_valid_descriptor_needs_a_device(gcs, built):
    capi = gcs.capi
    lib = capi.load()
    d, keep = _descriptor(capi)
    h = C.c_void_p()
    rc = lib.gcs_b200_program_create(C.byref(d), 0, C.byref(h))
    if lib.gcs_b200_device_count() == 0:
        assert rc == capi.GCS_E_NO_DEVICE and not h.value
    else:
        assert rc == capi.GCS_OK and h.value
        assert lib.gcs_b200_program_run_host(h, 0, None, None, None, 0, None) == capi.GCS_E_INVALID  # K < 1
        lib.gcs_b200_program_destroy(h)


def _one_wave(rows):
    """A one-wave program of K1 rows given as (solver, elem): solver 1 reads v0 v1 v2, solver 4 v1 v2."""
    r = np.zeros(len(rows), dtype=R.ROW)
    for i, (solver, elem) in enumerate(rows):
        r[i]["solver"], r[i]["elem"], r[i]["sign"] = solver, elem, 1.0
        r[i]["value"] = [3 * i, 3 * i + 1, 3 * i + 2] if solver == 1 else [-1, 3 * i + 1, 3 * i + 2]
    n_slots = int(r["elem"].max()) + 1
    return R.Arrays(r, [0] + [len(rows)] * 5, np.zeros(n_slots), np.zeros((n_slots, 4)), np.zeros(3 * len(rows)))


def _create(gcs, arrays):
    lib = gcs.capi.load()
    h = C.c_void_p()
    rc = lib.gcs_b200_program_create(C.byref(arrays.desc()), 0, C.byref(h))
    if h.value:
        lib.gcs_b200_program_destroy(h)
    return rc, lib.gcs_b200_last_error().decode()


def _valid(gcs):
    """what gcs_b200_program_create returns for a valid descriptor on this machine"""
    return gcs.capi.GCS_OK if gcs.capi.load().gcs_b200_device_count() > 0 else gcs.capi.GCS_E_NO_DEVICE


@pytest.mark.parametrize("rows,written,read", [
    ([(4, [0, 1, 4]), (4, [2, 3, 4])], "written by row 0", "written by row 1"),   # two rows target slot 4
    ([(1, [0, 1, 2]), (4, [3, 0, 4])], "written by row 0", "read by row 1"),      # row 0 anchors slot 0 that row 1 reads
    ([(4, [2, 3, 4]), (4, [0, 1, 2])], "read by row 0", "written by row 1"),      # row 1 targets slot 2 that row 0 reads
])
def test_rows_of_one_wave_with_overlapping_footprints_are_refused(gcs, built, rows, written, read):
    """The rows of a wave run concurrently: a slot two of them write, or one writes and another reads,
    would make the result depend on thread scheduling.  Refused before any device call, naming both rows."""
    rc, msg = _create(gcs, _one_wave(rows))
    assert rc == gcs.capi.GCS_E_INVALID
    assert written in msg and read in msg, msg
    # the same rows in two waves are a valid program
    two = _one_wave(rows)
    two = two.with_waves([[np.array([0]), *[np.zeros(0, dtype=np.int64)] * 4], [np.array([1]), *[np.zeros(0, dtype=np.int64)] * 4]])
    assert _create(gcs, two)[0] == _valid(gcs), _create(gcs, two)[1]


def test_rows_of_one_wave_may_share_what_they_read(gcs, built):
    assert _create(gcs, _one_wave([(4, [0, 1, 2]), (4, [1, 0, 3]), (4, [0, 1, 4])]))[0] == _valid(gcs)


@pytest.mark.parametrize("case", GOLDEN_SKETCHES + ["linkage20k"])
def test_compiled_programs_and_their_wave_layouts_pass_validation(gcs, host, case):
    """What SketchProgram::compile makes, and every layout of tests/program_restate.py (the layouts the
    GPU tests require to leave every result unchanged), passes the footprint rule."""
    if case == "linkage20k":
        el, edges = S.make_linkage(20000, seed=6)
        prog = PT.Program(el, edges)
    else:
        seed, first, n = case
        el, lv = S.make_sketch(n, seed=seed, first_shape=first)
        prog = PT.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    p = R.Arrays.from_desc(prog.desc())
    layouts = [("compiled", p)] + R.transforms(p) + [("relabelled", R.relabelled(p, seed=1)[0]),
                                                     ("no_rows", R.without_rows(p, 0)), ("no_rows_3_waves", R.without_rows(p, 3))]
    for name, q in layouts:
        rc, msg = _create(gcs, q)
        assert rc == _valid(gcs), (name, msg)
