"""Sketch programs on the GPU: a decomposed sketch planned once and solved for K sets of constraint
values must leave, per instance, exactly what the wave solver (and the reference's own loop) leaves
for those values - bit for bit, NaN with NaN."""

import numpy as np
import pytest

import host_lib as H
import program_lib as P
import oracle_lib as O
import sketch_gen as S
from test_gpu_host import WHOLE_SKETCHES, _ref_loops, _triangle_strip, config4_sample
from util import bits, digest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def host(gpu, built):
    built.build_host()
    return H.load()


def _table(out):
    """[n][4] positions of host_lib element dicts (NaN past a point's two coordinates), [n] solved flags."""
    pos = np.full((len(out), 4), np.nan)
    for i, e in enumerate(out):
        pos[i, :len(e["pos"])] = e["pos"]
    return pos, np.array([e["is_set"] for e in out], dtype=np.uint8)


def _instance(pos_k, elements):
    """One instance of a run as the same [n][4] table (NaN past a point's two coordinates)."""
    p = pos_k.copy()
    for i, e in enumerate(elements):
        if e["type"] == S.P:
            p[i, 2:] = np.nan
    return p


def _same(a, b):
    return bool(((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))).all())


def _with_values(edges, values):
    out, v = [], iter(values)
    for e in edges:
        e = dict(e)
        if e["type"] != S.VIRT:
            e["value"] = float(next(v))
        out.append(e)
    return out


def _perturbed(edges, K, seed):
    """K value sets: distances moved by up to 1e-3 relative, angles by up to 1e-2 rad; set 0 unmoved."""
    base = P.sketch_values(edges)
    is_angle = np.array([e["type"] == S.ANG for e in edges if e["type"] != S.VIRT])
    rng = np.random.default_rng(seed)
    u = rng.uniform(-1.0, 1.0, size=(K, len(base)))
    vals = np.where(is_angle, base + 1e-2 * u, base * (1.0 + 1e-3 * u))
    vals[0] = base
    return vals


def _assert_equals_host_path(el, edges, prog, vals, pos, what):
    d = prog.describe()
    for k in range(len(vals)):
        rc, out, _ = H.system_solve_ex(el, _with_values(edges, vals[k]))
        assert rc == 0, H.last_error()
        want, want_set = _table(out)
        assert np.array_equal(d["solved_after"], want_set), f"{what}: solved flags differ"
        assert _same(_instance(pos[k], el), want), f"{what}: instance {k} differs from the host path"


@pytest.mark.parametrize("seed,first,n", WHOLE_SKETCHES)
def test_one_instance_equals_the_reference_loop_on_golden_sketches(host, seed, first, n):
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    edges = S.sketch_graph(el, lv)
    prog = P.Program(el, edges)
    assert prog.rc == 0, prog.error
    rc, pos, nc, st = prog.run(P.sketch_values(edges))
    assert rc == 0, H.last_error()
    got = _instance(pos[0], el)
    ref = _ref_loops()
    assert np.array_equal(prog.describe()["solved_after"], ref[f"sketch{seed}_set"])
    assert digest(got) == str(ref[f"sketch{seed}_pos_sha256"]), "solved positions differ from the reference loop"
    rc, out, _ = H.system_solve_ex(el, edges)
    assert rc == 0 and _same(got, _table(out)[0])


def test_one_instance_equals_the_reference_loop_on_the_unchecked_linkage(host):
    el, edges = S.make_linkage_unchecked(6000, seed=4)
    prog = P.Program(el, edges)
    rc, pos, nc, _ = prog.run(P.sketch_values(edges))
    assert rc == 0, H.last_error()
    ref = _ref_loops()
    assert np.array_equal(prog.describe()["solved_after"], ref["unchecked_set"])
    assert digest(_instance(pos[0], el)) == str(ref["unchecked_pos_sha256"])
    assert nc[0] > 0  # the runs that spin to the iteration cap are reported


def test_one_instance_equals_the_reference_loop_on_the_100k_linkage(host):
    el, edges = S.make_linkage(100000, seed=4)
    prog = P.Program(el, edges)
    rc, pos, nc, st = prog.run(P.sketch_values(edges))
    assert rc == 0, H.last_error()
    xy = np.ascontiguousarray(pos[0, :, :2])
    ref = _ref_loops()
    idx = config4_sample(len(xy))
    assert np.array_equal(xy[idx].view(np.uint64), ref["config4_xy_sample"].view(np.uint64))
    assert digest(xy) == str(ref["config4_xy_sha256"])
    assert nc[0] == 0 and prog.describe()["solved_after"].all()
    rc, out, _ = H.system_solve_ex(el, edges)
    assert rc == 0 and _same(xy, np.array([e["pos"] for e in out]))


@pytest.mark.parametrize("case", ["sketch31", "sketch32", "sketch33", "linkage20k"])
def test_a_sweep_equals_the_host_path_instance_by_instance(host, case):
    seeds = {"sketch31": 131, "sketch32": 132, "sketch33": 133, "linkage20k": 120}
    if case == "linkage20k":
        el, edges = S.make_linkage(20000, seed=6)
    else:
        seed, first, n = {"sketch31": WHOLE_SKETCHES[0], "sketch32": WHOLE_SKETCHES[1], "sketch33": WHOLE_SKETCHES[2]}[case]
        el, lv = S.make_sketch(n, seed=seed, first_shape=first)
        edges = S.sketch_graph(el, lv)
    prog = P.Program(el, edges)
    vals = _perturbed(edges, 16, seed=seeds[case])
    rc, pos, nc, st = prog.run(vals)
    assert rc == 0, H.last_error()
    _assert_equals_host_path(el, edges, prog, vals, pos, case)


def test_instances_are_independent_of_k_and_of_their_position(host):
    el, lv = S.make_sketch(3000, seed=32, first_shape=2)
    edges = S.sketch_graph(el, lv)
    prog = P.Program(el, edges)
    vals = _perturbed(edges, 257, seed=7)
    rc, full, nc_full, _ = prog.run(vals)
    assert rc == 0, H.last_error()
    for K in (1, 3, 33):
        rc, pos, nc, _ = prog.run(vals[:K])
        assert rc == 0 and _same(pos, full[:K]) and np.array_equal(nc, nc_full[:K]), K
    rc, pos, nc, _ = prog.run(vals[100:101])
    assert rc == 0 and _same(pos[0], full[100]) and nc[0] == nc_full[100]
    rc, pos, nc, _ = prog.run(vals[::-1].copy())
    assert rc == 0 and _same(pos, full[::-1]) and np.array_equal(nc, nc_full[::-1])


def test_an_unrealisable_instance_is_reported_and_leaves_its_neighbours_alone(host, gcs):
    """Instance 1 gives one point a distance the triangle inequality rules out: its circles do not
    meet, the chosen run spins to the cap.  That instance still equals the host path, its count is
    positive and equals what the CPU oracle finds re-solving every K1 row from the final positions
    (every element of a linkage is written once, so the final positions are the rows' inputs); the
    instances beside it are the drawn linkage and report 0."""
    el, edges = S.make_linkage(3000, seed=11)
    prog = P.Program(el, edges)
    d = prog.describe()
    vals = np.repeat(P.sketch_values(edges)[None, :], 3, axis=0)
    # a leaf in the middle of the construction: its new point's first distance made far too long
    r = d["rows"] // 2
    v1 = int(d["row_values"][r][1])
    vals[1, v1] = 1e4 * vals[1, v1]
    rc, pos, nc, _ = prog.run(vals)
    assert rc == 0, H.last_error()
    assert nc[0] == 0 and nc[2] == 0 and nc[1] > 0
    _assert_equals_host_path(el, edges, prog, vals, pos, "unrealisable")
    # the oracle on the K1 rows of instance 1
    rows = np.arange(d["rows"])
    solver = d["row_solver"]
    assert set(solver) <= {1, 4}
    a, b = d["row_elems"][:, 0], d["row_elems"][:, 1]
    p = pos[1]
    v = vals[1]
    zero = solver == 1
    cols = [np.where(zero, 0.0, p[a, 0]), np.where(zero, 0.0, p[a, 1]), v[d["row_values"][:, 1]],
            np.where(zero, v[np.maximum(d["row_values"][:, 0], 0)], p[b, 0]), np.where(zero, 0.0, p[b, 1]), v[d["row_values"][:, 2]]]
    hb = gcs.capi.HostBatch(1, 2, [np.ascontiguousarray(c) for c in cols], np.ascontiguousarray(d["row_code"]))
    O.solve(hb.alloc_outputs())
    chosen = hb.converged[hb.root_index.astype(np.int64), rows]
    assert int((chosen == 0).sum()) == int(nc[1])
    # and the oracle's roots are the positions the run wrote
    c = d["row_elems"][:, 2]
    assert _same(np.stack([hb.out[0], hb.out[1]], axis=1), p[c, :2])


def test_a_program_is_reusable_and_solve_follows_edits(host):
    el, lv = S.make_sketch(3000, seed=33, first_shape=3)
    edges = S.sketch_graph(el, lv)
    prog = P.Program(el, edges)
    vals = _perturbed(edges, 4, seed=3)
    rc, first, _, _ = prog.run(vals[:2])
    rc2, second, _, _ = prog.run(vals[2:])
    fresh = P.Program(el, edges)
    rc3, want, _, _ = fresh.run(vals[2:])
    assert rc == rc2 == rc3 == 0 and _same(second, want) and not _same(first, second)
    # the edit loop: SketchProgram::solve() with edited values equals solveGcs on the edited sketch
    rc, out = prog.solve(vals[3])
    assert rc == 0, H.last_error()
    rc, ref, _ = H.system_solve_ex(el, _with_values(edges, vals[3]))
    assert rc == 0
    for x, y in zip(out, ref):
        assert x["is_set"] == y["is_set"] and _same(np.array(x["pos"]), np.array(y["pos"]))


def test_the_contracted_class_agrees_to_the_tolerance(host):
    """The contracted class on the chain of 400 dependent leaves of
    test_solve_gcs_with_the_contracted_kernels_agrees_to_the_tolerance: each leaf's coordinates are the
    next leaf's inputs, and the program agrees with the bit-identical class to 1e-9 relative, for the
    drawn values and for value sets moved by up to 1e-7 relative.  Every contracted variant:
    GCS_VARIANT_CONTRACTED and the explicit mappings _STATIC, _SORTED, _SEQ and _LINEAR."""
    pts, el, lv = _triangle_strip(402)
    prog = P.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    base_vals = np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])
    u = np.random.default_rng(2).uniform(-1.0, 1.0, size=(4, len(base_vals)))
    vals = base_vals * (1.0 + 1e-7 * u)
    vals[0] = base_vals
    rc, base, nc_base, _ = prog.run(vals)
    assert rc == 0 and not nc_base.any()
    xy = base[:, :, :2]
    scale = max(1.0, float(np.abs(xy).max()))
    for variant in (5, 6, 7, 8, 10):
        old = host.gcs_host_set_variant(variant)
        try:
            rc2, fast, nc_fast, _ = prog.run(vals)
        finally:
            host.gcs_host_set_variant(old)
        assert old == 0 and rc2 == 0 and np.array_equal(nc_base, nc_fast), variant
        worst = float(np.abs(xy - fast[:, :, :2]).max()) / scale
        assert worst <= 1e-9, (variant, worst)


def test_results_do_not_depend_on_the_device_count(host, gcs):
    ndev = gcs.capi.load().gcs_b200_device_count()
    el, edges = S.make_linkage(20000, seed=6)
    prog = P.Program(el, edges)
    vals = _perturbed(edges, 8, seed=9)
    rc, one, nc1, _ = prog.run(vals, n_devices=1)
    rc2, many, ncm, st = prog.run(vals, n_devices=ndev)
    assert rc == rc2 == 0 and _same(one, many) and np.array_equal(nc1, ncm)


def test_launches_per_run_do_not_depend_on_k(host):
    el, lv = S.make_sketch(3000, seed=31, first_shape=1)
    edges = S.sketch_graph(el, lv)
    prog = P.Program(el, edges)
    waves = prog.describe()["waves"]
    vals = _perturbed(edges, 257, seed=1)
    rc, _, _, s1 = prog.run(vals[:1])
    rc2, _, _, s257 = prog.run(vals)
    assert rc == rc2 == 0
    assert 0 < s1["launches"] == s257["launches"] <= 7 * waves
