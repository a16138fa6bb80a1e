"""Host mirror on the GPU: the reference-shaped entry points (classifyAndSolve, the solver
structs, Equations::solve2D, DeficitStreeBasedTopDownStrategy::solveGcs,
GeometricConstraintSystem) run through the CUDA path and must leave the element state the
reference's own code leaves (golden fixtures made from the reference sources)."""
import json
import math
import os

import numpy as np
import pytest

import host_lib as H
import oracle_lib as O
import sketch_gen as S
from test_host_packer import GOLD, same_pos
from util import digest, positions

pytestmark = pytest.mark.gpu
WHOLE_SKETCHES = [(31, 1, 3000), (32, 2, 3000), (33, 3, 3000)]


def _ref_loops():
    """What the reference build's sequential loop left in the elements of the sketches below
    (oracle/make_golden_ref_loops.py)."""
    return np.load(os.path.join(GOLD, "ref_loops.npz"))


def _assert_same_elements(got, ref, name):
    """Solved flags equal, every position bit for bit (NaN with NaN) through the stored digest."""
    pos, is_set = positions(got)
    assert np.array_equal(is_set, ref[f"{name}_set"]), np.nonzero(is_set != ref[f"{name}_set"])[0][:8]
    assert digest(pos) == str(ref[f"{name}_pos_sha256"]), f"{name}: solved positions differ from the reference loop"


def config4_sample(n):
    """The fixed sample of the 100k-point linkage whose coordinates are stored beside their digest."""
    return np.sort(np.random.default_rng(4).choice(n, 4096, replace=False))


@pytest.fixture(scope="module")
def host(gpu, built):
    built.build_host()
    return H.load()


def test_classify_and_solve_matches_reference_components(host):
    items = json.load(open(os.path.join(GOLD, "components.json")))["items"]
    for it in items:
        status, els = H.component_solve(it["elements"], it["edges"])
        assert status == it["status"], (it["shape"], status, H.last_error())
        if status != 0:
            continue
        for got, exp in zip(els, it["expected"]):
            assert got["is_set"] == exp["is_set"]
            if exp["is_set"]:
                assert same_pos(got["pos"], exp["pos"]), (it["shape"], got, exp)


def test_baseline_config_1_single_triangle_through_the_whole_pipeline(host):
    """BASELINE configs[0]: points (100,100), (200,100), (150,200), distances 3-4-5, through
    GeometricConstraintSystem -> DeficitStreeBasedTopDownStrategy -> solveGcs."""
    el = [{"type": 0, "canvas": [100.0, 100.0]}, {"type": 0, "canvas": [200.0, 100.0]}, {"type": 0, "canvas": [150.0, 200.0]}]
    ed = [{"a": 0, "b": 1, "type": 0, "value": 3.0}, {"a": 0, "b": 2, "type": 0, "value": 4.0}, {"a": 1, "b": 2, "type": 0, "value": 5.0}]
    rc, out = H.system_solve(el, ed)
    assert rc == 0, H.last_error()
    assert out[0]["pos"] == [0.0, 0.0] and out[1]["pos"] == [3.0, 0.0]
    assert out[2]["pos"][1] == 4.0 and abs(out[2]["pos"][0]) < 1e-12
    # under-constrained (an edge missing): the driver throws like the reference
    rc, _ = H.system_solve(el, ed[:2])
    assert rc == -1 and "not well-constrained" in H.last_error()


@pytest.mark.parametrize("pair,kind", [(1, 1), (2, 2), (3, 3), (4, 4), (5, 5)])
def test_solve2d_mirror_equals_the_oracle(host, gcs, pair, kind):
    rng = np.random.default_rng(pair)
    for _ in range(40):
        if pair == 1:
            params = [*rng.uniform(-50, 50, 2), rng.uniform(60, 90), *rng.uniform(-50, 50, 2), rng.uniform(60, 90)]
            consts, guesses = params, None
        elif pair == 2:
            th = rng.uniform(0, 6.28)
            params = [*rng.uniform(-80, 80, 2), *rng.uniform(-30, 30, 2)]
            guesses = [np.cos(th), np.sin(th), -np.cos(th), -np.sin(th)]
            consts = params
        elif pair == 3:
            xa, ya, xb, yb = rng.uniform(-100, 100, 4)
            ln = float(np.sqrt((xb - xa) * (xb - xa) + (yb - ya) * (yb - ya)))
            params = [*rng.uniform(-50, 50, 2), rng.uniform(150, 250), xa, ya, xb, yb, rng.uniform(-20, 20), ln]
            consts, guesses = params, None
        elif pair == 4:
            l = rng.uniform(-100, 100, 8)
            l1 = float(np.sqrt((l[2] - l[0]) ** 2 + (l[3] - l[1]) ** 2))
            l2 = float(np.sqrt((l[6] - l[4]) ** 2 + (l[7] - l[5]) ** 2))
            s1, s2 = rng.uniform(-30, 30, 2)
            params = [*l[:4], s1, l1, *l[4:], s2, l2]
            consts, guesses = params, None
        else:
            fd = rng.uniform(-100, 100, 2)
            th = rng.uniform(0, 6.28)
            ln = float(np.sqrt(fd[0] * fd[0] + fd[1] * fd[1]))
            params = [fd[0], fd[1], ln, np.cos(rng.uniform(0.2, 2.9))]
            guesses = [np.cos(th), np.sin(th), -np.cos(th), -np.sin(th)]
            consts = params
        rc, cand, it, cv = H.solve2d(pair, params, guesses)
        assert rc == 0, H.last_error()
        g = guesses if guesses is not None else [20000.0, 20000.0, -20000.0, -20000.0]
        for s in range(2):
            x, y, oit, ocv = O.newton2d(kind, consts, g[2 * s], g[2 * s + 1])
            assert (it[s], cv[s]) == (oit, ocv)
            assert same_pos([cand[s, 0], cand[s, 1]], [x, y])
    # a length that is not the direction's length is refused, not silently recomputed
    if pair == 3:
        params[8] *= 1.5
        rc, *_ = H.solve2d(pair, params, None)
        assert rc == -1 and "length" in H.last_error()


def test_solve_gcs_batched_equals_the_reference_loop_on_golden_sketches(host):
    data = json.load(open(os.path.join(GOLD, "sketch_leaves.json")))["items"]
    for sk in data:
        for mode in (0, 1):
            r = H.leaves_solve(sk["elements"], sk["leaves"], mode)
            assert r["rc"] == 0, H.last_error()
            assert r["status"] == sk["status"]
            for got, exp in zip(r["elements"], sk["expected"]):
                assert got["is_set"] == exp["is_set"] and same_pos(got["pos"], exp["pos"])
            if mode == 1:
                assert r["launches"] <= 5 * r["waves"] and r["waves"] < len(sk["leaves"])


def _triangle_strip(n_points):
    """A consistent linkage: points on two rows, every new point hung on the previous two with its
    true distances; the canvas is the true layout.  From the default guesses the two seeds of every
    leaf sit on opposite sides of the fixed pair, so each leaf has its two distinct roots and the
    orientation heuristic picks the drawn one - unlike the random sketches of sketch_gen, whose
    later leaves inherit a wrong root and then never converge (as they do in the reference)."""
    pts = [(5.0 * i, 0.0 if i % 2 == 0 else 8.0 + 0.01 * i) for i in range(n_points)]
    el = [{"type": 0, "canvas": [x + 100.0, y + 50.0]} for x, y in pts]
    dist = lambda i, j: math.dist(pts[i], pts[j])
    e = lambda i, j: {"a": i, "b": j, "type": 0, "value": dist(i, j), "flip": False}
    leaves = [{"elems": [0, 1, 2], "edges": [e(0, 1), e(0, 2), e(1, 2)]}]
    for k in range(3, n_points):
        leaves.append({"elems": [k - 2, k - 1, k], "edges": [e(k - 2, k), e(k - 1, k), {"a": k - 2, "b": k - 1, "type": 2, "value": 0.0, "flip": False}]})
    return pts, el, leaves


def test_solve_gcs_with_the_contracted_kernels_agrees_to_the_tolerance(host):
    """Gcs::B200::setKernelVariant(GCS_VARIANT_CONTRACTED): each leaf's coordinates are the next
    leaf's inputs, so a whole sketch agrees with the bit-identical run to the north star's 1e-9
    relative (statuses and solved flags identical), here over a chain of 400 dependent leaves."""
    lib = H.load()
    pts, el, lv = _triangle_strip(402)
    base = H.leaves_solve(el, lv, 1)
    old = lib.gcs_host_set_variant(5)
    try:
        fast = H.leaves_solve(el, lv, 1)
    finally:
        lib.gcs_host_set_variant(old)
    assert old == 0 and base["rc"] == 0 and fast["rc"] == 0 and base["status"] == fast["status"] and set(base["status"]) == {0}
    # the base run reproduces the drawn linkage (so the comparison below is about a real solution)
    xy = np.array([e_["pos"] for e_ in base["elements"]])
    for i, j in ((0, 1), (100, 101), (399, 401), (400, 401)):
        assert abs(math.dist(xy[i], xy[j]) - math.dist(pts[i], pts[j])) < 1e-6
    scale = float(np.abs(xy).max())
    worst = 0.0
    for x, y in zip(base["elements"], fast["elements"]):
        assert x["is_set"] and y["is_set"]
        worst = max(worst, max(abs(a - b) for a, b in zip(x["pos"], y["pos"])) / max(1.0, scale))
    assert worst <= 1e-9, worst


def test_solve_gcs_batched_equals_sequential_at_scale(host):
    """20k leaves: one launch per kind per wave (a few hundred launches) against one launch per
    leaf; the final element state must be bit-identical."""
    el, lv = S.make_sketch(20000, seed=5, first_shape=2)
    a = H.leaves_solve(el, lv, 1)
    assert a["rc"] == 0 and a["solved"] == len(lv)
    sub_el, sub_lv = S.make_sketch(1500, seed=6, first_shape=3, locality=40)
    b0 = H.leaves_solve(sub_el, sub_lv, 0)
    b1 = H.leaves_solve(sub_el, sub_lv, 1)
    assert b0["rc"] == 0 and b1["rc"] == 0
    for x, y in zip(b0["elements"], b1["elements"]):
        assert x["is_set"] and y["is_set"] and same_pos(x["pos"], y["pos"])
    assert a["launches"] < 0.05 * len(lv)
    # the reference build itself (oracle/_ref, where it travelled to this box) on all 20k leaves
    import ref_lib as R
    if R.available():
        rc, status, exp = R.leaves_solve(el, lv)
        assert rc == 0 and status == a["status"]
        for got, e in zip(a["elements"], exp):
            assert got["is_set"] == e["is_set"] and same_pos(got["pos"], e["pos"])


def test_an_exception_mid_list_stops_the_loop_like_the_reference(host):
    el, lv = S.make_sketch(60, seed=9, p_line=0.0)
    bad = {"elems": lv[30]["elems"], "edges": [dict(e) for e in lv[30]["edges"] if e["type"] != 2]}
    # remove one of the two real constraints of leaf 30: getConstraintBetweenNodes throws there
    real = [e for e in bad["edges"] if e["type"] == 0 and max(e["a"], e["b"]) == max(bad["elems"])]
    bad["edges"].remove(real[0])
    lv2 = lv[:30] + [bad] + lv[31:]
    seq = H.leaves_solve(el, lv2, 0)
    bat = H.leaves_solve(el, lv2, 1)
    assert seq["rc"] == -1 and bat["rc"] == -1
    for x, y in zip(seq["elements"], bat["elements"]):
        assert x["is_set"] == y["is_set"] and (not x["is_set"] or same_pos(x["pos"], y["pos"]))
    assert sum(e["is_set"] for e in bat["elements"]) == 32  # leaves 0..29 only


@pytest.mark.parametrize("seed,first,n", WHOLE_SKETCHES)
def test_whole_sketch_pipeline_equals_reference_loop_on_the_same_leaves(host, seed, first, n):
    """GeometricConstraintSystem::solveGeometricConstraintSystem on a whole sketch (check ->
    peel decomposition -> batched solveGcs on the GPU) against what the reference build's sequential
    loop over the same leaves left (tests/golden/ref_loops.npz), bit for bit."""
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    edges = S.sketch_graph(el, lv)
    rc, got, stats = H.system_solve_ex(el, edges)
    assert rc == 0, H.last_error()
    assert stats["leaves"] == len(el) - 2 and stats["solved"] == stats["leaves"]
    assert stats["launches"] <= 5 * stats["waves"] and stats["waves"] < 0.2 * stats["leaves"]
    assert all(e["is_set"] for e in got)
    ref = _ref_loops()
    _assert_same_elements(got, ref, f"sketch{seed}")


def test_config4_linkage_100k_points(host):
    """BASELINE config 4 at full size: a rigid linkage of 100k points and 199,997 distances through
    the public entry point (check -> decomposition -> wave-batched solveGcs on the GPU).  The sketch
    is one the reference itself solves consistently (sketch_gen.make_linkage), so (i) EVERY distance
    constraint holds in the result to 1e-6 and (ii) every solved position equals, bit for bit, what
    the reference build's sequential loop leaves in the same elements (stored as a digest of all of them
    and a fixed sample, tests/golden/ref_loops.npz)."""
    el, edges = S.make_linkage(100000, seed=4)
    rc, got, stats = H.system_solve_ex(el, edges)
    assert rc == 0, H.last_error()
    assert stats["leaves"] == 99998 and stats["solved"] == 99998
    assert stats["launches"] == stats["waves"] < 200
    assert all(e["is_set"] for e in got)
    xy = np.array([e["pos"] for e in got])
    ea = np.array([[e["a"], e["b"], e["value"]] for e in edges])
    d = np.hypot(*(xy[ea[:, 0].astype(int)] - xy[ea[:, 1].astype(int)]).T)
    resid = np.abs(d - ea[:, 2]) / np.maximum(1.0, ea[:, 2])
    assert (resid < 1e-6).all(), f"{int((resid >= 1e-6).sum())} of {len(edges)} distances do not hold, worst {resid.max():.3e}"
    ref = _ref_loops()
    idx = config4_sample(len(xy))
    sample = ref["config4_xy_sample"]
    assert np.array_equal(xy[idx].view(np.uint64), sample.view(np.uint64)), \
        f"{int((xy[idx].view(np.uint64) != sample.view(np.uint64)).any(axis=1).sum())} of {len(idx)} sampled points differ from the reference loop"
    assert digest(xy) == str(ref["config4_xy_sha256"]), "the points outside the stored sample differ from the reference loop"


def test_unchecked_linkage_runs_into_the_cap_like_the_reference(host):
    """The stress case: a linkage drawn without regard for the reference's unchecked candidate-1 pick
    (heuristics.hpp:56).  Some leaf returns the mirrored root, the circles below it no longer meet
    and those runs spin to the iteration cap - in the reference and here alike, bit for bit."""
    el, edges = S.make_linkage_unchecked(6000, seed=4)
    rc, got, stats = H.system_solve_ex(el, edges)
    assert rc == 0, H.last_error()
    assert stats["solved"] == stats["leaves"] == 5998
    ref = _ref_loops()
    _assert_same_elements(got, ref, "unchecked")


def test_one_sketch_over_several_devices_equals_one_device(host, gcs):
    """DeficitStreeBasedTopDownStrategy::setDeviceCount / solveLeavesOnDevices: the waves of ONE sketch
    cut into index ranges over the GPUs of the box (gcs_b200_solve_sharded per kind batch; the solved
    positions meet again in the host's elements).  Same result as on one device, bit for bit.  On a
    one-GPU box the device list has one entry and the call degenerates to the single-device path."""
    capi = gcs.capi
    ndev = capi.load().gcs_b200_device_count()
    capi.init(list(range(ndev)))
    el, edges = S.make_linkage(20000, seed=6)
    try:
        os.environ["GCS_HOST_DEVICES"], os.environ["GCS_HOST_MIN_ROWS"] = str(ndev), "64"
        rc, many, st_many = H.system_solve_ex(el, edges)
        assert rc == 0, H.last_error()
    finally:
        os.environ.pop("GCS_HOST_DEVICES", None), os.environ.pop("GCS_HOST_MIN_ROWS", None)
        capi.init([0])
    rc, one, st_one = H.system_solve_ex(el, edges)
    assert rc == 0, H.last_error()
    assert st_one["sharded_launches"] == 0
    if ndev > 1:
        assert st_many["sharded_launches"] > 0
    for a, b in zip(many, one):
        assert a["is_set"] and same_pos(a["pos"], b["pos"])
