"""Bottom-up Merge3 numeric helpers of the host mirror (host/src/bottom_up/merge3_solver_common.cpp;
SURVEY.md section 8f rank 3) against golden vectors produced by the reference's own
merge3_solver_common.cpp (tests/golden/merge3.npz, oracle/make_golden_merge3.py).

CPU side: the packer half of each helper (canvas-side signs, flags, nullopt decisions) is finished
by the CPU oracle - this is a test; the product has no host Newton iteration - and must reproduce
the reference's results bit for bit; the Procrustes fit and the pose score are host arithmetic and
are compared directly.  GPU side: the same rows through Merge3Batch (one launch per kind) and
through the single-call functions with the reference's signatures."""
import os

import numpy as np
import pytest

import host_lib as H
import oracle_lib as O
from util import bits, digest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "merge3.npz")
CASES = [1, 2, 3, 4]


@pytest.fixture(scope="module")
def gold():
    return np.load(GOLD)


@pytest.fixture(scope="module")
def host(built):
    built.build_host()
    return H.load()


def same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return (bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))


@pytest.mark.parametrize("kase", CASES)
def test_packed_rows_finished_by_the_oracle_match_the_reference(gcs, host, gold, kase):
    capi = gcs.capi
    rows, exp, exp_ok = gold[f"rows{kase}"], gold[f"out{kase}"], gold[f"ok{kase}"]
    rc, packed, code, needs = H.m3_pack(kase, rows)
    assert rc == 0, H.last_error()
    assert np.array_equal(needs, exp_ok), "nullopt decisions differ from the reference"
    kind = H.M3_KIND[kase]
    sel = np.nonzero(needs)[0]
    hb = capi.HostBatch(kind, 2, [np.ascontiguousarray(packed[sel, c]) for c in range(capi.IN_COLS[kind])],
                        np.ascontiguousarray(code[sel]))
    O.solve(hb.alloc_outputs())
    got = np.stack(hb.out, axis=1)
    bad = ~same(got, exp[sel]).all(axis=1)
    assert not bad.any(), (kase, sel[bad][:8], got[bad][:2], exp[sel][bad][:2])
    if kase in (1, 3):
        # both roots must be exercised, or the orientation code is not being tested (case 4 is a
        # linear system: both seeds reach the same point; case 2 is checked through its signs)
        assert 0.2 < hb.root_index.mean() < 0.8


def test_rigid_transform_matches_the_reference(host, gold):
    n_bad = 0
    for i, n in enumerate(gold["rigid_n"]):
        rc, out = H.m3_rigid_transform(gold["rigid_src"][i, :n], gold["rigid_dst"][i, :n])
        assert rc == gold["rigid_rc"][i]
        n_bad += int(not same(out, gold["rigid_out"][i]).all())
        # a proper rotation whatever the inputs
        r = out[:4].reshape(2, 2)
        assert abs(np.linalg.det(r) - 1.0) < 1e-9 and np.allclose(r @ r.T, np.eye(2), atol=1e-9)
    assert n_bad == 0
    assert H.m3_rigid_transform(np.zeros((0, 2)), np.zeros((0, 2)))[0] == 0  # empty input -> nullopt


def test_rigid_transform_recovers_a_known_motion(host):
    rng = np.random.default_rng(5)
    src = rng.uniform(-100, 100, (5, 2))
    th = 0.7
    rot = np.array([[np.cos(th), -np.sin(th)], [np.sin(th), np.cos(th)]])
    dst = src @ rot.T + np.array([30.0, -12.0])
    rc, out = H.m3_rigid_transform(src, dst)
    assert rc == 1
    assert np.allclose(out[:4].reshape(2, 2), rot, atol=1e-12) and np.allclose(out[4:], [30.0, -12.0], atol=1e-9)


def test_pose_score_matches_the_reference(host, gold):
    for i in range(len(gold["score"])):
        got = H.m3_score(gold["score_types"][i], gold["score_canvas"][i], gold["score_pose"][i], gold["score_in"][i])
        exp = float(gold["score"][i])
        # same container, hash and insertion order as the reference's ClusterPose, so the sum runs
        # in the same order: bit-identical
        assert np.float64(got).view(np.uint64) == np.float64(exp).view(np.uint64) or (np.isinf(got) and np.isinf(exp)), (i, got, exp)


def test_degenerate_fixed_line_is_refused_not_guessed(host):
    # fixed line shorter than 1e-9 and no intersection frame: the reference solves a rank-deficient
    # system with L = MIN_LINE_LENGTH; the mirror throws (documented difference)
    row = np.array([[0, 0, 5, 5, 5 + 4e-10, 5 + 3e-10, 3.0, 1.0, 10, 10, 20, 20, 30, 25, 12, 18]], dtype=np.float64)
    rc, *_ = H.m3_pack(3, row)
    assert rc == -1 and "fixed line" in H.last_error()


# ---------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("kase", CASES)
def test_cuda_batch_matches_the_reference(gpu, host, gold, kase):
    rows, exp, exp_ok = gold[f"rows{kase}"], gold[f"out{kase}"], gold[f"ok{kase}"]
    rc, out, ok, launches = H.m3_solve(kase, rows, mode=1)
    assert rc == 0, H.last_error()
    assert launches == 1, "a Merge3 enumeration must cost one launch per kind"
    assert np.array_equal(ok, exp_ok)
    sel = exp_ok == 1
    assert same(out[sel], exp[sel]).all()
    # the north star's coordinate tolerance, spelled out (bit equality above implies it)
    assert np.all(np.abs(out[sel] - exp[sel]) <= 1e-9 * np.maximum(1.0, np.abs(exp[sel])))


@pytest.mark.gpu
@pytest.mark.parametrize("kase", CASES)
def test_cuda_single_call_functions_match_the_reference(gpu, host, gold, kase):
    rows, exp, exp_ok = gold[f"rows{kase}"][:24], gold[f"out{kase}"][:24], gold[f"ok{kase}"][:24]
    rc, out, ok, launches = H.m3_solve(kase, rows, mode=2)
    assert rc == 0, H.last_error()
    assert np.array_equal(ok, exp_ok)
    assert same(out[exp_ok == 1], exp[exp_ok == 1]).all()


def _ref_loops():
    """What the reference build returned for the fresh rows and the PPP merges below (oracle/make_golden_ref_loops.py)."""
    return np.load(os.path.join(os.path.dirname(GOLD), "ref_loops.npz"))


def fresh_rows():
    """Seeded rows beyond merge3.npz, per case, from the fixture's own generators (oracle/make_golden_merge3.py).
    Case 4 leaves out the rows the host refuses: the documented difference, a fixed line shorter than 1e-9 that the
    reference still solves (no intersection frame -> nearest-to-canvas on arbitrary candidates)."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("mg3", os.path.join(os.path.dirname(GOLD), "..", "..", "oracle", "make_golden_merge3.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    mg.N = 2048
    rng = np.random.default_rng(77)
    out = []
    for kase, gen in ((1, mg.rows_pp), (2, mg.rows_line), (3, mg.rows_pl), (4, mg.rows_ll)):
        rows = gen(rng)
        if kase == 4:
            tiny = np.nonzero(np.hypot(rows[:, 2] - rows[:, 0], rows[:, 3] - rows[:, 1]) < 1e-9)[0]
            refused = [i for i in tiny if H.m3_pack(4, rows[i:i + 1])[0] != 0]
            assert len(refused) < 0.01 * len(rows)
            rows = np.delete(rows, refused, axis=0)
        out.append((kase, rows))
    return out


@pytest.mark.gpu
def test_cuda_batch_equals_reference_build_on_fresh_rows(gpu, host):
    """Beyond merge3.npz: 2048 more seeded rows per case against what the reference build returned for them."""
    ref = _ref_loops()
    for kase, rows in fresh_rows():
        rc, out, ok, launches = H.m3_solve(kase, rows, mode=1)
        assert rc == 0 and launches == 1
        assert np.array_equal(ok, ref[f"m3fresh_k{kase}_ok"])
        assert digest(out[ok == 1]) == str(ref[f"m3fresh_k{kase}_out_sha256"]), kase


def _ppp_scenario(rng, n_ref_only=1, n_shared_ra=2, n_shared_rb=2, n_free=2, n_a_only=1, n_b_only=1, lines=True, coincide=False):
    """Three solved clusters of one sketch: a reference cluster and two moving clusters that share
    points with it and with each other.  Every cluster holds the true layout under its own rigid
    motion (a solved cluster is rigid; its frame is arbitrary); the canvas is the true layout under
    another motion, with noise.  Returns (types, canvas4, [cluster 0, 1, 2] as (id, pose4) lists)."""
    groups = {}
    nid = 0
    for name, k in (("r", n_ref_only), ("ra", n_shared_ra), ("rb", n_shared_rb), ("f", n_free), ("a", n_a_only), ("b", n_b_only)):
        groups[name] = list(range(nid, nid + k))
        nid += k
    line_ids = []
    if lines:  # a line inside moving cluster A and one inside the reference: transformed and scored, never an anchor
        line_ids = [nid, nid + 1]
        nid += 2
    true = rng.uniform(-300, 300, size=(nid, 4))
    types = np.zeros(nid, dtype=np.int32)
    for l in line_ids:
        types[l] = 1
    if coincide and groups["f"]:  # a free candidate sitting on a fixed point of A: distance < EPSILON, skipped by the loop
        true[groups["f"][0], :2] = true[groups["ra"][0], :2]

    def motion():
        th = rng.uniform(0, 2 * np.pi)
        c, s = np.cos(th), np.sin(th)
        t = rng.uniform(-500, 500, size=2)
        return lambda p: np.array([c * p[0] - s * p[1] + t[0], s * p[0] + c * p[1] + t[1]])

    def pose_of(ids, mv):
        out = []
        for i in ids:
            p4 = np.zeros(4)
            p4[:2] = mv(true[i, :2])
            if types[i] == 1:
                p4[2:] = mv(true[i, 2:])
            out.append((int(i), p4))
        return out

    ref_ids = groups["r"] + groups["ra"] + groups["rb"] + line_ids[1:2]
    a_ids = groups["ra"] + groups["f"] + groups["a"] + line_ids[0:1]
    b_ids = groups["rb"] + groups["f"] + groups["b"]
    clusters = [pose_of(list(rng.permutation(ids)), motion()) for ids in (ref_ids, a_ids, b_ids)]
    order = rng.permutation(3)  # which child is the reference must not matter: the loop tries all three
    clusters = [clusters[k] for k in order]
    cm = motion()
    canvas4 = np.zeros((nid, 4))
    for i in range(nid):
        canvas4[i, :2] = cm(true[i, :2]) + rng.normal(0, 2.0, size=2)
        if types[i] == 1:
            canvas4[i, 2:] = cm(true[i, 2:]) + rng.normal(0, 2.0, size=2)
    return types, canvas4, clusters


PPP_SHAPES = [dict(), dict(n_shared_ra=3, n_shared_rb=2, n_free=3), dict(n_shared_ra=1, n_shared_rb=1, n_free=1, lines=False),
              dict(n_free=0), dict(n_shared_rb=0), dict(coincide=True), dict(n_shared_ra=3, n_shared_rb=3, n_free=4, n_ref_only=3)]


def ppp_scenarios():
    rng = np.random.default_rng(77)
    return [_ppp_scenario(rng, **kw) for rep in range(6) for kw in PPP_SHAPES]


@pytest.mark.gpu
def test_ppp_merge_enumeration_loop_equals_the_reference_solver(gpu, host):
    """The reference's real candidate enumeration (Merge3PppSolver::solve, merge3_ppp_solver.cpp:18-214:
    reference cluster x shared fixed points x free candidates, one solve2D + pickByTriangleOrientation
    per candidate, two-point anchor placement, merge, score, first best wins) against its batched form
    Gcs::B200::solveMerge3Ppp, which collects every candidate of a merge in a Merge3Batch and solves
    them with ONE kernel launch: the merged pose must come out as the reference's solver returned it
    (tests/golden/ref_loops.npz), bit for bit, over scenarios with 8..72 candidates, lines riding along,
    a coincident candidate the loop skips, and merges without any candidate."""
    ref = _ref_loops()
    scenarios = ppp_scenarios()
    assert len(scenarios) == len(ref["ppp_n"])
    total, at = 0, 0
    for (types, canvas4, clusters), n_ref in zip(scenarios, ref["ppp_n"]):
        ids_ref, pose_ref = ref["ppp_ids"][at:at + n_ref], ref["ppp_pose4"][at:at + n_ref]
        at += n_ref
        n, ids, pose, score, (cands, scored, launches) = H.m3_ppp_merge(types, canvas4, clusters)
        assert n >= 0, H.last_error()
        assert n == n_ref and np.array_equal(ids, ids_ref), (n, n_ref)
        assert same(pose, pose_ref).all(), (pose, pose_ref)
        assert launches == (1 if cands else 0), "every candidate of a merge goes through one launch"
        total += cands
    assert total > 500


# ---- the Merge3 cases with a line in them, the fallback and the case order of a merge node ----
def _m3_scenario(rng, spec, coincide=False, permute=True):
    """Three solved clusters of one sketch.  spec: group -> (points, lines) for the groups r (reference only),
    ra / rb (shared by the reference and moving cluster A / B), f (shared by A and B, outside the reference),
    a / b (A / B only).  Every cluster holds the true layout under its own rigid motion, the canvas the true
    layout under another motion with noise.  Returns (types, canvas4, [cluster 0, 1, 2] as (id, pose4) lists)."""
    groups, types = {}, []
    for name in ("r", "ra", "rb", "f", "a", "b"):
        n_pt, n_ln = spec.get(name, (0, 0))
        groups[name] = list(range(len(types), len(types) + n_pt + n_ln))
        types += [0] * n_pt + [1] * n_ln
    nid = len(types)
    types = np.array(types, dtype=np.int32)
    true = rng.uniform(-300, 300, size=(nid, 4))
    for i in np.nonzero(types == 1)[0]:  # lines of a sensible length
        d = rng.uniform(-1, 1, size=2)
        true[i, 2:] = true[i, :2] + d / np.hypot(*d) * rng.uniform(60, 400)
    if coincide and groups["f"] and groups["ra"]:  # a free point sitting on a fixed point of A
        f0, a0 = groups["f"][0], groups["ra"][0]
        if types[f0] == 0 and types[a0] == 0:
            true[f0, :2] = true[a0, :2]

    def motion():
        th = rng.uniform(0, 2 * np.pi)
        c, s = np.cos(th), np.sin(th)
        t = rng.uniform(-500, 500, size=2)
        return lambda p: np.array([c * p[0] - s * p[1] + t[0], s * p[0] + c * p[1] + t[1]])

    def pose_of(ids, mv):
        out = []
        for i in ids:
            p4 = np.zeros(4)
            p4[:2] = mv(true[i, :2])
            if types[i] == 1:
                p4[2:] = mv(true[i, 2:])
            out.append((int(i), p4))
        return out

    members = (groups["r"] + groups["ra"] + groups["rb"], groups["ra"] + groups["f"] + groups["a"], groups["rb"] + groups["f"] + groups["b"])
    clusters = [pose_of(list(rng.permutation(ids)) if ids else [], motion()) for ids in members]
    if permute:  # which child is the reference must not matter: the loops try all three
        clusters = [clusters[k] for k in rng.permutation(3)]
    cm = motion()
    canvas4 = np.zeros((nid, 4))
    for i in range(nid):
        canvas4[i, :2] = cm(true[i, :2]) + rng.normal(0, 2.0, size=2)
        if types[i] == 1:
            canvas4[i, 2:] = cm(true[i, 2:]) + rng.normal(0, 2.0, size=2)
    return types, canvas4, clusters


P, L = (1, 0), (0, 1)
M3_SHAPES = {
    # two fixed points, a free line
    "pll": [dict(r=(1, 1), ra=(2, 0), rb=(2, 0), f=(0, 2), a=(1, 0), b=(0, 1)), dict(ra=P, rb=P, f=L), dict(ra=(3, 0), rb=(2, 0), f=(0, 3), r=(2, 0)),
            dict(ra=P, rb=P, f=(0, 0)), dict(ra=P, rb=(0, 0), f=L)],
    # a fixed point in one moving cluster, a fixed line in the other, a free point
    "lpp": [dict(r=(1, 0), ra=(2, 0), rb=(0, 2), f=(2, 0), a=(0, 1), b=(1, 0)), dict(ra=P, rb=L, f=P), dict(ra=(0, 2), rb=(3, 0), f=(3, 0), r=(1, 1)),
            dict(ra=(1, 1), rb=(1, 1), f=(2, 0)), dict(ra=P, rb=L, f=(0, 0))],
    # two fixed lines, a free point
    "llp": [dict(r=(1, 0), ra=(0, 2), rb=(0, 2), f=(2, 0), a=(1, 0), b=(0, 1)), dict(ra=L, rb=L, f=P), dict(ra=(0, 3), rb=(0, 2), f=(3, 0), r=(0, 2)),
            dict(ra=L, rb=L, f=(0, 0)), dict(ra=L, rb=(0, 0), f=P)],
}


def _quiet_stderr():
    import contextlib

    @contextlib.contextmanager
    def cm():
        devnull = os.open(os.devnull, os.O_WRONLY)
        saved = os.dup(2)
        os.dup2(devnull, 2)  # the reference prints a line per candidate
        try:
            yield
        finally:
            os.dup2(saved, 2)
            os.close(devnull)
            os.close(saved)
    return cm()


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["pll", "lpp", "llp"])
def test_line_case_enumeration_loops_equal_the_reference_solvers(gpu, host, case):
    """Merge3PllSolver / Merge3LppSolver / Merge3LlpSolver::solve (merge3_pll_solver.cpp:15-189,
    merge3_lpp_solver.cpp:15-208, merge3_llp_solver.cpp:15-190) against their batched forms: every candidate
    of a merge through ONE kernel launch of its kind (K2 / K3 / K4), the merged pose bit for bit - over the
    committed merges of every M3_SHAPES shape (1..36 candidates, passengers of both types, merges without any
    candidate) and what the reference's classes returned for them."""
    scenarios = [g for g in _golden_nodes() if g[0] == case]
    assert len(scenarios) >= 15
    total = 0
    for _, types, canvas4, clusters, n_ref, ids_ref, pose_ref, _ in scenarios:
        n, ids, pose, score, (cands, scored, launches, by) = H.m3_merge(case, types, canvas4, clusters)
        assert n >= 0, H.last_error()
        assert n == n_ref and np.array_equal(ids, ids_ref), (case, n, n_ref)
        assert same(pose, pose_ref).all(), (case, pose, pose_ref)
        assert launches == (1 if cands else 0), "every candidate of a merge goes through one launch"
        total += cands
    assert total > 5 * len(scenarios)


M3_NODE_SHAPES = [
    ("ppp", dict(r=(1, 1), ra=(2, 0), rb=(2, 0), f=(2, 1), a=(1, 0), b=(0, 1))),   # points everywhere: the first case wins
    ("ppp", dict(ra=(1, 1), rb=(1, 1), f=(1, 1))),                                  # every case has candidates: still PPP
    ("pll", dict(ra=(2, 0), rb=(1, 0), f=(0, 2), r=(0, 1))),
    ("pll", dict(ra=(1, 1), rb=(1, 1), f=(0, 1))),                                  # PLL before LLP-style lines
    # a point, a line and a point shared pairwise: the LPP shape - and, seen from another child, the PLL shape
    # (two points with the reference, a line between the moving clusters), which the case order tries first
    ("pll", dict(ra=(1, 0), rb=(0, 1), f=(2, 0), a=(0, 1))),
    ("pll", dict(ra=(0, 2), rb=(2, 0), f=(1, 0))),
    ("llp", dict(ra=(0, 2), rb=(0, 1), f=(2, 0), r=(1, 0))),
    ("unsolvable", dict(ra=(0, 1), rb=(0, 1), f=(0, 1))),                           # three lines: detectUnsolvableMerge3Lll
    ("fallback", dict(ra=(2, 0), rb=(2, 0), f=(0, 0), a=(1, 0))),                   # nothing free: rigid fits over the shared points
    ("fallback", dict(ra=(1, 1), rb=(0, 2), r=(1, 0))),
    ("unsolvable", dict(r=(1, 0), a=(1, 0), b=(1, 0))),                             # nothing shared at all: the fallback has nothing to fit
]


def _golden_merge_nodes():
    """The committed merge-node scenarios as (case the shape is built for, scenario): the fixture holds
    M3_NODE_SHAPES in order, repeated."""
    nodes = [g for g in _golden_nodes() if g[0] == "node"]
    return [(M3_NODE_SHAPES[k % len(M3_NODE_SHAPES)][0], g) for k, g in enumerate(nodes)]


@pytest.mark.gpu
def test_merge_node_case_order_equals_the_reference(gpu, host):
    """What a Merge3 plan node does (bottom_up_plan_solver.cpp:393-431): PPP, PLL, LPP, LLP in that order, the LLL
    detector, the rigid fallback.  Gcs::B200::solveMerge3Node (PPP with its own launch; the three line cases
    enumerated into ONE batch, at most a launch per kind) against what the same sequence over the reference's own
    classes returned for the committed merge nodes: the same case decides and the merged pose is the same bit for bit."""
    names = {0: "ppp", 1: "pll", 2: "lpp", 3: "llp", 4: "fallback", 5: "unsolvable"}
    seen = set()
    for expect, (_, types, canvas4, clusters, n_ref, ids_ref, pose_ref, by_ref) in _golden_merge_nodes():
        n, ids, pose, score, (cands, scored, launches, by) = H.m3_merge("node", types, canvas4, clusters)
        assert n >= 0, H.last_error()
        assert names[by] == names[by_ref] == expect, (expect, names[by], names[by_ref])
        assert n == n_ref and np.array_equal(ids, ids_ref), (expect, n, n_ref)
        assert same(pose, pose_ref).all(), expect
        assert launches <= 4
        seen.add(expect)
    assert seen == {"ppp", "pll", "llp", "fallback", "unsolvable"}  # LPP is shadowed by PLL in this order (see the shapes)


@pytest.mark.gpu
def test_a_level_of_merge_nodes_shares_one_batch(gpu, host):
    """Gcs::B200::solveMerge3Level: every merge node of a plan-tree level - all shapes mixed, the committed merge
    nodes - through ONE Merge3Batch, at most one launch per equation-pair kind for the whole level; node by node the
    result is what the reference's case order over its own classes returned, bit for bit."""
    golden = [g for _, g in _golden_merge_nodes()]
    nodes = [(types, canvas4, clusters) for _, types, canvas4, clusters, *_ in golden]
    rc, got, (n_nodes, cands, launches) = H.m3_level(nodes)
    assert rc == 0, H.last_error()
    assert n_nodes == len(nodes) >= 33 and cands > 2.5 * len(nodes)
    assert launches <= 4, "one launch per kind for the whole level"
    for (_, _, _, _, n_ref, ids_ref, pose_ref, by_ref), (n, ids, pose, by) in zip(golden, got):
        assert by == by_ref and n == n_ref and np.array_equal(ids, ids_ref)
        assert same(pose, pose_ref).all()


def test_fallback_merge_equals_the_reference(host):
    """Merge3FallbackSolver::solve (merge3_fallback_solver.cpp:61-78): child 1, then child 2, fitted onto child 0
    over the elements they share - host arithmetic only, so this one runs without a device.  Over the committed
    fallback merges and the committed merge nodes the fallback decides (their result is the fallback's)."""
    scenarios = [g for g in _golden_nodes() if g[0] == "fallback"] + [g for e, g in _golden_merge_nodes() if e == "fallback"]
    assert len(scenarios) >= 12
    hits = 0
    for _, types, canvas4, clusters, n_ref, ids_ref, pose_ref, _ in scenarios:
        n, ids, pose, score, stats = H.m3_merge("fallback", types, canvas4, clusters)
        assert n >= 0, H.last_error()
        assert n == n_ref and np.array_equal(ids, ids_ref), (n, n_ref)
        assert same(pose, pose_ref).all()
        assert stats[2] == 0  # no kernel launch
        hits += n > 0
    assert hits > 0.2 * len(scenarios)


def test_a_level_without_candidates_needs_no_device(host):
    """solveMerge3Level on nodes that no enumeration has a candidate for (the fallback's and the unsolvable shapes,
    and no node at all): nothing is packed, nothing is launched - so this runs without a device - and every node
    is the reference's outcome."""
    rc, got, stats = H.m3_level([])
    assert rc == 0 and got == [] and stats == (0, 0, 0)
    chosen = [(e, g) for e, g in _golden_merge_nodes() if e in ("fallback", "unsolvable")]
    assert len(chosen) >= 9
    nodes = [(types, canvas4, clusters) for _, (_, types, canvas4, clusters, *_) in chosen]
    rc, got, (n_nodes, cands, launches) = H.m3_level(nodes)
    assert rc == 0, H.last_error()
    assert (n_nodes, cands, launches) == (len(nodes), 0, 0)
    names = {4: "fallback", 5: "unsolvable"}
    for (expect, (_, _, _, _, n_ref, ids_ref, pose_ref, by_ref)), (n, ids, pose, by) in zip(chosen, got):
        assert names[by] == names[by_ref] == expect
        assert n == n_ref and np.array_equal(ids, ids_ref) and same(pose, pose_ref).all()


# ---- golden merge nodes: outputs of the reference's own solver classes, committed (oracle/make_golden_merge3_nodes.py) ----
def _golden_nodes():
    z = np.load(os.path.join(os.path.dirname(GOLD), "merge3_nodes.npz"))
    names = {v: k for k, v in H.M3_CASES.items()}
    el0 = mem0 = out0 = 0
    for k in range(len(z["which"])):
        n_el, counts, n = int(z["n_el"][k]), z["counts"][k], int(z["ref_n"][k])
        types, canvas4 = z["types"][el0:el0 + n_el], z["canvas4"][el0:el0 + n_el]
        clusters, at = [], mem0
        for c in counts:
            clusters.append([(int(i), p) for i, p in zip(z["ids"][at:at + c], z["pose4"][at:at + c])])
            at += int(c)
        yield names[int(z["which"][k])], types, canvas4, clusters, n, z["ref_ids"][out0:out0 + n], z["ref_pose4"][out0:out0 + n], int(z["ref_by"][k])
        el0, mem0, out0 = el0 + n_el, at, out0 + n


def test_golden_fallback_nodes(host):
    """The committed reference outputs of Merge3FallbackSolver::solve: host arithmetic only, no device."""
    seen = 0
    for which, types, canvas4, clusters, n_ref, ids_ref, pose_ref, by_ref in _golden_nodes():
        if which != "fallback":
            continue
        n, ids, pose, score, stats = H.m3_merge(which, types, canvas4, clusters)
        assert n == n_ref and np.array_equal(ids, ids_ref) and same(pose, pose_ref).all()
        seen += 1
    assert seen >= 6


@pytest.mark.gpu
def test_golden_merge_nodes(gpu, host):
    """Every committed scenario - the four enumeration loops, the fallback, the merge node - against what the
    reference's own classes returned when the fixture was generated: merged pose bit for bit, same deciding case.
    Needs no oracle/_ref at run time."""
    seen = {}
    for which, types, canvas4, clusters, n_ref, ids_ref, pose_ref, by_ref in _golden_nodes():
        n, ids, pose, score, stats = H.m3_merge(which, types, canvas4, clusters)
        assert n >= 0, H.last_error()
        assert n == n_ref and np.array_equal(ids, ids_ref), (which, n, n_ref)
        assert same(pose, pose_ref).all(), which
        if which == "node":
            assert stats[3] == by_ref
        seen[which] = seen.get(which, 0) + 1
    assert set(seen) == {"ppp", "pll", "lpp", "llp", "fallback", "node"} and sum(seen.values()) == 90
