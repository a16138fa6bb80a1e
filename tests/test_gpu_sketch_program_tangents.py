"""Sketch-program tangents on the GPU: a tangent run leaves the positions of a plain run untouched,
its tangents equal a wave-by-wave CPU restatement (numpy gather + gcs_oracle_solve + the tangent
restatement of tests/tangent_oracle.py) bit for bit, and they are the derivatives of the positions: central differences
through the program agree with them, and every satisfied constraint's linearisation holds."""

import ctypes as C

import numpy as np
import pytest

import host_lib as H
import oracle_lib as O
import program_tangents_lib as P
import sketch_gen as S
from test_gpu_host import WHOLE_SKETCHES, _ref_loops, _triangle_strip
from program_restate import restate, rows
from util import bits, digest

pytestmark = pytest.mark.gpu

@pytest.fixture(scope="module")
def host(gpu, built):
    built.build_host()
    return H.load()


def _same(a, b):
    return bool(((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))).all())


def _golden(seed, first, n):
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    return el, S.sketch_graph(el, lv)


def _directions(nv, K, T, seed):
    return np.random.default_rng(seed).standard_normal((K, nv, T))


# ---- 1. the primal is untouched ----

@pytest.mark.parametrize("case", ["sketch31", "sketch32", "sketch33", "linkage100k", "unchecked6000"])
def test_a_tangent_run_leaves_the_positions_of_a_plain_run(host, case):
    if case == "linkage100k":
        el, edges = S.make_linkage(100000, seed=4)
    elif case == "unchecked6000":
        el, edges = S.make_linkage_unchecked(6000, seed=4)
    else:
        el, edges = _golden(*WHOLE_SKETCHES[int(case[-1]) - 1])
    prog = P.Program(el, edges)
    vals = P.sketch_values(edges)[None, :]
    rc, pos, nc, _ = prog.run(vals)
    rc2, tpos, dpos, tnc, _ = prog.run_tangents(vals, _directions(vals.shape[1], 1, 2, seed=1))
    assert rc == rc2 == 0, H.last_error()
    assert _same(pos, tpos) and np.array_equal(nc, tnc)
    if case == "linkage100k":
        xy = np.ascontiguousarray(tpos[0, :, :2])
        assert digest(xy) == str(_ref_loops()["config4_xy_sha256"])
        assert np.isfinite(dpos).all()


# ---- 2. device equals the CPU restatement, bit for bit ----

def _desc_run(desc, vals, dvals, gcs):
    """gcs_b200_program_run_tangents_host on a C-ABI program built from `desc`."""
    lib = gcs.capi.load()
    h = C.c_void_p()
    assert lib.gcs_b200_program_create(C.byref(desc), 0, C.byref(h)) == 0, lib.gcs_b200_last_error()
    K, T = dvals.shape[0], dvals.shape[2]
    pos = np.zeros((K, desc.n_slots, 4))
    dpos = np.zeros((K, desc.n_slots, 4, T))
    nc = np.zeros(K, dtype=np.uint32)
    vals, dvals = np.ascontiguousarray(vals), np.ascontiguousarray(dvals)
    try:
        rc = lib.gcs_b200_program_run_tangents_host(h, K, vals.ctypes.data, pos.ctypes.data, nc.ctypes.data, T, dvals.ctypes.data,
                                                    dpos.ctypes.data, 0, None)
        assert rc == 0, lib.gcs_b200_last_error()
    finally:
        lib.gcs_b200_program_destroy(h)
    return pos, dpos, nc


def _leaf_program(seed, first, n):
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    return P.Program(el, leaves=lv), np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])


@pytest.mark.parametrize("seed,first,n", WHOLE_SKETCHES)
def test_device_tangents_equal_the_cpu_restatement(host, gcs, seed, first, n):
    """The leaf lists of the golden sketches (all eight solvers occur across them); K = 4 instances,
    values moved by up to 1e-7 relative, T = 3 random directions; cos values and d(cos) directions
    computed here.  Every position and every tangent equal, NaN with NaN."""
    prog, base = _leaf_program(seed, first, n)
    assert prog.rc == 0, prog.error
    desc = prog.desc()
    rng = np.random.default_rng(seed)
    K, T = 4, 3
    v = base * (1.0 + 1e-7 * rng.uniform(-1, 1, size=(K, len(base))))
    dv = rng.standard_normal((K, len(base), T))
    angle = np.array([desc.value_is_angle[i] for i in range(desc.n_values)], dtype=bool)
    cv = np.where(angle, np.cos(v), v)
    dcv = np.where(angle[None, :, None], -np.sin(v)[:, :, None] * dv, dv)
    pos, dpos, nc = _desc_run(desc, cv, dcv, gcs)
    want, dwant, wnc = restate(desc, cv, dcv)
    assert _same(pos, want)
    assert _same(dpos, dwant)
    assert np.array_equal(nc, wnc)
    assert set(rows(desc)["solver"]) <= set(range(1, 9))


def test_all_solvers_occur_in_the_restated_sketches(host):
    solvers = set()
    for case in WHOLE_SKETCHES:
        solvers |= set(int(s) for s in _leaf_program(*case)[0].describe()["row_solver"])
    assert solvers == set(range(1, 9))


# ---- 3. central differences through the program ----

def _central(prog, vals, T, seed):
    """One run of 2T instances at v +- h_t dir_t, h_t = 1e-3 / max(1, largest finite |tangent| along t)
    so that no position moves by more than 1e-3, and runTangents along the directions those value sets
    actually differ by, (v+ - v-) / 2h_t (with tangents of 1e9, h_t is small enough for the rounding
    of v +- h_t dir_t to matter)."""
    dirs = vals[None, :] * np.random.default_rng(seed).standard_normal((T, len(vals)))
    rc, _, dpos, _, _ = prog.run_tangents(vals[None, :], dirs.T[None, :, :])
    assert rc == 0, H.last_error()
    big = np.where(np.isfinite(dpos[0]), np.abs(dpos[0]), 0.0).reshape(-1, T).max(axis=0)
    h = 1e-3 / np.maximum(1.0, big)
    vp, vm = vals + h[:, None] * dirs, vals - h[:, None] * dirs
    rc, pos, dpos, _, _ = prog.run_tangents(vals[None, :], np.ascontiguousarray(((vp - vm) / (2 * h[:, None])).T[None, :, :]))
    assert rc == 0, H.last_error()
    rc, pm, _, _ = prog.run(np.concatenate([vp, vm]))
    assert rc == 0, H.last_error()
    return pos[0], dpos[0], pm[:T], pm[T:], h


@pytest.mark.parametrize("case", ["sketch31", "sketch32", "sketch33", "strip"])
def test_tangents_agree_with_central_differences_through_the_program(host, case):
    """Directions: each value times a normal random number; the step h_t keeps every position change
    within 1e-3 (the linkages' tangents reach 1e6: a fixed step leaves the linear range).  Tolerance
    1e-4 max(1, |tangent|) (the difference quotient carries the chain's rounding amplified by 1/h).  A
    coordinate whose +- positions are more than 0.1 apart, far beyond 2e-3, took another root on one
    side (a root flip): excluded and counted; none on the strip.  NaN tangents (rows without a
    derivative) are excluded too.
    The linkages are not in this list: their tangents span 1 to 1e9 along one direction, and no single
    step resolves the insensitive coordinates above their rounding while keeping the sensitive ones
    linear (profiles/r4_sketch_program_tangents.md: up to 2.8 relative on the 100 k linkage, 0.03 on
    the 20 k one).  test_the_linearised_constraints_hold checks their tangents exactly instead."""
    if case == "strip":
        _, el, lv = _triangle_strip(402)
        prog = P.Program(el, leaves=lv)
        vals = np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])
    else:
        el, edges = _golden(*WHOLE_SKETCHES[int(case[-1]) - 1])
        prog = P.Program(el, edges)
        vals = P.sketch_values(edges)
    T = 3
    pos, dpos, pp, pm, h = _central(prog, vals, T, seed=3)
    jumps = nan = compared = 0
    for t in range(T):
        tan = dpos[..., t]
        flip = np.abs(pp[t] - pm[t]) > 0.1
        ok = np.isfinite(tan) & np.isfinite(pp[t]) & np.isfinite(pm[t]) & ~flip
        fd = (pp[t] - pm[t]) / (2 * h[t])
        bad = ok & ~(np.abs(fd - tan) <= 1e-4 * np.maximum(1.0, np.abs(tan)))
        assert not bad.any(), (case, t, np.argwhere(bad)[:5], fd[bad][:5], tan[bad][:5])
        jumps += int((flip & np.isfinite(tan)).sum())
        nan += int((~np.isfinite(tan)).sum())
        compared += int(ok.sum())
    print(f"{case}: {compared} coordinates compared, {jumps} excluded as root flips, {nan} without a derivative")
    assert compared > 0
    if case == "strip":
        assert jumps == 0 and nan == 0


# ---- 4. linearised constraints ----

def _constraint_tangents(el, edges, pos, dpos, vals, dvals):
    """For every distance and angle constraint the solved positions satisfy to 1e-9 relative: (the
    tangent of its constraint function, its value tangent, a scale for the comparison)."""
    out = []
    real = [e for e in edges if e["type"] != S.VIRT]
    for v, e in enumerate(real):
        a, b = e["a"], e["b"]
        ta, tb = el[a]["type"], el[b]["type"]
        A, B, dA, dB = pos[a], pos[b], dpos[a], dpos[b]
        if not (np.isfinite(dA).all() and np.isfinite(dB).all()):
            continue
        if e["type"] == S.DIST and ta == S.P and tb == S.P:
            u = A[:2] - B[:2]
            f = np.hypot(*u)
            if abs(f - vals[v]) > 1e-9 * max(1.0, vals[v]):
                continue
            lhs = u @ (dA[:2] - dB[:2])
            out.append((lhs, f * dvals[v], max(1.0, f) * max(1.0, np.abs(dA).max() + np.abs(dB).max())))
        elif e["type"] == S.DIST and ta != tb:
            (Pp, dP), (L, dL) = ((A, dA), (B, dB)) if ta == S.P else ((B, dB), (A, dA))
            ex, ey, dex, dey = L[2] - L[0], L[3] - L[1], dL[2] - dL[0], dL[3] - dL[1]
            wx, wy, dwx, dwy = Pp[0] - L[0], Pp[1] - L[1], dP[0] - dL[0], dP[1] - dL[1]
            n = np.hypot(ex, ey)
            cr = ex * wy - ey * wx
            g = cr / n
            if abs(abs(g) - vals[v]) > 1e-9 * max(1.0, vals[v]):
                continue
            dcr = (dex * wy + ex * dwy) - (dey * wx + ey * dwx)
            dn = (ex * dex + ey * dey) / n
            dg = (dcr - g * dn) / n
            scale = max(1.0, np.abs(dP).max() + np.abs(dL).max()) * (1.0 + np.hypot(wx, wy) / n)
            out.append((np.sign(g) * dg, dvals[v], scale))
        elif e["type"] == S.ANG and ta == S.L and tb == S.L:
            d1, d2 = A[2:] - A[:2], B[2:] - B[:2]
            dd1, dd2 = dA[2:] - dA[:2], dB[2:] - dB[:2]
            n1, n2 = np.hypot(*d1), np.hypot(*d2)
            c = (d1 @ d2) / (n1 * n2)
            s = 1.0 if abs(c - np.cos(vals[v])) <= abs(c + np.cos(vals[v])) else -1.0
            if abs(c - s * np.cos(vals[v])) > 1e-9:
                continue
            dc = (dd1 @ d2 + d1 @ dd2) / (n1 * n2) - c * ((d1 @ dd1) / n1 ** 2 + (d2 @ dd2) / n2 ** 2)
            out.append((dc, s * -np.sin(vals[v]) * dvals[v], max(1.0, np.abs(dd1).max() / n1 + np.abs(dd2).max() / n2)))
    return out


@pytest.mark.parametrize("case", ["sketch31", "sketch32", "sketch33", "linkage20k", "linkage100k"])
def test_the_linearised_constraints_hold(host, case):
    """T = 4 random directions over all values (radians for angles).  Point-point: (P-Q).(P'-Q') = d d';
    point-line: the signed distance's tangent, signed like the solved distance, equals d'; angle:
    the tangent of cos(angle) equals -sin(theta) theta', signed like the solved configuration.
    Tolerance 1e-9 relative to the scale of the tangents involved."""
    if case.startswith("linkage"):
        el, edges = S.make_linkage(100000, seed=4) if case == "linkage100k" else S.make_linkage(20000, seed=6)
    else:
        el, edges = _golden(*WHOLE_SKETCHES[int(case[-1]) - 1])
    prog = P.Program(el, edges)
    vals = P.sketch_values(edges)
    T = 4
    dv = _directions(len(vals), 1, T, seed=5)
    rc, pos, dpos, nc, _ = prog.run_tangents(vals[None, :], dv)
    assert rc == 0, H.last_error()
    checked = 0
    for t in range(T):
        for lhs, rhs, scale in _constraint_tangents(el, edges, pos[0], dpos[0, ..., t], vals, dv[0, :, t]):
            assert abs(lhs - rhs) <= 1e-9 * scale, (case, t, lhs, rhs, scale)
            checked += 1
    print(f"{case}: {checked} constraint tangents checked")
    assert checked > 0


# ---- 5. independence ----

def test_each_direction_and_each_instance_is_independent(host):
    el, lv = S.make_sketch(3000, seed=32, first_shape=2)
    edges = S.sketch_graph(el, lv)
    prog = P.Program(el, edges)
    base = P.sketch_values(edges)
    rng = np.random.default_rng(7)
    u = rng.uniform(-1.0, 1.0, size=(257, len(base)))
    is_angle = np.array([e["type"] == S.ANG for e in edges if e["type"] != S.VIRT])
    vals = np.where(is_angle, base + 1e-2 * u, base * (1.0 + 1e-3 * u))
    vals[0] = base
    dv = rng.standard_normal((257, len(base), 8))
    rc, full, dfull, ncf, _ = prog.run_tangents(vals, dv)
    assert rc == 0, H.last_error()
    for t in (0, 5, 7):  # column t of T = 8 is a T = 1 run along direction t
        rc, _, d1, _, _ = prog.run_tangents(vals[:5], np.ascontiguousarray(dv[:5, :, t:t + 1]))
        assert rc == 0 and _same(d1[..., 0], dfull[:5, ..., t]), t
    for K in (1, 3, 33):
        rc, pos, d, nc, _ = prog.run_tangents(vals[:K], dv[:K])
        assert rc == 0 and _same(pos, full[:K]) and _same(d, dfull[:K]) and np.array_equal(nc, ncf[:K]), K
    rc, pos, d, nc, _ = prog.run_tangents(vals[100:101], dv[100:101])
    assert rc == 0 and _same(d[0], dfull[100]) and nc[0] == ncf[100]
    rc, pos, d, nc, _ = prog.run_tangents(vals[::-1].copy(), dv[::-1].copy())
    assert rc == 0 and _same(d, dfull[::-1]) and np.array_equal(nc, ncf[::-1])


# ---- 6. an unrealisable instance ----

def test_rows_without_a_root_have_nan_tangents_and_leave_their_neighbours_alone(host, gcs):
    """The instance of test_an_unrealisable_instance_is_reported_and_leaves_its_neighbours_alone: the
    rows whose chosen run the oracle finds unconverged, re-solving from the final positions, are
    exactly `nonconverged` many, and their targets' tangents are NaN; instances 0 and 2 are finite and
    equal their single-instance runs bit for bit."""
    el, edges = S.make_linkage(3000, seed=11)
    prog = P.Program(el, edges)
    d = prog.describe()
    vals = np.repeat(P.sketch_values(edges)[None, :], 3, axis=0)
    r = d["rows"] // 2
    v1 = int(d["row_values"][r][1])
    vals[1, v1] = 1e4 * vals[1, v1]
    dv = _directions(vals.shape[1], 3, 2, seed=8)
    rc, pos, dpos, nc, _ = prog.run_tangents(vals, dv)
    assert rc == 0, H.last_error()
    assert nc[0] == 0 and nc[2] == 0 and nc[1] > 0
    rows = np.arange(d["rows"])
    solver = d["row_solver"]
    a, b = d["row_elems"][:, 0], d["row_elems"][:, 1]
    p, v = pos[1], vals[1]
    zero = solver == 1
    cols = [np.where(zero, 0.0, p[a, 0]), np.where(zero, 0.0, p[a, 1]), v[d["row_values"][:, 1]],
            np.where(zero, v[np.maximum(d["row_values"][:, 0], 0)], p[b, 0]), np.where(zero, 0.0, p[b, 1]), v[d["row_values"][:, 2]]]
    hb = gcs.capi.HostBatch(1, 2, [np.ascontiguousarray(c) for c in cols], np.ascontiguousarray(d["row_code"]))
    O.solve(hb.alloc_outputs())
    failed = hb.converged[hb.root_index.astype(np.int64), rows] == 0
    assert int(failed.sum()) == int(nc[1])
    targets = d["row_elems"][failed, 2]
    assert np.isnan(dpos[1, targets, :2]).all()
    for k in (0, 2):
        assert np.isfinite(dpos[k]).all()
        rc, p1, d1, n1, _ = prog.run_tangents(vals[k:k + 1], dv[k:k + 1])
        assert rc == 0 and _same(p1[0], pos[k]) and _same(d1[0], dpos[k]) and n1[0] == 0


# ---- 7. launches, 8. devices, 9. the contracted class ----

def test_launches_of_a_tangent_run_add_at_most_one_per_wave(host):
    el, lv = S.make_sketch(3000, seed=31, first_shape=1)
    edges = S.sketch_graph(el, lv)
    prog = P.Program(el, edges)
    waves = prog.describe()["waves"]
    vals = np.repeat(P.sketch_values(edges)[None, :], 257, axis=0)
    dv = _directions(vals.shape[1], 257, 8, seed=2)
    rc, _, _, plain = prog.run(vals[:1])
    launches = set()
    for K, T in ((1, 1), (1, 8), (257, 1), (257, 8)):
        rc2, _, _, _, st = prog.run_tangents(vals[:K], np.ascontiguousarray(dv[:K, :, :T]))
        assert rc == rc2 == 0
        launches.add(st["launches"])
    assert len(launches) == 1 and plain["launches"] < launches.pop() <= plain["launches"] + waves


def test_tangents_do_not_depend_on_the_device_count(host, gcs):
    ndev = gcs.capi.load().gcs_b200_device_count()
    el, edges = S.make_linkage(20000, seed=6)
    prog = P.Program(el, edges)
    vals = np.repeat(P.sketch_values(edges)[None, :], 8, axis=0)
    vals *= 1.0 + 1e-4 * np.random.default_rng(9).uniform(-1, 1, size=vals.shape)
    dv = _directions(vals.shape[1], 8, 4, seed=9)
    rc, one, d1, nc1, _ = prog.run_tangents(vals, dv, n_devices=1)
    rc2, many, dm, ncm, _ = prog.run_tangents(vals, dv, n_devices=ndev)
    assert rc == rc2 == 0 and _same(one, many) and _same(d1, dm) and np.array_equal(nc1, ncm)


def test_the_contracted_class_agrees_on_tangents(host):
    """The contracted class on the 400-leaf strip: positions within 1e-9 and tangents within 1e-8
    relative of the bit-identical class (the tangent of a chain amplifies the positions' differences by
    the same factor it amplifies their derivatives).  Every contracted variant: GCS_VARIANT_CONTRACTED
    and the explicit mappings _STATIC, _SORTED, _SEQ and _LINEAR."""
    pts, el, lv = _triangle_strip(402)
    prog = P.Program(el, leaves=lv)
    vals = np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])
    u = np.random.default_rng(2).uniform(-1.0, 1.0, size=(4, len(vals)))
    vals = vals * (1.0 + 1e-7 * u)
    dv = _directions(vals.shape[1], 4, 3, seed=4)
    rc, base, dbase, nc_base, _ = prog.run_tangents(vals, dv)
    assert rc == 0 and not nc_base.any()
    scale = max(1.0, float(np.abs(dbase).max()))
    pscale = max(1.0, float(np.abs(base[:, :, :2]).max()))
    for variant in (5, 6, 7, 8, 10):
        old = host.gcs_host_set_variant(variant)
        try:
            rc2, fast, dfast, nc_fast, _ = prog.run_tangents(vals, dv)
        finally:
            host.gcs_host_set_variant(old)
        assert rc2 == 0 and np.array_equal(nc_base, nc_fast), variant
        assert float(np.abs(base[:, :, :2] - fast[:, :, :2]).max()) / pscale <= 1e-9, variant
        worst = float(np.abs(dbase - dfast).max()) / scale
        print(f"contracted variant {variant}: tangents within {worst:.3e} relative")
        assert worst <= 1e-8, (variant, worst)
