"""Sketch-program fits on the GPU: the device equals the CPU restatement (tests/program_restate_fit.py)
bit for bit, recovers the values that produced its targets, reaches the least-squares optimum, keeps
every instance independent, returns a plain run's positions, respects boxes and refuses trials that
break a row."""
import ctypes as C

import numpy as np
import pytest

import host_lib as H
import program_fit_lib as F
import sketch_gen as S
from program_restate import Arrays
from program_restate_fit import COST, FTOL, GTOL, START_FAILED, XTOL, Fit, restate_fit
from test_gpu_host import WHOLE_SKETCHES, _triangle_strip
from util import bits

pytestmark = pytest.mark.gpu
CONVERGED = (COST, GTOL, FTOL, XTOL)


@pytest.fixture(scope="module")
def host(gpu, built):
    built.build_host()
    return H.load()


def _same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return bool(((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))).all())


def _same_results(got, want):
    for g, w in zip(got, want):
        assert g["status"] == w["status"] and g["iterations"] == w["iterations"], (g, w)
        assert _same([g["cost"], g["grad_inf"], g["lambda_"]], [w["cost"], w["grad_inf"], w["lambda_"]]), (g, w)


def _golden(case):
    """the solvable part of a golden sketch's leaf list, its values (C-ABI units) [1][n_values]"""
    seed, first, n = case
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    prog = F.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    p = Arrays.from_desc(prog.desc())
    base = np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])
    cv = np.where(p.value_is_angle.astype(bool), np.cos(base), base)[None]
    return F.solvable(p, cv), cv


def _starts(dp, cv, free, K, rng, lo=1e-3, hi=1e-2):
    """K starts: cv with the free values moved by lo .. hi relative, each drawn until it solves every row"""
    out = np.repeat(cv, K, axis=0)
    for k in range(K):
        for _ in range(50):
            x = cv[0, free] * (1.0 + rng.uniform(lo, hi, len(free)) * rng.choice([-1.0, 1.0], len(free)))
            out[k, free] = x
            if dp.run(out[k:k + 1])[1][0] == 0:
                break
        else:
            raise AssertionError("no solvable start")
    return out


# ---- 1. bit for bit with the restatement; 5. final positions; 4. independence ----

@pytest.mark.parametrize("case", WHOLE_SKETCHES)
@pytest.mark.parametrize("reach", ["reachable", "unreachable"])
def test_device_fit_equals_the_cpu_restatement(host, case, reach):
    p, cv = _golden(case)
    free, os_, oc, _ = F.problem(p, cv, 5, seed=case[0])
    rng = np.random.default_rng(case[0])
    dp = F.DescProgram(p)
    K = 4
    start = _starts(dp, cv, free, K, rng)
    if reach == "reachable":
        moved = _starts(dp, cv, free, K, rng)
        targets = dp.run(moved)[0][:, os_, oc]
    else:
        pos = dp.run(cv)[0][0, os_, oc]
        targets = pos[None] + rng.standard_normal((K, len(os_))) * (1e-2 * (1.0 + np.abs(pos)))
    fit = Fit(free, os_, oc, weights=rng.uniform(0.5, 2.0, len(os_)), max_iterations=10)
    rc, vals, pos, nc, res = dp.fit(start, targets, fit)
    assert rc == 0, F.capi.load().gcs_b200_last_error()
    wv, wpos, wnc, wres = restate_fit(p, start, targets, fit)
    assert _same(vals, wv) and _same(pos, wpos) and np.array_equal(nc, wnc)
    _same_results(res, wres)
    assert p.value_is_angle[free].any() or not p.value_is_angle[p.rows["value"][p.rows["value"] >= 0]].any()
    # 5: positions and counts are those of a plain run at the returned values
    ppos, pnc = dp.run(vals)
    assert _same(pos, ppos) and np.array_equal(nc, pnc)
    # 4: an instance alone, the instances reversed, and other targets for the other instances
    rc, v1, p1, _, r1 = dp.fit(start[2:3], targets[2:3], fit)
    assert rc == 0 and _same(v1[0], vals[2]) and _same(p1[0], pos[2])
    _same_results(r1, res[2:3])
    rc, vr, _, _, rr = dp.fit(start[::-1], targets[::-1], fit)
    assert rc == 0 and _same(vr, vals[::-1])
    _same_results(rr, res[::-1])
    other = targets.copy()
    other[[0, 1, 3]] += 1.0
    rc, vo, _, _, ro = dp.fit(start, other, fit)
    assert rc == 0 and _same(vo[2], vals[2])
    _same_results(ro[2:3], res[2:3])


def test_all_solvers_occur_in_the_fitted_programs(host):
    solvers = set()
    for case in WHOLE_SKETCHES:
        solvers |= set(int(s) for s in _golden(case)[0].rows["solver"])
    assert solvers == set(range(1, 9))


# ---- 2. recovery ----

@pytest.mark.parametrize("case", WHOLE_SKETCHES)
def test_the_fit_recovers_the_values_of_its_targets_on_the_golden_sketches(host, case):
    p, cv = _golden(case)
    free, os_, oc, J = F.problem(p, cv, 8, seed=7)
    assert np.linalg.matrix_rank(J) == len(free)
    dp = F.DescProgram(p)
    rng = np.random.default_rng(11)
    K = 8
    start = _starts(dp, cv, free, K, rng)
    targets = np.repeat(dp.run(cv)[0][:, os_, oc], K, axis=0)
    rc, vals, _, nc, res = dp.fit(start, targets, Fit(free, os_, oc, max_iterations=60))
    assert rc == 0
    assert all(r["status"] in CONVERGED for r in res), res
    assert not nc.any()
    err = np.abs(vals[:, free] - cv[:, free]) / np.maximum(np.abs(cv[:, free]), 1e-300)
    assert err.max() <= 1e-9, err.max()


def _linkage_fit(n, seed, K, n_free, rng_seed):
    el, edges = S.make_linkage(n, seed=seed)
    prog = F.Program(el, edges)
    v = F.sketch_values(edges)
    p = Arrays.from_desc(prog.desc())
    cv = np.where(p.value_is_angle.astype(bool), np.cos(v), v)[None]
    free, os_, oc, J = F.problem(p, cv, n_free, seed=rng_seed)
    assert np.linalg.matrix_rank(J) == n_free
    rc, pos, nc, _ = prog.run(v[None])
    assert rc == 0 and nc[0] == 0
    rng = np.random.default_rng(rng_seed)
    start = np.repeat(v[None], K, axis=0)
    for k in range(K):
        for _ in range(50):
            start[k, free] = v[free] * (1.0 + rng.uniform(1e-3, 1e-2, n_free) * rng.choice([-1.0, 1.0], n_free))
            if prog.run(start[k:k + 1])[2][0] == 0:
                break
    targets = np.repeat(pos[:, os_, oc], K, axis=0)
    return prog, v, start, targets, Fit(free, os_, oc, max_iterations=30)


@pytest.mark.parametrize("n,seed,K,n_free", [(20000, 6, 16, 8), (100000, 4, 1, 8)])
def test_the_fit_recovers_the_values_of_its_targets_on_the_linkages(host, n, seed, K, n_free):
    prog, v, start, targets, fit = _linkage_fit(n, seed, K, n_free, rng_seed=5)
    rc, vals, pos, nc, res, st = prog.fit(start, targets, fit)
    assert rc == 0, H.last_error()
    assert all(r["status"] in CONVERGED for r in res), res
    err = np.abs(vals[:, fit.free] - v[fit.free]) / np.abs(v[fit.free])
    assert err.max() <= 1e-9, err.max()
    rc, ppos, pnc, _ = prog.run(vals)
    assert rc == 0 and _same(pos, ppos) and np.array_equal(nc, pnc)
    if K == 1:
        # launches: one more iteration costs one tangent run + 2
        tan = prog.run_tangents(start, np.zeros((1, len(v), n_free)))[4]["launches"]
        counts = []
        for m in (2, 3):
            f = Fit(fit.free, fit.obs_slots, fit.obs_coords, max_iterations=m, xtol=0.0, ftol=0.0)
            counts.append(prog.fit(start, targets, f)[5]["launches"])
        assert counts[1] - counts[0] == tan + 2, (counts, tan)


# ---- 3. the least-squares optimum ----

def test_unreachable_targets_end_at_the_least_squares_optimum(host):
    from scipy.optimize import least_squares
    p, cv = _golden(WHOLE_SKETCHES[0])
    free, os_, oc, _ = F.problem(p, cv, 4, seed=3, max_obs=24)
    dp = F.DescProgram(p)
    rng = np.random.default_rng(4)
    pos0 = dp.run(cv)[0][0, os_, oc]
    targets = (pos0 + 1e-3 * (1.0 + np.abs(pos0)) * rng.standard_normal(len(os_)))[None]
    w = rng.uniform(0.5, 2.0, len(os_))
    fit = Fit(free, os_, oc, weights=w, max_iterations=40)
    rc, vals, _, _, res = dp.fit(cv, targets, fit)
    assert rc == 0 and res[0]["status"] in CONVERGED, res
    sel = np.zeros((1, p.n_values, len(free)))
    sel[0, free, np.arange(len(free))] = 1.0

    def at(x):
        v = cv.copy()
        v[0, free] = x
        return v

    def fun(x):
        return np.sqrt(w) * (dp.run(at(x))[0][0, os_, oc] - targets[0])

    def jac(x):
        return np.sqrt(w)[:, None] * dp.tangents(at(x), sel)[1][0, os_, oc, :]

    ls = least_squares(fun, cv[0, free], jac=jac, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15)
    assert abs(res[0]["cost"] - 2 * ls.cost) <= 1e-9 * 2 * ls.cost, (res[0]["cost"], 2 * ls.cost)
    costs = []
    for m in range(1, 9):
        fit.max_iterations = m
        rc, _, _, _, r = dp.fit(cv, targets, fit)
        costs.append(r[0]["cost"])
    assert all(b <= a for a, b in zip(costs, costs[1:])), costs


# ---- 4. the early stop of the _host entry point and the device entry point ----

def test_the_host_entry_point_equals_the_device_entry_point(host):
    import torch
    p, cv = _golden(WHOLE_SKETCHES[1])
    free, os_, oc, _ = F.problem(p, cv, 4, seed=2)
    dp = F.DescProgram(p)
    rng = np.random.default_rng(6)
    K = 3
    start = _starts(dp, cv, free, K, rng)
    targets = np.repeat(dp.run(cv)[0][:, os_, oc], K, axis=0)
    fit = Fit(free, os_, oc, max_iterations=25)
    rc, vals, pos, nc, res = dp.fit(start, targets, fit)
    assert rc == 0 and all(r["status"] in CONVERGED for r in res)
    dev = torch.device("cuda", 0)
    v = torch.from_numpy(start.copy()).to(dev)
    t = torch.from_numpy(targets).to(dev)
    dpos = torch.empty((K, p.n_slots, 4), dtype=torch.float64, device=dev)
    dnc = torch.empty(K, dtype=torch.int32, device=dev)
    dres = torch.empty((K, C.sizeof(F.capi.CFitResult)), dtype=torch.uint8, device=dev)
    lib = F.capi.load()
    rc = lib.gcs_b200_program_fit(dp.h, C.byref(F.cfit(fit)), K, v.data_ptr(), t.data_ptr(), dpos.data_ptr(), dnc.data_ptr(),
                                  dres.data_ptr(), 0, None)
    assert rc == 0, lib.gcs_b200_last_error()
    torch.cuda.synchronize()
    raw = dres.cpu().numpy().tobytes()
    dr = F.results((F.capi.CFitResult * K).from_buffer_copy(raw))
    assert _same(v.cpu().numpy(), vals) and _same(dpos.cpu().numpy(), pos) and np.array_equal(dnc.cpu().numpy().astype(np.uint32), nc)
    _same_results(dr, res)


def test_fits_do_not_depend_on_the_device_count(host, gcs):
    ndev = gcs.capi.load().gcs_b200_device_count()
    prog, v, start, targets, fit = _linkage_fit(20000, 6, 4, 6, rng_seed=8)
    one = prog.fit(start, targets, fit, n_devices=1)
    many = prog.fit(start, targets, fit, n_devices=ndev)
    assert one[0] == many[0] == 0 and _same(one[1], many[1]) and _same(one[2], many[2])
    _same_results(many[4], one[4])


# ---- 6. bounds and failures ----

def test_boxes_hold_and_a_target_beyond_a_bound_ends_at_the_bound(host):
    p, cv = _golden(WHOLE_SKETCHES[2])
    free, os_, oc, _ = F.problem(p, cv, 4, seed=9)
    dp = F.DescProgram(p)
    x = cv[0, free]
    moved = cv.copy()
    moved[0, free] = x * (1.0 + 5e-3)
    targets = dp.run(moved)[0][:, os_, oc]  # reached by a move of 5e-3 in every free value
    lo, hi = x - 2e-3 * np.abs(x), x + 2e-3 * np.abs(x)
    ang = p.value_is_angle[free].astype(bool)
    rc, vals, _, nc, res = dp.fit(cv, targets, Fit(free, os_, oc, lower=lo, upper=hi, max_iterations=30))
    assert rc == 0 and res[0]["status"] != START_FAILED and nc[0] == 0
    got = vals[0, free]
    assert ((got >= lo) & (got <= hi)).all()
    assert (np.abs(got[ang]) <= 1.0).all()
    assert ((got == hi) | (got == lo)).any(), (got, lo, hi)


def test_a_start_without_a_root_fails_and_keeps_its_values(host):
    p, cv = _golden(WHOLE_SKETCHES[0])
    free, os_, oc, _ = F.problem(p, cv, 3, seed=1)
    row = p.rows[np.flatnonzero(p.rows["solver"] == 4)[0]]  # two circles about fixed points
    v1, v2 = int(row["value"][1]), int(row["value"][2])
    free = np.unique(np.concatenate([[v1], free]))
    dp = F.DescProgram(p)
    start = np.repeat(cv, 2, axis=0)
    start[1, v1] = 1e3 * (abs(cv[0, v1]) + abs(cv[0, v2]) + 1.0)  # one circle holds the other: no intersection
    assert dp.run(start[1:2])[1][0] > 0
    targets = np.repeat(dp.run(cv)[0][:, os_, oc], 2, axis=0)
    rc, vals, _, _, res = dp.fit(start, targets, Fit(free, os_, oc, max_iterations=5))
    assert rc == 0 and res[1]["status"] == START_FAILED and res[1]["iterations"] == 1
    assert _same(vals[1], start[1]) and res[0]["status"] != START_FAILED


def test_the_returned_values_solve_every_row_after_every_iteration_count(host):
    """lambda0 = 0 and targets far beyond what the sketch reaches, so that the steps are long.  After
    every iteration count the returned values solve every row: a trial that breaks a row is never
    accepted."""
    p, cv = _golden(WHOLE_SKETCHES[0])
    free, os_, oc, _ = F.problem(p, cv, 4, seed=5)
    dp = F.DescProgram(p)
    pos = dp.run(cv)[0][0, os_, oc]
    targets = (pos + 10.0 * (1.0 + np.abs(pos)))[None]
    for m in range(1, 7):
        rc, vals, _, nc, res = dp.fit(cv, targets, Fit(free, os_, oc, lambda0=0.0, max_iterations=m))
        assert rc == 0 and nc[0] == 0 and dp.run(vals)[1][0] == 0, m


# ---- 7. the contracted class ----

def test_the_contracted_class_fits_the_same_values(host):
    _, el, lv = _triangle_strip(402)
    prog = F.Program(el, leaves=lv)
    v = np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])
    p = Arrays.from_desc(prog.desc())
    free, os_, oc, _ = F.problem(p, v[None], 8, seed=3)
    rc, pos, _, _ = prog.run(v[None])
    targets = pos[:, os_, oc]
    start = v[None].copy()
    start[0, free] *= 1.0 + 3e-3
    fit = Fit(free, os_, oc, max_iterations=30, xtol=1e-12)
    rc, base, _, _, res, _ = prog.fit(start, targets, fit)
    assert rc == 0 and res[0]["status"] in CONVERGED
    old = host.gcs_host_set_variant(F.capi.VARIANT_CONTRACTED)
    try:
        rc, fast, _, _, rf, _ = prog.fit(start, targets, fit)
    finally:
        host.gcs_host_set_variant(old)
    assert rc == 0 and rf[0]["status"] in CONVERGED
    assert (np.abs(fast - base) <= 1e-9 * np.abs(base)).all()
