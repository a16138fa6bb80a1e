"""Sketch-program fits on the GPU against the high-precision reference (tests/fit_reference.py), step
by step.  A fit with max_iterations = m is a prefix of a longer one (finished instances freeze, and
the last iteration writes the accepted values), so the fits for m = 0 .. M read off the device's
trajectory: x_m, c_m, max|g|_m, lambda_m and the status.  J and p at x_m come from a tangent run along
the selector (the run the fit itself makes there), and the shadow replay checks every decision,
value and damping the device took against the reference and its a-priori bounds."""
import math

import numpy as np
import pytest

import host_lib as H
import program_fit_lib as F
import sketch_gen as S
from fit_reference import Mismatch, Normal, Shadow, Step
from program_restate import Arrays
from program_restate_fit import COST, FTOL, GTOL, RUNNING, STALLED, START_FAILED, XTOL, Fit
from util import bits

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def host(gpu, built):
    built.build_host()
    return H.load()


def _same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return bool(((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))).all())


@pytest.fixture(scope="module")
def linkage(host):
    el, edges = S.make_linkage(20000, seed=6)
    prog = F.Program(el, edges)
    p = Arrays.from_desc(prog.desc())
    v = F.sketch_values(edges)
    cv = np.where(p.value_is_angle.astype(bool), np.cos(v), v)[None]
    dp = F.DescProgram(p)
    assert dp.run(cv)[1][0] == 0
    return dp, cv


def _golden(seed, first, n):
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    prog = F.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    p = Arrays.from_desc(prog.desc())
    base = np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])
    cv = np.where(p.value_is_angle.astype(bool), np.cos(base), base)[None]
    p = F.solvable(p, cv)
    return F.DescProgram(p), cv


@pytest.fixture(scope="module")
def golden(host):
    return [_golden(31, 1, 300), _golden(33, 3, 300)]


def _selector(dp, free):
    sel = np.zeros((1, dp.p.n_values, len(free)))
    sel[0, free, np.arange(len(free))] = 1.0
    return sel


def _choose(dp, cv, n_free, seed, per_value=3):
    """n_free distinct values read by the program and, for each, per_value observed coordinates whose
    tangent along it is nonzero, drawn until J has full column rank: (free, slots, coords)"""
    rng = np.random.default_rng(seed)
    read = np.unique(dp.p.rows["value"][dp.p.rows["value"] >= 0])
    for _ in range(20):
        free = rng.choice(read, size=min(n_free, len(read)), replace=False)
        J = dp.tangents(cv, _selector(dp, free))[1][0].reshape(-1, len(free))
        ok = np.isfinite(J).all(axis=1)
        obs = set()
        for i in range(len(free)):
            rows = np.flatnonzero(ok & (J[:, i] != 0))
            obs |= set(rng.choice(rows, size=min(per_value, len(rows)), replace=False).tolist()) if len(rows) else set()
        obs = np.array(sorted(obs))
        if len(obs) >= len(free) and np.linalg.matrix_rank(J[obs]) == len(free):
            return free, obs // 4, obs % 4
    raise AssertionError("no full-rank fit problem found")


def _start(dp, cv, free, rng, lo=1e-3, hi=1e-2):
    """cv with the free values moved by lo .. hi relative, the move shrunk until every row solves"""
    x = cv.copy()
    for q in range(50):
        move = rng.uniform(lo, hi, len(free)) * 0.7 ** q
        x[0, free] = cv[0, free] * (1.0 + move * rng.choice([-1.0, 1.0], len(free)))
        if dp.run(x)[1][0] == 0:
            return x
    raise AssertionError("no solvable start")


def _box(dp, fit):
    lo = np.full(len(fit.free), -np.inf) if fit.lower is None else np.array(fit.lower)
    hi = np.full(len(fit.free), np.inf) if fit.upper is None else np.array(fit.upper)
    ang = dp.p.value_is_angle[fit.free].astype(bool)
    return np.where(ang, np.maximum(lo, -1.0), lo), np.where(ang, np.minimum(hi, 1.0), hi)


def _normal(dp, vals, fit, targets, w):
    """(Normal at vals or None, failed): the tangent run the fit makes at vals"""
    pos, dpos, nc = dp.tangents(vals, _selector(dp, fit.free))
    obs = np.array(fit.obs_slots) * 4 + np.array(fit.obs_coords)
    p = pos[0].reshape(-1)[obs]
    J = dpos[0].reshape(-1, len(fit.free))[obs]
    failed = nc[0] > 0 or not (np.isfinite(p).all() and np.isfinite(J).all())
    return (None if failed else Normal(p, J, targets[0], w)), failed


def _check_reject(dp, sh, fit, targets, w, vals):
    """A reject is wrong when the program solves every row at the rounded reference trial and its cost
    there is below the accepted cost by more than the bounds.  The device's trial is within bt_i of the
    reference trial; the cost change over that distance is estimated by the Gauss-Newton model
    2 |g|^T bt + bt^T |A| bt (g, A at the reference trial).  That model leaves out the residual
    curvature sum_o w_o r_o grad^2 r_o and higher orders, so it is an estimate, not an a-priori bound;
    the check is one-sided (it can only flag a reject of a clearly cheaper trial), so an estimate
    that is too small can cost power or flag a reject wrongly, and never lets a wrong reject pass
    that a true bound would catch."""
    st = sh.pending
    if st is None or st.xt is None or not all(math.isfinite(b) for b in st.bt):
        return
    x = vals.copy()
    x[0, fit.free] = [float(v) for v in st.xt]
    nm, failed = _normal(dp, x, fit, targets, w)
    if failed:
        return
    bt = np.array(st.bt)
    carried = 2.0 * float(np.abs([float(v) for v in nm.g]) @ bt) + float(bt @ np.abs(np.array(nm.A.tolist(), dtype=float)) @ bt)
    if nm.c + nm.bc + carried < sh.acc.c - sh.acc.bc:
        raise Mismatch(f"it {sh.it}: rejected a trial whose cost {float(nm.c)!r} is below {float(sh.acc.c)!r}")


def trajectory(dp, start, targets, fit, M):
    """The device's fit of one instance read off for m = 0 .. M and replayed by the shadow; the last fit
    is also run inside a K = 65 batch (_in_batch).  Returns (shadow, results of the last fit, values of
    the last fit)."""
    w = np.ones(len(fit.obs_slots)) if fit.weights is None else np.array(fit.weights)
    lo, hi = _box(dp, fit)
    sh = Shadow(start[0, fit.free], lo, hi, fit.lambda0, fit.cost_tol, fit.ftol, fit.xtol, fit.gtol)
    prev = None
    for m in range(M + 1):
        f = Fit(fit.free, fit.obs_slots, fit.obs_coords, fit.lower, fit.upper, fit.weights, m, fit.lambda0,
                fit.cost_tol, fit.ftol, fit.xtol, fit.gtol)
        rc, vals, _, _, res = dp.fit(start, targets, f)
        assert rc == 0, F.capi.load().gcs_b200_last_error()
        r = res[0]
        assert r["iterations"] == m + 1, r
        x = vals[0, fit.free]
        dev = dict(status=r["status"], lambda_=r["lambda_"], x=x, cost=r["cost"], grad_inf=r["grad_inf"])
        if m == 0:
            x0 = start.copy()
            x0[0, fit.free] = np.clip(start[0, fit.free], lo, hi)
            nm, failed = _normal(dp, x0, fit, targets, w)
            sh.step(dev, trial=nm, trial_x=x0[0, fit.free], failed=failed)
        elif not np.array_equal(bits(x), bits(prev)):
            nm, failed = _normal(dp, vals, fit, targets, w)
            sh.step(dev, trial=nm, trial_x=x, failed=failed)
        else:
            _check_reject(dp, sh, fit, targets, w, vals)
            sh.step(dev)
        prev = x
        if r["status"] != RUNNING:
            break
    _in_batch(dp, start, targets, f, np.random.default_rng(m))
    return sh, r, vals


def _in_batch(dp, start, targets, fit, rng, K=65, at=(0, 31, 64)):
    """the instance at each position of a K-instance fit whose other instances start elsewhere equals
    the K = 1 fit bit for bit"""
    rc, v1, p1, n1, r1 = dp.fit(start, targets, fit)
    assert rc == 0
    starts = np.repeat(start, K, axis=0)
    starts[:, fit.free] *= 1.0 + rng.uniform(-1e-3, 1e-3, (K, len(fit.free)))
    tg = np.repeat(targets, K, axis=0)
    for k in at:
        starts[k] = start[0]
    rc, vk, pk, nk, rk = dp.fit(starts, tg, fit)
    assert rc == 0
    for k in at:
        assert _same(vk[k], v1[0]) and _same(pk[k], p1[0]) and nk[k] == n1[0], k
        assert rk[k]["status"] == r1[0]["status"] and rk[k]["iterations"] == r1[0]["iterations"]
        assert _same([rk[k][q] for q in ("cost", "grad_inf", "lambda_")], [r1[0][q] for q in ("cost", "grad_inf", "lambda_")])


# ---- sizes: 1 .. 32 free values on the 20k linkage, and every readable value of two golden sketches ----

@pytest.mark.parametrize("n_free", [1, 2, 8, 9, 16, 31, 32])
def test_linkage_fits_follow_the_reference(linkage, n_free):
    dp, cv = linkage
    rng = np.random.default_rng(n_free)
    free, os_, oc = _choose(dp, cv, n_free, seed=n_free)
    start = _start(dp, cv, free, rng)
    pos = dp.run(cv)[0][0, os_, oc]
    targets = (pos + (1e-4 * (1.0 + np.abs(pos)) * rng.standard_normal(len(os_)) if n_free % 2 else 0.0))[None]
    fit = Fit(free, os_, oc, weights=rng.uniform(0.5, 2.0, len(os_)), lambda0=1e-3)
    M = 12 if n_free <= 9 else 4
    sh, r, _ = trajectory(dp, start, targets, fit, M)
    print(f"n_free {n_free}: statuses {sorted(sh.seen)}, worst error / bound {sh.worst:.3e}")


def test_golden_sketch_fits_of_every_readable_value_follow_the_reference(golden):
    for dp, cv in golden:
        read = np.unique(dp.p.rows["value"][dp.p.rows["value"] >= 0])
        n = min(len(read), 32)
        free, os_, oc = _choose(dp, cv, n, seed=n)
        rng = np.random.default_rng(n)
        start = _start(dp, cv, free, rng)
        targets = dp.run(cv)[0][:, os_, oc]
        trajectory(dp, start, targets, Fit(free, os_, oc, lambda0=1e-3), 6)


# ---- rank, damping, weights ----

def _with_unobserved(dp, cv, n_free, seed):
    """free values with one more value that no observed coordinate depends on"""
    free, os_, oc = _choose(dp, cv, n_free, seed)
    read = np.setdiff1d(np.unique(dp.p.rows["value"][dp.p.rows["value"] >= 0]), free)
    obs = os_ * 4 + oc
    rng = np.random.default_rng(seed)
    for v in rng.permutation(read)[:200]:
        J = dp.tangents(cv, _selector(dp, [v]))[1][0].reshape(-1)
        if not J[obs].any():
            return np.append(free, v), os_, oc
    raise AssertionError("every value reaches an observation")


def test_an_unobserved_value_never_moves_and_the_rest_follow_the_reduced_system(golden):
    dp, cv = golden[0]
    free, os_, oc = _with_unobserved(dp, cv, 4, seed=3)
    rng = np.random.default_rng(3)
    start = _start(dp, cv, free, rng)
    targets = dp.run(cv)[0][:, os_, oc]
    fit = Fit(free, os_, oc, lambda0=1e-3)
    sh, r, vals = trajectory(dp, start, targets, fit, 8)
    assert vals[0, free[-1]] == start[0, free[-1]]
    # the reduced system: the same fit without the unobserved value, the same values and costs
    red = Fit(free[:-1], os_, oc, lambda0=1e-3, max_iterations=8)
    rc, rv, _, _, rr = dp.fit(start, targets, red)
    assert rc == 0 and rr[0]["status"] == r["status"]
    assert _same(rv[0, free[:-1]], vals[0, free[:-1]]) and _same(rr[0]["cost"], r["cost"])


def test_a_zero_column_under_gauss_newton_fails_once_then_damps_at_the_floor(golden):
    """lambda0 = 0 with a value no observation sees: the first factorisation has a zero pivot, so
    lambda becomes exactly 10 * 1e-12, and the step then solves the system damped by the floor"""
    dp, cv = golden[0]
    free, os_, oc = _with_unobserved(dp, cv, 3, seed=5)
    rng = np.random.default_rng(5)
    start = _start(dp, cv, free, rng)
    targets = dp.run(cv)[0][:, os_, oc]
    fit = Fit(free, os_, oc, lambda0=0.0)
    rc, _, _, _, res = dp.fit(start, targets, Fit(free, os_, oc, lambda0=0.0, max_iterations=0))
    assert rc == 0 and res[0]["lambda_"] == 10.0 * 1e-12, res
    trajectory(dp, start, targets, fit, 6)


def test_gauss_newton_steps_on_a_full_rank_problem(golden):
    dp, cv = golden[1]
    free, os_, oc = _choose(dp, cv, 5, seed=8)
    rng = np.random.default_rng(8)
    start = _start(dp, cv, free, rng)
    pos = dp.run(cv)[0][0, os_, oc]
    targets = (pos + 1e-3 * rng.standard_normal(len(os_)))[None]
    sh, _, _ = trajectory(dp, start, targets, Fit(free, os_, oc, lambda0=0.0), 8)
    assert sh.it >= 2


def test_weights_across_twelve_decades_and_duplicated_observations(golden):
    dp, cv = golden[1]
    free, os_, oc = _choose(dp, cv, 6, seed=9)
    os_, oc = np.concatenate([os_, os_[:4]]), np.concatenate([oc, oc[:4]])
    rng = np.random.default_rng(9)
    w = 10.0 ** rng.uniform(-6.0, 6.0, len(os_))
    start = _start(dp, cv, free, rng)
    pos = dp.run(cv)[0][0, os_, oc]
    targets = (pos + 1e-3 * rng.standard_normal(len(os_)))[None]
    trajectory(dp, start, targets, Fit(free, os_, oc, weights=w, lambda0=1e-2), 10)


def test_a_near_singular_normal_matrix_under_the_smallest_damping(golden):
    """As many observed coordinates as free values (a square J), one of them weighted down a decade at
    a time until cond(J^T W J) at the start lies in 1e10 .. 1e12, and lambda0 = 1e-12, the damping's
    own floor.  The shadow's bounds widen with ||M^-1||; it allows a device step or decision to differ
    from the exact one only as far as they say."""
    dp, cv = golden[1]
    free, os_, oc = _choose(dp, cv, 4, seed=12, per_value=1)
    assert len(os_) == len(free)
    rng = np.random.default_rng(12)
    start = _start(dp, cv, free, rng)
    J = dp.tangents(start, _selector(dp, free))[1][0].reshape(-1, len(free))[os_ * 4 + oc]
    w = np.ones(len(os_))
    for _ in range(40):
        kappa = np.linalg.cond((J * w[:, None]).T @ J)
        if kappa >= 1e10:
            break
        w[0] /= 10.0
    assert 1e10 <= kappa <= 1e12, kappa
    targets = dp.run(cv)[0][:, os_, oc]
    sh, _, _ = trajectory(dp, start, targets, Fit(free, os_, oc, weights=w, lambda0=1e-12), 8)
    print(f"cond(A) {kappa:.2e}: statuses {sorted(sh.seen)}, worst error / bound {sh.worst:.3e}")


@pytest.mark.parametrize("e", [-20, 0, 20])
def test_the_same_fit_with_lengths_and_positions_scaled_by_a_power_of_two(golden, e):
    """golden[0] with every length value and every initial position times 2^e (angles unchanged), and
    the start and targets scaled alike: the absolute parts of the bounds (underflow, the 1e-12 floors
    of D and lambda, xtol (max|x| + xtol)) meet a different scale while the reference still holds"""
    dp0, cv0 = golden[0]
    s = 2.0 ** e
    p0 = dp0.p
    p = Arrays(p0.rows, p0.offsets, p0.slot_is_line, p0.initial * s, p0.value_is_angle)
    ang = p.value_is_angle.astype(bool)
    dp = F.DescProgram(p)
    cv = np.where(ang, cv0, cv0 * s)
    assert dp.run(cv)[1][0] == 0
    free, os_, oc = _choose(dp0, cv0, 5, seed=13)
    start = _start(dp0, cv0, free, np.random.default_rng(13))
    start = np.where(ang, start, start * s)
    pos = dp.run(cv)[0][0, os_, oc]
    targets = (pos + 1e-3 * s * np.random.default_rng(14).standard_normal(len(os_)))[None]
    sh, r, _ = trajectory(dp, start, targets, Fit(free, os_, oc, lambda0=1e-3), 10)
    print(f"scale 2^{e}: final {r}, worst error / bound {sh.worst:.3e}")


# ---- boxes ----

def test_boxes_equal_bounds_a_start_outside_and_a_wide_angle_box(golden):
    dp, cv = golden[0]
    free, os_, oc = _choose(dp, cv, 6, seed=4)
    ang = dp.p.value_is_angle[free].astype(bool)
    x = cv[0, free]
    lo, hi = x - 5e-3 * np.abs(x), x + 5e-3 * np.abs(x)
    lo[ang], hi[ang] = -5.0, 5.0  # wider than [-1, 1]: the device meets it with [-1, 1]
    k = int(np.flatnonzero(~ang)[0])
    lo[k] = hi[k] = x[k]  # lo == hi
    q = int(np.flatnonzero(~ang)[1])
    rng = np.random.default_rng(4)
    start = _start(dp, cv, free, rng)
    start[0, free[q]] = hi[q] + 1e-3 * abs(hi[q])  # outside its box: clamped before the first run
    pos = dp.run(cv)[0][0, os_, oc]
    targets = (pos + 1e-2 * (1.0 + np.abs(pos)) * rng.standard_normal(len(os_)))[None]
    sh, r, vals = trajectory(dp, start, targets, Fit(free, os_, oc, lower=lo, upper=hi, lambda0=1e-3), 10)
    got = vals[0, free]
    blo, bhi = _box(dp, Fit(free, os_, oc, lower=lo, upper=hi))
    assert got[k] == x[k] and got[q] <= hi[q]
    assert (np.abs(got[ang]) <= 1.0).all() and ((got >= blo) & (got <= bhi)).all()


def _decoupled(dp, cv, n_free, seed):
    """n_free values and, for each, up to 3 observed coordinates that depend on it and on no other
    free value, so that J^T W J is diagonal at every point"""
    rng = np.random.default_rng(seed)
    read = np.unique(dp.p.rows["value"][dp.p.rows["value"] >= 0])
    for _ in range(20):
        free = rng.choice(read, size=n_free, replace=False)
        J = dp.tangents(cv, _selector(dp, free))[1][0].reshape(-1, n_free)
        nz = np.isfinite(J).all(axis=1)[:, None] & (J != 0)
        own = [np.flatnonzero(nz[:, i] & (nz.sum(axis=1) == 1)) for i in range(n_free)]
        if all(len(o) for o in own):
            obs = np.sort(np.concatenate([rng.choice(o, size=min(3, len(o)), replace=False) for o in own]))
            return free, obs // 4, obs % 4
    raise AssertionError("no decoupled fit problem found")


def _bounded_fit(dp, cv, free, os_, oc, move):
    """targets reached by moving free value i by move[i] relative, a box of 1e-5 relative about cv"""
    x = cv[0, free]
    lo, hi = x - 1e-5 * np.abs(x), x + 1e-5 * np.abs(x)
    moved = cv.copy()
    moved[0, free] = x * (1.0 + move)
    targets = dp.run(moved)[0][:, os_, oc]
    return targets, Fit(free, os_, oc, lower=lo, upper=hi, max_iterations=100, xtol=1e-13, ftol=0.0)


@pytest.mark.parametrize("n_free", [16, 32])
def test_an_optimum_with_active_bounds_meets_kkt_and_scipy(linkage, n_free):
    """Observations that each depend on one free value, so J^T W J is diagonal and the clamped step of
    one value does not depend on the others: the clamped iteration reaches the constrained optimum.
    Half the values have targets 3e-5 away, beyond the box of 1e-5, the other half 3e-6 away, inside.
    At the end (XTOL, the only test that can stop it with cost_tol = ftol = gtol = 0):
      at an active bound the exact gradient points out of the box;
      elsewhere the last step d_i = -g_i / M_ii (M = A + lambda D diagonal) was not clamped, so
      |g_i| <= M_ii (xtol (max|x| + xtol) + be), be the reference's bound on the device's step;
      and the cost is no more than scipy's trust-region reflective fit's plus the first-order change
      2 |g|^T |x - x_scipy| that separates two points of a locally convex cost."""
    from scipy.optimize import least_squares
    dp, cv = linkage
    free, os_, oc = _decoupled(dp, cv, n_free, seed=40 + n_free)
    signs = np.random.default_rng(n_free).choice([-1.0, 1.0], n_free)
    move = np.where(np.arange(n_free) % 2 == 0, 3e-5, 3e-6) * signs
    targets, fit = _bounded_fit(dp, cv, free, os_, oc, move)
    rc, vals, _, nc, res = dp.fit(cv, targets, fit)
    assert rc == 0 and nc[0] == 0 and res[0]["status"] == XTOL, res
    nm, failed = _normal(dp, vals, fit, targets, np.ones(len(os_)))
    assert not failed
    got = vals[0, free]
    lo, hi = np.array(fit.lower), np.array(fit.upper)
    at_lo, at_hi = got == lo, got == hi
    assert (at_lo | at_hi)[::2].all() and not (at_lo | at_hi)[1::2].any(), (at_lo, at_hi)
    g = np.array([float(v) for v in nm.g])
    assert (g[at_lo] >= 0).all() and (g[at_hi] <= 0).all(), g
    lam = res[0]["lambda_"]
    st = Step(nm, got, lam, lo, hi, fit.xtol)
    A = np.array([float(nm.A[i, i]) for i in range(n_free)])
    Mii = A + lam * np.maximum(A, 1e-12 * A.max())
    tau = fit.xtol * (np.abs(got).max() + fit.xtol)
    inside = ~(at_lo | at_hi)
    assert (np.abs(g[inside]) <= (Mii[inside] * (tau + st.be)) * (1.0 + 1e-10) + nm.bg[inside]).all(), g[inside]
    sel = _selector(dp, free)

    def at(z):
        v = cv.copy()
        v[0, free] = z
        return v

    ls = least_squares(lambda z: dp.run(at(z))[0][0, os_, oc] - targets[0], cv[0, free], bounds=(lo, hi), method="trf",
                       jac=lambda z: dp.tangents(at(z), sel)[1][0, os_, oc, :], xtol=1e-15, ftol=1e-15, gtol=1e-15)
    assert float(nm.c) <= 2 * ls.cost + 2 * float(np.abs(g) @ np.abs(got - ls.x)) + nm.bc, (float(nm.c), 2 * ls.cost)


@pytest.mark.xfail(strict=True, reason="the documented iteration clamps the whole step into the box: when a value at its "
                   "bound is coupled to the others through J^T W J, it can report convergence where the gradient still points "
                   "into the box")
@pytest.mark.parametrize("n_free", [16, 32])
def test_a_coupled_active_bound_ends_at_a_kkt_point(linkage, n_free):
    """Every value's targets 3e-5 away, beyond a box of 1e-5, with observations that depend on several
    free values.  The fit reports a converged status, but at some active bound the exact gradient
    points into the box: the end point is not the constrained optimum.  Kept as an expected failure
    so that a change to the box handling shows up here."""
    dp, cv = linkage
    free, os_, oc = _choose(dp, cv, n_free, seed=40 + n_free)
    move = 3e-5 * np.random.default_rng(n_free).choice([-1.0, 1.0], n_free)
    targets, fit = _bounded_fit(dp, cv, free, os_, oc, move)
    rc, vals, _, nc, res = dp.fit(cv, targets, fit)
    assert rc == 0 and nc[0] == 0 and res[0]["status"] in (COST, GTOL, FTOL, XTOL), res
    nm, failed = _normal(dp, vals, fit, targets, np.ones(len(os_)))
    got = vals[0, free]
    at_lo, at_hi = got == np.array(fit.lower), got == np.array(fit.upper)
    g = np.array([float(v) for v in nm.g])
    assert (g[at_lo] >= 0).all() and (g[at_hi] <= 0).all(), g


# ---- every status ----

@pytest.mark.parametrize("want", [COST, GTOL, FTOL, XTOL, STALLED, START_FAILED, RUNNING])
def test_every_status_occurs_and_follows_the_reference(golden, want):
    dp, cv = golden[0]
    rng = np.random.default_rng(want)
    free, os_, oc = _choose(dp, cv, 4, seed=20 + want)
    start = _start(dp, cv, free, rng)
    targets = dp.run(cv)[0][:, os_, oc]
    M = 20
    fit = Fit(free, os_, oc)
    if want == COST:
        fit.cost_tol = 1e-20
    elif want == GTOL:
        fit = Fit(free, os_, oc, gtol=1e3)
    elif want == FTOL:
        pos = targets[0]
        targets = (pos + 1e-2 * (1.0 + np.abs(pos)) * rng.standard_normal(len(os_)))[None]
        fit = Fit(free, os_, oc, ftol=1e-3)
    elif want == XTOL:
        fit = Fit(free, os_, oc, xtol=1e-10)
    elif want == STALLED:
        # lambda0 = 1e16 and targets 1e20 away: the first step, about 1e20 / 1e16 times a value's
        # size, leaves two circles without an intersection; the failed trial is a reject, and lambda
        # goes to 1e17 > 1e16
        row = dp.p.rows[np.flatnonzero(dp.p.rows["solver"] == 4)[0]]
        free = np.array([int(row["value"][1]), int(row["value"][2])])
        J = dp.tangents(cv, _selector(dp, free))[1][0].reshape(-1, 2)
        obs = np.flatnonzero(np.isfinite(J).all(axis=1) & (np.abs(J).max(axis=1) > 0))
        os_, oc = obs // 4, obs % 4
        start, M = cv, 3
        targets = dp.run(cv)[0][:, os_, oc] + 1e20
        fit = Fit(free, os_, oc, lambda0=1e16, xtol=0.0, ftol=0.0)
    elif want == START_FAILED:
        row = dp.p.rows[np.flatnonzero(dp.p.rows["solver"] == 4)[0]]  # two circles about fixed points
        v1, v2 = int(row["value"][1]), int(row["value"][2])
        free = np.unique(np.concatenate([[v1], free]))
        start = cv.copy()
        start[0, v1] = 1e3 * (abs(cv[0, v1]) + abs(cv[0, v2]) + 1.0)  # one circle holds the other
        fit = Fit(free, os_, oc)
    elif want == RUNNING:
        M = 2
        fit = Fit(free, os_, oc, ftol=0.0, xtol=0.0)
    sh, r, _ = trajectory(dp, start, targets, fit, M)
    assert r["status"] == want, (r, sh.seen)


def test_all_free_values_unobserved_is_gtol_at_iteration_zero(golden):
    dp, cv = golden[0]
    free, os_, oc = _with_unobserved(dp, cv, 2, seed=6)
    fit = Fit(free[-1:], os_, oc)
    targets = dp.run(cv)[0][:, os_, oc] + 1.0
    sh, r, vals = trajectory(dp, cv, targets, fit, 2)
    assert r["status"] == GTOL and r["iterations"] == 1 and r["grad_inf"] == 0.0


# ---- the 2^31 boundary of the working state ----

def _fit_host_bytes(p, K, n, n_obs):
    """device memory of gcs_b200_program_fit_host for K instances (csrc/sketch_program.cu's buffers):
    values and positions; counts; value and position tangents along n directions; the working state
    (3 n^2 + 5 n + 3 doubles an instance); targets; results (32 bytes); the kind batches of a tangent
    run, per kind cap = the kind's largest wave x K sub-systems of (in + out) columns of doubles, four
    byte planes and (bounded here for every kind) four candidate doubles.  1 MiB covers the
    descriptor tables, the running counts and each buffer's 256-byte alignment."""
    lib = F.capi.load()
    widest = [max((p.segment(wv, k)[1] - p.segment(wv, k)[0] for wv in range(p.n_waves)), default=0) for k in range(1, 6)]
    per = 8 * p.n_values + 32 * p.n_slots + 4 + n * (8 * p.n_values + 32 * p.n_slots) + 8 * (3 * n * n + 5 * n + 3) + 8 * n_obs + 32
    batches = sum(((widest[k] * K + 31) // 32 * 32) * (8 * (lib.gcs_b200_kind_in_cols(k + 1) + lib.gcs_b200_kind_out_cols(k + 1)) + 4 + 32)
                  for k in range(5))
    return K * per + batches + 2 ** 20


def test_a_fit_whose_working_state_crosses_2_31_doubles(host):
    import torch
    dp, cv = _golden(31, 1, 40)
    n = 32
    read = np.unique(dp.p.rows["value"][dp.p.rows["value"] >= 0])
    if len(read) < n:
        pytest.skip("the program reads fewer than 32 values")
    free, os_, oc = _choose(dp, cv, n, seed=1)
    stride = 3 * n * n + 5 * n + 3
    kb = (2 ** 31) // stride + 1  # instance kb - 1's state straddles 2^31 doubles, instance kb's starts past it
    K = kb + 64
    need = _fit_host_bytes(dp.p, K, n, len(os_))
    free_bytes = torch.cuda.mem_get_info(0)[0]
    if need > free_bytes:
        pytest.skip(f"needs about {need / 2 ** 30:.1f} GiB of device memory, {free_bytes / 2 ** 30:.1f} GiB free")
    rng = np.random.default_rng(2)
    starts = [_start(dp, cv, free, rng) for _ in range(4)]
    targets = dp.run(cv)[0][:, os_, oc]
    fit = Fit(free, os_, oc, max_iterations=2)
    ones = [dp.fit(s, targets, fit) for s in starts]
    big = np.repeat(cv, K, axis=0)
    for k in range(K):
        big[k] = starts[k % 4][0]
    rc, vals, pos, nc, res = dp.fit(big, np.repeat(targets, K, axis=0), fit)
    assert rc == 0, F.capi.load().gcs_b200_last_error()
    for k in (0, 1, kb - 2, kb - 1, kb, kb + 1, K - 1):
        one = ones[k % 4]
        assert _same(vals[k], one[1][0]) and _same(pos[k], one[2][0]) and nc[k] == one[3][0], k
        assert res[k]["status"] == one[4][0]["status"] and _same(res[k]["cost"], one[4][0]["cost"]), k
