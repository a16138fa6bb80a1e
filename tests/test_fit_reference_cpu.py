"""The high-precision fit reference (tests/fit_reference.py) without a device: on synthetic problems
(n = 1 .. 32 free values, n .. 4n observations, cond(J) 1 .. 1e6, zero columns, boxes, weights across
decades) it accepts every iteration of the CPU restatement of the fit kernels, which the device equals
bit for bit, and it rejects each of a list of plausible mistakes in that restatement, which a
bit-for-bit comparison cannot see."""
import inspect
import math

import numpy as np
import pytest

import program_restate_fit as R
from fit_reference import Mismatch, Normal, Shadow
from program_restate_fit import RUNNING, XTOL, Fit


class Problem:
    """p(x) = J0 x + h b * (J0 x)^2 at m observed coordinates, J(x) its exact derivative evaluated in
    float64; NaN outside |x_i| <= reach (a trial that fails).  A plateau keeps p and J at their values
    at x0."""

    def __init__(self, n, m, cond, seed, zero_col=False, box=None, lambda0=1e-3, ftol=1e-15, xtol=1e-15, h=0.05,
                 weights=True, plateau=False, reach=math.inf, M=8, x0=None, targets=None, J0=None):
        rng = np.random.default_rng(seed)
        u, _ = np.linalg.qr(rng.standard_normal((m, n)))
        v, _ = np.linalg.qr(rng.standard_normal((n, n)))
        s = np.logspace(0.0, -math.log10(cond), n) * 2.0 ** rng.integers(-4, 5)
        self.J0 = (u * s) @ v.T if J0 is None else np.asarray(J0, dtype=np.float64)
        if zero_col:
            self.J0[:, rng.integers(n)] = 0.0
        self.b = rng.uniform(-1.0, 1.0, m)
        self.h, self.plateau, self.reach = h, plateau, reach
        self.n, self.m, self.M = n, m, M
        self.x0 = rng.standard_normal(n) if x0 is None else np.asarray(x0, dtype=np.float64)
        xs = self.x0 + rng.uniform(-0.3, 0.3, n)
        self.targets = (self.p(xs) + 1e-2 * rng.standard_normal(m)) if targets is None else np.asarray(targets)
        self.w = 10.0 ** rng.uniform(-3, 3, m) if weights else np.ones(m)
        self.lo, self.hi = (np.full(n, -np.inf), np.full(n, np.inf)) if box is None else box(rng, self.x0)
        self.lambda0, self.ftol, self.xtol = lambda0, ftol, xtol

    def p(self, x):
        y = self.J0 @ (self.x0 if self.plateau else x)
        return y + self.h * self.b * y * y

    def jac(self, x):
        y = self.J0 @ (self.x0 if self.plateau else x)
        out = self.J0 * (1.0 + 2.0 * self.h * self.b * y)[:, None]
        if np.abs(x).max() > self.reach:
            return np.full(self.m, np.nan), out
        return self.p(x), out


def _box_with_equal_and_outside(rng, x0):
    n = len(x0)
    lo, hi = x0 - rng.uniform(0.05, 0.5, n), x0 + rng.uniform(0.05, 0.5, n)
    lo[0] = hi[0] = x0[0] + 0.01  # lo == hi, the start outside it
    if n > 1:
        lo[1] = x0[1] + 0.1      # the start below its box
    return lo, hi


def _tight_box(rng, x0):
    return x0 - 1e-3, x0 + 1e-3


def _problems():
    out = []
    seed = 0
    for n in (1, 2, 7, 8, 9, 16, 31, 32):
        M = 8 if n <= 9 else (4 if n <= 16 else 2)
        for cond in (1.0, 1e3, 1e6):
            seed += 1
            m = (n, 2 * n, 4 * n)[seed % 3]
            out.append(Problem(n, m, cond, seed, M=M, zero_col=n > 2 and cond == 1e3,
                               box=_box_with_equal_and_outside if cond == 1e6 else None,
                               lambda0=(1e-3, 0.0, 10.0)[seed % 3]))
    # targets out of reach with a large ftol: FTOL decided against c_old.  c(x) = 2 x^2 + 2 from x =
    # 0.9: the first step gains 1.62 of 3.62, within ftol = 0.5 of c_old and not of c
    out += [Problem(n, 3 * n, 10.0, 100 + n, ftol=0.5, h=0.2, M=10) for n in (2, 3, 4, 5)]
    out += [Problem(1, 2, 1.0, 104, J0=[[1.0], [1.0]], h=0.0, x0=[0.9], targets=[1.0, -1.0], weights=False, ftol=0.5)]
    # the same in two values: c = 2 x^2 + 2 + 2 y^2 + 8 from (0.9, 1.7) gains 7.4 of 17.4
    out += [Problem(2, 4, 1.0, 105, J0=[[1.0, 0.0], [1.0, 0.0], [0.0, 1.0], [0.0, 1.0]], h=0.0, x0=[0.9, 1.7],
                    targets=[1.0, -1.0, 2.0, -2.0], weights=False, ftol=0.5)]
    # every value pushed out of a tight box: XTOL on the clamped step
    out += [Problem(n, 2 * n, 10.0, 200 + n, box=_tight_box, xtol=1e-12, M=6) for n in (2, 3)]
    # a flat cost: every trial costs what the accepted point costs, bit for bit, and from x = 0 no
    # step rounds away, so lambda climbs to STALLED
    out += [Problem(n, 2 * n, 10.0, 300 + n, plateau=True, x0=np.zeros(n), xtol=0.0, M=24) for n in (2, 3)]
    # trials that fail, and a zero column under damping
    out += [Problem(4, 8, 10.0, 400, reach=1.5, lambda0=0.0, M=8), Problem(5, 10, 1.0, 401, zero_col=True, lambda0=1.0, M=6)]
    return out


PROBLEMS = _problems()


def replay(State, prob):
    """the fit of `prob` by the restatement's update (State), each iteration checked by the shadow;
    returns the shadow"""
    n, m = prob.n, prob.m
    obs = np.arange(m)
    fit = Fit(list(range(n)), obs // 4, obs % 4, lower=prob.lo, upper=prob.hi, weights=prob.w, max_iterations=prob.M,
              lambda0=prob.lambda0, ftol=prob.ftol, xtol=prob.xtol)
    box = fit.box(np.zeros(n, dtype=np.int32))
    st = State(list(prob.x0), box, fit.lambda0)
    sh = Shadow(prob.x0, prob.lo, prob.hi, fit.lambda0, ftol=fit.ftol, xtol=fit.xtol)
    rows = -(-m // 4) * 4
    xt = list(st.x)
    for it in range(prob.M + 1):
        p, J = prob.jac(np.array(xt))
        pos, dpos = np.zeros(rows), np.zeros((rows, n))
        pos[:m], dpos[:m] = p, J
        trial = R._normal(fit, pos, dpos, 0, prob.targets)
        nxt = st.update(fit, box, it, it == prob.M, trial)
        failed = trial[3]
        dev = dict(status=st.status, lambda_=st.lam, x=st.x, cost=st.cost, grad_inf=st.grad_inf,
                   xt=st.xt if st.status in (RUNNING, XTOL) else None)
        sh.step(dev, trial=None if failed else Normal(p, J, prob.targets, prob.w), trial_x=xt, failed=failed, A=st.A, g=st.g)
        if st.status != RUNNING:
            break
        xt = list(nxt)
    return sh


def test_the_reference_accepts_every_iteration_of_the_restatement():
    worst, seen = 0.0, set()
    for prob in PROBLEMS:
        sh = replay(R._State, prob)
        worst, seen = max(worst, sh.worst), seen | sh.seen
    # the shadow raises Mismatch at any error above its bound, so worst <= 1 here
    print(f"worst device error / bound over {len(PROBLEMS)} problems: {worst:.3e}")
    assert {R.RUNNING, R.FTOL, R.XTOL, R.STALLED} <= seen, seen


def _mutant(old, new):
    """program_restate_fit's _State with `old` (which occurs once in the module) replaced by `new`"""
    src = inspect.getsource(R)
    assert src.count(old) == 1, old
    ns = {"__name__": "program_restate_fit_mutant"}
    exec(compile(src.replace(old, new), "program_restate_fit_mutant", "exec"), ns)
    return ns["_State"]


MUTATIONS = {
    "back solve reads L[i][q] for L[q][i]": ("t = t - L[q][i] * d[q]", "t = t - L[i][q] * d[q]"),
    "damping lambda I for lambda D": ("s = ajj + lam * (ajj if ajj > floor else floor)", "s = ajj + lam"),
    "no floor: D_jj = A_jj": ("s = ajj + lam * (ajj if ajj > floor else floor)", "s = ajj + lam * ajj"),
    "FTOL against c for c_old": ("c_old - ct <= fit.ftol * c_old", "c_old - ct <= fit.ftol * ct"),
    "XTOL on the step before the clamp": (
        "d[i] = _clamp(self.x[i] + d[i], *box[i])\n                a, b = abs(d[i] - self.x[i]), abs(self.x[i])",
        "a, b = abs(d[i]), abs(self.x[i])\n                d[i] = _clamp(self.x[i] + d[i], *box[i])"),
    "g with its sign flipped": ("t = -self.g[i]", "t = self.g[i]"),
    "accept on ct <= c": ("ct < self.c", "ct <= self.c"),
}


@pytest.mark.parametrize("name", sorted(MUTATIONS))
def test_the_reference_rejects_a_mutated_restatement(name):
    """each mutation is caught on at least two problems of the set"""
    State = _mutant(*MUTATIONS[name])
    caught = 0
    for k, prob in enumerate(PROBLEMS):
        try:
            replay(State, prob)
        except Mismatch as e:
            print(f"caught '{name}' on problem {k} (n = {prob.n}): {e}")
            caught += 1
            if caught == 2:
                return
    pytest.fail(f"'{name}' is caught on {caught} problem(s), not 2")
