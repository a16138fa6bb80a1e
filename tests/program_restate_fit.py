"""The fit of gcs_b200_program_fit restated on the CPU: per iteration one restated tangent run
(program_restate.restate, the selector as directions), then the arithmetic of program_fit_normal_kernel
and program_fit_update_kernel (csrc/sketch_program.cu) in their stated order, in scalar float64, and
at the end one restated plain run.  Every instance runs on its own: the kernels share nothing across
instances."""
import math

import numpy as np

from program_restate import Arrays, restate

RUNNING, COST, GTOL, FTOL, XTOL, STALLED, START_FAILED = range(7)


class Fit:
    """A fit descriptor in Python: free value slots, box (None: unbounded), observations (slot,
    coordinate, weight) and the controls.  Units are the C ABI's (cos for an angle slot)."""

    def __init__(self, free, obs_slots, obs_coords, lower=None, upper=None, weights=None, max_iterations=20, lambda0=1e-3,
                 cost_tol=0.0, ftol=1e-15, xtol=1e-15, gtol=0.0):
        self.free = [int(v) for v in free]
        self.obs_slots = [int(s) for s in obs_slots]
        self.obs_coords = [int(c) for c in obs_coords]
        self.lower = None if lower is None else [float(x) for x in lower]
        self.upper = None if upper is None else [float(x) for x in upper]
        self.weights = None if weights is None else [float(x) for x in weights]
        self.max_iterations, self.lambda0 = int(max_iterations), float(lambda0)
        self.cost_tol, self.ftol, self.xtol, self.gtol = float(cost_tol), float(ftol), float(xtol), float(gtol)

    def box(self, angle):
        """[(lo, hi)] per free value as the device uses it: an angle slot's box meets [-1, 1]"""
        out = []
        for i, v in enumerate(self.free):
            lo = -math.inf if self.lower is None else self.lower[i]
            hi = math.inf if self.upper is None else self.upper[i]
            if angle[v]:
                lo, hi = (lo if lo > -1.0 else -1.0), (hi if hi < 1.0 else 1.0)
            out.append((lo, hi))
        return out


def _clamp(x, lo, hi):
    return lo if x < lo else (hi if x > hi else x)


def _normal(fit, pos, dpos, nc, target):
    """program_fit_normal_kernel for one instance: (At [n][n] upper, gt [n], ct, failed)"""
    n = len(fit.free)
    obs = [s * 4 + c for s, c in zip(fit.obs_slots, fit.obs_coords)]
    w = [1.0] * len(obs) if fit.weights is None else fit.weights
    p = pos.reshape(-1)
    J = dpos.reshape(-1, n)
    A = [[0.0] * n for _ in range(n)]
    for i in range(n):
        for j in range(i, n):
            a = 0.0
            for o, q in enumerate(obs):
                a = a + (w[o] * float(J[q, i])) * float(J[q, j])
            A[i][j] = a
    g = []
    for i in range(n):
        a = 0.0
        for o, q in enumerate(obs):
            a = a + (w[o] * float(J[q, i])) * (float(p[q]) - float(target[o]))
        g.append(a)
    c, failed = 0.0, int(nc) > 0
    for o, q in enumerate(obs):
        r = float(p[q]) - float(target[o])
        c = c + (w[o] * r) * r
        failed |= not math.isfinite(float(p[q]))
        failed |= not all(math.isfinite(float(x)) for x in J[q])
    return A, g, c, failed


def _cholesky(A, lam, floor):
    n = len(A)
    L = [[0.0] * n for _ in range(n)]
    for j in range(n):
        ajj = A[j][j]
        s = ajj + lam * (ajj if ajj > floor else floor)
        for q in range(j):
            s = s - L[j][q] * L[j][q]
        if not s > 0.0:
            return None
        d = math.sqrt(s)
        L[j][j] = d
        for i in range(j + 1, n):
            t = A[j][i]
            for q in range(j):
                t = t - L[i][q] * L[j][q]
            L[i][j] = t / d
    return L


class _State:
    def __init__(self, x0, box, lambda0):
        self.x0 = list(x0)
        self.x = [_clamp(v, lo, hi) for v, (lo, hi) in zip(x0, box)]
        self.xt = list(self.x)
        self.A = self.g = None
        self.c = 0.0
        self.status, self.iterations, self.cost, self.grad_inf, self.lam = RUNNING, 0, math.nan, math.nan, lambda0

    def update(self, fit, box, it, last, trial):
        """program_fit_update_kernel; returns the free values the next run reads"""
        if self.status != RUNNING:
            return self.x0 if self.status == START_FAILED else self.x
        n = len(self.x)
        At, gt, ct, failed = trial
        self.iterations += 1
        if it == 0 and failed:
            self.status = START_FAILED
            return self.x0
        status, lam = RUNNING, self.lam

        def reject(lam):
            lam = 10.0 * (lam if lam > 1e-12 else 1e-12)
            return lam, (STALLED if lam > 1e16 else RUNNING)

        if not failed and (it == 0 or ct < self.c):
            c_old = self.c
            self.x, self.g, self.A, self.c = list(self.xt), list(gt), [list(r) for r in At], ct
            if it > 0:
                lam = lam / 10.0 if lam / 10.0 > 1e-12 else 1e-12
            gi = 0.0
            for v in self.g:
                gi = abs(v) if abs(v) > gi else gi
            if ct <= fit.cost_tol:
                status = COST
            elif gi <= fit.gtol:
                status = GTOL
            elif it > 0 and c_old - ct <= fit.ftol * c_old:
                status = FTOL
            self.cost, self.grad_inf = ct, gi
        else:
            lam, status = reject(lam)
        L = None
        if status == RUNNING:
            amax = 0.0
            for j in range(n):
                amax = self.A[j][j] if self.A[j][j] > amax else amax
            floor = 1e-12 * amax
            while status == RUNNING:
                L = _cholesky(self.A, lam, floor)
                if L is not None:
                    break
                lam, status = reject(lam)
        if status == RUNNING:
            d = [0.0] * n
            for i in range(n):
                t = -self.g[i]
                for q in range(i):
                    t = t - L[i][q] * d[q]
                d[i] = t / L[i][i]
            for i in range(n - 1, -1, -1):
                t = d[i]
                for q in range(i + 1, n):
                    t = t - L[q][i] * d[q]
                d[i] = t / L[i][i]
            step = xmax = 0.0
            for i in range(n):
                d[i] = _clamp(self.x[i] + d[i], *box[i])
                a, b = abs(d[i] - self.x[i]), abs(self.x[i])
                step = a if a > step else step
                xmax = b if b > xmax else xmax
            self.xt = d
            if step <= fit.xtol * (xmax + fit.xtol):
                status = XTOL
        self.status, self.lam = status, lam
        return self.xt if status == RUNNING and not last else self.x


def restate_fit(p, values, targets, fit):
    """The fit of program `p` (Arrays, or a C-ABI descriptor) for values [K][n_values] (C-ABI units)
    and targets [K][n_obs].  Returns (values, positions, nonconverged, results), results [K] of dict
    (status, iterations, cost, grad_inf, lambda)."""
    if not isinstance(p, Arrays):
        p = Arrays.from_desc(p)
    vals = np.array(values, dtype=np.float64)
    K, n = vals.shape[0], len(fit.free)
    box = fit.box(p.value_is_angle)
    sel = np.zeros((K, p.n_values, n))
    for t, v in enumerate(fit.free):
        sel[:, v, t] = 1.0
    states = [_State([float(vals[k, v]) for v in fit.free], box, fit.lambda0) for k in range(K)]
    for k, s in enumerate(states):
        vals[k, fit.free] = s.x
    for it in range(fit.max_iterations + 1):
        pos, dpos, nc = restate(p, vals, sel)
        for k, s in enumerate(states):
            trial = _normal(fit, pos[k], dpos[k], nc[k], targets[k]) if s.status == RUNNING else None
            vals[k, fit.free] = s.update(fit, box, it, it == fit.max_iterations, trial)
    pos, _, nc = restate(p, vals)
    results = [dict(status=s.status, iterations=s.iterations, cost=s.cost, grad_inf=s.grad_inf, lambda_=s.lam) for s in states]
    return vals, pos, nc, results
