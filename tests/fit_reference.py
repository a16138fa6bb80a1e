"""A high-precision reference of one iteration of gcs_b200_program_fit (include/gcs_b200.h, the comment
above it), written from the documented algorithm and not from the kernels' loops, and a shadow replay
that walks a fit's trajectory against it.

Every input is a float64 number taken as exact: the observed positions p and tangents J at a point,
the targets t and weights w, the free values x, the damping lambda and the box.  The exact quantities
(c, g, A, D, M = A + lambda D, the step d = -M^-1 g, the clamped trial, the tolerance tests) are
computed with mpmath at DPS digits; their own relative error, 10^-DPS, is far below every bound
here.  Next to each quantity stands an a-priori bound on the difference between it and what a
float64 implementation of the documented operation order may return (Higham, Accuracy and Stability
of Numerical Algorithms, 2nd ed.: u = 2^-53, gamma_k = k u / (1 - k u)).  Underflow adds at most
ETA / 2 per rounded product and nothing to a sum (a subnormal sum is exact); the Cholesky and solve
bounds assume no underflow inside the factorisation, which the problems here never come near.

A decision the device makes from rounded numbers is three-valued here: True or False when the
exact quantity is beyond its threshold by more than its bound, EITHER when it lies within it."""
import math

import mpmath as mp
import numpy as np

from program_restate_fit import COST, FTOL, GTOL, RUNNING, STALLED, START_FAILED, XTOL

DPS = 60
U = 2.0 ** -53
ETA = 2.0 ** -1074
EITHER = None
NAMES = {RUNNING: "RUNNING", COST: "COST", GTOL: "GTOL", FTOL: "FTOL", XTOL: "XTOL", STALLED: "STALLED",
         START_FAILED: "START_FAILED"}


def gamma(k):
    return k * U / (1.0 - k * U)


def _up(x):
    """x rounded up a little: float64 sums of non-negative terms used inside a bound are within
    gamma_k of their value; every such sum here has k <= 4 n_obs + 8, so this factor covers it"""
    return float(x) * (1.0 + 1e-10)


class Mismatch(AssertionError):
    pass


def leq(value, bound, threshold, tbound=0.0):
    """the device's test `value <= threshold` for a value within `bound` and a threshold within
    `tbound` of the exact ones: True, False or EITHER"""
    gap = mp.mpf(threshold) - mp.mpf(value)
    b = bound + tbound
    if b == 0:
        return bool(gap >= 0)
    if gap > b:
        return True
    if gap < -b:
        return False
    return EITHER


def lam_accept(lam):
    """the lambda rule on an accepted trial, in float64: max(lambda / 10, 1e-12)"""
    return lam / 10.0 if lam / 10.0 > 1e-12 else 1e-12


def lam_reject(lam):
    """the lambda rule on a rejected trial or a failed factorisation: 10 max(lambda, 1e-12)"""
    return 10.0 * (lam if lam > 1e-12 else 1e-12)


class Normal:
    """c = sum w r^2, g = J^T W r, A = J^T W J at one point, exact, with the bounds bc, bg [n], bA [n][n]
    on a float64 evaluation that rounds r = p - t, then forms each term as (w a) b and adds the terms
    one at a time from 0.0 (any order of the n_obs terms: recursive summation of m terms is within
    gamma_{m-1} of the sum of their absolute values, Higham 4.2).
      term of c: r rounded once (it appears twice), w r once, (w r) r once: gamma_4 |w r^2|.
      term of g: r, w J and the product: gamma_3 |w J r|.
      term of A: w J_i and the product: gamma_2 |w J_i J_j|.
    Adding gamma_{m-1} gives gamma_{m+3}, gamma_{m+2} and gamma_{m+1} of the absolute sums; underflow
    adds ETA (1 + max|r| or max|J|) per term."""

    def __init__(self, p, J, t, w):
        with mp.workdps(DPS):
            p, t, w = (np.asarray(a, dtype=np.float64) for a in (p, t, w))
            J = np.asarray(J, dtype=np.float64).reshape(len(p), -1)
            m, n = J.shape
            self.m, self.n = m, n
            r = [mp.mpf(float(a)) - mp.mpf(float(b)) for a, b in zip(p, t)]
            wm = [mp.mpf(float(a)) for a in w]
            cols = [[mp.mpf(float(J[o, i])) for o in range(m)] for i in range(n)]
            wcols = [[wm[o] * cols[i][o] for o in range(m)] for i in range(n)]
            self.r = r
            self.c = mp.fdot(wm, [a * a for a in r])
            self.g = [mp.fdot(wcols[i], r) for i in range(n)]
            self.A = mp.matrix(n, n)
            for i in range(n):
                for j in range(i, n):
                    self.A[i, j] = self.A[j, i] = mp.fdot(wcols[i], cols[j])
            self.gi = max((abs(v) for v in self.g), default=mp.mpf(0))
        ra = np.abs(p - t)
        aJ = np.abs(J)
        und_r = 2 * m * ETA * (1.0 + _up(ra.max()))
        und_j = 2 * m * ETA * (1.0 + _up(aJ.max()))
        self.bc = gamma(m + 3) * _up(np.sum(w * ra * ra)) + und_r
        self.bg = gamma(m + 2) * np.array([_up(v) for v in (w * ra) @ aJ]) + und_r
        self.bA = gamma(m + 1) * ((aJ * w[:, None]).T @ aJ) * (1.0 + 1e-10) + und_j
        self.bgi = float(self.bg.max()) if n else 0.0
        self.zero_cols = [i for i in range(n) if not J[:, i].any()]
        self.key = (p.tobytes(), J.tobytes())


def _fro(rows):
    return math.sqrt(sum(float(v) ** 2 for v in rows))


class Step:
    """One step from an accepted point (its Normal `nm`, free values x) at damping lam in the box
    [lo, hi]: the factorisation's decision, the step d = -(A + lam D)^-1 g, the clamped trial and the
    XTOL test, each with its bound.

    D_jj = max(A_jj, floor), floor = 1e-12 max_j A_jj.  On the device A_jj is within bA_jj, so max_j
    A_jj is within max_j bA_jj; floor is that times the double 1e-12, rounded once; max(., floor) is
    1-Lipschitz in both arguments, so D_jj is within bD_j = max(bA_jj, bfloor).  The diagonal the
    factorisation reads, A_jj + lam D_jj, rounds twice: bM_jj = bA_jj + lam bD_j + gamma_2 (M_jj + bA_jj
    + lam bD_j).  Off the diagonal bM_ij = bA_ij.

    pivot: False when the exact M has a zero column (J's column j is all zero, so the float64 A has
    an exact zero row, and lam D_jj = 0 exactly: every pivot of that column is 0 - sum L^2 <= 0).  True
    when Demmel's condition (Higham Thm 10.7) holds for the matrix the device factors: with H =
    diag(M)^-1/2 M diag(M)^-1/2, the factorisation of M + dM succeeds when
        min_j M_jj / (M_jj + bM_jj) * (1 / ||H^-1||_F - ||E||_F) > n gamma_{n+1} / (1 - n gamma_{n+1}),
    E_ij = bM_ij / sqrt(M_ii M_jj) (lambda_min(H) >= 1 / ||H^-1||_F; Weyl for E; the rescaling by the
    perturbed diagonal moves the smallest eigenvalue by at most that factor).  EITHER otherwise.

    step: a successful factorisation and the two triangular solves give (M + dM + dC) d^ = -(g + dg)
    with |dC| <= gamma_{3n+1} |L^||L^T| (Higham Thm 10.4) and || |L^||L^T| ||_2 <= n ||M + dM||_2 /
    (1 - n gamma_{n+1}) (Higham 10.1).  With dM' = dM + dC and ||M^-1||_2 <= ||L^-1||_F^2,
        ||d^ - d||_2 <= ||M^-1|| (||dM'|| ||d|| + ||dg||) / (1 - ||M^-1|| ||dM'||)
    (M (d^ - d) = -dM' d^ - dg, and ||d^|| <= ||d|| + ||d^ - d||); infinite when the denominator is
    not positive.  The trial clamp(x + d) rounds x + d once and clamp is 1-Lipschitz: bt_i = be + u
    (|x_i + d_i| + be).

    XTOL: the device tests max_i |xt_i - x_i| <= xtol (max_i |x_i| + xtol): the left side within
    max_i (bt_i + u (|xt_i - x_i| + bt_i)) (one rounding of each difference), the right side rounded
    twice, gamma_2 of its value."""

    def __init__(self, nm, x, lam, lo, hi, xtol):
        n = nm.n
        self.lam = lam
        with mp.workdps(DPS):
            A = nm.A
            diag = [A[j, j] for j in range(n)]
            amax = max(diag, default=mp.mpf(0))
            floor = mp.mpf(1e-12) * amax
            bA = nm.bA
            bamax = float(max(bA[j, j] for j in range(n)))
            bfloor = 1e-12 * bamax + U * (float(floor) + 1e-12 * bamax) + ETA
            D = [a if a > floor else floor for a in diag]
            bD = [max(float(bA[j, j]), bfloor) for j in range(n)]
            M = A.copy()
            for j in range(n):
                M[j, j] = A[j, j] + mp.mpf(lam) * D[j]
            bM = np.array(bA, dtype=np.float64)
            for j in range(n):
                bM[j, j] = bA[j, j] + lam * bD[j] + gamma(2) * (float(M[j, j]) + bA[j, j] + lam * bD[j]) + ETA
            self.bM = bM
            self.zero_pivot = any(M[j, j] == 0 for j in nm.zero_cols)
            try:
                L = mp.cholesky(M)
                Linv = mp.inverse(L)
            except (ValueError, ZeroDivisionError):
                L = Linv = None
            if self.zero_pivot or L is None:
                self.pivot = False if self.zero_pivot else EITHER
                self.minv = math.inf
                self.d = None
            else:
                minv = mp.mpf(0)
                for i in range(n):
                    for j in range(i + 1):
                        minv += Linv[i, j] ** 2
                self.minv = float(minv) * (1.0 + 1e-10)
                # ||H^-1||_F with H^-1 = diag(M)^1/2 M^-1 diag(M)^1/2
                Minv = Linv.T * Linv
                hinv = mp.sqrt(sum((Minv[i, j] * mp.sqrt(M[i, i] * M[j, j])) ** 2 for i in range(n) for j in range(n)))
                E = math.sqrt(sum((bM[i, j] / math.sqrt(float(M[i, i]) * float(M[j, j]))) ** 2 for i in range(n) for j in range(n)))
                shrink = min(float(M[j, j]) / (float(M[j, j]) + bM[j, j]) for j in range(n))
                need = n * gamma(n + 1) / (1.0 - n * gamma(n + 1))
                self.pivot = True if shrink * (1.0 / float(hinv) * (1 - 1e-10) - E) > need else EITHER
                self.d = Linv.T * (Linv * mp.matrix([-v for v in nm.g]))
            mnorm = _fro(M[i, j] for i in range(n) for j in range(n)) * (1 + 1e-10) + float(np.sqrt((bM ** 2).sum()))
            dC = gamma(3 * n + 1) * n * mnorm / (1.0 - n * gamma(n + 1))
            dMp = float(np.sqrt((bM ** 2).sum())) + dC
            if self.d is None:
                self.be = math.inf
            else:
                dn = _fro(self.d) * (1 + 1e-10)
                den = 1.0 - self.minv * dMp
                self.be = self.minv * (dMp * dn + float(np.sqrt((nm.bg ** 2).sum()))) / den if den > 0 else math.inf
            # the trial and the XTOL test
            xm = [mp.mpf(float(v)) for v in x]
            if self.d is None:
                self.xt, self.bt = None, [math.inf] * n
                self.xtol = EITHER
                return
            raw = [xm[i] + self.d[i] for i in range(n)]
            self.xt = [min(max(raw[i], mp.mpf(lo[i])), mp.mpf(hi[i])) for i in range(n)]
            self.bt = [self.be + U * (abs(float(raw[i])) + self.be) for i in range(n)]
            step = max((abs(self.xt[i] - xm[i]) for i in range(n)), default=mp.mpf(0))
            bstep = max((self.bt[i] + U * (abs(float(self.xt[i] - xm[i])) + self.bt[i]) for i in range(n)), default=0.0)
            xmax = max((abs(v) for v in xm), default=mp.mpf(0))
            rhs = mp.mpf(xtol) * (xmax + mp.mpf(xtol))
            exact_step = all(b == 0 for b in self.bt)
            self.xtol = leq(step, 0.0 if exact_step else bstep, rhs, gamma(2) * float(rhs) + ETA)

    def trial_within(self, xt):
        """the largest |xt_i - exact trial_i| / bound_i, or Mismatch where a bound excludes xt"""
        worst = 0.0
        for i, v in enumerate(xt):
            err = abs(mp.mpf(float(v)) - self.xt[i])
            if self.bt[i] == 0:
                if err != 0:
                    raise Mismatch(f"trial value {i}: {float(v)!r} is not the exact {float(self.xt[i])!r}")
                continue
            ratio = float(err) / self.bt[i]
            if ratio > 1.0:
                raise Mismatch(f"trial value {i}: {float(v)!r} is {float(err):.3e} from {float(self.xt[i])!r}, bound {self.bt[i]:.3e}")
            worst = max(worst, ratio)
        return worst


class Shadow:
    """Walks one instance's fit iteration by iteration.  step() takes what the device evaluated at its
    trial (trial_x, its Normal, whether the trial failed) and what it reported after the update (status,
    lambda, accepted x, cost, grad_inf and, where known, the next trial xt).  Where a decision is EITHER
    the shadow follows the device; otherwise the first device decision, value or number that the
    reference excludes raises Mismatch.  worst is the largest observed error as a fraction of its
    bound."""

    def __init__(self, x0, lo, hi, lambda0, cost_tol=0.0, ftol=1e-15, xtol=1e-15, gtol=0.0):
        self.lo, self.hi = [float(v) for v in lo], [float(v) for v in hi]
        self.x = [min(max(float(v), a), b) for v, a, b in zip(x0, self.lo, self.hi)]
        self.lam = float(lambda0)
        self.cost_tol, self.ftol, self.xtol, self.gtol = float(cost_tol), float(ftol), float(xtol), float(gtol)
        self.it = 0
        self.status = RUNNING
        self.acc = None      # Normal at the accepted x
        self.pending = None  # Step whose trial the device evaluates next
        self.worst = 0.0
        self.seen = set()

    def _ratio(self, what, dev, exact, bound):
        err = abs(mp.mpf(float(dev)) - exact)
        if bound == 0:
            if err != 0:
                raise Mismatch(f"it {self.it}: {what} {float(dev)!r} is not the exact {float(exact)!r}")
            return
        if float(err) > bound:
            raise Mismatch(f"it {self.it}: {what} {float(dev)!r} is {float(err):.3e} from {float(exact)!r}, bound {bound:.3e}")
        self.worst = max(self.worst, float(err) / bound)

    @staticmethod
    def _allow(decision, taken, what):
        if decision is not EITHER and decision != taken:
            raise Mismatch(f"{what}: the device took {taken}, the reference requires {decision}")

    def step(self, dev, trial=None, trial_x=None, failed=False, A=None, g=None):
        """dev: dict(status, lambda_, x, cost, grad_inf[, xt]).  trial: the Normal at the evaluated
        trial, or None when the device rejected a trial the caller did not evaluate.  A, g: the
        device's accepted normal equations where it exposes them."""
        if self.status != RUNNING:
            raise Mismatch("step() after the fit finished")
        it = self.it
        if trial_x is not None:
            want = self.x if it == 0 else None
            if want is not None:
                if any(float(a) != float(b) for a, b in zip(trial_x, want)):
                    raise Mismatch(f"it 0: the start {list(trial_x)} is not the clamped start {want}")
            elif self.pending is not None:
                self.worst = max(self.worst, self.pending.trial_within(trial_x))
        status = dev["status"]
        if it == 0 and failed:
            self._allow(START_FAILED, status, "it 0 failed start")
            self.status = status
            self.seen.add(status)
            return
        # accept or reject
        if it == 0:
            accept = True
        elif failed:
            accept = False
        elif trial is None:
            accept = EITHER
        elif trial.key == self.acc.key:
            accept = False  # the same inputs give the same float64 cost: ct < c is false
        else:
            accept = _less(trial, self.acc)
        dev_x = [float(v) for v in dev["x"]]
        taken = dev_x != self.x if it > 0 else True
        if it > 0 and trial is not None and taken and [float(v) for v in trial_x] != dev_x:
            raise Mismatch(f"it {it}: the accepted values are not the trial's")
        self._allow(accept, taken, f"it {it}: accept")
        if taken and trial is None:
            raise Mismatch(f"it {it}: an accepted trial needs its normal equations")
        lam = self.lam
        stage = [RUNNING]
        if taken:
            c_old = self.acc.c if self.acc else None
            bc_old = self.acc.bc if self.acc else 0.0
            self.acc, self.x = trial, dev_x
            if it > 0:
                lam = lam_accept(lam)
            self._ratio("cost", dev["cost"], trial.c, trial.bc)
            self._ratio("grad_inf", dev["grad_inf"], trial.gi, trial.bgi)
            if A is not None:
                for i in range(trial.n):
                    for j in range(i, trial.n):
                        self._ratio(f"A[{i}][{j}]", A[i][j], trial.A[i, j], float(trial.bA[i, j]))
            if g is not None:
                for i in range(trial.n):
                    self._ratio(f"g[{i}]", g[i], trial.g[i], float(trial.bg[i]))
            tests = [(COST, leq(trial.c, trial.bc, self.cost_tol)), (GTOL, leq(trial.gi, trial.bgi, self.gtol))]
            if it > 0:
                # c_old - c <= ftol c_old: the difference of two rounded costs rounds once, the product once
                gain = c_old - trial.c
                bgain = bc_old + trial.bc + U * (abs(float(gain)) + bc_old + trial.bc)
                rhs = mp.mpf(self.ftol) * c_old
                brhs = self.ftol * bc_old + U * (float(rhs) + self.ftol * bc_old)
                tests.append((FTOL, leq(gain, bgain, rhs, brhs)))
            for st, dec in tests:
                if status == st:
                    self._allow(dec, True, f"it {it}: {NAMES[st]}")
                    stage = None
                    break
                self._allow(dec, False, f"it {it}: {NAMES[st]} (the device says {NAMES.get(status)})")
        else:
            lam = lam_reject(lam)
            if lam > 1e16:
                stage = None
                self._allow(STALLED, status, f"it {it}: lambda {lam} above 1e16")
        if stage is not None:
            self._step_phase(dev, status, lam, it)
        elif dev["lambda_"] != lam:
            raise Mismatch(f"it {it}: lambda {dev['lambda_']!r}, the rule gives {lam!r}")
        self.status = status
        self.lam = dev["lambda_"]
        self.seen.add(status)
        self.it += 1

    def _step_phase(self, dev, status, lam, it):
        for _ in range(64):
            if lam > 1e16:
                self._allow(STALLED, status, f"it {it}: lambda {lam} above 1e16")
                break
            st = Step(self.acc, self.x, lam, self.lo, self.hi, self.xtol)
            if status == STALLED or dev["lambda_"] != lam:
                self._allow(st.pivot, False, f"it {it}: factorisation at lambda {lam!r}")
                lam = lam_reject(lam)
                continue
            self._allow(st.pivot, True, f"it {it}: factorisation at lambda {lam!r}")
            self._allow(st.xtol, status == XTOL, f"it {it}: XTOL")
            if status not in (XTOL, RUNNING):
                raise Mismatch(f"it {it}: status {NAMES.get(status)} after a step")
            if dev.get("xt") is not None:
                self.worst = max(self.worst, st.trial_within(dev["xt"]))
            self.pending = st
            break
        if dev["lambda_"] != lam:
            raise Mismatch(f"it {it}: lambda {dev['lambda_']!r}, the rule gives {lam!r}")


def _less(trial, acc):
    """the accept test ct < c: True when ct + bct < c - bc, False when ct - bct >= c + bc"""
    gap = acc.c - trial.c
    b = acc.bc + trial.bc
    if b == 0:
        return bool(gap > 0)
    if gap > b:
        return True
    if gap <= -b:
        return False
    return EITHER
