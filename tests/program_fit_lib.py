"""ctypes binding of sketch-program fits: gcs_b200_program_fit[_host] and gcs_b200_fit_check at the C
ABI (DescProgram, over a gcs_b200_program_desc), SketchProgram::fit through gcs_host_program_fit
(Program), and the solvable part of a program (the rows a run solves)."""
import ctypes as C

import numpy as np

import program_adjoints_lib
from host_lib import _dp, load
from program_lib import sketch_values  # noqa: F401  (re-exported for the fit tests)
from program_restate import Arrays, restate
from program_restate_fit import Fit
from program_tangents_lib import capi


def cfit(fit):
    """capi.CFitDesc over a program_restate_fit.Fit (its tables live as long as the descriptor)."""
    keep = {"free": np.array(fit.free, dtype=np.int32), "slots": np.array(fit.obs_slots, dtype=np.int32),
            "coords": np.array(fit.obs_coords, dtype=np.int32)}
    for name in ("lower", "upper", "weights"):
        if getattr(fit, name) is not None:
            keep[name] = np.array(getattr(fit, name), dtype=np.float64)
    ip, dp = C.POINTER(C.c_int32), C.POINTER(C.c_double)
    d = capi.CFitDesc(n_free=len(fit.free), n_obs=len(fit.obs_slots), max_iterations=fit.max_iterations, lambda0=fit.lambda0,
                      cost_tol=fit.cost_tol, ftol=fit.ftol, xtol=fit.xtol, gtol=fit.gtol)
    d.free_values, d.obs_slots, d.obs_coords = (keep[k].ctypes.data_as(ip) for k in ("free", "slots", "coords"))
    for name in ("lower", "upper", "weights"):
        if name in keep:
            setattr(d, name, keep[name].ctypes.data_as(dp))
    d._keep = keep
    return d


def results(res):
    """capi.CFitResult array -> [dict(status, iterations, cost, grad_inf, lambda_)]"""
    return [dict(status=r.status, iterations=r.iterations, cost=r.cost, grad_inf=r.grad_inf, lambda_=r.lambda_) for r in res]


class DescProgram:
    """A C-ABI program (gcs_b200_program_create) over an Arrays or a descriptor, on device 0."""

    def __init__(self, p):
        self.p = p if isinstance(p, Arrays) else Arrays.from_desc(p)
        self.lib = capi.load()
        self.h = C.c_void_p()
        rc = self.lib.gcs_b200_program_create(C.byref(self.p.desc()), 0, C.byref(self.h))
        assert rc == 0, self.lib.gcs_b200_last_error()

    def __del__(self):
        if getattr(self, "h", None) and self.h.value:
            self.lib.gcs_b200_program_destroy(self.h)

    def run(self, cv, variant=0):
        """gcs_b200_program_run_host: (positions, nonconverged)"""
        cv = np.ascontiguousarray(cv, dtype=np.float64)
        K = cv.shape[0]
        pos = np.zeros((K, self.p.n_slots, 4))
        nc = np.zeros(K, dtype=np.uint32)
        rc = self.lib.gcs_b200_program_run_host(self.h, K, cv.ctypes.data, pos.ctypes.data, nc.ctypes.data, variant, None)
        assert rc == 0, self.lib.gcs_b200_last_error()
        return pos, nc

    def tangents(self, cv, dcv):
        """gcs_b200_program_run_tangents_host: (positions, dpositions, nonconverged)"""
        cv, dcv = np.ascontiguousarray(cv, dtype=np.float64), np.ascontiguousarray(dcv, dtype=np.float64)
        K, T = dcv.shape[0], dcv.shape[2]
        pos, dpos = np.zeros((K, self.p.n_slots, 4)), np.zeros((K, self.p.n_slots, 4, T))
        nc = np.zeros(K, dtype=np.uint32)
        rc = self.lib.gcs_b200_program_run_tangents_host(self.h, K, cv.ctypes.data, pos.ctypes.data, nc.ctypes.data, T, dcv.ctypes.data,
                                                         dpos.ctypes.data, 0, None)
        assert rc == 0, self.lib.gcs_b200_last_error()
        return pos, dpos, nc

    def fit(self, cv, targets, fit, variant=0):
        """gcs_b200_program_fit_host: (rc, values, positions, nonconverged, results)"""
        vals = np.array(cv, dtype=np.float64)
        targets = np.ascontiguousarray(targets, dtype=np.float64)
        K = vals.shape[0]
        pos = np.zeros((K, self.p.n_slots, 4))
        nc = np.zeros(K, dtype=np.uint32)
        res = (capi.CFitResult * K)()
        d = cfit(fit)
        rc = self.lib.gcs_b200_program_fit_host(self.h, C.byref(d), K, vals.ctypes.data, targets.ctypes.data, pos.ctypes.data,
                                                nc.ctypes.data, res, variant, None)
        return rc, vals, pos, nc, results(res)


def check(p, fit):
    """gcs_b200_fit_check: (rc, message)"""
    lib = capi.load()
    p = p if isinstance(p, Arrays) else Arrays.from_desc(p)
    rc = lib.gcs_b200_fit_check(C.byref(p.desc()), C.byref(cfit(fit)))
    return rc, lib.gcs_b200_last_error().decode()


def solvable(p, cv):
    """The rows of `p` whose target has a finite tangent in a restated run at cv [1][n_values] (the row
    has a root and so has every row it depends on), as a program of their own: a program without the
    rows that have no root there.  Dropping a row and everything downstream of it leaves every other
    row's inputs as they were."""
    p = p if isinstance(p, Arrays) else Arrays.from_desc(p)
    _, dpos, _ = restate(p, cv, np.ones((1, p.n_values, 1)))
    ok = np.isfinite(dpos[0, :, :, 0]).all(axis=1)
    keep = ok[p.rows["elem"][:, 2]]
    return p.with_waves([[idx[keep[idx]] for idx in wave] for wave in p.waves()])


class Program(program_adjoints_lib.Program):
    """program_adjoints_lib.Program plus fit() (SketchProgram::fit)."""

    def fit(self, values, targets, fit, n_devices=1):
        """values [K][n_values] (radians for angles), targets [K][n_obs].  Returns (rc, values, positions,
        nonconverged, results, stats)."""
        lib = load()
        if not getattr(lib, "_fit_api", False):
            lib.gcs_host_program_fit.argtypes = [C.c_void_p, C.POINTER(capi.CFitDesc), C.c_int64, C.POINTER(C.c_double),
                                                 C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p, C.POINTER(C.c_uint32),
                                                 C.c_int, C.POINTER(C.c_int64)]
            lib._fit_api = True
        vals = np.array(np.atleast_2d(values), dtype=np.float64)
        targets = np.ascontiguousarray(np.atleast_2d(targets), dtype=np.float64)
        K = vals.shape[0]
        pos = np.zeros((K, self.describe()["slots"], 4))
        nc = np.zeros(K, dtype=np.uint32)
        res = (capi.CFitResult * K)()
        stats = np.zeros(7, dtype=np.int64)
        rc = lib.gcs_host_program_fit(self.handle, C.byref(cfit(fit)), K, _dp(vals), _dp(targets), _dp(pos), res,
                                      nc.ctypes.data_as(C.POINTER(C.c_uint32)), n_devices, stats.ctypes.data_as(C.POINTER(C.c_int64)))
        return rc, vals, pos, nc, results(res), dict(zip(program_adjoints_lib._KEYS, (int(v) for v in stats)))


def problem(p, cv, n_free, seed, max_obs=48):
    """A fit problem on program `p` (Arrays) at cv [1][n_values]: n_free distinct values read by its rows,
    and up to max_obs observed coordinates that depend on them, drawn until J (the restated tangents
    along the free values) has full column rank.  Returns (free, obs_slots, obs_coords, J)."""
    rng = np.random.default_rng(seed)
    read = np.unique(p.rows["value"][p.rows["value"] >= 0])
    for _ in range(20):
        free = rng.choice(read, size=n_free, replace=False)
        angles = np.setdiff1d(read[p.value_is_angle[read] == 1], free)
        if len(angles) and not p.value_is_angle[free].any():
            free[0] = rng.choice(angles)  # an angle cosine among the free values wherever the program reads one
        sel = np.zeros((1, p.n_values, n_free))
        sel[0, free, np.arange(n_free)] = 1.0
        _, dpos, _ = restate(p, cv, sel)
        J = dpos[0].reshape(-1, n_free)
        live = np.flatnonzero(np.isfinite(J).all(axis=1) & (np.abs(J).max(axis=1) > 0))
        if len(live) < n_free:
            continue
        obs = np.sort(rng.choice(live, size=min(max_obs, len(live)), replace=False))
        if np.linalg.matrix_rank(J[obs]) == n_free:
            return free, obs // 4, obs % 4, J[obs]
    raise AssertionError("no full-rank fit problem found")
