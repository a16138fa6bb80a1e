"""Sketch-program fits without a device: every malformed fit descriptor is refused before any device
call (gcs_b200_fit_check, SketchProgram::fit, gcs_b200_program_fit[_host]), and the CPU restatement
of the fit (tests/program_restate_fit.py) recovers the values that produced its targets."""
import ctypes as C
import math

import numpy as np
import pytest

import host_lib as H
import program_fit_lib as F
import sketch_gen as S
from program_restate import Arrays, restate
from program_restate_fit import XTOL, Fit, restate_fit


@pytest.fixture(scope="module")
def host(built):
    built.build_host()
    return H.load()


@pytest.fixture(scope="module")
def small(host):
    el, lv = S.make_sketch(300, seed=31, first_shape=1)
    prog = F.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    return prog, Arrays.from_desc(prog.desc())


def _malformed(p):
    point = int(np.flatnonzero(p.slot_is_line == 0)[0])
    angle = int(np.flatnonzero(p.value_is_angle)[0])
    ok = dict(free=[0, 1], obs_slots=[point], obs_coords=[0])
    return [
        (dict(ok, free=[]), "n_free must be in 1..32"),
        (dict(ok, free=list(range(33))), "n_free must be in 1..32"),
        (dict(ok, free=[0, 0]), "is already free value 0"),
        (dict(ok, free=[p.n_values]), "out of range"),
        (dict(ok, free=[-1]), "out of range"),
        (dict(ok, obs_slots=[], obs_coords=[]), "n_obs must be >= 1"),
        (dict(ok, obs_slots=[p.n_slots]), "out of range"),
        (dict(ok, obs_coords=[2]), "coordinate 2 of a point slot"),
        (dict(ok, obs_coords=[-1]), "coordinate -1"),
        (dict(ok, weights=[0.0]), "not finite and positive"),
        (dict(ok, weights=[-1.0]), "not finite and positive"),
        (dict(ok, weights=[math.inf]), "not finite and positive"),
        (dict(ok, weights=[math.nan]), "not finite and positive"),
        (dict(ok, lower=[1.0, 0.0], upper=[0.0, 1.0]), "above upper bound"),
        (dict(ok, lower=[math.nan, 0.0]), "NaN bound"),
        (dict(ok, upper=[0.0, math.nan]), "NaN bound"),
        (dict(ok, free=[angle], lower=[1.5]), "does not meet [-1, 1]"),
        (dict(ok, max_iterations=-1), "max_iterations must be >= 0"),
        (dict(ok, lambda0=-1.0), "lambda0 must be finite"),
        (dict(ok, lambda0=math.inf), "lambda0 must be finite"),
        (dict(ok, cost_tol=-1e-9), "cost_tol must be finite"),
        (dict(ok, ftol=math.nan), "ftol must be finite"),
        (dict(ok, xtol=-1.0), "xtol must be finite"),
        (dict(ok, gtol=math.inf), "gtol must be finite"),
    ]


def test_malformed_fit_descriptors_are_refused_before_any_device_call(small):
    """The same messages from gcs_b200_fit_check and from SketchProgram::fit, which throws
    std::invalid_argument before it looks for a device; a well-formed descriptor passes the check."""
    prog, p = small
    K = 1
    vals = np.zeros((K, p.n_values))
    for spec, message in _malformed(p):
        fit = Fit(**spec)
        rc, msg = F.check(p, fit)
        assert rc == F.capi.GCS_E_INVALID and message in msg, (spec, msg)
        targets = np.zeros((K, max(len(fit.obs_slots), 1)))
        rc, _, _, _, _, _ = prog.fit(vals, targets, fit)
        assert rc == -1 and message in H.last_error() and "SketchProgram::fit" in H.last_error(), (spec, H.last_error())
    assert F.check(p, Fit([0, 1], [int(np.flatnonzero(p.slot_is_line)[0])], [3]))[0] == 0


def test_fit_entry_points_refuse_bad_arguments(gcs, built):
    capi = gcs.capi
    lib = capi.load()
    buf = (C.c_double * 8)()
    res = (capi.CFitResult * 1)()
    d = F.cfit(Fit([0], [0], [0]))
    for fn, last in ((lib.gcs_b200_program_fit, None), (lib.gcs_b200_program_fit_host, (C.c_float * 3)())):
        assert fn(None, C.byref(d), 1, buf, buf, buf, None, res, 0, last) == capi.GCS_E_INVALID
        assert b"null program" in lib.gcs_b200_last_error()


def test_the_restated_fit_recovers_the_values_of_its_targets(small):
    """The solvable rows of a small golden-style sketch, four free values (an angle cosine among them
    where the program reads one), starts 1e-3 .. 1e-2 away that solve every row: XTOL within 1e-9."""
    _, p0 = small
    base = np.zeros(p0.n_values)
    el, lv = S.make_sketch(300, seed=31, first_shape=1)
    base[:] = [e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT]
    cv = np.where(p0.value_is_angle.astype(bool), np.cos(base), base)[None]
    p = F.solvable(p0, cv)
    assert p.n_rows > 0 and restate(p, cv)[2][0] == 0
    free, os_, oc, J = F.problem(p, cv, 4, seed=2)
    assert np.linalg.matrix_rank(J) == 4
    targets = restate(p, cv)[0][:, os_, oc]
    rng = np.random.default_rng(1)
    start = cv.copy()
    start[0, free] *= 1.0 + rng.uniform(1e-3, 1e-2, 4) * rng.choice([-1.0, 1.0], 4)
    assert restate(p, start)[2][0] == 0
    vals, pos, nc, res = restate_fit(p, start, targets, Fit(free, os_, oc, max_iterations=20))
    assert res[0]["status"] == XTOL and nc[0] == 0, res
    assert (np.abs(vals[0, free] - cv[0, free]) <= 1e-9 * np.abs(cv[0, free])).all()
    # the accepted cost never increases with the iteration budget
    costs = [restate_fit(p, start, targets, Fit(free, os_, oc, max_iterations=m))[3][0]["cost"] for m in range(4)]
    assert all(b <= a for a, b in zip(costs, costs[1:])), costs
