"""The gradient of a fit's first iteration, g = J^T W r, against the reverse-mode entry point on the same
program: recording a plain run at the start values and sweeping the cotangents W r over the observed
coordinates gives g as the adjoints of the free values.  The fit reports max_i |g_i| (grad_inf); with
one free value that is |g_i| itself."""
import numpy as np
import pytest

import program_fit_lib as F
from program_restate_fit import Fit
from test_gpu_host import WHOLE_SKETCHES
from test_gpu_sketch_program_fit import _golden, _starts, host  # noqa: F401  (fixture)

pytestmark = pytest.mark.gpu


def _reverse_gradient(dp, start, targets, fit):
    """g [K][n_free] from gcs_b200_program_run_recorded_host + gcs_b200_program_adjoints_host, and the
    terms w_o r_o J_oi [K][n_obs][n_free] (J from a tangent run along the free values)"""
    lib = dp.lib
    K, n_slots = start.shape[0], dp.p.n_slots
    vals = np.ascontiguousarray(start)
    pos = np.zeros((K, n_slots, 4))
    nc = np.zeros(K, dtype=np.uint32)
    assert lib.gcs_b200_program_run_recorded_host(dp.h, K, vals.ctypes.data, pos.ctypes.data, nc.ctypes.data, 0, None) == 0
    assert not nc.any()
    w = np.asarray(fit.weights)
    wr = w * (pos[:, fit.obs_slots, fit.obs_coords] - targets)
    ob = np.zeros((K, n_slots, 4, 1))
    np.add.at(ob, (slice(None), fit.obs_slots, fit.obs_coords, 0), wr)
    av = np.full((K, dp.p.n_values, 1), np.nan)
    assert lib.gcs_b200_program_adjoints_host(dp.h, 1, ob.ctypes.data, av.ctypes.data, None) == 0, lib.gcs_b200_last_error()
    sel = np.zeros((K, dp.p.n_values, len(fit.free)))
    sel[:, fit.free, np.arange(len(fit.free))] = 1.0
    J = dp.tangents(start, sel)[1][:, fit.obs_slots, fit.obs_coords, :]
    return av[:, fit.free, 0], wr[:, :, None] * J


@pytest.mark.parametrize("case", WHOLE_SKETCHES)
def test_the_first_fit_gradient_equals_the_reverse_mode_gradient(host, case):
    """K = 3 instances, max_iterations = 0 (one tangent run, the start accepted): per instance grad_inf
    equals max_i |g_i| of the sweep, and a fit of each free value alone gives |g_i|, within 1e-9 of
    sum_o |w_o r_o J_oi| (the tolerance of the reverse-mode dot-product tests).  The one-value fits'
    |g_i| are the components of the full fit's gradient: their maximum is its grad_inf bit for bit."""
    p, cv = _golden(case)
    free, os_, oc, _ = F.problem(p, cv, 5, seed=case[0] + 1)
    dp = F.DescProgram(p)
    rng = np.random.default_rng(case[0])
    K = 3
    start = _starts(dp, cv, free, K, rng)
    pos = dp.run(cv)[0][0, os_, oc]
    targets = pos[None] + rng.standard_normal((K, len(os_))) * (1e-2 * (1.0 + np.abs(pos)))
    fit = Fit(free, os_, oc, weights=rng.uniform(0.5, 2.0, len(os_)), max_iterations=0)
    g, terms = _reverse_gradient(dp, start, targets, fit)
    scale = np.abs(terms).sum(axis=1)  # [K][n_free]
    assert (scale > 0).all()
    rc, _, _, _, res = dp.fit(start, targets, fit)
    assert rc == 0, F.capi.load().gcs_b200_last_error()
    full = np.array([r["grad_inf"] for r in res])
    assert (np.abs(full - np.abs(g).max(axis=1)) <= 1e-9 * scale.max(axis=1)).all(), (full, g)
    one = np.zeros((K, len(free)))
    for i, v in enumerate(free):
        f1 = Fit([v], os_, oc, weights=fit.weights, max_iterations=0)
        rc, _, _, _, r1 = dp.fit(start, targets, f1)
        assert rc == 0 and all(r["iterations"] == 1 for r in r1), r1
        one[:, i] = [r["grad_inf"] for r in r1]
    gap = np.abs(one - np.abs(g)) / scale
    print(f"seed {case[0]}: worst gap {gap.max():.2e} of sum |w r J|")
    assert (gap <= 1e-9).all(), gap
    assert np.array_equal(one.max(axis=1), full)
