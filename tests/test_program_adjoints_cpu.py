"""Sketch-program adjoints without a device: the CPU restatement of a row's adjoint
(tests/adjoint_oracle.py) is the transpose of the row's tangent (tests/tangent_oracle.py), the
restated sweep (tests/program_restate_adjoints.py) is the transpose of the restated tangent run, and
the adjoint entry points check their arguments before any device is touched."""
import ctypes as C
import os

import numpy as np
import pytest

import host_lib as H
import oracle_lib as O
import program_adjoints_lib as P
import sketch_gen as S
from adjoint_oracle import adjoint
from program_restate import Arrays, restate
from program_restate_adjoints import restate_adjoints
from tangent_oracle import tangent

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
OUT_COLS = {1: 2, 2: 4, 3: 2, 4: 2, 5: 4}
SKETCHES = [(31, 1, 3000), (32, 2, 3000), (33, 3, 3000)]  # the golden whole sketches (tests/test_gpu_host.py)


def _duality(fwd, rev):
    """|<o, J k> - <J^T o, k>| over sum |terms| of both, per contraction; fwd / rev: the terms [m][...]"""
    gap = np.abs(fwd.sum(axis=0) - rev.sum(axis=0))
    scale = np.abs(fwd).sum(axis=0) + np.abs(rev).sum(axis=0)
    return gap, scale


@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_row_adjoint_is_the_transpose_of_the_row_tangent(built, kind):
    """The golden per-kind batches solved by the CPU oracle; random input tangents over every column
    and random output adjoints, T = 3.  Every converged sub-system: <ob, tangent(kd)> = <adjoint(ob), kd>
    to 1e-13 of the sum of the two contractions' |terms|."""
    z = np.load(os.path.join(GOLD, f"numeric_k{kind}.npz"))
    cols, code = z["cols"].astype(np.float64), z["code"]
    nin, n = cols.shape
    T = 3
    rng = np.random.default_rng(200 + kind)
    hb = O.solve(O.capi.HostBatch(kind, 2, [np.ascontiguousarray(c) for c in cols], code).alloc_outputs())
    kd = rng.standard_normal((nin, n, T))
    ob = rng.standard_normal((OUT_COLS[kind], n, T))
    dout = tangent(hb, kd)
    kb, live = adjoint(hb, ob)
    gap, scale = _duality(ob * dout, kb * kd)
    ok = live[:, None] & np.isfinite(scale)
    assert ok.sum() > 0.9 * ok.size, (int(ok.sum()), ok.size)
    bad = ok & ~(gap <= 1e-13 * scale)
    assert not bad.any(), (np.argwhere(bad)[:5], gap[bad][:5], scale[bad][:5])
    print(f"K{kind}: {int(ok.sum())} contractions, worst {float((gap[ok] / scale[ok]).max()):.2e} of the terms")


def _leaf_program(seed, first, n):
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    return P.Program(el, leaves=lv), np.array([e["value"] for lf in lv for e in lf["edges"] if e["type"] != S.VIRT])


@pytest.fixture(scope="module")
def host(built):
    built.build_host()
    return H.load()


@pytest.mark.parametrize("seed,first,n", SKETCHES)
def test_restated_sweep_is_the_transpose_of_the_restated_tangent_run(host, seed, first, n):
    """The leaf lists of the golden sketches (all eight solvers, zero-fixed anchors included), K = 2
    instances, T = 2: for random value directions dv and position cotangents ob, <ob, J dv> (the
    restated tangent run) equals <J^T ob, dv> (the restated sweep) to 1e-12 of the sum of both
    contractions' |terms|.  The cotangents weigh only the coordinates whose forward tangents are finite
    (the golden sketches have rows without a root); with that support the sweep gives no NaN either.
    Then the same with every coordinate weighted: the sweep's NaN pairs are the forward run's."""
    prog, base = _leaf_program(seed, first, n)
    assert prog.rc == 0, prog.error
    p = Arrays.from_desc(prog.desc())
    rng = np.random.default_rng(seed)
    K, T = 2, 2
    v = base * (1.0 + 1e-7 * rng.uniform(-1, 1, size=(K, len(base))))
    cv = np.where(p.value_is_angle.astype(bool), np.cos(v), v)
    dv = rng.standard_normal((K, p.n_values, T))
    _, dpos, _ = restate(p, cv, dv)
    finite = np.isfinite(dpos).all(axis=3, keepdims=True)
    assert finite.sum() > 1000
    ob = rng.standard_normal((K, p.n_slots, 4, T)) * finite
    av = restate_adjoints(p, cv, ob)
    assert np.isfinite(av).all()
    fwd = (ob * np.where(finite, dpos, 0.0)).reshape(K, -1, T).transpose(1, 0, 2)
    rev = (av * dv).transpose(1, 0, 2)
    gap, scale = _duality(fwd, rev)
    assert (gap <= 1e-12 * scale).all(), (gap, scale)
    full = rng.standard_normal((K, p.n_slots, 4, T))
    av = restate_adjoints(p, cv, full)
    assert np.array_equal(np.isnan(full * dpos).reshape(K, -1, T).any(axis=1), np.isnan(av).any(axis=1))


def test_adjoint_entry_points_refuse_bad_arguments(gcs, built):
    """Without a device (and with one: the checks run first): no cotangents, null tables, a null
    program."""
    capi = gcs.capi
    lib = capi.load()
    buf = (C.c_double * 8)()
    ms = (C.c_float * 3)()
    for fn, last in ((lib.gcs_b200_program_adjoints, None), (lib.gcs_b200_program_adjoints_host, ms)):
        cases = [
            ((None, 0, buf, buf, last), b"n_cotangents must be >= 1"),
            ((None, -2, buf, buf, last), b"n_cotangents must be >= 1"),
            ((None, 1, None, buf, last), b"null adjoint table"),
            ((None, 1, buf, None, last), b"null adjoint table"),
            ((None, 1, buf, buf, last), b"null program"),
        ]
        for args, message in cases:
            assert fn(*args) == capi.GCS_E_INVALID, message
            assert message in lib.gcs_b200_last_error(), (message, lib.gcs_b200_last_error())
    for fn, last in ((lib.gcs_b200_program_run_recorded, None), (lib.gcs_b200_program_run_recorded_host, ms)):
        assert fn(None, 1, buf, buf, None, 0, last) == capi.GCS_E_INVALID
        assert b"null program" in lib.gcs_b200_last_error()
        assert fn(None, 1, buf, buf, None, 11, last) == capi.GCS_E_INVALID


def test_adjoints_before_a_recorded_run_fail_with_a_message(host):
    """SketchProgram::adjoints throws std::logic_error before any device call when nothing was
    recorded; the plain-C export returns -1 with the message."""
    el, lv = S.make_sketch(300, seed=31, first_shape=1)
    prog = P.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    d = prog.describe()
    rc, _, _ = prog.adjoints(np.zeros((1, d["slots"], 4, 2)))
    assert rc == -1 and "no recorded run" in H.last_error(), H.last_error()
