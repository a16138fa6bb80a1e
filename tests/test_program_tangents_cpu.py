"""Sketch-program tangents without a device: the CPU restatement of a row's tangent
(tests/tangent_oracle.py) against central differences of the oracle's own solve, and the argument checks
of the tangent entry points, which run before any device is touched."""
import ctypes as C
import os

import numpy as np
import pytest

import host_lib as H
import oracle_lib as O
import program_tangents_lib as P
import sketch_gen as S
from tangent_oracle import tangent

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
# input columns that carry values or solved positions; the others (canvas normals, canvas lengths,
# canvas points and directions) are constants of a program and have no tangent
MOVING = {1: range(6), 2: range(6), 3: range(8), 4: range(10), 5: (0, 1, 2, 7, 8, 9, 10, 11)}
EPS = np.finfo(np.float64).eps


def jacobian(kind, k, x, y):
    """(a, b, c, d) of Sys<KIND>::eval at (x, y), per sub-system."""
    if kind == 1:
        return 2 * (x - k[0]), 2 * (y - k[1]), 2 * (x - k[3]), 2 * (y - k[4])
    if kind == 2:
        return k[2] - k[0], k[3] - k[1], 2 * x, 2 * y
    if kind == 3:
        return 2 * (x - k[0]), 2 * (y - k[1]), -(k[6] - k[4]), k[5] - k[3]
    if kind == 4:
        return -(k[3] - k[1]), k[2] - k[0], -(k[8] - k[6]), k[7] - k[5]
    return k[1], -k[0], 2 * x, 2 * y


def _solve(kind, cols, code):
    return O.solve(O.capi.HostBatch(kind, 2, [np.ascontiguousarray(c) for c in cols], code).alloc_outputs())


def _chosen_converged(b):
    r = b.root_index.astype(np.int64)
    return (r < 2) & (b.converged[np.minimum(r, 1), np.arange(b.n)] == 1)


@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_restated_tangents_agree_with_central_differences(built, kind):
    """Central differences D(h) with h = 1e-5 and 2h along normal random directions of the moving
    columns, extrapolated to (4 D(h) - D(2h)) / 3 so that the h^2 term cancels (some sub-systems of
    these batches have third derivatives large enough to dominate a plain central difference).  A
    sub-system is compared when its chosen run and the four perturbed ones converge on the same root
    index, |det J| is at least 1e-6 of |ad| + |bc|, and the second difference (f(+h) + f(-h) - 2 f(0)) / h
    stays below 1e-2 max(1, |tangent|) (near a tangency, where two roots meet, the curvature swamps any
    difference quotient).  Tolerance per output: 1e-6 max(1, |tangent|) plus the quotient's
    rounding, 4 eps S / (h c), with S the sub-system's largest input or output magnitude and
    c = |det J| / (|ad| + |bc|)."""
    z = np.load(os.path.join(GOLD, f"numeric_k{kind}.npz"))
    cols, code = z["cols"].astype(np.float64), z["code"]
    nin, n = cols.shape
    T, h = 3, 1e-5
    rng = np.random.default_rng(100 + kind)
    din = np.zeros((nin, n, T))
    for c in MOVING[kind]:
        din[c] = rng.standard_normal((n, T))
    base = _solve(kind, cols, code)
    dout = tangent(base, din)
    root = np.minimum(base.root_index.astype(np.int64), 1)
    line = kind in (2, 5)
    x = base.cand[root, 0, np.arange(n)] if line else base.out[0]
    y = base.cand[root, 1, np.arange(n)] if line else base.out[1]
    a, b, c, d = jacobian(kind, cols, x, y)
    cond = np.abs(a * d - b * c) / (np.abs(a * d) + np.abs(b * c))
    f0 = np.array(base.out)
    scale = np.maximum(1.0, np.maximum(np.abs(cols).max(axis=0), np.abs(f0).max(axis=0)))
    compared = excluded = 0
    for t in range(T):
        runs = [_solve(kind, cols + s * h * din[:, :, t], code) for s in (1, -1, 2, -2)]
        fp, fm, fp2, fm2 = (np.array(r.out) for r in runs)
        tan = dout[:, :, t]
        mag = np.maximum(1.0, np.abs(tan)).max(axis=0)
        ok = _chosen_converged(base) & (cond >= 1e-6)
        for r in runs:
            ok &= _chosen_converged(r) & (r.root_index == base.root_index)
        ok &= np.abs(fp + fm - 2 * f0).max(axis=0) / h <= 1e-2 * mag
        fd = (4 * (fp - fm) / (2 * h) - (fp2 - fm2) / (4 * h)) / 3
        err = np.abs(fd - tan).max(axis=0)
        with np.errstate(divide="ignore"):
            tol = 1e-6 * mag + 4 * EPS * scale / (h * cond)
        bad = np.where(ok & ~(err <= tol))[0]
        assert len(bad) == 0, [(int(i), float(err[i]), float(tol[i])) for i in bad[:5]]
        compared += int(ok.sum())
        excluded += int((~ok).sum())
    print(f"kind {kind}: {compared} sub-system directions compared, {excluded} excluded")
    assert excluded <= 0.1 * (compared + excluded), excluded


def test_the_tangent_entry_points_check_their_arguments_without_a_device(gcs, built):
    """n_tangents < 1, null tangent tables, a null program and an unknown variant are GCS_E_INVALID
    with a message; the checks that need no program come before the null-program check."""
    capi = gcs.capi
    lib = capi.load()
    buf = (C.c_double * 8)()
    ms = (C.c_float * 3)()
    for fn, last in ((lib.gcs_b200_program_run_tangents, None), (lib.gcs_b200_program_run_tangents_host, ms)):
        cases = [
            ((None, 1, buf, buf, None, 0, buf, buf, 0, last), b"n_tangents must be >= 1"),
            ((None, 1, buf, buf, None, -3, buf, buf, 0, last), b"n_tangents must be >= 1"),
            ((None, 1, buf, buf, None, 2, buf, buf, 11, last), b"unknown variant 11"),
            ((None, 1, buf, buf, None, 2, None, buf, 0, last), b"null tangent table"),
            ((None, 1, buf, buf, None, 2, buf, None, 0, last), b"null tangent table"),
            ((None, 1, buf, buf, None, 2, buf, buf, 0, last), b"null program"),
        ]
        for args, message in cases:
            assert fn(*args) == capi.GCS_E_INVALID, message
            assert message in lib.gcs_b200_last_error(), (message, lib.gcs_b200_last_error())


@pytest.fixture(scope="module")
def host(built):
    built.build_host()
    return H.load()


def test_host_tangent_run_refuses_no_directions_and_its_descriptor_is_valid(host, gcs):
    """runTangents with T = 0 throws std::invalid_argument before any device call, and the descriptor
    gcs_host_program_desc hands out passes gcs_b200_program_create's validation: without a device the
    call gets as far as GCS_E_NO_DEVICE (with one, it creates the program)."""
    el, lv = S.make_sketch(300, seed=31, first_shape=1)
    prog = P.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    d = prog.describe()
    vals = np.ones((1, d["values"]))
    rc, *_ = prog.run_tangents(vals, np.zeros((1, d["values"], 0)))
    assert rc == -1 and "T must be >= 1" in H.last_error()
    desc = prog.desc()
    assert (desc.n_waves, desc.n_slots, desc.n_values, desc.n_rows) == (d["waves"], d["slots"], d["values"], d["rows"])
    assert [desc.offsets[i] for i in range(len(d["offsets"]))] == list(d["offsets"])
    assert [desc.rows[r].solver for r in range(d["rows"])] == list(d["row_solver"])
    lib = gcs.capi.load()
    h = C.c_void_p()
    rc = lib.gcs_b200_program_create(C.byref(desc), 0, C.byref(h))
    if lib.gcs_b200_device_count() == 0:
        assert rc == gcs.capi.GCS_E_NO_DEVICE and not h.value, lib.gcs_b200_last_error()
    else:
        assert rc == gcs.capi.GCS_OK and h.value
        lib.gcs_b200_program_destroy(h)
