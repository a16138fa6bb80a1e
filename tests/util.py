"""Shared helpers for the parity tests."""
import hashlib

import numpy as np


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def digest(a):
    """sha256 of an array's bytes, every NaN made the same NaN: a stored fingerprint of an output too large for
    tests/golden/ that still compares bit for bit, NaN with NaN."""
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.nan, a)
    return hashlib.sha256(a.tobytes()).hexdigest()


def positions(elements):
    """[n][4] solved positions of host_lib element dicts (NaN past a point's two coordinates) and [n] is_set."""
    pos = np.full((len(elements), 4), np.nan)
    for i, e in enumerate(elements):
        pos[i, :len(e["pos"])] = e["pos"]
    return pos, np.array([e["is_set"] for e in elements], dtype=np.uint8)


def assert_batches_identical(got, ref, what=""):
    """Discrete outputs and coordinates bit-identical (NaNs compare by bit pattern class)."""
    assert np.array_equal(got.iters, ref.iters), f"{what}: iters differ at {np.nonzero(got.iters != ref.iters)}"
    assert np.array_equal(got.converged, ref.converged), f"{what}: converged flags differ"
    assert np.array_equal(got.root_index, ref.root_index), f"{what}: root index differs"
    for c, (a, b) in enumerate(zip(got.out, ref.out)):
        same = (bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))
        assert same.all(), f"{what}: out[{c}] differs at {np.nonzero(~same)[0][:8]}"
    if got.cand is not None and ref.cand is not None:
        same = (bits(got.cand) == bits(ref.cand)) | (np.isnan(got.cand) & np.isnan(ref.cand))
        assert same.all(), f"{what}: candidates differ"


def rel_err(a, b, scale):
    """|a-b| / max(1, |b|, scale): SURVEY section 7's relative-error definition."""
    den = np.maximum(np.maximum(1.0, np.abs(b)), scale)
    return np.abs(a - b) / den


def assert_batches_within_contract(got, ref, what="", rel=1e-9):
    """The north star's contract, no more: iteration counts, convergence flags and root indices
    identical; coordinates within `rel` relative (rel_err with the sub-system's largest input
    magnitude as scale); a NaN only where the reference has one."""
    assert np.array_equal(got.iters, ref.iters), f"{what}: iters differ at {np.nonzero(got.iters != ref.iters)}"
    assert np.array_equal(got.converged, ref.converged), f"{what}: converged flags differ"
    assert np.array_equal(got.root_index, ref.root_index), f"{what}: root index differs at {np.nonzero(got.root_index != ref.root_index)[0][:8]}"
    with np.errstate(invalid="ignore", over="ignore"):
        finite_cols = [np.where(np.isfinite(c), np.abs(c), 0.0) for c in ref.dense_cols()]
        scale = np.max(np.stack(finite_cols), axis=0)

        def close(a, b, sc):
            nan = np.isnan(b)
            assert np.array_equal(np.isnan(a), nan), f"{what}: NaN pattern differs"
            fin = np.isfinite(b)
            assert np.array_equal(a[~fin & ~nan], b[~fin & ~nan]), f"{what}: infinities differ"
            sc = np.broadcast_to(sc, b.shape)
            err = rel_err(a[fin], b[fin], sc[fin])
            assert err.size == 0 or err.max() <= rel, f"{what}: max relative error {err.max():.3e}"
            return float(err.max()) if err.size else 0.0

        worst = 0.0
        for a, b in zip(got.out, ref.out):
            worst = max(worst, close(a, b, scale))
        if got.cand is not None and ref.cand is not None:
            worst = max(worst, close(got.cand, ref.cand, scale))
    return worst
