"""Oracle (CPU) against the golden vectors generated from the reference's own sources
(oracle/make_golden.py -> tests/golden/).  The GPU twin of this file is test_gpu_golden.py."""
import json
import os

import numpy as np
import pytest

import oracle_lib as O
from util import bits, digest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load_numeric(capi, kind):
    z = np.load(os.path.join(GOLD, f"numeric_k{kind}.npz"))
    cols = [np.ascontiguousarray(c) for c in z["cols"]]
    hb = capi.HostBatch(kind, 2, cols, np.ascontiguousarray(z["code"]))
    return hb, z


def check_against_golden(hb, z, kind, what):
    cand_same = (bits(hb.cand) == bits(z["cand"])) | (np.isnan(hb.cand) & np.isnan(z["cand"]))
    assert cand_same.all(), f"{what}: candidates differ from the reference"
    git, gcv = z["iters"], z["converged"]
    capped = git >= 999  # the reference's count cannot tell i=999 from the cap (see ref_driver.cpp)
    assert np.array_equal(hb.iters[~capped], git[~capped]), f"{what}: iteration counts differ"
    assert (hb.iters[capped] >= 999).all()
    assert np.array_equal(hb.converged[~capped], gcv[~capped])
    seen = z["root"] != 2  # 2 = both candidates identical, root unobservable in the reference
    assert np.array_equal(hb.root_index[seen], z["root"][seen]), f"{what}: chosen root differs"
    if kind in (1, 3, 4):
        for c in range(2):
            same = (bits(hb.out[c]) == bits(z["out"][c])) | (np.isnan(hb.out[c]) & np.isnan(z["out"][c]))
            assert same.all(), f"{what}: chosen point differs"
    else:
        # golden out = (nx, ny, offset): the chosen normal must be the chosen candidate
        r = hb.root_index.astype(int)
        idx = np.arange(hb.n)
        assert np.array_equal(bits(hb.cand[r, 0, idx]), bits(z["out"][0]))
        assert np.array_equal(bits(hb.cand[r, 1, idx]), bits(z["out"][1]))


def check_against_golden_contract(hb, z, kind, what, rel=1e-9):
    """The north star's contract against reference outputs: iteration counts, convergence flags and
    the chosen root equal; candidates and the chosen result within `rel` relative, NaN where the
    reference has NaN.  (For the contracted kernel variants.)  Returns the largest relative error."""
    git, gcv = z["iters"], z["converged"]
    capped = git >= 999  # the reference's count cannot tell i=999 from the cap (see ref_driver.cpp)
    assert np.array_equal(hb.iters[~capped], git[~capped]), f"{what}: iteration counts differ"
    assert (hb.iters[capped] >= 999).all()
    assert np.array_equal(hb.converged[~capped], gcv[~capped])
    seen = z["root"] != 2  # 2 = both candidates identical, root unobservable in the reference
    assert np.array_equal(hb.root_index[seen], z["root"][seen]), f"{what}: chosen root differs"
    worst = 0.0
    with np.errstate(invalid="ignore", over="ignore"):
        scale = np.maximum(1.0, np.max(np.stack([np.where(np.isfinite(c), np.abs(c), 0.0) for c in hb.cols]), axis=0))

        def close(a, b):
            nonlocal worst
            assert np.array_equal(np.isnan(a), np.isnan(b)), f"{what}: NaN pattern differs"
            fin = np.isfinite(b)
            sc = np.broadcast_to(scale, b.shape)
            err = np.abs(a[fin] - b[fin]) / np.maximum(sc[fin], np.abs(b[fin]))
            assert err.size == 0 or err.max() <= rel, f"{what}: max relative error {err.max():.3e}"
            if err.size:
                worst = max(worst, float(err.max()))

        close(hb.cand, z["cand"])
        if kind in (1, 3, 4):
            for c in range(2):
                close(hb.out[c], z["out"][c])
        else:
            r = hb.root_index.astype(int)
            idx = np.arange(hb.n)
            close(hb.cand[r, 0, idx], z["out"][0])
            close(hb.cand[r, 1, idx], z["out"][1])
    return worst


@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_oracle_matches_reference_golden(gcs, built, kind):
    hb, z = load_numeric(gcs.capi, kind)
    O.solve(hb.alloc_outputs())
    check_against_golden(hb, z, kind, f"oracle kind {kind}")


def test_golden_contains_the_known_answers(gcs):
    hb, z = load_numeric(gcs.capi, 1)
    # rows 0..2 are the hand-made 3-4-5 (both canvas signs) and equilateral-100 triangles
    assert z["iters"][:, 0].tolist() == [18, 18] and z["iters"][:, 2].tolist() == [13, 13]
    assert z["out"][1][0] == 4.0 and z["out"][1][1] == -4.0
    assert z["out"][0][2] == 50.0 and abs(z["out"][1][2] - 86.60254037844386) < 1e-12


def test_reference_build_agrees_with_oracle_at_scale(gcs, built):
    """20k instances per kind against what the reference build returned for them (digests in
    tests/golden/ref_loops.npz, oracle/make_golden_ref_loops.py): candidates bit for bit, iteration counts
    where below the reference's cap, chosen roots."""
    ref = np.load(os.path.join(GOLD, "ref_loops.npz"))
    for kind in (1, 2, 3, 4, 5):
        a = O.solve(gcs.synth.make(kind, 20000, seed=77 + kind).alloc_outputs())
        cand, iters, root = ref[f"scale_k{kind}_sha256"]
        assert digest(a.cand) == cand, kind
        # the reference's count cannot tell i=999 from the cap (see ref_driver.cpp)
        assert digest(np.minimum(a.iters, 999)) == iters, kind
        assert digest(a.root_index) == root, kind


def test_components_fixture_is_complete():
    items = json.load(open(os.path.join(GOLD, "components.json")))["items"]
    shapes = {}
    for it in items:
        shapes[it["shape"]] = shapes.get(it["shape"], 0) + 1
        assert it["status"] in (0, 1)
    assert all(shapes.get(s, 0) >= 96 for s in range(1, 9)) and shapes[0] == 2
