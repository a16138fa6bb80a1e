"""Kernel parity across the exponent range: every kind and every kernel mapping on rescaled, translated
and mixed-magnitude sub-systems, against the CPU oracle.

The fast paths of the Newton kernels are exact only inside operand ranges that integer tests on high
words enforce (csrc/newton_core.cuh, qr_fast_core R0-R4), and the guards of the contracted class
scale with a per-kind coordinate scale S (csrc/newton_relaxed.cuh, RelaxGuard::init).  The synthetic
batches sit a few hundred units from the origin, where every one of those tests passes.  Here the same
batches are moved to where they fail:

- `scaled(hb, e)`: every length, point and canvas coordinate times exactly 2^e.  The same geometry,
  with every product's exponent shifted; EXPONENTS names the bound each exponent sits next to.
- `translated(hb, ox, oy)`: every solver-space point moved by (ox, oy), 2^10 .. 2^40 from the origin,
  from the default seeds (the "far seed" regime for every run) and from the oracle's own roots of the
  untranslated batch, perturbed and moved along.
- `mixed(hb, name)`: one element of each sub-system at another magnitude than the rest (needle
  triangles, short and long lines, close fixed points far out, a short direction vector).

Bit-identical mappings (1, 2, 3, 4, 9) must equal the oracle bit for bit.  Contracted mappings (5 - 8,
and 10 for K4) must keep the contract (util.assert_batches_within_contract) and, on runs that decided
on quadratic convergence, a scale-relative bound without the floor at 1 (see `_floor_free`).

The part without the gpu mark checks the transforms themselves and runs without a device.
"""
import ctypes as C
import functools

import numpy as np
import pytest

import oracle_lib as O
from util import assert_batches_identical, assert_batches_within_contract, bits

gcs = O.gcs
capi = O.capi

TOL = 1e-5  # GCS_CONVERGENCE_THRESHOLD
BITWISE = [1, 2, 3, 4, 9]        # static, refill, sorted, pair, sequential
CONTRACTED = [5, 6, 7, 8]        # contracted default, static, sorted, sequential
LINEAR = 10                      # K4 only: the contracted linear kernel
SORTED = (3, 7)                  # these get a batch of 2^16 sub-systems (full tiles) where runs converge

# ---- column roles ------------------------------------------------------------------------------
# points: solver-space (x, y) column pairs - scaled and translated.  lengths: radii, signed distances,
# the K5 fixed-direction vector and canvas lengths - scaled, never translated.  canvas: canvas points
# (nearest-to-canvas selection) - scaled with the sketch, never translated.  Every other column (unit
# normals, cosines, canvas directions) never moves.
ROLES = {
    1: dict(points=[(0, 1), (3, 4)], lengths=[2, 5], canvas=[]),
    2: dict(points=[(0, 1), (2, 3)], lengths=[4, 5, 8], canvas=[]),
    3: dict(points=[(0, 1), (3, 4), (5, 6)], lengths=[2, 7], canvas=[(8, 9)]),
    4: dict(points=[(0, 1), (2, 3), (5, 6), (7, 8)], lengths=[4, 9], canvas=[(10, 11)]),
    5: dict(points=[(7, 8), (10, 11)], lengths=[0, 1, 9, 12], canvas=[]),
}
POINT_UNKNOWNS = (1, 3, 4)  # K2 and K5 solve for a unit normal: their guesses never scale or move


def _flat(pairs):
    return [c for p in pairs for c in p]


def scaled_cols(kind):
    r = ROLES[kind]
    return sorted(_flat(r["points"]) + r["lengths"] + _flat(r["canvas"]))


def _copy(hb, cols=None, guesses=None):
    cols = [np.array(c, dtype=np.float64, copy=True) for c in (hb.cols if cols is None else cols)]
    g = hb.guesses if guesses is None else guesses
    g = None if g is None else np.ascontiguousarray(g, dtype=np.float64)
    return capi.HostBatch(hb.kind, hb.n_seeds, cols, hb.code.copy(), g)


def scaled(hb, e):
    """Lengths, points and canvas coordinates times exactly 2^e (and explicit point guesses with them)."""
    out = _copy(hb)
    for c in scaled_cols(hb.kind):
        out.cols[c] = np.ldexp(out.cols[c], e)
    if out.guesses is not None and hb.kind in POINT_UNKNOWNS:
        out.guesses = np.ldexp(out.guesses, e)
    return out


def translated(hb, ox, oy, guesses=None):
    """Every solver-space point moved by (ox, oy); `guesses` [n_seeds][2][n]: explicit guesses, used as given."""
    out = _copy(hb, guesses=guesses)
    for cx, cy in ROLES[hb.kind]["points"]:
        out.cols[cx] = out.cols[cx] + ox
        out.cols[cy] = out.cols[cy] + oy
    return out


def moved_roots(base, ox, oy, seed):
    """The oracle's candidates of `base`, perturbed by 2^-20 relative and moved by (ox, oy) for the kinds
    whose unknown is a point: the same runs, started next to their roots, far from the origin."""
    ref = O.solve(_copy(base).alloc_outputs(), threads=0)
    g = ref.cand * (1.0 + 2.0 ** -20 * np.random.default_rng(seed).standard_normal(ref.cand.shape))
    g = np.where(np.isfinite(g), g, 1.0)
    if base.kind in POINT_UNKNOWNS:
        g[:, 0] += ox
        g[:, 1] += oy
    return np.ascontiguousarray(g)


def _pow2(rng, lo, hi, n):
    return np.ldexp(1.0, rng.integers(lo, hi + 1, size=n))


def _shrink(c, a, b, ratio):
    """Segment (a, b) (column pairs) shrunk about its midpoint by `ratio`: the same infinite line."""
    for i in range(2):
        m = 0.5 * (c[a[i]] + c[b[i]])
        c[a[i]][:], c[b[i]][:] = m + (c[a[i]] - m) * ratio, m + (c[b[i]] - m) * ratio


def _stretch(c, a, b, ratio):
    """Endpoint b pushed out along the line to a + (b - a) * ratio: the same infinite line."""
    for i in range(2):
        c[b[i]][:] = c[a[i]] + (c[b[i]] - c[a[i]]) * ratio


def mixed(hb, name, seed=5):
    """One element of every sub-system at another magnitude than the rest (MIXED)."""
    out = _copy(hb)
    c, n = out.cols, hb.n
    rng = np.random.default_rng(seed)
    if name == "k1_needle_2^-30..-40":
        # the free point 2^-30 .. 2^-40 of |AB| from A or B: radii 2^30 .. 2^40 apart
        ax, ay, ra, bx, by, rb = c
        d = np.hypot(bx - ax, by - ay)
        rho = d * _pow2(rng, -40, -30, n) * rng.uniform(1.0, 2.0, n)
        phi = rng.uniform(0.02, np.pi - 0.02, n) * np.where(rng.random(n) < 0.5, 1.0, -1.0)
        near_b = rng.random(n) < 0.5
        px = np.where(near_b, bx, ax) + rho * np.cos(phi)
        py = np.where(near_b, by, ay) + rho * np.sin(phi)
        ra[:], rb[:] = np.hypot(px - ax, py - ay), np.hypot(px - bx, py - by)
    elif name == "k2_points_2^-20_apart_at_1e3":
        # the two fixed points 2^-21 .. 2^-20 apart, 1e3 from the origin; the signed distances keep their
        # difference in proportion (a power-of-two factor), so the line stays feasible
        r = np.ldexp(1.0, np.floor(np.log2(2.0 ** -20 / np.hypot(c[2] - c[0], c[3] - c[1]))).astype(int))
        dx, dy, ds = (c[2] - c[0]) * r, (c[3] - c[1]) * r, (c[5] - c[4]) * r
        c[0][:], c[1][:] = c[0] + 1e3, c[1] + 1e3
        c[2][:], c[3][:], c[5][:] = c[0] + dx, c[1] + dy, c[4] + ds
    elif name == "k3_line_2^-10..-30_of_its_distance":
        _shrink(c, (3, 4), (5, 6), _pow2(rng, -30, -10, n))
    elif name == "k3_line_2^10..30_long":
        _stretch(c, (3, 4), (5, 6), _pow2(rng, 10, 30, n))
    elif name == "k4_lines_2^-10..-30_of_their_distance":
        _shrink(c, (0, 1), (2, 3), _pow2(rng, -30, -10, n))
        _shrink(c, (5, 6), (7, 8), _pow2(rng, -30, -10, n))
    elif name == "k4_lines_2^10..30_long":
        # the second endpoints far out: the guard scale S of K4 is built from the first endpoints only
        _stretch(c, (0, 1), (2, 3), _pow2(rng, 10, 30, n))
        _stretch(c, (5, 6), (7, 8), _pow2(rng, 10, 30, n))
    elif name == "k5_direction_2^-10..-30":
        # the fixed direction vector 2^-10 .. 2^-30 of its usual length, the points 1e3 out
        r = _pow2(rng, -30, -10, n)
        c[0][:], c[1][:] = c[0] * r, c[1] * r
        for col in (7, 8, 10, 11):
            c[col][:] = c[col] + 1e3
    else:
        raise KeyError(name)
    return out


MIXED = {1: ["k1_needle_2^-30..-40"], 2: ["k2_points_2^-20_apart_at_1e3"],
         3: ["k3_line_2^-10..-30_of_its_distance", "k3_line_2^10..30_long"],
         4: ["k4_lines_2^-10..-30_of_their_distance", "k4_lines_2^10..30_long"], 5: ["k5_direction_2^-10..-30"]}

# ---- the exponent grid -------------------------------------------------------------------------
# The synthetic batches' inputs lie between 2^-3 and 2^10 (mostly 2^5 .. 2^9), so at a scale of 2^e a
# quantity of nominal size 2^(e + 8) spreads over about six binades around it: each exponent below puts
# a share of the batch on either side of the bound it names.  "Entries" are Jacobian entries, "q_p" the
# pivot column's squared norm, "numerators" the transformed right-hand side (R4).  R0 - R4:
# newton_core.cuh, qr_fast_core; R3 of K2 / K5 mixes a row of size 2^(e+8) with the unit-normal row.
# The bounds are sufficient, not tight: R1 moved out by one binade at either end changes no result on
# this grid, because the square-root and division sequences stay exact well beyond 2^-800 .. 2^800 (the
# sqrt sequence from 2^-970, the divisions under R2 - R4).  A mutation of R1 therefore cannot be caught
# here; one of R2 - R4 or of the sequences themselves is (csrc/selftest.cu and these cases).
EXPONENTS = {
    -560: "below every lower bound: K4 q_p ~2^-1100, first-update numerators ~2^-537",
    -524: "R4 low, K4 first update from the seed: numerators ~2^(e+23) cross 2^-500",
    -523: "R4 low, K4 first update (crossing)",
    -522: "R4 low, K4 first update",
    -513: "fused column norms: x^2 subnormal for |x| < 2^-511 where (2x)^2 is not",
    -512: "fused column norms: the subnormal-square edge",
    -511: "fused column norms: x^2 normal again",
    -508: "R2 |p_c| >= 2^-500, K4 entries ~2^(e+8)",
    -507: "R2 (crossing)",
    -506: "R2",
    -501: "R2 / R4 bound 2^-500 for unit-sized operands",
    -500: "R2 / R4 bound 2^-500 (crossing)",
    -499: "R2 / R4 bound 2^-500",
    -409: "R1 low q_p >= 2^-800, K4 q_p ~2^(2e+16)",
    -408: "R1 low, K4 (crossing)",
    -407: "R1 low, K4",
    -401: "R1 low for unit-sized entries: |entry| 2^-400",
    -400: "R1 low for unit-sized entries (crossing)",
    -399: "R1 low for unit-sized entries",
    -300: "between the R1 and R4 lower crossings",
    -233: "R4 low, K4 after the landing: residuals of rounding size ~2^(2e+16-52)",
    -232: "R4 low, K4 after the landing (crossing)",
    -231: "R4 low, K4 after the landing",
    -100: "systems far under the tolerance: runs converge while halving in from the seed",
    -60: "R3 of K3 where the iterate stops ~1e-5 out: d'^2 >= 2^-70 q_p",
    -59: "R3 of K3 (crossing)",
    -58: "R3 of K3",
    -45: "R3 of K2 / K5: the scaled row's share of the determinant passes 2^-35",
    -44: "R3 of K2 / K5 (crossing)",
    -43: "R3 of K2 / K5",
    -20: "systems at the tolerance: both convergence regimes",
    -10: "small systems, roots 2^10 tol apart: the scale-relative check applies",
    0: "the synthetic batches as generated",
    10: "large systems, every range test passes",
    20: "large systems: coordinates' ulp 2^-24 next to the tolerance",
    27: "R3 of K2 / K5 from above; coordinates' ulp crosses the tolerance (2^-17)",
    28: "R3 of K2 / K5 from above (crossing)",
    29: "R3 of K2 / K5 from above; K1 / K3 / K4 runs converge only on exact fixed points",
    100: "huge systems, inside the ranges of q_p and the numerators",
    240: "R4 high, K1 / K3 / K4: residuals ~2^(2e+18) cross 2^500",
    241: "R4 high, squared residuals (crossing)",
    242: "R4 high, squared residuals",
    300: "between the R4 and R1 upper crossings",
    390: "R1 high q_p < 2^800, squared norms ~2^(2e+18)",
    391: "R1 high (crossing)",
    392: "R1 high",
    399: "R1 high for unit-sized entries: |entry| 2^400",
    400: "R1 high for unit-sized entries (crossing)",
    401: "R1 high for unit-sized entries",
    491: "R4 high, K2 / K5 linear residuals ~2^(e+8) cross 2^500; guard kBigH 2^500",
    492: "R4 high, linear residuals (crossing)",
    493: "R4 high, linear residuals",
    499: "the 2^500 bound for unit-sized operands",
    500: "the 2^500 bound for unit-sized operands (crossing)",
    501: "the 2^500 bound for unit-sized operands",
    511: "squares of inputs overflow (inputs 2^(e+10) >= 2^512)",
    512: "squares of unit-sized inputs overflow (crossing)",
    513: "every square overflows",
}
SHIFTS = [10, 20, 26, 30, 33, 36, 40]


def _base(kind, n, n_seeds=2):
    kw = {} if n_seeds == 2 else dict(n_seeds=n_seeds)
    return gcs.synth.make(kind, n, **kw)


@functools.lru_cache(maxsize=4)
def _moved_roots_of(kind, k, n, n_seeds):
    """moved_roots of the generator batch, once per (kind, shift, size): every mapping starts from the same
    guesses, and the oracle solves the untranslated batch once (read-only: `translated` copies it)."""
    g = moved_roots(_base(kind, n, n_seeds), np.ldexp(1.0, k), -0.75 * np.ldexp(1.0, k), seed=k)
    g.flags.writeable = False
    return g


def make_case(kind, case, n, n_seeds=2):
    """A fresh batch for the case `case` = (what, arg) of `kind` with n sub-systems."""
    what, arg = case
    hb = _base(kind, n, n_seeds)
    if what == "scale":
        return scaled(hb, arg)
    if what in ("shift", "shift_seeded"):
        ox, oy = np.ldexp(1.0, arg), -0.75 * np.ldexp(1.0, arg)
        g = _moved_roots_of(kind, arg, n, n_seeds) if what == "shift_seeded" else None
        return translated(hb, ox, oy, g)
    assert what == "mixed"
    return mixed(hb, arg)


# ---- the part without a device: the transforms -------------------------------------------------

def test_column_roles_cover_the_soaks_length_columns():
    """The scaled columns are the soak's rescaled columns (tests/test_gpu_soak.py LENGTH_COLS) plus all of K1."""
    from test_gpu_soak import LENGTH_COLS
    for kind in (2, 3, 4, 5):
        assert scaled_cols(kind) == sorted(LENGTH_COLS[kind]), kind
    assert scaled_cols(1) == list(range(6))
    for kind, r in ROLES.items():
        used = scaled_cols(kind)
        assert len(set(used)) == len(used) and max(used) < capi.IN_COLS[kind]


@pytest.mark.parametrize("e", [-560, -512, -408, -1, 0, 241, 513])
@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_scaling_keeps_every_mantissa(kind, e):
    hb = _base(kind, 999)
    if kind in POINT_UNKNOWNS:
        hb.guesses = np.ascontiguousarray(np.random.default_rng(e & 0xFF).uniform(-3e3, 3e3, size=(2, 2, hb.n)))
    s = scaled(hb, e)
    moved = set(scaled_cols(kind))
    for c, (a, b) in enumerate(zip(hb.cols, s.cols)):
        if c not in moved:
            assert np.array_equal(bits(a), bits(b)), f"column {c} moved"
            continue
        fin = np.isfinite(b) & (a != 0)
        if e < 0:  # every input of the generators is at least 2^-60 or zero: nothing goes subnormal
            assert fin.all() or (a[~fin] == 0).all()
        ma, ea = np.frexp(a[fin])
        mb, eb = np.frexp(b[fin])
        assert np.array_equal(ma, mb) and np.array_equal(eb - ea, np.full_like(ea, e)), f"column {c}"
        assert np.array_equal(bits(np.ldexp(b[fin], -e)), bits(a[fin]))
        assert np.array_equal(b[a == 0], a[a == 0])
    assert np.array_equal(s.code, hb.code)
    if kind in POINT_UNKNOWNS:
        assert np.array_equal(bits(np.ldexp(s.guesses, -e)), bits(hb.guesses))
    assert (hb.cols[0] is not s.cols[0]) and np.array_equal(bits(hb.cols[0]), bits(_base(kind, 999).cols[0])), "input batch modified"


@pytest.mark.parametrize("k", [10, 40])
@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_translation_keeps_lengths_signed_distances_and_canvas_columns(kind, k):
    hb = _base(kind, 999)
    ox, oy = np.ldexp(1.0, k), -0.75 * np.ldexp(1.0, k)
    t = translated(hb, ox, oy)
    pts = _flat(ROLES[kind]["points"])
    for c, (a, b) in enumerate(zip(hb.cols, t.cols)):
        if c in pts:
            off = ox if c in [p[0] for p in ROLES[kind]["points"]] else oy
            assert np.array_equal(bits(b), bits(a + off)), f"column {c}"
        else:
            assert np.array_equal(bits(a), bits(b)), f"column {c} moved"
    assert np.array_equal(t.code, hb.code) and t.guesses is None


@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_moved_roots_start_next_to_the_oracles_roots(kind):
    n, k = 257, 20
    hb = _base(kind, n)
    ox, oy = np.ldexp(1.0, k), -0.75 * np.ldexp(1.0, k)
    g = moved_roots(hb, ox, oy, seed=1)
    ref = O.solve(_copy(hb).alloc_outputs(), threads=0)
    want = ref.cand.copy()
    if kind in POINT_UNKNOWNS:
        want[:, 0] += ox
        want[:, 1] += oy
    fin = np.isfinite(ref.cand)
    scale = np.abs(ref.cand[fin]) + (0.0 if kind in (2, 5) else np.ldexp(1.0, k))
    assert (np.abs(g[fin] - want[fin]) <= 2.0 ** -17 * scale).all()
    t = translated(hb, ox, oy, g)
    assert t.guesses.shape == (2, 2, n)


@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_mixed_batches_keep_their_roots_where_they_should(kind):
    """Shrinking or stretching a line along itself keeps the infinite line, so K3 / K4 keep their roots;
    every mixed batch of every kind solves on the oracle."""
    n = 512
    base = O.solve(_base(kind, n).alloc_outputs(), threads=0)
    for name in MIXED[kind]:
        m = O.solve(mixed(_base(kind, n), name).alloc_outputs(), threads=0)
        assert ((m.iters >= 0) & (m.iters <= 1000)).all() and (m.root_index < 2).all()
        assert m.converged.mean() > 0.5, name
        if kind == 4:
            ok = (base.converged[0] == 1) & (m.converged[0] == 1) & (base.iters[0] < 5)
            assert ok.mean() > 0.8
            d = np.hypot(m.cand[0, 0, ok] - base.cand[0, 0, ok], m.cand[0, 1, ok] - base.cand[0, 1, ok])
            assert np.median(d) < 1e-3, name


@pytest.mark.parametrize("case", [("scale", -560), ("scale", -512), ("scale", -408), ("scale", 28), ("scale", 241),
                                  ("scale", 513), ("shift", 40), ("shift_seeded", 33)], ids=str)
@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_transformed_batches_solve_on_the_oracle(kind, case):
    hb = make_case(kind, case, 97)
    O.solve(hb.alloc_outputs(), threads=0)
    assert ((hb.iters >= 0) & (hb.iters <= 1000)).all() and (hb.root_index < 2).all()
    assert set(np.unique(hb.converged)) <= {0, 1}


# ---- the GPU part -----------------------------------------------------------------------------

def _reset_stats(lib):
    st = (C.c_uint64 * 8)()
    lib.gcs_b200_contracted_stats_ex(0, st, 1)
    return st


def _literal_runs(lib):
    st = (C.c_uint64 * 8)()
    assert lib.gcs_b200_contracted_stats_ex(0, st, 1) == 0
    return int(sum(st))


def _floor_free(got, ref, kind):
    """|got - ref| <= 1e-9 S_sub on the runs that decided on quadratic convergence: the chosen run
    converged and the roots lie at least 2^10 tol apart on the oracle's two candidates (the half chord
    for K1 / K3, the distance of the two unit normals for K2 / K5; K4 has one root).  There both
    arithmetics sit within eps * cond of the same root, cond <= 2^14 by the (G1) floor.  S_sub: the
    sub-system's largest finite input magnitude.  Returns (runs checked, worst |got - ref| / S_sub).

    Newton corrects its own step errors: a solve whose reciprocal is left at its 2^-20 MUFU seed still
    ends within 2^-20 of the last update (< tol) of the root, about 1e-11, and the roots being 2^10 tol
    apart puts S_sub above 5e-3, so this bound cannot see it (worst 1.3e-13 with such a reciprocal).
    Such an arithmetic moves the landing from the far seed instead, and the iteration counts that
    assert_batches_within_contract compares catch it."""
    n = ref.n
    idx = np.arange(n)
    root = ref.root_index.astype(np.int64)
    conv = ref.converged[np.minimum(root, ref.n_seeds - 1), idx] == 1
    if kind == 4:
        sep_ok = np.ones(n, bool)
    else:
        with np.errstate(invalid="ignore", over="ignore"):
            sep = np.hypot(ref.cand[0, 0] - ref.cand[1, 0], ref.cand[0, 1] - ref.cand[1, 1])
        if kind in (1, 3):
            sep = 0.5 * sep
        sep_ok = sep >= 1024.0 * TOL
    with np.errstate(invalid="ignore", over="ignore"):
        s_sub = np.max(np.stack([np.where(np.isfinite(c), np.abs(c), 0.0) for c in ref.dense_cols()]), axis=0)
        sel = conv & sep_ok & (s_sub > 0)
        pairs = [(a[sel], b[sel]) for a, b in zip(got.out, ref.out)]
        pairs += [(got.cand[root[sel], i, idx[sel]], ref.cand[root[sel], i, idx[sel]]) for i in range(2)]
        worst = 0.0
        for a, b in pairs:
            fin = np.isfinite(b)
            if fin.any():
                worst = max(worst, float((np.abs(a[fin] - b[fin]) / s_sub[sel][fin]).max()))
    return int(sel.sum()), worst


def _label(kind, case, n_seeds=2):
    what, arg = case
    tag = {"scale": f"x2^{arg}", "shift": f"+2^{arg}", "shift_seeded": f"+2^{arg} seeded", "mixed": arg}[what]
    return f"K{kind} {tag}" + (f" x{n_seeds} seeds" if n_seeds != 2 else "")


def _sizes(kind, case, n_seeds):
    """(n, n for the sorted mappings): 4099 (a ragged tail) and 2^16 (full tiles) where runs converge;
    2003 for both where they take 1000 iterations on the oracle too (a 64-row probe decides)."""
    probe = O.solve(make_case(kind, case, 64, n_seeds).alloc_outputs(), threads=0)
    if probe.iters.mean() > 200:
        return 2003, 2003
    return 4099, 1 << 16


def _run_case(gpu, kind, case, n_seeds=2, contracted=True):
    lib = gpu.load()
    what = _label(kind, case, n_seeds)
    n_small, n_sorted = _sizes(kind, case, n_seeds)
    refs = {}
    for n in sorted({n_small, n_sorted}):
        refs[n] = O.solve(make_case(kind, case, n, n_seeds).alloc_outputs(), threads=0)
    for v in BITWISE:
        n = n_sorted if v in SORTED else n_small
        hb = make_case(kind, case, n, n_seeds)
        hb.variant = v
        gpu.solve_host(hb.alloc_outputs(), 0)
        assert_batches_identical(hb, refs[n], f"{what} variant {v}")
        print(f"[ranges] {what:40s} variant {v:2d} n {n:6d}: {n * n_seeds} runs bit-identical, "
              f"{float(refs[n].converged.mean()):.3f} converged")
    if not contracted:
        return
    for v in CONTRACTED + ([LINEAR] if kind == 4 else []):
        n = n_sorted if v in SORTED else n_small
        hb = make_case(kind, case, n, n_seeds)
        hb.variant = v
        _reset_stats(lib)
        gpu.solve_host(hb.alloc_outputs(), 0)
        literal = _literal_runs(lib)
        worst = assert_batches_within_contract(hb, refs[n], f"{what} variant {v}")
        checked, rel = _floor_free(hb, refs[n], kind)
        print(f"[ranges] {what:40s} variant {v:2d} n {n:6d}: {n * n_seeds} runs within contract (worst {worst:.2e}), "
              f"{literal} literal, {checked} scale-relative checks, worst {rel:.2e}")
        assert rel <= 1e-9, f"{what} variant {v}: |got - ref| / S_sub = {rel:.3e} on runs that converged quadratically"


# ---- regression tests: what the grid found in the contracted class ----

@pytest.mark.gpu
@pytest.mark.parametrize("kind", [2, 5])
def test_contracted_unit_normal_kinds_with_a_tiny_linear_row(gpu, kind):
    """K2 / K5 whose linear row is 2^-37 .. 2^-35 of the unit-normal row: the literal QR rounds that
    row's equation relative to the larger row, so its iteration counts carry an error the guards did not
    budget for, and every contracted mapping decided some runs differently.  Such runs now go literal
    (newton_relaxed.cuh, rows_comparable)."""
    _run_case(gpu, kind, ("scale", -44))


@pytest.mark.gpu
def test_contracted_k2_with_fixed_points_2_20_apart(gpu):
    """K2 with its fixed points 2^-21 .. 2^-20 apart, 1e3 out: coordinates were more than 1e-9 off on
    every contracted mapping (the same row-size mismatch)."""
    _run_case(gpu, 2, ("mixed", "k2_points_2^-20_apart_at_1e3"))


@pytest.mark.gpu
@pytest.mark.parametrize("e", [-300, 200])
def test_contracted_sorted_k2_far_from_unit_scale(gpu, e):
    """K2 through the contracted-sorted mapping at 2^-300 and 2^200: unit normals up to 7.5e-6 off."""
    _run_case(gpu, 2, ("scale", e))


@pytest.mark.gpu
@pytest.mark.parametrize("e", [-300, -100])
def test_contracted_k4_systems_under_the_landing_noise(gpu, e):
    """K4 at 2^-300 and 2^-100: the landing from the default seeds carries more rounding noise than the
    system is large, and the static / sorted / sequential mappings chose other roots
    (newton_relaxed.cuh, kMinLinearScale)."""
    _run_case(gpu, 4, ("scale", e))


@pytest.mark.gpu
@pytest.mark.parametrize("e", list(EXPONENTS), ids=[f"e{e}" for e in EXPONENTS])
@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_scaled_systems(gpu, kind, e):
    """Every length, point and canvas coordinate x 2^e: bit-identical mappings bit for bit, contracted ones
    to the contract and the scale-relative bound."""
    _run_case(gpu, kind, ("scale", e))


@pytest.mark.gpu
@pytest.mark.parametrize("seeded", [False, True], ids=["default_seeds", "moved_roots"])
@pytest.mark.parametrize("k", SHIFTS)
@pytest.mark.parametrize("kind", [1, 2, 3, 4, 5])
def test_translated_systems(gpu, kind, k, seeded):
    """Whole systems 2^k from the origin: from the default seeds every run starts in the far-seed regime;
    from the oracle's own roots of the untranslated batch (moved along) the same runs happen far out."""
    _run_case(gpu, kind, ("shift_seeded" if seeded else "shift", k))


@pytest.mark.gpu
@pytest.mark.parametrize("kind,name", [(k, m) for k in MIXED for m in MIXED[k]])
def test_mixed_magnitude_systems(gpu, kind, name):
    _run_case(gpu, kind, ("mixed", name))


@pytest.mark.gpu
@pytest.mark.parametrize("e", [-408, -232, -20, 0, 20, 241, 391])
@pytest.mark.parametrize("kind", [1, 3, 4])
def test_eight_seeds_across_exponents(gpu, kind, e):
    _run_case(gpu, kind, ("scale", e), n_seeds=8, contracted=False)


# ---- sketch programs at scale -----------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("e", [-40, -20, 20, 40])
@pytest.mark.parametrize("seed", [31, 32, 33])
def test_sketch_programs_at_scale_equal_the_cpu_restatements(gpu, built, seed, e):
    """The golden leaf programs with every length value and every initial position x 2^e, K = 4: device run,
    tangents and the adjoints of a recorded run equal the CPU restatements bit for bit, NaN with NaN."""
    import program_restate as R
    import program_tangents_lib as PT
    import sketch_gen as S
    from program_restate_adjoints import restate_adjoints
    from test_gpu_host import WHOLE_SKETCHES
    from test_gpu_sketch_program_abi import Prog, _directions, _values
    from test_gpu_sketch_program_adjoints import _adjoints, _record

    def same(a, b):
        return a.shape == b.shape and bool(((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))).all())

    built.build_host()
    first, n = {s: (f, m) for s, f, m in WHOLE_SKETCHES}[seed][:2]
    el, lv = S.make_sketch(n, seed=seed, first_shape=first)
    prog = PT.Program(el, leaves=lv)
    assert prog.rc == 0, prog.error
    p0 = R.Arrays.from_desc(prog.desc())
    base = np.array([x["value"] for lf in lv for x in lf["edges"] if x["type"] != S.VIRT])
    angle = p0.value_is_angle.astype(bool)
    p = R.Arrays(p0.rows, p0.offsets, p0.slot_is_line, np.ldexp(p0.initial, e), p0.value_is_angle)
    vals, _ = _values(p, base, 4, seed=seed)
    vals = np.where(angle[None, :], vals, np.ldexp(vals, e))
    dvals = _directions(p, 4, 3, seed=seed + 1)
    with Prog(gpu.load(), p) as dev:
        pos, dpos, nc, _ = dev.run_host(vals, dvals)
        ob = np.random.default_rng(seed + 2).standard_normal((4, p.n_slots, 4, 2))
        ob[..., 1:] *= np.isfinite(dpos[..., :1])
        rpos, rnc, _ = _record(dev, vals)
        adj, _ = _adjoints(dev, ob)
    want, dwant, wnc = R.restate(p, vals, dvals)
    assert same(pos, want) and np.array_equal(nc, wnc), f"positions, 2^{e}"
    assert same(dpos, dwant), f"tangents, 2^{e}"
    assert same(rpos, want) and np.array_equal(rnc, wnc), f"recorded run, 2^{e}"
    assert same(adj, restate_adjoints(p, vals, ob)), f"adjoints, 2^{e}"
    fin = float(np.isfinite(pos[..., :2]).mean())
    print(f"[ranges] sketch {seed} x2^{e}: {pos.shape[0]} instances, {fin:.3f} of the coordinates finite, "
          f"{int(nc.sum())} rows without a converged root")
    assert fin > 0.5
