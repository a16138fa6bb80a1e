// newton_relaxed.cuh — the tolerance-class arithmetic of GCS_VARIANT_CONTRACTED (sm_100a).
//
// The bit-identical kernels spend 35 of their 72 FP64 instructions per update on the four IEEE
// divisions and the square root of Eigen's Householder QR, and may not contract a*b+c.  The
// correctness contract of the path (BASELINE.json north_star) is narrower than bit identity:
//     iteration count, convergence flag, chosen root   identical to the reference,
//     solved coordinates                               within 1e-9 relative.
// This file solves the same 2x2 Newton system in closed form (Cramer's rule on fused
// multiply-adds, one reciprocal refined to ~2^-60) - about 21 FP64 instructions per update - and
// keeps the discrete outputs identical by construction:
//
//   * every decision that could come out differently under a perturbation of the iterate is
//     detected and the run is redone with the literal device functions of newton_core.cuh
//     (newton_run, the same code the bit-identical kernels execute).  Detected means:
//       (G1) |det J| has fallen under 2^-10 of its size at a well-conditioned root of this system
//            (per-system constant): the step is sensitive to rounding;
//       (G2) |det J| has grown 16x over its smallest value so far: the iterate has been thrown
//            back out from near the line where J is singular - the one event that amplifies a
//            deviation between the two arithmetics (and the signature of a run without real roots);
//       (G3) the length of an update lies inside a band around the convergence threshold
//            (newton_raphson.hpp:83-88).  First level, integer tests: band = 2^-16 tol + 2^-36 S with
//            S the magnitude of the system's coordinates.  Second level, for the update that falls
//            into that band: | m - tol | <= 2^-44 S dr/|det| + 2^-40 tol, 32x the bound on how far
//            the two arithmetics' updates can be apart from the same iterate;
//       (G4) no convergence after kRelaxCap updates (slow or chaotic runs: no real root, tangent
//            circles), or a non-finite / huge update;
//       (G5) in the root selection, an orientation (or a distance difference) within 2^-24
//            relative of zero: the sign (or the comparison) could flip.
//   * why that suffices - an argument, backed by the tests, not a machine-checked proof.  Both
//     arithmetics are backward stable on a 2x2 system, so from the same iterate their updates
//     differ by O(cond(J) (eps |step| + ulp(S))).  Every equation pair of the path is a circle and
//     a line (newton_kernels.cuh, "Prediction"): the first update lands on the line, and along it
//     Newton's map is w <- (w^2 + h^2)/(2w), +-h the roots, with derivative (1 - h^2/w^2)/2.
//       - Landing from a far seed (|seed| = G) is itself ill conditioned (cond ~ G/d): the two
//         arithmetics land a RELATIVE eps G/d apart.  While |w| >> h the map halves w and the
//         deviation alike: the relative deviation is carried, not grown.  A system smaller than
//         the tolerance (h <~ 1e-5) meets `< tol` while still in that phase, so the carried
//         deviation eps cond(J_seed) * |update| is part of both levels of (G3)
//         (RelaxGuard::add_carry; found by a 1.1e8-system soak: one run in 4.2e6 at scale 1e-6
//         had decided differently before this term existed).
//       - Once |w| ~ h the map contracts quadratically: the deviation is multiplied by
//         (w - h)/h per update, so at the deciding update (the first one shorter than tol) what is
//         left of the history is below eps (G/d) sqrt(2 h tol) times further factors < 0.4 - orders
//         of magnitude under the band at every scale the soak covers (1e-6 .. 1e6).
//       - The only amplifying event is a landing (or a seed) with |w| << h, which throws the
//         iterate out to h^2/(2w): |det| grows by (h/w)^2/2.  (G2) sends those runs to the
//         literal code, so nothing is amplified by more than 4x on the closed-form path.
//       - At the deciding update the fresh difference between the two arithmetics is
//         ~8 (dr/|det|) 2^-52 S with dr/|det| <= 2^10 by (G1): 2^-39 S against a first-level band
//         of 2^-36 S, and the second level scales its margin with the actual dr/|det|.
//       - Runs without real roots never meet the threshold and leave by (G2) / (G4); non-finite
//         values by (G4).
//   * tests/test_gpu_relaxed.py and the soak (profiles/) compare iteration counts, flags and root
//     indices for equality and coordinates to 1e-9 against the CPU checker on every parity case;
//     bench.py re-checks its whole batch against the bit-identical kernels in every run.
#pragma once

#include <type_traits>

#include "newton_core.cuh"

namespace gcsk {

constexpr int kRelaxCap = 64;  // updates a run may take on the closed-form path (G4)
constexpr int kBounce = 4 << 20;  // (G2) four binades of growth of |det| over its running minimum
#ifndef GCS_CAREFUL_BINADES
#define GCS_CAREFUL_BINADES 4
#endif
constexpr int kCarefulBinades = GCS_CAREFUL_BINADES;  // careful mode reaches this many binades under the (G1) line 2^-10 dr (0: off)

// How often the guards hand work to the literal code (read by gcs_b200_contracted_stats[_ex]), by
// reason (kWhy*): touched on the rare path only.
enum : int {
    kWhyCond = 0,       // (G1) |det J| under its floor: conditioning past what the margins cover
    kWhySelection = 1,  // (G5) root selection within its margin
    kWhyBounce = 2,     // (G2) |det J| grew 16x over its running minimum
    kWhyBand = 3,       // (G3) update length inside the second-level margin around the threshold
    kWhyCap = 4,        // (G4) kRelaxCap updates without convergence
    kWhyHuge = 5,       // (G4) non-finite / huge update
    kWhyCount = 8
};
__device__ unsigned long long g_relax_reruns[kWhyCount];

// 1/b to ~2^-60 relative: MUFU.RCP64H seed (>= 20 bits) and one cubic refinement
__device__ __forceinline__ double rcp_relaxed(double b)
{
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(b));
    double e = __fma_rn(-b, r, 1.0);
    e = __fma_rn(e, e, e);
    return __fma_rn(r, e, r);
}

// |v|^-1/2 refined to an ulp or two (MUFU.RSQ64H seed, one cubic step: 2^-60 before the roundings of the step itself)
__device__ __forceinline__ double rsqrt_relaxed(double v)
{
    double r;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(v));
    const double e = __fma_rn(-v * r, r, 1.0);           // 1 - v r^2
    return __fma_rn(r * __fma_rn(0.375, e, 0.5), e, r);  // r (1 + e/2 + 3 e^2 / 8)
}

__device__ __forceinline__ int abs_hi(double v) { return __double2hiint(v) & 0x7fffffff; }

// high word of a non-negative double, rounded outwards (thresholds of integer comparisons)
__device__ __forceinline__ int hi_floor(double v) { return v > 0.0 ? __double2hiint(v) : 0; }

// K2 / K5 pair a linear row of size L with the unit-normal row (size 2).  The literal solve's column-
// pivoted QR rounds relative to the columns' norms, which the larger row dominates: its error in the
// smaller row's equation is eps times the ratio of the rows, which the guards' eps S cond budget does not
// contain.  Where the ratio leaves 2^-16 .. 2^16 the run goes to the literal code (det_root < 0 below:
// G1 on the first update).  Found by tests/test_gpu_ranges.py at 2^-45 .. 2^-43 and on K2 fixed points
// 2^-20 apart.
__device__ __forceinline__ bool rows_comparable(double len) { return len >= 0x1p-16 && len <= 0x1p16; }

// K4 lands with its first update; from a seed at |G| (20000 for the default seeds) the landing carries an
// absolute rounding error ~eps cond |G|, and a system whose coordinates are smaller than that is solved
// to noise in both arithmetics: the two seeds' candidates differ by that noise and the nearest-to-canvas
// selection decides on it, beyond what (G5) budgets (2^-36 S).  Under 2^-20 the run goes literal.
// Found by tests/test_gpu_ranges.py at 2^-513 .. 2^-100.
constexpr double kMinLinearScale = 0x1p-20;

// Per-run constants of the guards, derived once per run from the system's scale.
struct RelaxGuard {
    int lo_h, hi_h;  // hi(|s|) < lo_h: converged for certain; >= hi_h: not converged for certain
    int det_h;       // hi(|det|) must reach this (G1)
    double pm;       // 2^-44 S dr: numerator of the second-level margin (S coordinate scale, dr = |det| at a well-conditioned root)
    double band;     // first-level band of this system before the run's own carry term
    double carry;    // 2^-48 cond(J at the seed): relative deviation the run carries from its first update (x4 margin)
    static constexpr int kBigH = 0x5F300000;  // 2^500: anything from here on is "non-finite / huge" (G4)
    // thresholds of the integer tests for a first-level band of `b` around tol; step_scale: the
    // closed-form solve returns step / step_scale (K1 works on J/2)
    __device__ __forceinline__ void set_band(double b, double step_scale)
    {
        const double inv = 1.0 / step_scale;  // 1 or 2: exact
        lo_h = hi_floor((kTol - b) * inv) - 1;
        hi_h = hi_floor((kTol + b) * inv) + 1;
        if (!(b < kTol)) lo_h = 0;  // also catches a NaN band: never "certain"
        if (lo_h < 0) lo_h = 0;
        if (!(hi_h > 0 && hi_h < kBigH)) hi_h = kBigH;
    }
    __device__ __forceinline__ void init(double coord_scale, double det_root, double step_scale)
    {
        pm = 0x1p-44 * coord_scale * det_root;
        band = __fma_rn(0x1p-36, coord_scale, 0x1p-16 * kTol);
        carry = 0.0;
        set_band(band, step_scale);
        det_h = hi_floor(0x1p-10 * det_root) + 1;
        if (!(det_root > 0.0 && det_root < 0x1p900)) det_h = 0x7ff00000;  // degenerate / NaN / inf scale: always uncertain
    }
    // The update from the seed is as ill conditioned as the seed is far (cond ~ |seed| / d for the
    // default seeds): the two arithmetics land a RELATIVE 2^-53 cond(J_seed) apart, and that relative
    // deviation rides along while the iteration halves its way in.  Where the roots are closer
    // together than the tolerance (small systems: h <~ 1e-5) the deciding update happens in that
    // phase, before the quadratic contraction has wiped the history out, and the update length then
    // differs by ~2^-53 cond * 2 |update|.  With c = cond(J_seed) = |J|_F^2 / |det|:
    //     carry = 2^-48 c   (2^-53 c, x2 for |w| ~ 2 |update|, x4 for the halving-phase updates'
    //                        own contributions, x4 margin),
    // added as carry * tol to the first-level band and as carry * m to the second-level margin.
    __device__ __forceinline__ void add_carry(double c, double step_scale)
    {
        carry = c;
        set_band(__fma_rn(c, kTol, band), step_scale);
    }
    // Second level of (G3), reached only by an update whose length fell between lo_h and hi_h (the
    // first-level band, integer tests on high words, is 2^-36 S wide; about one run in a thousand
    // gets here).  From the same iterate the two arithmetics' updates differ by at most
    // ~8 (dr/|det|) 2^-52 S: the residuals carry O(ulp(S)) rounding, the solve divides by det
    // (newton_relaxed.cuh header; dr/|det| <= 2^10 by G1).  With 32x margin:
    //     | m - tol | > 2^-44 S dr/|det| + 2^-40 tol   ->   `m < tol` is the literal code's decision too.
    // Returns +1 converged for certain, -1 not converged for certain, 0 undecided.
    // `extra`: an absolute term on top (the deviation carried over from the PREVIOUS update, see
    // relaxed_updates: carry * |previous update|, which matters when that update dwarfs this one).
    __device__ __forceinline__ int precise(double m, double det, double extra = 0.0) const
    {
        const double margin = __fma_rn(carry, m, __fma_rn(pm, rcp_relaxed(fabs(det)), 0x1p-40 * kTol)) + extra;
        const double gap = m - kTol;
        if (gap > margin) return -1;
        if (-gap > margin) return 1;
        return 0;  // NaN margins land here
    }
};

// ------------------------------------------------------------------------------------------
// The five equation pairs with fused multiply-adds: J = [[a b],[c d]], right-hand side (-f, -g).
// load() takes the same input columns as Sys<KIND>::load.
// ------------------------------------------------------------------------------------------
template <int KIND>
struct Rsys;

// K1: two circles.  Works on J/2 = [[dxa dya],[dxb dyb]]: the solve returns twice the step.
template <>
struct Rsys<GCS_KIND_PP> {
    static constexpr double kStepScale = 0.5;
    double ax, ay, qa, bx, by, qb;
    // kGuard = false: only the system's constants (the guard comes from where it was stashed)
    template <bool kGuard = true>
    __device__ __forceinline__ void load(const double* k, RelaxGuard& g)
    {
        ax = k[0], ay = k[1], qa = k[2] * k[2];
        bx = k[3], by = k[4], qb = k[5] * k[5];
        // at a root det(J/2) = (P-A) x (P-B) = ra rb sin(angle at P)
        if constexpr (kGuard) g.init(fabs(ax) + fabs(ay) + fabs(bx) + fabs(by) + fabs(k[2]) + fabs(k[5]), fabs(k[2] * k[5]), kStepScale);
    }
    __device__ __forceinline__ void eval(
        double x, double y, double& a, double& b, double& c, double& d, double& r0, double& r1) const
    {
        a = x - ax, b = y - ay, c = x - bx, d = y - by;
        r0 = __fma_rn(-b, b, __fma_rn(-a, a, qa));
        r1 = __fma_rn(-d, d, __fma_rn(-c, c, qb));
    }
};

// K2: signed-distance difference (linear) + unit normal
template <>
struct Rsys<GCS_KIND_SDD> {
    static constexpr double kStepScale = 1.0;
    double dX, dY, c0;
    // kGuard = false: only the system's constants (the guard comes from where it was stashed)
    template <bool kGuard = true>
    __device__ __forceinline__ void load(const double* k, RelaxGuard& g)
    {
        dX = k[2] - k[0], dY = k[3] - k[1];
        c0 = k[4] - k[5];
        const double l1 = fabs(dX) + fabs(dY);
        // iterates are unit normals; the linear residual carries the offsets in units of |delta|.
        // Rows far apart in size (|delta| outside 2^-16 .. 2^16 of the unit-normal row): run literally.
        if constexpr (kGuard)
            g.init(1.0 + (fabs(k[4]) + fabs(k[5])) * rcp_relaxed(l1), rows_comparable(l1) ? 2.0 * l1 * 0.70710678118654746 : -1.0,
                kStepScale);
    }
    __device__ __forceinline__ void eval(
        double x, double y, double& a, double& b, double& c, double& d, double& r0, double& r1) const
    {
        a = dX, b = dY, c = x + x, d = y + y;
        r0 = -__fma_rn(dX, x, __fma_rn(dY, y, c0));
        r1 = __fma_rn(-x, x, __fma_rn(-y, y, 1.0));
    }
};

struct RP2L {
    double xa, ya, ex, ey, ld, len, rl;
    __device__ __forceinline__ void set(double xa_, double ya_, double xb_, double yb_, double s_)
    {
        xa = xa_, ya = ya_;
        ex = xb_ - xa_, ey = yb_ - ya_;
        // |e| to an ulp or two without the 40 instructions of an IEEE square root (the literal code's
        // length is correctly rounded: the difference is an ulp of the coordinate scale, in the budget)
        const double l2 = __fma_rn(ex, ex, ey * ey);
        rl = rsqrt_relaxed(l2);  // a point for a line: inf, len = NaN -> (G4)
        len = l2 * rl;
        ld = len * s_;
    }
    // -f of pointToLineDistance: ld - uy ex + ux ey
    __device__ __forceinline__ double neg_f(double x, double y) const
    {
        return __fma_rn(x - xa, ey, __fma_rn(-(y - ya), ex, ld));
    }
};

// K3: circle + point-to-line (linear)
template <>
struct Rsys<GCS_KIND_PPL> {
    static constexpr double kStepScale = 1.0;
    double px, py, q;
    RP2L l;
    // kGuard = false: only the system's constants (the guard comes from where it was stashed)
    template <bool kGuard = true>
    __device__ __forceinline__ void load(const double* k, RelaxGuard& g)
    {
        px = k[0], py = k[1], q = k[2] * k[2];
        l.set(k[3], k[4], k[5], k[6], k[7]);
        // at a root det J = 2 (P - C) . e = 2 r L cos(.)
        if constexpr (kGuard) g.init(fabs(px) + fabs(py) + fabs(k[2]) + fabs(k[3]) + fabs(k[4]) + fabs(k[7]), 2.0 * fabs(k[2]) * l.len, kStepScale);
    }
    __device__ __forceinline__ void eval(
        double x, double y, double& a, double& b, double& c, double& d, double& r0, double& r1) const
    {
        const double dx = x - px, dy = y - py;
        a = dx + dx, b = dy + dy, c = -l.ey, d = l.ex;
        r0 = __fma_rn(-dy, dy, __fma_rn(-dx, dx, q));
        r1 = l.neg_f(x, y);
    }
};

// K4: two point-to-line equations (linear system, constant Jacobian)
template <>
struct Rsys<GCS_KIND_PLL> {
    static constexpr double kStepScale = 1.0;
    RP2L l1, l2;
    // kGuard = false: only the system's constants (the guard comes from where it was stashed)
    template <bool kGuard = true>
    __device__ __forceinline__ void load(const double* k, RelaxGuard& g)
    {
        l1.set(k[0], k[1], k[2], k[3], k[4]);
        l2.set(k[5], k[6], k[7], k[8], k[9]);
        // Systems under 2^-20 in their coordinates: run literally (see kMinLinearScale).
        const double sc = fabs(k[0]) + fabs(k[1]) + fabs(k[5]) + fabs(k[6]) + fabs(k[4]) + fabs(k[9]);
        if constexpr (kGuard) g.init(sc, sc >= kMinLinearScale ? l1.len * l2.len : -1.0, kStepScale);
    }
    __device__ __forceinline__ void eval(
        double x, double y, double& a, double& b, double& c, double& d, double& r0, double& r1) const
    {
        a = -l1.ey, b = l1.ex, c = -l2.ey, d = l2.ex;
        r0 = l1.neg_f(x, y);
        r1 = l2.neg_f(x, y);
    }
};

// K5: normal-angle (linear) + unit normal
template <>
struct Rsys<GCS_KIND_ANG> {
    static constexpr double kStepScale = 1.0;
    double fdx, fdy, cl, len, rl;
    // kGuard = false: only the system's constants (the guard comes from where it was stashed)
    template <bool kGuard = true>
    __device__ __forceinline__ void load(const double* k, RelaxGuard& g)
    {
        fdx = k[0], fdy = k[1];
        const double l2 = __fma_rn(fdx, fdx, fdy * fdy);
        rl = rsqrt_relaxed(l2);  // see RP2L::set
        len = l2 * rl;
        cl = k[2] * len;
        // unit normals; the linear residual is L (cos(phi) - cosA): scale 2; det J = 2 L sin(.).
        // Rows far apart in size (L outside 2^-16 .. 2^16): run literally, as K2.
        if constexpr (kGuard) g.init(2.0, rows_comparable(len) ? 2.0 * len : -1.0, kStepScale);
    }
    __device__ __forceinline__ void eval(
        double x, double y, double& a, double& b, double& c, double& d, double& r0, double& r1) const
    {
        a = fdy, b = -fdx, c = x + x, d = y + y;
        r0 = __fma_rn(fdx, y, __fma_rn(-fdy, x, cl));
        r1 = __fma_rn(-x, x, __fma_rn(-y, y, 1.0));
    }
};

// Outcome of a stretch of closed-form updates.  Uncertain outcomes carry the reason:
// state = kRlxUncertain + kWhy*.
enum : int { kRlxRunning = 0, kRlxConverged = 1, kRlxUncertain = 2, kRlxWantCareful = 32 };
__device__ __forceinline__ bool rlx_uncertain(int state) { return state >= kRlxUncertain; }

// Up to `limit` closed-form updates from (x, y), `it` updates applied so far.  Returns
//   kRlxConverged : the last update was shorter than the threshold for certain (and no guard fired)
//   kRlxUncertain : a guard fired - the caller redoes the run from its seed with newton_run
//   kRlxRunning   : `limit` reached, every update so far longer than the threshold for certain.
// d2 / d3 (optional): squared lengths of the last two updates, for the sort key of the sorted kernel.
// dmin_io (optional): the running minimum of hi(|det|) after the seed, carried from one stretch of a
// run to the next so that (G2) sees growth across the hand-off.
template <int KIND, bool kTrack>
__device__ __forceinline__ int relaxed_updates(const Rsys<KIND>& rs, RelaxGuard& g, double& x, double& y, int& it,
    int limit, double& d2, double& d3, int* dmin_io = nullptr, int* trace = nullptr)
{
    // trace (test hook, rare path only): |= 1 when a decision went to the second-level margin test
    unsigned span = (unsigned)(RelaxGuard::kBigH - g.hi_h);
    // smallest hi(|det|) at the iterates after the seed, and its largest growth over that running
    // minimum; the determinant AT THE SEED (d1) counts for (G1) only: both arithmetics start from
    // the same seed, so a badly conditioned first update creates a deviation (eps cond, carried
    // and then contracted) but has none to amplify, and |det| growing from the seed to the
    // landing point is routine (a seed that happens to lie near the singular line).
    int dmin = 0x7fffffff, grow = 0, d1 = 0x7fffffff;
    if (dmin_io && it > 0) dmin = *dmin_io;  // a run continued from an earlier stretch (sorted kernel)
    int state = kRlxRunning;
    if (it >= limit) return (limit >= kRelaxCap) ? kRlxUncertain + kWhyCap : kRlxRunning;
    int mh, dh;
    double s0, s1, det;
    // one closed-form update; leaves mh = larger high word of the update's components, dh = hi(|det|)
    auto update = [&](auto from_seed) {
        double a, b, c, d, r0, r1;
        rs.eval(x, y, a, b, c, d, r0, r1);
        det = __fma_rn(a, d, -(b * c));
        const double r = rcp_relaxed(det);
        if constexpr (decltype(from_seed)::value) {
            // the carry term of this run (RelaxGuard::add_carry): cond(J_seed) = |J|_F^2 / |det|
            const double q = __fma_rn(a, a, __fma_rn(b, b, __fma_rn(c, c, d * d)));
            g.add_carry(0x1p-48 * q * fabs(r), Rsys<KIND>::kStepScale);
            span = (unsigned)(RelaxGuard::kBigH - g.hi_h);
        }
        const double n0 = __fma_rn(r0, d, -(r1 * b));
        const double n1 = __fma_rn(a, r1, -(c * r0));
        s0 = n0 * r, s1 = n1 * r;
        if constexpr (Rsys<KIND>::kStepScale == 1.0) {
            x += s0, y += s1;
        } else {
            x = __fma_rn(s0, Rsys<KIND>::kStepScale, x);
            y = __fma_rn(s1, Rsys<KIND>::kStepScale, y);
        }
        ++it;
        if constexpr (kTrack) {
            d2 = d3;
            d3 = __fma_rn(s0, s0, s1 * s1) * (Rsys<KIND>::kStepScale * Rsys<KIND>::kStepScale);
        }
        dh = abs_hi(det);  // a NaN determinant shows up in mh
        mh = max(abs_hi(s0), abs_hi(s1));
    };
    bool in_loop = true;
    // The update AFTER the one from the seed is decided with a wider margin.  From the same iterate
    // the two arithmetics' updates differ by ~eps cond (|this update| + |previous update|): the part
    // that scales with the previous update is the rounding of the step before, re-solved now.  Where
    // updates shrink by halves or faster that is covered by the carry * m term; it is not when the
    // update from the seed dwarfs what follows - a LINEAR pair (K4) lands on its solution at once,
    // from a seed 1e9 away with an error of eps cond 1e9 ~ 1e-6 .. 1e-4, and its second update is that
    // error: pure rounding noise sitting around the threshold (found by tests/test_gpu_soak.py: one
    // run in 65536 with a different iteration count).  So the second update, peeled like the first,
    // is compared against a band widened by w1 = carry * |first update|, and so is its margin test.
    double extra = 0.0;   // absolute add-on of the decision in flight (w1 for the second update, else 0)
    int lo_cur = g.lo_h;  // "converged for certain" threshold of the decision in flight
    if (it == 0) {  // the update from the seed, peeled (see above)
        update(std::true_type {});
        d1 = dh;
        in_loop = (unsigned)(mh - g.hi_h) < span && it < limit;
        if (in_loop) {
            const double w1 = g.carry * fmax(fabs(s0), fabs(s1)) * Rsys<KIND>::kStepScale;
            RelaxGuard g2 = g;
            g2.set_band(__fma_rn(g.carry, kTol, g.band) + w1, Rsys<KIND>::kStepScale);
            update(std::false_type {});
            dmin = min(dmin, dh);  // first iterate after the seed: nothing to have grown from yet
            if ((unsigned)(mh - g2.hi_h) < (unsigned)(RelaxGuard::kBigH - g2.hi_h)) {
                in_loop = it < limit;  // longer than the threshold for certain, carried deviation included
            } else {
                in_loop = false;  // decided below, against the widened band and margin
                extra = fmax(w1, 0x1p-1000), lo_cur = g2.lo_h;
            }
        }
    }
#pragma unroll 1
    for (;;) {
        // hot loop: one update per trip, left when the update is no longer longer than the
        // threshold for certain (or is non-finite / huge), or at the limit
        if (in_loop) {
#pragma unroll 1
            do {
                update(std::false_type {});
                grow = max(grow, dh - dmin);  // (G2), in high-word units (2^20 per binade)
                dmin = min(dmin, dh);
            } while ((unsigned)(mh - g.hi_h) < span && it < limit);
        }
        in_loop = true;
        // ---- rare from here ----
        if (extra == 0.0 && (unsigned)(mh - g.hi_h) < span) break;  // limit reached, every update longer than the threshold
        if (mh >= RelaxGuard::kBigH || grow > kBounce) {  // (G4) / (G2)
            state = kRlxUncertain + (mh >= RelaxGuard::kBigH ? kWhyHuge : kWhyBounce);
            break;
        }
        if (min(dmin, d1) < g.det_h) {  // (G1): careful mode if the caller runs whole runs and the floor holds, else literal
            state = (!kTrack && kCarefulBinades > 0 && limit >= kRelaxCap && min(dmin, d1) >= g.det_h - (kCarefulBinades << 20))
                ? kRlxWantCareful : kRlxUncertain + kWhyCond;
            break;
        }
        if (mh < lo_cur) {
            state = kRlxConverged;
            break;
        }
        const int verdict = g.precise(fmax(fabs(s0), fabs(s1)) * Rsys<KIND>::kStepScale, det, extra);
        if (trace) *trace |= 1;
        if (verdict >= 0) {
            state = verdict > 0 ? kRlxConverged : kRlxUncertain + kWhyBand;
            break;
        }
        extra = 0.0, lo_cur = g.lo_h;
        if (it >= limit) break;  // not converged for certain, and out of updates
    }
    if (state == kRlxRunning && (min(dmin, d1) < g.det_h || grow > kBounce || limit >= kRelaxCap))
        state = kRlxUncertain + (min(dmin, d1) < g.det_h ? kWhyCond : grow > kBounce ? kWhyBounce : kWhyCap);
    if (dmin_io) *dmin_io = dmin;
    return state;
}

// ------------------------------------------------------------------------------------------
// The line form of a run.
//
// Every equation pair with a quadratic in it is a circle and a line (K2, K3, K5), or two circles
// whose difference is a line (K1: the radical line).  Newton's method is affine covariant: the
// update from the seed lands ON that line, and from there on the iteration is the scalar map of
// this file's header,
//        w  <-  w - (w^2 - h^2) / (2 w),
// w the coordinate along the line from the foot F of the circle's centre, +-h the two roots.  The
// literal arithmetic walks the same points with a 2x2 solve per update; the closed form above it
// (relaxed_updates) with Cramer's rule, 21 FP64 operations per update.  The scalar map needs 8, and
// its deviation from the literal arithmetic is of the kind the guards already budget for:
//   * the landing point of the first update is projected onto the line; what is dropped is the
//     component ACROSS the line, which is the landing's own rounding error (eps cond(J_seed) times
//     the first update): the literal arithmetic removes it with its second update, whose length
//     therefore differs from the scalar map's by at most that much - exactly the w1 term the second
//     update's band and margin are widened by (relaxed_updates);
//   * from the same point on the line the two arithmetics' updates differ by the rounding of F, of
//     the direction and of h^2 (a few ulp of the coordinate scale, amplified by the conditioning the
//     way a 2x2 solve amplifies its own rounding) - the O(cond eps S) of the header, under the
//     first-level band for cond <= 2^10 (G1) and scaled with the actual conditioning by the
//     second-level margin;
//   * |det J| at F + w u is |w| times a constant of the system (RLine::dscale), so (G1) and (G2)
//     watch the same quantity as before.
// The guards, their thresholds and the order of the decisions are those of relaxed_updates, line
// for line; careful mode and the literal re-run are unchanged (both restart from the seed).
// An argument backed by the same tests and soaks, not a proof - like the rest of this file.
// ------------------------------------------------------------------------------------------
template <int KIND>
struct RLine {
    static constexpr bool kHas = false;
};

struct RLineData {
    double fx, fy;   // foot of the circle's centre on the line
    double ux, uy;   // unit direction of the line
    double h2;       // squared half chord (negative: the line misses the circle, no real root)
    double dscale;   // |det| of the matrix the closed form solves, at F + w u, is |w| dscale
    double mscale;   // larger component of what that solve returns is |(w^2 - h^2) / w| mscale
    __device__ __forceinline__ double project(double x, double y) const { return __fma_rn(x - fx, ux, (y - fy) * uy); }
    __device__ __forceinline__ void point(double w, double& x, double& y) const { x = __fma_rn(w, ux, fx), y = __fma_rn(w, uy, fy); }
};

// How the constants are formed matters as much as the map.  The half chord h enters every late
// update as (w^2 - h^2) / w, so an absolute error dh in it moves those updates by ~2 dh: it has to
// stay within what the guards budget, eps S cond.  "h^2 = ra^2 - t0^2" does not: next to one of the
// centres (P close to B: rb << ra) it cancels to eps ra^2 / (2 h), orders of magnitude over the
// literal arithmetic's own error there (the first soak of this form: coordinates 1.1e-9 off on flat
// triangles).  So h^2 comes from factors that are each a sum of INPUTS (Heron's product for K1,
// (r - c)(r + c) for a circle of radius r at distance c from the line): relative error
// eps S / (smallest factor), and h / (smallest factor) <= 2 dr / |det| at the roots - the same
// amplification a 2x2 solve applies to its own rounding (checked for the needle P -> B and the
// flat P -> AB shapes in DESIGN.md).  The foot likewise from (ra - rb)(ra + rb), not qa - qb.

// K1: the radical line of the two circles, perpendicular to A -> B at t0 = (d^2 + ra^2 - rb^2) / (2 d) from A
template <>
struct RLine<GCS_KIND_PP> : RLineData {
    static constexpr bool kHas = true;
    __device__ __forceinline__ void set(const Rsys<GCS_KIND_PP>& rs, const double* k)
    {
        const double dx = rs.bx - rs.ax, dy = rs.by - rs.ay;
        const double d2 = __fma_rn(dx, dx, dy * dy);
        const double rd = rsqrt_relaxed(d2);  // concentric circles: inf -> NaN everywhere -> (G4)
        const double d = d2 * rd;
        const double px = dx * rd, py = dy * rd;
        const double ra = fabs(k[2]), rb = fabs(k[5]);
        const double sum = ra + rb, dif = ra - rb;
        const double hr = 0.5 * rd;
        const double t0 = __fma_rn(dif, sum, d2) * hr;
        fx = __fma_rn(t0, px, rs.ax), fy = __fma_rn(t0, py, rs.ay);
        ux = -py, uy = px;
        // 16 area^2 = (ra + rb - d)(ra + rb + d)(d + ra - rb)(d - ra + rb);  h = 2 area / d
        h2 = (((sum - d) * (sum + d)) * hr) * (((d + dif) * (d - dif)) * hr);
        dscale = d;                            // det(J/2) = (P - A) x (P - B) = w d
        mscale = fmax(fabs(ux), fabs(uy));     // the solve of J/2 returns twice the step
    }
};

// the unit circle and the line N . n = t0, N = (nx, ny) / |(nx, ny)| (K2, K5: the unknown is a unit normal)
struct RLineUnit : RLineData {
    __device__ __forceinline__ void set_unit(double nx, double ny, double c)  // line: nx x + ny y = c
    {
        const double l2 = __fma_rn(nx, nx, ny * ny);
        const double rl = rsqrt_relaxed(l2);
        set_unit(nx, ny, c, l2 * rl, rl);
    }
    __device__ __forceinline__ void set_unit(double nx, double ny, double c, double len, double rl)  // len = |(nx, ny)| = 1 / rl
    {
        const double Nx = nx * rl, Ny = ny * rl;
        const double t0 = c * rl;
        fx = t0 * Nx, fy = t0 * Ny;
        ux = -Ny, uy = Nx;
        h2 = (1.0 - t0) * (1.0 + t0);
        dscale = 2.0 * len;                    // det J = 2 |(nx, ny)| w
        mscale = 0.5 * fmax(fabs(ux), fabs(uy));
    }
};

// K2: dX x + dY y + c0 = 0 and the unit circle
template <>
struct RLine<GCS_KIND_SDD> : RLineUnit {
    static constexpr bool kHas = true;
    __device__ __forceinline__ void set(const Rsys<GCS_KIND_SDD>& rs, const double*) { set_unit(rs.dX, rs.dY, -rs.c0); }
};

// K5: fdy x - fdx y = cos(A) |fd| and the unit circle
template <>
struct RLine<GCS_KIND_ANG> : RLineUnit {
    static constexpr bool kHas = true;
    __device__ __forceinline__ void set(const Rsys<GCS_KIND_ANG>& rs, const double*) { set_unit(rs.fdy, -rs.fdx, rs.cl, rs.len, rs.rl); }
};

// K3: the circle (C, r) and the line at signed distance -s from A -> B
template <>
struct RLine<GCS_KIND_PPL> : RLineData {
    static constexpr bool kHas = true;
    __device__ __forceinline__ void set(const Rsys<GCS_KIND_PPL>& rs, const double* k)
    {
        ux = rs.l.ex * rs.l.rl, uy = rs.l.ey * rs.l.rl;
        // offset of the centre from the line along N = (uy, -ux):  N . (C - A) + s
        const double c = __fma_rn(rs.px - rs.l.xa, uy, __fma_rn(-(rs.py - rs.l.ya), ux, k[7]));
        fx = __fma_rn(-c, uy, rs.px), fy = __fma_rn(c, ux, rs.py);
        const double r = fabs(k[2]), ca = fabs(c);
        h2 = (r - ca) * (r + ca);
        dscale = 2.0 * rs.l.len;               // det J = 2 (P - C) . e = 2 |e| w
        mscale = 0.5 * fmax(fabs(ux), fabs(uy));
    }
};

// relaxed_updates for a whole run (it == 0 on entry) of a kind with a line form: the update from the
// seed in closed form, everything after it on the line.  Same outcomes, same guards.
template <int KIND>
__device__ __forceinline__ int relaxed_updates_line(const Rsys<KIND>& rs, const RLine<KIND>& ln, RelaxGuard& g, double& x, double& y,
    int& it, int limit, int* trace = nullptr)
{
    static_assert(RLine<KIND>::kHas, "no line form for this kind");
    int dmin = 0x7fffffff, grow = 0, d1 = 0x7fffffff;
    int state = kRlxRunning;
    if (it >= limit) return (limit >= kRelaxCap) ? kRlxUncertain + kWhyCap : kRlxRunning;
    int mh, dh;
    double sm, det;  // larger component of the update in flight, in the units of the closed-form solve; det at its iterate
    {  // the update from the seed (relaxed_updates, update(true_type))
        double a, b, c, d, r0, r1;
        rs.eval(x, y, a, b, c, d, r0, r1);
        det = __fma_rn(a, d, -(b * c));
        const double r = rcp_relaxed(det);
        const double q = __fma_rn(a, a, __fma_rn(b, b, __fma_rn(c, c, d * d)));
        g.add_carry(0x1p-48 * q * fabs(r), Rsys<KIND>::kStepScale);
        const double s0 = __fma_rn(r0, d, -(r1 * b)) * r, s1 = __fma_rn(a, r1, -(c * r0)) * r;
        if constexpr (Rsys<KIND>::kStepScale == 1.0) {
            x += s0, y += s1;
        } else {
            x = __fma_rn(s0, Rsys<KIND>::kStepScale, x);
            y = __fma_rn(s1, Rsys<KIND>::kStepScale, y);
        }
        ++it;
        sm = fmax(fabs(s0), fabs(s1));
        dh = abs_hi(det);
        mh = max(abs_hi(s0), abs_hi(s1));
    }
    const unsigned span = (unsigned)(RelaxGuard::kBigH - g.hi_h);
    d1 = dh;
    bool in_loop = (unsigned)(mh - g.hi_h) < span && it < limit;
    double w = ln.project(x, y);
    // one update on the line; leaves mh, dh, sm, det like the closed-form update does
    auto update = [&]() {
        const double f = __fma_rn(w, w, -ln.h2);
        det = w * ln.dscale;
        const double t = f * rcp_relaxed(w);
        w = __fma_rn(-0.5, t, w);
        ++it;
        sm = t * ln.mscale;
        dh = abs_hi(det);
        mh = abs_hi(sm);
    };
    double extra = 0.0;   // absolute add-on of the decision in flight (w1 for the second update, else 0)
    int lo_cur = g.lo_h;  // "converged for certain" threshold of the decision in flight
    if (in_loop) {  // the second update, against a band widened by w1 (see relaxed_updates)
        const double w1 = g.carry * sm * Rsys<KIND>::kStepScale;
        RelaxGuard g2 = g;
        g2.set_band(__fma_rn(g.carry, kTol, g.band) + w1, Rsys<KIND>::kStepScale);
        update();
        dmin = min(dmin, dh);  // first iterate after the seed: nothing to have grown from yet
        if ((unsigned)(mh - g2.hi_h) < (unsigned)(RelaxGuard::kBigH - g2.hi_h)) {
            in_loop = it < limit;
        } else {
            in_loop = false;
            extra = fmax(w1, 0x1p-1000), lo_cur = g2.lo_h;
        }
    }
#pragma unroll 1
    for (;;) {
        if (in_loop) {
#pragma unroll 1
            do {
                update();
                grow = max(grow, dh - dmin);  // (G2), in high-word units (2^20 per binade)
                dmin = min(dmin, dh);
            } while ((unsigned)(mh - g.hi_h) < span && it < limit);
        }
        in_loop = true;
        // ---- rare from here: relaxed_updates' decisions, in its order ----
        if (extra == 0.0 && (unsigned)(mh - g.hi_h) < span) break;
        if (mh >= RelaxGuard::kBigH || grow > kBounce) {
            state = kRlxUncertain + (mh >= RelaxGuard::kBigH ? kWhyHuge : kWhyBounce);
            break;
        }
        if (min(dmin, d1) < g.det_h) {
            state = (kCarefulBinades > 0 && limit >= kRelaxCap && min(dmin, d1) >= g.det_h - (kCarefulBinades << 20))
                ? kRlxWantCareful : kRlxUncertain + kWhyCond;
            break;
        }
        if (mh < lo_cur) {
            state = kRlxConverged;
            break;
        }
        const int verdict = g.precise(fabs(sm) * Rsys<KIND>::kStepScale, det, extra);
        if (trace) *trace |= 1;
        if (verdict >= 0) {
            state = verdict > 0 ? kRlxConverged : kRlxUncertain + kWhyBand;
            break;
        }
        extra = 0.0, lo_cur = g.lo_h;
        if (it >= limit) break;
    }
    if (state == kRlxRunning && (min(dmin, d1) < g.det_h || grow > kBounce || limit >= kRelaxCap))
        state = kRlxUncertain + (min(dmin, d1) < g.det_h ? kWhyCond : grow > kBounce ? kWhyBounce : kWhyCap);
    ln.point(w, x, y);
    return state;
}

// whole runs: the line form where the kind has one (GCS_RELAX_LINE=0 builds without it)
#ifndef GCS_RELAX_LINE
#define GCS_RELAX_LINE 1
#endif
// What a sub-system's runs share: the equations on fused multiply-adds, the guard before any run's own
// carry term, the constants of the line form.  One per (sub-system, seed) lane in the static mapping,
// one per sub-system - set once, used by every seed - in the sequential one.
template <int KIND>
struct RelaxedSystem {
    static constexpr bool kLine = RLine<KIND>::kHas && GCS_RELAX_LINE;
    Rsys<KIND> rs;
    RelaxGuard g0;
    RLine<KIND> ln;
    __device__ __forceinline__ void load(const double* k)
    {
        rs.load(k, g0);
        if constexpr (kLine) ln.set(rs, k);
    }
    // one run from (x, y) with it == 0; g: the run's own guard (a copy of g0 on entry)
    __device__ __forceinline__ int run(RelaxGuard& g, double& x, double& y, int& it, int* trace) const
    {
        if constexpr (kLine) {
            return relaxed_updates_line<KIND>(rs, ln, g, x, y, it, kRelaxCap, trace);
        } else {
            double u0, u1;
            return relaxed_updates<KIND, false>(rs, g, x, y, it, kRelaxCap, u0, u1, nullptr, trace);
        }
    }
};

// Careful mode: a whole run from its seed with EVERY convergence decision taken by the
// conditioning-scaled margin test (RelaxGuard::precise) instead of the fixed first-level band.
//
// A run whose |det J| falls under the (G1) line 2^-10 dr - flat triangles, lines that nearly touch
// their circle - used to be redone literally: one long chain of dependent FP64 operations that
// outlived its launch (DESIGN.md: the re-run tail).  Its decisions are still certifiable: the
// second-level margin of (G3), 2^-44 S dr/|det J| + 2^-40 tol (+ the carry term), scales with the
// actual conditioning at every update; what does not is the first-level band of the hot loop, which
// is only wide enough for dr/|det| <= 2^10.  So relaxed_updates hands such a run back
// (kRlxWantCareful) and the caller replays it here: the closed-form arithmetic is deterministic, the
// replay visits the same iterates, and now no decision rests on the fixed band.  The floor
// |det| >= 2^-14 dr stays (the coordinates of the two arithmetics differ by ~8 (dr/|det|) 2^-52 S:
// 2^-35 S there, a factor 30 inside the 1e-9 tolerance); below it, and for everything else the
// guards do not vouch for, the literal code.  Out of line and by value: one run in a few thousand
// comes here, and the hot loop of relaxed_updates keeps its registers.
struct CarefulOut {
    double x, y;
    int it, state, trace;
};

template <int KIND>
static __device__ __noinline__ CarefulOut relaxed_careful(Rsys<KIND> rs, RelaxGuard g, double x, double y)
{
    CarefulOut o;
    o.trace = 2;
    int it = 0, state = kRlxRunning;
    int dmin = 0x7fffffff, grow = 0, d1 = 0x7fffffff;
    double mprev = 0.0;  // length of the previous update: its rounding is what this update re-solves (see relaxed_updates)
#pragma unroll 1
    while (it < kRelaxCap) {
        double a, b, c, d, r0, r1;
        rs.eval(x, y, a, b, c, d, r0, r1);
        const double det = __fma_rn(a, d, -(b * c));
        const double r = rcp_relaxed(det);
        if (it == 0) {
            const double q = __fma_rn(a, a, __fma_rn(b, b, __fma_rn(c, c, d * d)));
            g.add_carry(0x1p-48 * q * fabs(r), Rsys<KIND>::kStepScale);
        }
        const double n0 = __fma_rn(r0, d, -(r1 * b));
        const double n1 = __fma_rn(a, r1, -(c * r0));
        const double s0 = n0 * r, s1 = n1 * r;
        if constexpr (Rsys<KIND>::kStepScale == 1.0) {
            x += s0, y += s1;
        } else {
            x = __fma_rn(s0, Rsys<KIND>::kStepScale, x);
            y = __fma_rn(s1, Rsys<KIND>::kStepScale, y);
        }
        const int dh = abs_hi(det), mh = max(abs_hi(s0), abs_hi(s1));
        if (it == 0) {
            d1 = dh;  // the determinant at the seed counts for the floor only (see relaxed_updates)
        } else {
            grow = max(grow, dh - dmin);
            dmin = min(dmin, dh);
        }
        ++it;
        if (mh >= RelaxGuard::kBigH || grow > kBounce) {  // (G4) / (G2)
            state = kRlxUncertain + (mh >= RelaxGuard::kBigH ? kWhyHuge : kWhyBounce);
            break;
        }
        if (min(dmin, d1) < g.det_h - (kCarefulBinades << 20)) {  // under the careful floor (or a degenerate scale)
            state = kRlxUncertain + kWhyCond;
            break;
        }
        const double m = fmax(fabs(s0), fabs(s1)) * Rsys<KIND>::kStepScale;
        const int verdict = g.precise(m, det, g.carry * mprev);
        mprev = m;
        if (verdict >= 0) {
            state = verdict > 0 ? kRlxConverged : kRlxUncertain + kWhyBand;
            break;
        }
    }
    if (state == kRlxRunning) state = kRlxUncertain + kWhyCap;
    o.x = x, o.y = y, o.it = it, o.state = state;
    return o;
}

// seed `seed` of sub-system `gi` as the kernels take it (kUniformSeed: `seed` is the same in every
// lane of the warp and not a compile-time constant - the sequential kernel's loop over seeds)
template <int KIND, bool kUniformSeed = false>
__device__ __forceinline__ void run_seed(
    const double* guesses, long long stride, long long gi, const double* k, int seed, double& x, double& y)
{
    if (guesses) {
        x = __ldg(guesses + ((long long)seed * 2 + 0) * stride + gi);
        y = __ldg(guesses + ((long long)seed * 2 + 1) * stride + gi);
    } else if constexpr (Sys<KIND>::kGuessFromCols) {
        column_seed<KIND>(k, seed, x, y);
    } else if constexpr (kUniformSeed) {
        default_seed_uniform(seed, x, y);
    } else {
        default_seed(seed, x, y);
    }
}

// The literal run of one seed (what an uncertain closed-form run is replaced by).  Inlined: the
// columns are in registers at every call site, and the kernels' register budgets are those of the
// literal kernels anyway.
template <int KIND>
__device__ __forceinline__ void literal_rerun(const double* guesses, long long stride, long long gi, const double* k,
    int seed, double runtime_zero, double& x, double& y, int& it, int& conv, int why = 0)
{
    Sys<KIND> sys;
    sys.load(k);
    FastConsts fc;
    fc.init(runtime_zero);
    run_seed<KIND>(guesses, stride, gi, k, seed, x, y);
    newton_run<KIND>(sys, fc, x, y, it, conv);
    atomicAdd(&g_relax_reruns[why], 1ull);
}

// (G5) is the root selection safe against a perturbation of the candidates by 2^-36 of the
// coordinate scale?  Mirrors the tests of select_and_finish with a margin of 2^-24 relative.
template <int KIND, int NS>
__device__ __forceinline__ bool selection_is_robust(const double* k, uint8_t code, const double* cx, const double* cy)
{
    constexpr double kMargin = 0x1p-24;
    bool ok = true;
    if constexpr (KIND == GCS_KIND_PP || KIND == GCS_KIND_PPL || KIND == GCS_KIND_PLL) {
        bool nearest = false;
        double ax = 0, ay = 0, bx = 0, by = 0;
        if constexpr (KIND != GCS_KIND_PP) {
            nearest = (code & GCS_CODE_COLLINEAR) != 0;
            if constexpr (KIND == GCS_KIND_PLL) nearest = nearest || (code & GCS_CODE_CANVAS_PARALLEL);
        }
        if (!nearest) nearest = !orientation_frame<KIND>(k, ax, ay, bx, by);
        if (nearest) {
            constexpr int cf = (KIND == GCS_KIND_PPL) ? 8 : 10;
            const double fx = (KIND == GCS_KIND_PP) ? 0.0 : k[cf];
            const double fy = (KIND == GCS_KIND_PP) ? 0.0 : k[cf + 1];
            double dd[NS], sc = fabs(fx) + fabs(fy);
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const double dx = cx[s] - fx, dy = cy[s] - fy;
                dd[s] = dx * dx + dy * dy;
                sc = fmax(sc, fabs(cx[s]) + fabs(cy[s]));
            }
            const double floor_ = 0x1p-44 * sc * sc;
#pragma unroll
            for (int s = 0; s < NS; ++s)
#pragma unroll
                for (int t = s + 1; t < NS; ++t)
                    ok = ok && (fabs(dd[s] - dd[t]) > 0x1p-22 * (dd[s] + dd[t]) + floor_);
        } else {
            const double ab = fabs(bx - ax) + fabs(by - ay);
            const double sa = fabs(ax) + fabs(ay) + fabs(bx) + fabs(by);
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const double ori = triangle_orientation(ax, ay, bx, by, cx[s], cy[s]);
                ok = ok && (fabs(ori) > kMargin * ab * (sa + fabs(cx[s]) + fabs(cy[s])));
            }
        }
    } else if constexpr (KIND == GCS_KIND_SDD) {
        const double dot0 = cx[0] * k[0] + cy[0] * k[1];
        const double p0 = dot0 - k[4];
        const double d1 = dot0 - p0;
        const double d2 = (cx[0] * k[2] + cy[0] * k[3]) - p0;
        const double sc = kMargin * (fabs(k[0]) + fabs(k[1]) + fabs(k[2]) + fabs(k[3]) + fabs(k[4]));
        ok = (fabs(d1) > sc) && (fabs(d2) > sc);
    } else {
        const double cross0 = (k[5] * cx[0]) + (k[6] * cy[0]);
        ok = fabs(cross0) > kMargin * (fabs(k[5]) + fabs(k[6]));
    }
    return ok;
}

}  // namespace gcsk
