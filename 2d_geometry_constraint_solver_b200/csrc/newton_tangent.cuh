// newton_tangent.cuh — forward-mode derivatives of one solved sub-system (sketch-program tangents,
// include/gcs_b200.h).
//
// A converged row satisfies F(u, k) = 0 at its chosen root u, with k its input columns.  By the
// implicit function theorem its tangent along input tangents k' is u' = -J^-1 (dF/dk k'), J = dF/du
// at u as Sys<KIND>::eval computes it.  The output columns are then the forward-mode tangent of what
// select_and_finish writes: u itself for the point kinds, the reconstructed endpoints for K2 / K5,
// where u is the normal of the chosen seed.
//
// Operation order (the test suite's CPU restatement follows it; built with --fmad=false there and
// -ffp-contract=off on the CPU, both round alike, one rounding per operation):
//   residual tangent, u held fixed (a b; c d = J):
//     K1   rf = -((a*kd0 + b*kd1) + (2.0*k2)*kd2),  rg = -((c*kd3 + d*kd4) + (2.0*k5)*kd5)
//     K2   rf = (((-kd5) + (kd2 - kd0)*x) + (kd3 - kd1)*y) + kd4,  rg = 0
//     K3   rf as K1 over (k0, k1, k2),  rg = p2l(k3..k7)
//     K4   rf = p2l(k0..k4),  rg = p2l(k5..k9)
//     K5   len = sqrt(k0*k0 + k1*k1), dlen = (k0*kd0 + k1*kd1)/len,
//          rf = ((-(kd2*len + k2*dlen)) + kd0*(-y)) + kd1*x,  rg = 0
//     p2l over a line (xa, ya)-(xb, yb) and signed distance s (P2L::eval):
//          ex = xb - xa, ey = yb - ya, len = sqrt(ex*ex + ey*ey), ux = x - xa, uy = y - ya,
//          dex = dxb - dxa, dey = dyb - dya, dlen = (ex*dex + ey*dey)/len, dld = dlen*s + len*ds,
//          r = ((-dld) + (uy*dex - dya*ex)) - (ux*dey - dxa*ey)
//   solve:  det = a*d - b*c,  dx = (b*rg - d*rf)/det,  dy = (c*rf - a*rg)/det
//   K2 / K5 outputs: p = (nx*c1x + ny*c1y) - q with (c1, c2, q, canvas_len) = (k0 k1, k2 k3, k4, k8)
//   for K2 and (k7 k8, k10 k11, k9, k12) for K5, dp = ((dnx*c1x + nx*dc1x) + (dny*c1y + ny*dc1y)) - dq,
//   then reconstruct_tangent below.
// Non-smooth points follow the primal's branch: `fabs(arg)` takes the sign of arg (0 as +), and
// max(canvas_len, span) the side the primal chose (the canvas length has tangent 0).
#pragma once

#include "newton_core.cuh"

namespace gcsk {

__device__ __forceinline__ double p2l_tangent(const double* k, const double* kd, double x, double y)
{
    const double ex = k[2] - k[0], ey = k[3] - k[1];
    const double len = sqrt(ex * ex + ey * ey);
    const double ux = x - k[0], uy = y - k[1];
    const double dex = kd[2] - kd[0], dey = kd[3] - kd[1];
    const double dlen = (ex * dex + ey * dey) / len;
    const double dld = dlen * k[4] + len * kd[4];
    return ((-dld) + (uy * dex - kd[1] * ex)) - (ux * dey - kd[0] * ey);
}

// tangent of reconstruct_line_endpoints (newton_core.cuh) at the same primal point
__device__ __forceinline__ void reconstruct_tangent(double c1x, double c1y, double c2x, double c2y, double nx, double ny,
    double p, double canvas_len, double dc1x, double dc1y, double dc2x, double dc2y, double dnx, double dny, double dp,
    double dout[4])
{
    const double sd1 = (nx * c1x + ny * c1y) - p;
    const double dsd1 = ((dnx * c1x + nx * dc1x) + (dny * c1y + ny * dc1y)) - dp;
    const double a1x = c1x - sd1 * nx, a1y = c1y - sd1 * ny;
    const double da1x = dc1x - (dsd1 * nx + sd1 * dnx), da1y = dc1y - (dsd1 * ny + sd1 * dny);
    const double sd2 = (nx * c2x + ny * c2y) - p;
    const double dsd2 = ((dnx * c2x + nx * dc2x) + (dny * c2y + ny * dc2y)) - dp;
    const double a2x = c2x - sd2 * nx, a2y = c2y - sd2 * ny;
    const double da2x = dc2x - (dsd2 * nx + sd2 * dnx), da2y = dc2y - (dsd2 * ny + sd2 * dny);
    const double dirx = -ny, diry = nx, ddirx = -dny, ddiry = dnx;
    const double dmidx = (da1x + da2x) / 2.0, dmidy = (da1y + da2y) / 2.0;
    const double ex = a2x - a1x, ey = a2y - a1y, dex = da2x - da1x, dey = da2y - da1y;
    const double arg = dirx * ex + diry * ey;
    const double darg = (ddirx * ex + dirx * dex) + (ddiry * ey + diry * dey);
    const double span = fabs(arg);
    const double dspan = (arg >= 0.0) ? darg : -darg;
    const bool wide = canvas_len < span;
    const double half = (wide ? span : canvas_len) / 2.0;
    const double dhalf = (wide ? dspan : 0.0) / 2.0;
    const double hx = dhalf * dirx + half * ddirx, hy = dhalf * diry + half * ddiry;
    dout[0] = dmidx - hx;
    dout[1] = dmidy - hy;
    dout[2] = dmidx + hx;
    dout[3] = dmidy + hy;
}

// The linearisation of one converged row: init() takes the input columns k and the unknown u at the
// chosen root and evaluates the Jacobian once; apply() maps one set of input tangents to output
// tangents (any number of times per init).
template <int KIND>
struct RowTangent {
    static constexpr int kIn = Sys<KIND>::kCols;
    static constexpr int kOut = Sys<KIND>::kOut;
    double k[kIn];
    double x, y, a, b, c, d, det;

    __device__ __forceinline__ void init(const double* cols, double ux, double uy)
    {
#pragma unroll
        for (int q = 0; q < kIn; ++q) k[q] = cols[q];
        x = ux, y = uy;
        Sys<KIND> sys;
        sys.load(k);
        double f, g;
        sys.eval(x, y, f, g, a, b, c, d);
        det = a * d - b * c;
    }

    __device__ __forceinline__ void apply(const double* kd, double dout[4]) const
    {
        double rf, rg = 0.0;
        if constexpr (KIND == GCS_KIND_PP) {
            rf = -((a * kd[0] + b * kd[1]) + (2.0 * k[2]) * kd[2]);
            rg = -((c * kd[3] + d * kd[4]) + (2.0 * k[5]) * kd[5]);
        } else if constexpr (KIND == GCS_KIND_SDD) {
            rf = (((-kd[5]) + (kd[2] - kd[0]) * x) + (kd[3] - kd[1]) * y) + kd[4];
        } else if constexpr (KIND == GCS_KIND_PPL) {
            rf = -((a * kd[0] + b * kd[1]) + (2.0 * k[2]) * kd[2]);
            rg = p2l_tangent(k + 3, kd + 3, x, y);
        } else if constexpr (KIND == GCS_KIND_PLL) {
            rf = p2l_tangent(k, kd, x, y);
            rg = p2l_tangent(k + 5, kd + 5, x, y);
        } else {
            const double len = sqrt(k[0] * k[0] + k[1] * k[1]);
            const double dlen = (k[0] * kd[0] + k[1] * kd[1]) / len;
            rf = ((-(kd[2] * len + k[2] * dlen)) + kd[0] * (-y)) + kd[1] * x;
        }
        const double dx = (b * rg - d * rf) / det;
        const double dy = (c * rf - a * rg) / det;
        if constexpr (KIND == GCS_KIND_SDD || KIND == GCS_KIND_ANG) {
            // columns of c1, q, c2 and the canvas length (see the header comment)
            constexpr int o = (KIND == GCS_KIND_SDD) ? 0 : 7;
            constexpr int oq = (KIND == GCS_KIND_SDD) ? 4 : 9;
            constexpr int o2 = (KIND == GCS_KIND_SDD) ? 2 : 10;
            constexpr int ol = (KIND == GCS_KIND_SDD) ? 8 : 12;
            const double p = (x * k[o] + y * k[o + 1]) - k[oq];
            const double dp = ((dx * k[o] + x * kd[o]) + (dy * k[o + 1] + y * kd[o + 1])) - kd[oq];
            reconstruct_tangent(k[o], k[o + 1], k[o2], k[o2 + 1], x, y, p, k[ol], kd[o], kd[o + 1], kd[o2], kd[o2 + 1], dx,
                dy, dp, dout);
        } else {
            dout[0] = dx, dout[1] = dy;
        }
    }
};

}  // namespace gcsk
