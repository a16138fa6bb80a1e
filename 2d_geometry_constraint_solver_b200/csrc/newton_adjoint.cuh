// newton_adjoint.cuh — reverse-mode derivatives of one solved sub-system (sketch-program adjoints,
// include/gcs_b200.h): the transpose of RowTangent<KIND>::apply (newton_tangent.cuh).
//
// RowTangent<KIND>::apply maps input-column tangents kd to output tangents dout, linearly.  Its
// transpose maps output adjoints ob (one weight per output column) to input-column adjoints kb with
// <ob, apply(kd)> = <kb, kd> for every kd.  Every forward statement y = f(x) becomes x_bar += df/dx *
// y_bar, the statements taken in reverse order.  The primal quantities (k, x, y, the Jacobian a b c d,
// det, and the reconstruction's sd1, sd2, dir, e, arg, span, half) are the forward ones, so
// non-smooth points take the primal's branch as forward mode does.
//
// Operation order (the test suite's CPU restatement follows it, one rounding per operation; "+="
// means one add into the running adjoint, in the order written):
//   K2 / K5 outputs (reconstruct_adjoint below; ob = o0 o1 o2 o3):
//     mx = o0 + o2, hx = o2 - o0, my = o1 + o3, hy = o3 - o1,
//     dhalf = hx*dirx + hy*diry, ddirx = half*hx, ddiry = half*hy,
//     dspan = wide ? dhalf/2.0 : 0, darg = arg >= 0 ? dspan : -dspan,
//     ddirx += ex*darg, dex = dirx*darg, ddiry += ey*darg, dey = diry*darg,
//     da2x = dex + mx/2.0, da1x = mx/2.0 - dex, da2y = dey + my/2.0, da1y = my/2.0 - dey,
//     dny = -ddirx, dnx = ddiry,
//     then per anchor i = 2, 1: dci_y = da_iy, dsd = -(ny*da_iy), dny += -(sd_i*da_iy),
//       dci_x = da_ix, dsd += -(nx*da_ix), dnx += -(sd_i*da_ix),
//       dnx += ci_x*dsd, dci_x += nx*dsd, dny += ci_y*dsd, dci_y += ny*dsd, dp += -dsd
//       (dp starts at 0 before anchor 2),
//     then p's tangent: dx = dnx + k[o]*dp, kb[o] = dc1x + x*dp, dy = dny + k[o+1]*dp,
//       kb[o+1] = dc1y + y*dp, kb[oq] = -dp; kb[o2] = dc2x, kb[o2+1] = dc2y.
//   Point kinds: dx, dy = ob0, ob1.
//   solve:  ub = dx/det, wb = dy/det, rf = (c*wb) - (d*ub), rg = (b*ub) - (a*wb)
//   residual tangents, in the same kinds as newton_tangent.cuh (s = -rf):
//     K1   kb0 = a*s, kb1 = b*s, kb2 = (2.0*k2)*s, and (c, d, k5; kb3..kb5) with -rg
//     K2   kb5 = -rf, kb2 += x*rf, kb0 += -(x*rf), kb3 += y*rf, kb1 += -(y*rf), kb4 += rf
//     K3   kb0..kb2 as K1, kb3..kb7 = p2l over rg
//     K4   kb0..kb4 = p2l over rf, kb5..kb9 = p2l over rg
//     K5   kb1 = x*rf, kb0 = (-y)*rf, s = -rf, kb2 = len*s, q = (k2*s)/len, kb0 += k0*q, kb1 += k1*q
//     p2l (r = the residual's adjoint): dex = uy*r, kb1 = -(ex*r), dey = -(ux*r), kb0 = ey*r,
//          dld = -r, kb4 = len*dld, q = (k4*dld)/len, dex += ex*q, dey += ey*q,
//          kb2 = dex, kb0 += -dex, kb3 = dey, kb1 += -dey
//   ("=" starts an entry, "+=" adds to one; entries never started are 0.)
#pragma once

#include "newton_tangent.cuh"

namespace gcsk {

// adjoint of p2l_tangent: r is the residual's adjoint, kb[0..4] are started (not added to)
__device__ __forceinline__ void p2l_adjoint(const double* k, double x, double y, double r, double* kb)
{
    const double ex = k[2] - k[0], ey = k[3] - k[1];
    const double len = sqrt(ex * ex + ey * ey);
    const double ux = x - k[0], uy = y - k[1];
    double dex = uy * r;
    kb[1] = -(ex * r);
    double dey = -(ux * r);
    kb[0] = ey * r;
    const double dld = -r;
    kb[4] = len * dld;
    const double q = (k[4] * dld) / len;
    dex = dex + ex * q;
    dey = dey + ey * q;
    kb[2] = dex;
    kb[0] = kb[0] + (-dex);
    kb[3] = dey;
    kb[1] = kb[1] + (-dey);
}

// adjoint of reconstruct_tangent at the same primal point: output adjoints o[4] to the adjoints of
// (dc1x, dc1y, dc2x, dc2y, dnx, dny, dp)
__device__ __forceinline__ void reconstruct_adjoint(double c1x, double c1y, double c2x, double c2y, double nx, double ny,
    double p, double canvas_len, const double o[4], double& dc1x, double& dc1y, double& dc2x, double& dc2y, double& dnx,
    double& dny, double& dp)
{
    const double sd1 = (nx * c1x + ny * c1y) - p;
    const double a1x = c1x - sd1 * nx, a1y = c1y - sd1 * ny;
    const double sd2 = (nx * c2x + ny * c2y) - p;
    const double a2x = c2x - sd2 * nx, a2y = c2y - sd2 * ny;
    const double dirx = -ny, diry = nx;
    const double ex = a2x - a1x, ey = a2y - a1y;
    const double arg = dirx * ex + diry * ey;
    const double span = fabs(arg);
    const bool wide = canvas_len < span;
    const double half = (wide ? span : canvas_len) / 2.0;
    const double mx = o[0] + o[2], hx = o[2] - o[0], my = o[1] + o[3], hy = o[3] - o[1];
    const double dhalf = hx * dirx + hy * diry;
    double ddirx = half * hx, ddiry = half * hy;
    const double dspan = wide ? dhalf / 2.0 : 0.0;
    const double darg = (arg >= 0.0) ? dspan : -dspan;
    ddirx = ddirx + ex * darg;
    const double dex = dirx * darg;
    ddiry = ddiry + ey * darg;
    const double dey = diry * darg;
    const double da2x = dex + mx / 2.0, da1x = mx / 2.0 - dex;
    const double da2y = dey + my / 2.0, da1y = my / 2.0 - dey;
    dny = -ddirx;
    dnx = ddiry;
    dp = 0.0;
    // anchor 2, then anchor 1
    double dsd = -(ny * da2y);
    dc2y = da2y;
    dny = dny + (-(sd2 * da2y));
    dc2x = da2x;
    dsd = dsd + (-(nx * da2x));
    dnx = dnx + (-(sd2 * da2x));
    dnx = dnx + c2x * dsd;
    dc2x = dc2x + nx * dsd;
    dny = dny + c2y * dsd;
    dc2y = dc2y + ny * dsd;
    dp = dp + (-dsd);
    dsd = -(ny * da1y);
    dc1y = da1y;
    dny = dny + (-(sd1 * da1y));
    dc1x = da1x;
    dsd = dsd + (-(nx * da1x));
    dnx = dnx + (-(sd1 * da1x));
    dnx = dnx + c1x * dsd;
    dc1x = dc1x + nx * dsd;
    dny = dny + c1y * dsd;
    dc1y = dc1y + ny * dsd;
    dp = dp + (-dsd);
}

// kb[0 .. kIn) = the transpose of lin.apply applied to the output adjoints ob[0 .. kOut)
template <int KIND>
__device__ __forceinline__ void row_adjoint(const RowTangent<KIND>& lin, const double ob[4], double* kb)
{
    constexpr int kIn = RowTangent<KIND>::kIn;
    const double* const k = lin.k;
    const double x = lin.x, y = lin.y, a = lin.a, b = lin.b, c = lin.c, d = lin.d;
#pragma unroll
    for (int q = 0; q < kIn; ++q) kb[q] = 0.0;
    double dx, dy;
    if constexpr (KIND == GCS_KIND_SDD || KIND == GCS_KIND_ANG) {
        constexpr int o = (KIND == GCS_KIND_SDD) ? 0 : 7;
        constexpr int oq = (KIND == GCS_KIND_SDD) ? 4 : 9;
        constexpr int o2 = (KIND == GCS_KIND_SDD) ? 2 : 10;
        constexpr int ol = (KIND == GCS_KIND_SDD) ? 8 : 12;
        const double p = (x * k[o] + y * k[o + 1]) - k[oq];
        double dc1x, dc1y, dc2x, dc2y, dnx, dny, dp;
        reconstruct_adjoint(k[o], k[o + 1], k[o2], k[o2 + 1], x, y, p, k[ol], ob, dc1x, dc1y, dc2x, dc2y, dnx, dny, dp);
        dx = dnx + k[o] * dp;
        kb[o] = dc1x + x * dp;
        dy = dny + k[o + 1] * dp;
        kb[o + 1] = dc1y + y * dp;
        kb[oq] = -dp;
        kb[o2] = dc2x, kb[o2 + 1] = dc2y;
    } else {
        dx = ob[0], dy = ob[1];
    }
    const double ub = dx / lin.det, wb = dy / lin.det;
    const double rf = (c * wb) - (d * ub);
    const double rg = (b * ub) - (a * wb);
    if constexpr (KIND == GCS_KIND_PP || KIND == GCS_KIND_PPL) {
        const double s = -rf;
        kb[0] = a * s, kb[1] = b * s, kb[2] = (2.0 * k[2]) * s;
    }
    if constexpr (KIND == GCS_KIND_PP) {
        const double s = -rg;
        kb[3] = c * s, kb[4] = d * s, kb[5] = (2.0 * k[5]) * s;
    } else if constexpr (KIND == GCS_KIND_SDD) {
        kb[5] = -rf;
        kb[2] = kb[2] + x * rf;
        kb[0] = kb[0] + (-(x * rf));
        kb[3] = kb[3] + y * rf;
        kb[1] = kb[1] + (-(y * rf));
        kb[4] = kb[4] + rf;
    } else if constexpr (KIND == GCS_KIND_PPL) {
        p2l_adjoint(k + 3, x, y, rg, kb + 3);
    } else if constexpr (KIND == GCS_KIND_PLL) {
        p2l_adjoint(k, x, y, rf, kb);
        p2l_adjoint(k + 5, x, y, rg, kb + 5);
    } else if constexpr (KIND == GCS_KIND_ANG) {
        const double len = sqrt(k[0] * k[0] + k[1] * k[1]);
        kb[1] = x * rf;
        kb[0] = (-y) * rf;
        const double s = -rf;
        kb[2] = len * s;
        const double q = (k[2] * s) / len;
        kb[0] = kb[0] + k[0] * q;
        kb[1] = kb[1] + k[1] * q;
    }
}

}  // namespace gcsk
