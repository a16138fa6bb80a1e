"""CPU restatement of a solved sub-system's forward-mode tangent (csrc/newton_tangent.cuh), in the
operation order written there.  numpy's float64 element-wise operations round once each and never
fuse a multiply with an add, so with the device built with --fmad=false the two agree bit for bit.
Test infrastructure only."""
import numpy as np


def _p2l(k, kd, x, y):
    """tangent of P2L::eval at fixed (x, y); k: xa ya xb yb s as [n][1] columns, kd as [n][T]"""
    ex, ey = k[2] - k[0], k[3] - k[1]
    length = np.sqrt(ex * ex + ey * ey)
    ux, uy = x - k[0], y - k[1]
    dex, dey = kd[2] - kd[0], kd[3] - kd[1]
    dlen = (ex * dex + ey * dey) / length
    dld = dlen * k[4] + length * kd[4]
    return ((-dld) + (uy * dex - kd[1] * ex)) - (ux * dey - kd[0] * ey)


def _reconstruct(c1x, c1y, c2x, c2y, nx, ny, p, canvas_len, dc1x, dc1y, dc2x, dc2y, dnx, dny, dp):
    sd1 = (nx * c1x + ny * c1y) - p
    dsd1 = ((dnx * c1x + nx * dc1x) + (dny * c1y + ny * dc1y)) - dp
    a1x, a1y = c1x - sd1 * nx, c1y - sd1 * ny
    da1x, da1y = dc1x - (dsd1 * nx + sd1 * dnx), dc1y - (dsd1 * ny + sd1 * dny)
    sd2 = (nx * c2x + ny * c2y) - p
    dsd2 = ((dnx * c2x + nx * dc2x) + (dny * c2y + ny * dc2y)) - dp
    a2x, a2y = c2x - sd2 * nx, c2y - sd2 * ny
    da2x, da2y = dc2x - (dsd2 * nx + sd2 * dnx), dc2y - (dsd2 * ny + sd2 * dny)
    dirx, diry, ddirx, ddiry = -ny, nx, -dny, dnx
    dmidx, dmidy = (da1x + da2x) / 2.0, (da1y + da2y) / 2.0
    ex, ey, dex, dey = a2x - a1x, a2y - a1y, da2x - da1x, da2y - da1y
    arg = dirx * ex + diry * ey
    darg = (ddirx * ex + dirx * dex) + (ddiry * ey + diry * dey)
    span = np.abs(arg)
    dspan = np.where(arg >= 0.0, darg, -darg)       # the sign of fabs' argument, 0 as +
    wide = canvas_len < span                        # the side of max(canvas_len, span) the primal took
    half = np.where(wide, span, canvas_len) / 2.0
    dhalf = np.where(wide, dspan, 0.0) / 2.0
    hx, hy = dhalf * dirx + half * ddirx, dhalf * diry + half * ddiry
    return [dmidx - hx, dmidy - hy, dmidx + hx, dmidy + hy]


def tangent(batch, din):
    """Output tangents [nout][n][T] of a capi.HostBatch solved with its candidate planes, root indices
    and flags (oracle_lib.solve), for input-column tangents din [nin][n][T].  A sub-system whose chosen
    run did not converge gets NaN."""
    kind, n = batch.kind, batch.n
    din = np.asarray(din, dtype=np.float64)
    cols = batch.dense_cols()
    k = [np.asarray(c, dtype=np.float64)[:, None] for c in cols]
    kd = [din[c] for c in range(len(cols))]
    root = batch.root_index.astype(np.int64)
    r = np.minimum(root, 1)
    live = (root < 2) & (batch.converged[r, np.arange(n)] == 1)
    line = kind in (2, 5)
    # the unknown at the chosen root: the output point, or the chosen seed's normal
    x = (batch.cand[r, 0, np.arange(n)] if line else batch.out[0])[:, None]
    y = (batch.cand[r, 1, np.arange(n)] if line else batch.out[1])[:, None]
    with np.errstate(all="ignore"):
        # the Jacobian as Sys<KIND>::eval computes it
        if kind == 1:
            a, b, c, d = 2.0 * (x - k[0]), 2.0 * (y - k[1]), 2.0 * (x - k[3]), 2.0 * (y - k[4])
        elif kind == 2:
            a, b, c, d = k[2] - k[0], k[3] - k[1], x + x, y + y
        elif kind == 3:
            a, b, c, d = 2.0 * (x - k[0]), 2.0 * (y - k[1]), -(k[6] - k[4]), k[5] - k[3]
        elif kind == 4:
            a, b, c, d = -(k[3] - k[1]), k[2] - k[0], -(k[8] - k[6]), k[7] - k[5]
        else:
            a, b, c, d = k[1], -k[0], x + x, y + y
        det = a * d - b * c
        rg = np.zeros_like(kd[0])
        if kind == 1:
            rf = -((a * kd[0] + b * kd[1]) + (2.0 * k[2]) * kd[2])
            rg = -((c * kd[3] + d * kd[4]) + (2.0 * k[5]) * kd[5])
        elif kind == 2:
            rf = (((-kd[5]) + (kd[2] - kd[0]) * x) + (kd[3] - kd[1]) * y) + kd[4]
        elif kind == 3:
            rf = -((a * kd[0] + b * kd[1]) + (2.0 * k[2]) * kd[2])
            rg = _p2l(k[3:8], kd[3:8], x, y)
        elif kind == 4:
            rf = _p2l(k[0:5], kd[0:5], x, y)
            rg = _p2l(k[5:10], kd[5:10], x, y)
        else:
            length = np.sqrt(k[0] * k[0] + k[1] * k[1])
            dlen = (k[0] * kd[0] + k[1] * kd[1]) / length
            rf = ((-(kd[2] * length + k[2] * dlen)) + kd[0] * (-y)) + kd[1] * x
        dx = (b * rg - d * rf) / det
        dy = (c * rf - a * rg) / det
        if line:
            # c1, q, c2, canvas length: K2 (k0 k1, k4, k2 k3, k8), K5 (k7 k8, k9, k10 k11, k12)
            o1, oq, o2, ol = (0, 4, 2, 8) if kind == 2 else (7, 9, 10, 12)
            p = (x * k[o1] + y * k[o1 + 1]) - k[oq]
            dp = ((dx * k[o1] + x * kd[o1]) + (dy * k[o1 + 1] + y * kd[o1 + 1])) - kd[oq]
            out = _reconstruct(k[o1], k[o1 + 1], k[o2], k[o2 + 1], x, y, p, k[ol], kd[o1], kd[o1 + 1], kd[o2], kd[o2 + 1], dx, dy, dp)
        else:
            out = [dx, dy]
    dout = np.stack([np.broadcast_to(q, din.shape[1:]) for q in out]).copy()
    dout[:, ~live, :] = np.nan
    return dout
