"""CPU restatement of a solved sub-system's reverse-mode adjoint (csrc/newton_adjoint.cuh), the
transpose of tests/tangent_oracle.py's tangent, in the operation order written there.  numpy's float64
element-wise operations round once each and never fuse a multiply with an add, so with the device
built with --fmad=false the two agree bit for bit.  Test infrastructure only."""
import numpy as np


def _p2l(k, x, y, r):
    """adjoint of P2L::eval's tangent at fixed (x, y); k: xa ya xb yb s as [n][1] columns, r [n][T].
    Returns kb[0..4]."""
    ex, ey = k[2] - k[0], k[3] - k[1]
    length = np.sqrt(ex * ex + ey * ey)
    ux, uy = x - k[0], y - k[1]
    kb = [None] * 5
    dex = uy * r
    kb[1] = -(ex * r)
    dey = -(ux * r)
    kb[0] = ey * r
    dld = -r
    kb[4] = length * dld
    q = (k[4] * dld) / length
    dex = dex + ex * q
    dey = dey + ey * q
    kb[2] = dex
    kb[0] = kb[0] + (-dex)
    kb[3] = dey
    kb[1] = kb[1] + (-dey)
    return kb


def _reconstruct(c1x, c1y, c2x, c2y, nx, ny, p, canvas_len, o):
    """adjoint of reconstruct_tangent: (dc1x, dc1y, dc2x, dc2y, dnx, dny, dp)"""
    sd1 = (nx * c1x + ny * c1y) - p
    a1x, a1y = c1x - sd1 * nx, c1y - sd1 * ny
    sd2 = (nx * c2x + ny * c2y) - p
    a2x, a2y = c2x - sd2 * nx, c2y - sd2 * ny
    dirx, diry = -ny, nx
    ex, ey = a2x - a1x, a2y - a1y
    arg = dirx * ex + diry * ey
    span = np.abs(arg)
    wide = canvas_len < span
    half = np.where(wide, span, canvas_len) / 2.0
    mx, hx, my, hy = o[0] + o[2], o[2] - o[0], o[1] + o[3], o[3] - o[1]
    dhalf = hx * dirx + hy * diry
    ddirx, ddiry = half * hx, half * hy
    dspan = np.where(wide, dhalf / 2.0, 0.0)
    darg = np.where(arg >= 0.0, dspan, -dspan)
    ddirx = ddirx + ex * darg
    dex = dirx * darg
    ddiry = ddiry + ey * darg
    dey = diry * darg
    da2x, da1x = dex + mx / 2.0, mx / 2.0 - dex
    da2y, da1y = dey + my / 2.0, my / 2.0 - dey
    dny, dnx, dp = -ddirx, ddiry, 0.0
    out = {}
    for (cx, cy, sd, dax, day, i) in ((c2x, c2y, sd2, da2x, da2y, 2), (c1x, c1y, sd1, da1x, da1y, 1)):
        dsd = -(ny * day)
        dcy = day
        dny = dny + (-(sd * day))
        dcx = dax
        dsd = dsd + (-(nx * dax))
        dnx = dnx + (-(sd * dax))
        dnx = dnx + cx * dsd
        dcx = dcx + nx * dsd
        dny = dny + cy * dsd
        dcy = dcy + ny * dsd
        dp = dp + (-dsd)
        out[i] = (dcx, dcy)
    return out[1][0], out[1][1], out[2][0], out[2][1], dnx, dny, dp


def adjoint(batch, ob):
    """Input-column adjoints [nin][n][T] of a capi.HostBatch solved with its candidate planes, root
    indices and flags (oracle_lib.solve), for output adjoints ob [nout][n][T].  Also returns live [n]:
    the sub-system's chosen run converged.  A sub-system that is not live gets 0 (the NaN rule is the
    caller's)."""
    kind, n = batch.kind, batch.n
    ob = np.asarray(ob, dtype=np.float64)
    T = ob.shape[2]
    cols = batch.dense_cols()
    k = [np.asarray(c, dtype=np.float64)[:, None] for c in cols]
    root = batch.root_index.astype(np.int64)
    r = np.minimum(root, 1)
    live = (root < 2) & (batch.converged[r, np.arange(n)] == 1)
    line = kind in (2, 5)
    x = (batch.cand[r, 0, np.arange(n)] if line else batch.out[0])[:, None]
    y = (batch.cand[r, 1, np.arange(n)] if line else batch.out[1])[:, None]
    zero = np.zeros((n, T))
    kb = [zero.copy() for _ in cols]
    with np.errstate(all="ignore"):
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
        if line:
            o, oq, o2, ol = (0, 4, 2, 8) if kind == 2 else (7, 9, 10, 12)
            p = (x * k[o] + y * k[o + 1]) - k[oq]
            dc1x, dc1y, dc2x, dc2y, dnx, dny, dp = _reconstruct(k[o], k[o + 1], k[o2], k[o2 + 1], x, y, p, k[ol], ob)
            dx = dnx + k[o] * dp
            kb[o] = dc1x + x * dp
            dy = dny + k[o + 1] * dp
            kb[o + 1] = dc1y + y * dp
            kb[oq] = -dp
            kb[o2], kb[o2 + 1] = dc2x, dc2y
        else:
            dx, dy = ob[0], ob[1]
        ub, wb = dx / det, dy / det
        rf = (c * wb) - (d * ub)
        rg = (b * ub) - (a * wb)
        if kind in (1, 3):
            s = -rf
            kb[0], kb[1], kb[2] = a * s, b * s, (2.0 * k[2]) * s
        if kind == 1:
            s = -rg
            kb[3], kb[4], kb[5] = c * s, d * s, (2.0 * k[5]) * s
        elif kind == 2:
            kb[5] = -rf
            kb[2] = kb[2] + x * rf
            kb[0] = kb[0] + (-(x * rf))
            kb[3] = kb[3] + y * rf
            kb[1] = kb[1] + (-(y * rf))
            kb[4] = kb[4] + rf
        elif kind == 3:
            kb[3:8] = _p2l(k[3:8], x, y, rg)
        elif kind == 4:
            kb[0:5] = _p2l(k[0:5], x, y, rf)
            kb[5:10] = _p2l(k[5:10], x, y, rg)
        elif kind == 5:
            length = np.sqrt(k[0] * k[0] + k[1] * k[1])
            kb[1] = x * rf
            kb[0] = (-y) * rf
            s = -rf
            kb[2] = length * s
            q = (k[2] * s) / length
            kb[0] = kb[0] + k[0] * q
            kb[1] = kb[1] + k[1] * q
    out = np.stack([np.broadcast_to(v, (n, T)) for v in kb]).copy()
    out[:, ~live, :] = 0.0
    return out, live
