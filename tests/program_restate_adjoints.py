"""The adjoint sweep of a sketch program (gcs_b200_program_adjoints) restated wave by wave on the CPU:
the forward run of tests/program_restate.py keeping every wave's solved batches, then the waves from
last to first with the row adjoint of tests/adjoint_oracle.py, the gather's transpose
(gather_row_transpose) and the reader lists' summation order of csrc/sketch_program.cu.  Also the forward/reverse contractions the duality
tests compare."""
import numpy as np

import oracle_lib as O
from adjoint_oracle import adjoint
from program_restate import KINDS, Arrays, gather_wave, not_converged

_LINE = {1: (0, 0, 0), 2: (0, 0, 1), 3: (1, 0, 1), 4: (0, 0, 0), 5: (0, 0, 1), 6: (0, 1, 0), 7: (1, 1, 0), 8: (1, 0, 1)}
_OUT = {1: 2, 2: 4, 3: 2, 4: 2, 5: 4}


def record(p, vals):
    """The forward run of `p` for vals [K][n_values], keeping per wave [(kind, lo, hi, solved HostBatch)].
    Returns (positions [K][n_slots][4], nonconverged [K], tape)."""
    K = vals.shape[0]
    pos = np.repeat(p.initial[None], K, axis=0)
    dpos = np.zeros((K, p.n_slots, 4, 1))
    dvals = np.zeros((K, p.n_values, 1))
    nc = np.zeros(K, dtype=np.uint32)
    tape = []
    for w in range(p.n_waves):
        batches, anchors = gather_wave(p, w, pos, dpos, vals, dvals)
        for _, _, _, hb, _ in batches:
            O.solve(hb.alloc_outputs())
        for slot, x, _ in anchors:
            for q in x:
                pos[:, slot, q] = x[q]
        for _, lo, hi, hb, _ in batches:
            nc += not_converged(hb).reshape(hi - lo, K).sum(axis=0).astype(np.uint32)
            for i in range(lo, hi):
                c, sl = p.rows["elem"][i, 2], slice((i - lo) * K, (i - lo + 1) * K)
                for q in range(len(hb.out)):
                    pos[:, c, q] = hb.out[q][sl]
        tape.append([(k, lo, hi, hb) for k, lo, hi, hb, _ in batches])
    return pos, nc, tape


def restate_adjoints(p, vals, adj_pos):
    """adj_values [K][n_values][T] of the program `p` (Arrays, or a C-ABI descriptor) at vals [K][n_values]
    (angle slots hold cos) for the cotangents adj_pos [K][n_slots][4][T], in the device's order."""
    if not isinstance(p, Arrays):
        p = Arrays.from_desc(p)
    K, T = vals.shape[0], adj_pos.shape[3]
    _, _, tape = record(p, vals)
    ap = np.array(adj_pos, dtype=np.float64, copy=True)
    av = np.zeros((K, p.n_values, T))
    flag = np.zeros((K, T), dtype=bool)
    rows = p.rows
    for w in range(p.n_waves - 1, -1, -1):
        wlo = p.segment(w, 1)[0]
        scon, vcon = {}, {}  # (row - wlo, role) -> [4][K][T]; (row - wlo, q) -> [K][T]
        for k, lo, hi, hb in tape[w]:
            nout = _OUT[k]
            ob = np.zeros((nout, (hi - lo) * K, T))
            anchor = {}
            for i in range(lo, hi):
                sl = slice((i - lo) * K, (i - lo + 1) * K)
                a, b, c = rows["elem"][i]
                solver = int(rows["solver"][i])
                for q in range(nout):
                    ob[q, sl] = ap[:, c, q]
                    ap[:, c, q] = 0.0
                if solver <= 3:
                    anchor[i] = ap[:, b, 1 if solver == 3 else 0].copy()
                    ap[:, a, :4 if solver == 3 else 2] = 0.0
                    ap[:, b, :2] = 0.0
            kb, live = adjoint(hb, ob)
            dead = ~live.reshape(hi - lo, K)
            touched = ~(ob == 0.0)  # NaN counts as non-zero
            for i in range(lo, hi):
                sl = slice((i - lo) * K, (i - lo + 1) * K)
                flag |= dead[i - lo][:, None] & touched[:, sl].any(axis=0)
                kr = kb[:, sl]
                solver = int(rows["solver"][i])
                s1, s2 = rows["sign"][i][1], rows["sign"][i][2]
                r = i - wlo
                z = np.zeros((K, T))
                sa = {}
                if solver == 1:
                    va = {0: kr[3] + anchor[i], 1: kr[2], 2: kr[5]}
                elif solver == 2:
                    va = {0: kr[2] + anchor[i], 1: s1 * kr[4], 2: s2 * kr[5]}
                elif solver == 3:
                    va = {0: kr[2], 1: s1 * (kr[8] + anchor[i]), 2: s2 * kr[9]}
                elif solver == 4:
                    sa = {0: [kr[0], kr[1], z, z], 1: [kr[3], kr[4], z, z]}
                    va = {1: kr[2], 2: kr[5]}
                elif solver == 5:
                    sa = {0: [kr[0], kr[1], z, z], 1: [kr[2], kr[3], z, z]}
                    va = {1: s1 * kr[4], 2: s2 * kr[5]}
                elif solver == 6:
                    sa = {0: [kr[0], kr[1], z, z], 1: [kr[3], kr[4], kr[5], kr[6]]}
                    va = {1: kr[2], 2: s2 * kr[7]}
                elif solver == 7:
                    sa = {0: [kr[0], kr[1], kr[2], kr[3]], 1: [kr[5], kr[6], kr[7], kr[8]]}
                    va = {1: s1 * kr[4], 2: s2 * kr[9]}
                else:
                    mx, my = kr[10] / 2.0, kr[11] / 2.0
                    sa = {0: [mx - kr[0], my - kr[1], mx + kr[0], my + kr[1]], 1: [kr[7], kr[8], z, z]}
                    va = {0: kr[2], 2: s2 * kr[9]}
                for role, v in sa.items():
                    scon[(r, role)] = v
                for q, v in va.items():
                    vcon[(r, q)] = v
        # the reduce: every entry's readers in ascending (row, role) order, one add at a time
        for (r, role) in sorted(scon):
            i = wlo + r
            slot = rows["elem"][i, role]
            for c in range(4 if _LINE[int(rows["solver"][i])][role] else 2):
                ap[:, slot, c] = ap[:, slot, c] + scon[(r, role)][c]
        for (r, q) in sorted(vcon):
            v = rows["value"][wlo + r, q]
            av[:, v] = av[:, v] + vcon[(r, q)]
    av[np.broadcast_to(flag[:, None, :], av.shape)] = np.nan
    return av
