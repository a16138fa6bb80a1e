"""Sketch programs at the C ABI, test side: a gcs_b200_program_desc as numpy arrays and back, the wave
layouts that must not change what a run computes, and a run restated wave by wave on the CPU (numpy
gather + gcs_oracle_solve + the tangent restatement of tests/tangent_oracle.py)."""
import ctypes as C
import importlib

import numpy as np

import oracle_lib as O
from tangent_oracle import tangent

capi = importlib.import_module("2d_geometry_constraint_solver_b200").capi

KINDS = 5
IN_COLS = {1: 6, 2: 9, 3: 10, 4: 12, 5: 13}
KIND_OF_SOLVER = {1: 1, 2: 2, 3: 5, 4: 1, 5: 2, 6: 3, 7: 4, 8: 5}
ROW = np.dtype(capi.CProgramRow)  # the layout of gcs_b200_program_row


class Arrays:
    """A program descriptor as numpy arrays: rows (structured, ROW) [n_rows], offsets [n_waves * 5 + 1],
    slot_is_line [n_slots], initial [n_slots][4], value_is_angle [n_values]."""

    def __init__(self, rows, offsets, slot_is_line, initial, value_is_angle):
        self.rows = np.ascontiguousarray(rows, dtype=ROW)
        self.offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        self.slot_is_line = np.ascontiguousarray(slot_is_line, dtype=np.uint8)
        self.initial = np.ascontiguousarray(initial, dtype=np.float64).reshape(-1, 4)
        self.value_is_angle = np.ascontiguousarray(value_is_angle, dtype=np.uint8)
        assert (len(self.offsets) - 1) % KINDS == 0

    n_waves = property(lambda self: (len(self.offsets) - 1) // KINDS)
    n_slots = property(lambda self: len(self.slot_is_line))
    n_values = property(lambda self: len(self.value_is_angle))
    n_rows = property(lambda self: len(self.rows))

    def segment(self, w, k):
        """rows [lo, hi) of (wave w, kind k), k = 1..5"""
        return int(self.offsets[KINDS * w + k - 1]), int(self.offsets[KINDS * w + k])

    @classmethod
    def from_desc(cls, d):
        def arr(ptr, ctype, n):
            return np.ctypeslib.as_array(ptr, shape=(n,)).copy() if n else np.zeros(0, dtype=np.ctypeslib.as_ctypes_type(ctype))

        rows = np.zeros(d.n_rows, dtype=ROW)
        if d.n_rows:
            rows[:] = np.frombuffer((capi.CProgramRow * d.n_rows).from_address(C.addressof(d.rows.contents)), dtype=ROW)
        return cls(rows, arr(d.offsets, C.c_int64, KINDS * d.n_waves + 1), arr(d.slot_is_line, C.c_uint8, d.n_slots),
                   arr(d.initial, C.c_double, 4 * d.n_slots), arr(d.value_is_angle, C.c_uint8, d.n_values))

    def desc(self):
        """capi.CProgramDesc over these arrays (they live as long as the descriptor)."""
        d = capi.CProgramDesc(n_waves=self.n_waves, n_slots=self.n_slots, n_values=self.n_values, n_rows=self.n_rows)
        d.rows = self.rows.ctypes.data_as(C.POINTER(capi.CProgramRow))
        d.offsets = self.offsets.ctypes.data_as(C.POINTER(C.c_int64))
        d.slot_is_line = self.slot_is_line.ctypes.data_as(C.POINTER(C.c_uint8))
        d.initial = self.initial.ctypes.data_as(C.POINTER(C.c_double))
        d.value_is_angle = self.value_is_angle.ctypes.data_as(C.POINTER(C.c_uint8))
        d._keep = self
        return d

    def waves(self):
        """[[row indices of kind 1..5] per wave]"""
        return [[np.arange(*self.segment(w, k)) for k in range(1, KINDS + 1)] for w in range(self.n_waves)]

    def with_waves(self, waves):
        """The same rows, slots and values laid out in `waves` ([[row indices of kind 1..5] per wave])."""
        order, offsets = [], [0]
        for wave in waves:
            for idx in wave:
                order += list(idx)
                offsets.append(len(order))
        return Arrays(self.rows[np.array(order, dtype=np.int64)], offsets, self.slot_is_line, self.initial, self.value_is_angle)


def rows(desc):
    """The rows of a C-ABI descriptor as a structured array (fields solver, elem, value, code, sign, canvas)."""
    return Arrays.from_desc(desc).rows


# ---- wave layouts that leave every result bit-identical ----
# The plan gives the rows of one wave disjoint footprints (gcs_b200_program_create refuses anything
# else), so how a wave's rows are grouped, ordered or split over consecutive waves changes nothing.

def split_by_kind(p, reverse=False):
    """every wave as one wave per kind present, in kind order (or reversed)"""
    out = []
    for wave in p.waves():
        ks = [k for k in range(KINDS) if len(wave[k])]
        for k in (ks[::-1] if reverse else ks):
            out.append([wave[k] if j == k else wave[k][:0] for j in range(KINDS)])
    return p.with_waves(out)


def one_row_per_wave(p):
    out = []
    for wave in p.waves():
        for k in range(KINDS):
            for r in wave[k]:
                out.append([np.array([r]) if j == k else np.zeros(0, dtype=np.int64) for j in range(KINDS)])
    return p.with_waves(out)


def with_empty_waves(p):
    """an empty wave before the first wave, between any two and after the last"""
    empty = [np.zeros(0, dtype=np.int64)] * KINDS
    out = [empty]
    for wave in p.waves():
        out += [wave, empty]
    return p.with_waves(out)


def reversed_segments(p):
    """the rows of every (wave, kind) segment in reverse order"""
    return p.with_waves([[idx[::-1] for idx in wave] for wave in p.waves()])


def relabelled(p, seed, extra_slots=7, extra_values=5):
    """Slots and values permuted, plus unused slots (NaN initial positions) and unused values.  Returns
    (program, slot_map, value_map): old slot s is new slot slot_map[s], old value v new value value_map[v]."""
    rng = np.random.default_rng(seed)
    ns, nv = p.n_slots + extra_slots, p.n_values + extra_values
    slot_map, value_map = rng.permutation(ns)[:p.n_slots], rng.permutation(nv)[:p.n_values]
    r = p.rows.copy()
    r["elem"] = slot_map[r["elem"]]
    r["value"] = np.where(r["value"] >= 0, value_map[np.maximum(r["value"], 0)], -1)
    is_line = rng.integers(0, 2, ns).astype(np.uint8)
    is_line[slot_map] = p.slot_is_line
    initial = np.full((ns, 4), np.nan)
    initial[slot_map] = p.initial
    angle = np.zeros(nv, dtype=np.uint8)
    angle[value_map] = p.value_is_angle
    return Arrays(r, p.offsets, is_line, initial, angle), slot_map, value_map


def without_rows(p, n_waves):
    """the program's slots and values, no rows, n_waves empty waves"""
    return Arrays(p.rows[:0], np.zeros(KINDS * n_waves + 1, dtype=np.int64), p.slot_is_line, p.initial, p.value_is_angle)


def transforms(p):
    """(name, program) for every layout above that keeps slot and value labels"""
    return [("split_by_kind", split_by_kind(p)), ("split_by_kind_reversed", split_by_kind(p, reverse=True)),
            ("one_row_per_wave", one_row_per_wave(p)), ("empty_waves", with_empty_waves(p)),
            ("reversed_segments", reversed_segments(p))]


# ---- the CPU restatement ----

def gather(solver, sign, cst, pa, pb, v, dpa, dpb, dv):
    """gather_row (csrc/sketch_program.cu) for one row over K instances and its tangent: (columns
    [nin][K], column tangents [nin][K][T], anchors {role: (position [K][4] writes, tangent writes)})."""
    K, T = v.shape[0], dv.shape[2]
    z, dz = np.zeros(K), np.zeros((K, T))
    v0, v1, v2 = v[:, 0], v[:, 1], v[:, 2]
    d0, d1, d2 = dv[:, 0], dv[:, 1], dv[:, 2]
    anchors = {}
    if solver in (1, 2):
        anchors = {0: ({0: z, 1: z}, {0: dz, 1: dz}), 1: ({0: v0, 1: z}, {0: d0, 1: dz})}
    if solver == 1:
        return [z, z, v1, v0, z, v2], [dz, dz, d1, d0, dz, d2], anchors
    if solver == 4:
        return [pa[:, 0], pa[:, 1], v1, pb[:, 0], pb[:, 1], v2], [dpa[:, 0], dpa[:, 1], d1, dpb[:, 0], dpb[:, 1], d2], anchors
    c = [np.full(K, x) for x in cst]
    if solver == 2:
        return ([z, z, v0, z, sign[1] * v1, sign[2] * v2, c[0], c[1], c[2]],
                [dz, dz, d0, dz, sign[1] * d1, sign[2] * d2, dz, dz, dz], anchors)
    if solver == 5:
        return ([pa[:, 0], pa[:, 1], pb[:, 0], pb[:, 1], sign[1] * v1, sign[2] * v2, c[0], c[1], c[2]],
                [dpa[:, 0], dpa[:, 1], dpb[:, 0], dpb[:, 1], sign[1] * d1, sign[2] * d2, dz, dz, dz], anchors)
    if solver == 6:
        return ([pa[:, 0], pa[:, 1], v1, pb[:, 0], pb[:, 1], pb[:, 2], pb[:, 3], sign[2] * v2, c[0], c[1]],
                [dpa[:, 0], dpa[:, 1], d1, dpb[:, 0], dpb[:, 1], dpb[:, 2], dpb[:, 3], sign[2] * d2, dz, dz], anchors)
    if solver == 7:
        return ([pa[:, 0], pa[:, 1], pa[:, 2], pa[:, 3], sign[1] * v1, pb[:, 0], pb[:, 1], pb[:, 2], pb[:, 3], sign[2] * v2, c[0], c[1]],
                [dpa[:, 0], dpa[:, 1], dpa[:, 2], dpa[:, 3], sign[1] * d1, dpb[:, 0], dpb[:, 1], dpb[:, 2], dpb[:, 3], sign[2] * d2, dz, dz],
                anchors)
    if solver == 3:
        sd1, dsd1 = sign[1] * v1, sign[1] * d1
        anchors = {0: ({0: c[7], 1: z, 2: c[8], 3: z}, {0: dz, 1: dz, 2: dz, 3: dz}), 1: ({0: z, 1: sd1}, {0: dz, 1: dsd1})}
        return ([c[5], c[6], v0, c[0], c[1], c[2], c[3], z, sd1, sign[2] * v2, z, z, c[4]],
                [dz, dz, d0, dz, dz, dz, dz, dz, dsd1, sign[2] * d2, dz, dz, dz], anchors)
    # solver 8
    return ([pa[:, 2] - pa[:, 0], pa[:, 3] - pa[:, 1], v0, c[0], c[1], c[2], c[3], pb[:, 0], pb[:, 1], sign[2] * v2,
             (pa[:, 0] + pa[:, 2]) / 2.0, (pa[:, 1] + pa[:, 3]) / 2.0, c[4]],
            [dpa[:, 2] - dpa[:, 0], dpa[:, 3] - dpa[:, 1], d0, dz, dz, dz, dz, dpb[:, 0], dpb[:, 1], sign[2] * d2,
             (dpa[:, 0] + dpa[:, 2]) / 2.0, (dpa[:, 1] + dpa[:, 3]) / 2.0, dz], anchors)


def gather_wave(p, w, pos, dpos, vals, dvals):
    """Wave w gathered from the state (pos [K][n_slots][4], dpos [K][n_slots][4][T]) the earlier waves left:
    ([(kind, lo, hi, HostBatch of (hi - lo) * K sub-systems without outputs, column tangents [nin][n][T])],
    [(slot, {coordinate: [K]}, {coordinate: [K][T]}) the zero-fixed anchors write])."""
    K, T = dvals.shape[0], dvals.shape[2]
    r = p.rows
    batches, anchors = [], []
    for k in range(1, KINDS + 1):
        lo, hi = p.segment(w, k)
        if hi == lo:
            continue
        cols, dcols = [[] for _ in range(IN_COLS[k])], [[] for _ in range(IN_COLS[k])]
        for i in range(lo, hi):
            a, b = r["elem"][i, 0], r["elem"][i, 1]
            vi = r["value"][i]
            v = np.stack([vals[:, j] if j >= 0 else np.zeros(K) for j in vi], axis=1)
            dv = np.stack([dvals[:, j, :] if j >= 0 else np.zeros((K, T)) for j in vi], axis=1)
            cs, dcs, anc = gather(r["solver"][i], r["sign"][i], r["canvas"][i], pos[:, a], pos[:, b], v, dpos[:, a], dpos[:, b], dv)
            for q in range(IN_COLS[k]):
                cols[q].append(cs[q])
                dcols[q].append(dcs[q])
            anchors += [(a if role == 0 else b, x, dx) for role, (x, dx) in anc.items()]
        code = np.repeat(r["code"][lo:hi].astype(np.uint8), K)  # sub-system (row i, instance j) at i * K + j
        hb = O.capi.HostBatch(k, 2, [np.ascontiguousarray(np.concatenate(c)) for c in cols], np.ascontiguousarray(code))
        batches.append((k, lo, hi, hb, np.stack([np.concatenate(c) for c in dcols])))
    return batches, anchors


def not_converged(hb):
    """[n]: the sub-system's chosen root is none (>= 2) or its chosen Newton run did not converge"""
    root = hb.root_index.astype(np.int64)
    return (root >= 2) | (hb.converged[np.minimum(root, 1), np.arange(hb.n)] == 0)


def restate(p, vals, dvals=None):
    """A run of the program `p` (Arrays, or a C-ABI descriptor) restated wave by wave on the CPU.  vals
    [K][n_values] (angle slots hold cos), dvals [K][n_values][T] (None: a plain run).  Returns (positions
    [K][n_slots][4], tangents [K][n_slots][4][T], nonconverged [K])."""
    if not isinstance(p, Arrays):
        p = Arrays.from_desc(p)
    K = vals.shape[0]
    if dvals is None:
        dvals = np.zeros((K, p.n_values, 1))
    T = dvals.shape[2]
    pos = np.repeat(p.initial[None], K, axis=0)
    dpos = np.zeros((K, p.n_slots, 4, T))
    nc = np.zeros(K, dtype=np.uint32)
    for w in range(p.n_waves):
        batches, anchors = gather_wave(p, w, pos, dpos, vals, dvals)  # reads the state the previous waves left
        for _, _, _, hb, dcols in batches:
            O.solve(hb.alloc_outputs())
        for slot, x, dx in anchors:
            for q in x:
                pos[:, slot, q] = x[q]
                dpos[:, slot, q] = dx[q]
        for _, lo, hi, hb, dcols in batches:  # the scatter and the tangent kernel
            dout = tangent(hb, dcols)
            nc += not_converged(hb).reshape(hi - lo, K).sum(axis=0).astype(np.uint32)
            for i in range(lo, hi):
                c, sl = p.rows["elem"][i, 2], slice((i - lo) * K, (i - lo + 1) * K)
                for q in range(len(hb.out)):
                    pos[:, c, q] = hb.out[q][sl]
                    dpos[:, c, q, :] = dout[q, sl, :]
    return pos, dpos, nc
