"""Sketch-program adjoints (SketchProgram::record / adjoints) against plain and tangent runs, in one process:
  1. the 100k-point linkage (configs[3]) at K = 1: run, record, the sweep at T = 1 and T = 8, and a
     tangent run at T = 32: device time (events), host clock and launches of each, and the tape's bytes;
  2. the 20k linkage at K = 64: run, record, the sweep at T = 1 and a tangent run at T = 32.
The gradient of one objective over every value by forward mode would take n_values / 32 tangent runs
at T = 32; that figure is an extrapolation from the measured tangent run, not a measurement.  Each
shape is warmed up; the paths alternate; medians of 7.  Prints the card and its power limit and the
library's source hash first, then one JSON line per measurement; with an output directory argument
also writes them there (sketch_program_adjoints_bench.jsonl).
Usage: python profiles/sketch_program_adjoints_bench.py [out_dir]"""
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
gcs = importlib.import_module("2d_geometry_constraint_solver_b200")
gcs.capi.init([0])
import host_lib as H  # noqa: E402
import program_adjoints_lib as P  # noqa: E402
import sketch_gen as S  # noqa: E402

lines = []
IN, OUT = {1: 6, 2: 9, 3: 10, 4: 12, 5: 13}, {1: 2, 2: 4, 3: 2, 4: 2, 5: 4}


def emit(d):
    print(json.dumps(d), flush=True)
    lines.append(d)


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
emit({"card": card.splitlines()[0] if card else "unknown", "library": gcs.capi.load().gcs_b200_version().decode()})


def median(xs):
    return float(np.median(np.asarray(xs, dtype=np.float64)))


def tape_bytes(offsets, K):
    """the tape of a recorded run (csrc/sketch_program.cu: tape_layout), from the program's offsets"""
    a256 = lambda v: (v + 255) // 256 * 256  # noqa: E731
    total = 0
    for s in range(len(offsets) - 1):
        k = s % 5 + 1
        cap = ((int(offsets[s + 1]) - int(offsets[s])) * K + 31) // 32 * 32
        total += a256((IN[k] + OUT[k]) * cap * 8) + 4 * a256(cap) + (a256(32 * cap) if k in (2, 5) else 0)
    return total


def summary(stats):
    return {"device_ms": median([s["device_us"] for s in stats]) / 1e3, "host_ms": median([s["run_us"] for s in stats]) / 1e3,
            "launches": stats[0]["launches"]}


def measure(name, prog, vals, sweeps, reps=7):
    K, nv = vals.shape
    d = prog.describe()
    rng = np.random.default_rng(K)
    obs = {T: rng.standard_normal((K, d["slots"], 4, T)) for T in sweeps}
    dirs = rng.standard_normal((K, nv, 32))
    for _ in range(2):  # warm-up of every shape
        prog.run(vals)
        prog.run_tangents(vals, dirs)
        prog.record(vals)
        for T in sweeps:
            prog.adjoints(obs[T])
    plain, rec, tang, sweep = [], [], [], {T: [] for T in sweeps}
    for _ in range(reps):
        rc, pos, nc, st = prog.run(vals)
        assert rc == 0, H.last_error()
        plain.append(st)
        rc, _, _, _, st = prog.run_tangents(vals, dirs)
        assert rc == 0, H.last_error()
        tang.append(st)
        rc, rpos, rnc, st = prog.record(vals)
        assert rc == 0, H.last_error()
        rec.append(st)
        for T in sweeps:
            rc, _, st = prog.adjoints(obs[T])
            assert rc == 0, H.last_error()
            sweep[T].append(st)
    t32 = summary(tang)
    emit({"measurement": name, "K": K, "waves": d["waves"], "rows": d["rows"], "values": nv,
          "run": summary(plain), "record": summary(rec),
          **{f"adjoints_T{T}": summary(sweep[T]) for T in sweeps},
          "tangents_T32": t32,
          "tape_bytes": tape_bytes(d["offsets"], K),
          "forward_gradient_extrapolated_device_ms": t32["device_ms"] * -(-nv // 32),
          "record_bit_identical": bool(np.array_equal(pos.view(np.uint64), rpos.view(np.uint64)) and np.array_equal(nc, rnc))})


el, edges = S.make_linkage(100000, seed=4)
prog = P.Program(el, edges)
assert prog.rc == 0, prog.error
measure("configs[3] K=1", prog, P.sketch_values(edges)[None, :], (1, 8))
del prog

el, edges = S.make_linkage(20000, seed=6)
prog = P.Program(el, edges)
base = P.sketch_values(edges)
vals = base * (1.0 + 1e-3 * np.random.default_rng(64).uniform(-1.0, 1.0, size=(64, len(base))))
vals[0] = base
measure("20k K=64", prog, vals, (1,))

if len(sys.argv) > 1:
    os.makedirs(sys.argv[1], exist_ok=True)
    with open(os.path.join(sys.argv[1], "sketch_program_adjoints_bench.jsonl"), "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")
