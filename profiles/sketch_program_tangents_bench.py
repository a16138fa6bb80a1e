"""Sketch-program tangents (SketchProgram::runTangents) against plain runs, in one process:
  1. the 100k-point linkage (configs[3]) at K = 1 and T = 1, 8, 32: device time (events) and host
     clock of run and runTangents, and launches per run;
  2. the 20k linkage at K = 64, T = 8: the same;
  3. for both, the same T directions by central differences through run (one run of 2T instances per
     base instance; directions are the values times normal random numbers, and the step of each
     instance and direction, 1e-3 / max(1, its largest |tangent|), moves no position by more than
     1e-3; the tangents compared are those along the directions the +- value sets actually differ
     by, (v+ - v-) / 2h, since with tangents of 1e9 the rounding of v +- h dir matters): time, and the largest deviation from the tangents relative to max(1, |tangent|) over the
     coordinates whose +- positions stay within 0.1 of each other (the rest are counted as root flips)
     and that the step moves by at least 1e-6 max(1, |position|) (the rest are below its resolution).
Each shape is warmed up; the two paths alternate; medians of 7.  Prints the card and its power limit
and the library's source hash first, then one JSON line per measurement; with an output directory
argument also writes them there (sketch_program_tangents_bench.jsonl).
Usage: python profiles/sketch_program_tangents_bench.py [out_dir]"""
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
import program_tangents_lib as P  # noqa: E402
import sketch_gen as S  # noqa: E402

lines = []


def emit(d):
    print(json.dumps(d), flush=True)
    lines.append(d)


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
emit({"card": card.splitlines()[0] if card else "unknown", "library": gcs.capi.load().gcs_b200_version().decode()})


def median(xs):
    return float(np.median(np.asarray(xs, dtype=np.float64)))


def measure(name, prog, vals, T, reps=7):
    K, nv = vals.shape
    dirs = vals[:, :, None] * np.random.default_rng(T).standard_normal((K, nv, T))
    rc, _, dpos, _, _ = prog.run_tangents(vals, dirs)
    assert rc == 0, H.last_error()
    h = 1e-3 / np.maximum(1.0, np.where(np.isfinite(dpos), np.abs(dpos), 0.0).reshape(K, -1, T).max(axis=1))  # [K][T]
    step = np.moveaxis(dirs, 2, 1) * h[:, :, None]  # [K][T][nv]
    vp, vm = vals[:, None, :] + step, vals[:, None, :] - step
    dirs = np.ascontiguousarray(np.moveaxis((vp - vm) / (2 * h[:, :, None]), 1, 2))
    plus_minus = np.concatenate([vp, vm], axis=1).reshape(K * 2 * T, nv)
    for _ in range(2):  # warm-up of every shape
        prog.run(vals)
        prog.run_tangents(vals, dirs)
        prog.run(plus_minus)
    plain, tang, fd = [], [], []
    for _ in range(reps):
        rc, pos, nc, st = prog.run(vals)
        assert rc == 0, H.last_error()
        plain.append(st)
        rc, tpos, dpos, tnc, st = prog.run_tangents(vals, dirs)
        assert rc == 0, H.last_error()
        tang.append(st)
        rc, pm, _, st = prog.run(plus_minus)
        assert rc == 0, H.last_error()
        fd.append(st)
    pm = pm.reshape(K, 2, T, *pm.shape[1:])
    pp, mm = np.moveaxis(pm[:, 0], 1, -1), np.moveaxis(pm[:, 1], 1, -1)  # [K][slots][4][T]
    flip = np.abs(pp - mm) > 0.1
    resolved = h[:, None, None, :] * np.abs(dpos) >= 1e-6 * np.maximum(1.0, np.abs(tpos))[..., None]
    ok = np.isfinite(dpos) & ~flip & resolved
    dev = np.abs((pp - mm) / (2 * h[:, None, None, :]) - dpos) / np.maximum(1.0, np.abs(dpos))
    emit({"measurement": name, "K": K, "T": T,
          "run_device_ms": median([s["device_us"] for s in plain]) / 1e3, "run_host_ms": median([s["run_us"] for s in plain]) / 1e3,
          "run_launches": plain[0]["launches"],
          "tangents_device_ms": median([s["device_us"] for s in tang]) / 1e3, "tangents_host_ms": median([s["run_us"] for s in tang]) / 1e3,
          "tangents_launches": tang[0]["launches"],
          "central_differences_device_ms": median([s["device_us"] for s in fd]) / 1e3,
          "central_differences_host_ms": median([s["run_us"] for s in fd]) / 1e3,
          "primal_bit_identical": bool(np.array_equal(pos.view(np.uint64), tpos.view(np.uint64)) and np.array_equal(nc, tnc)),
          "fd_max_rel_deviation": float(dev[ok].max()) if ok.any() else None,
          "fd_root_flip_coordinates": int((flip & np.isfinite(dpos)).sum()),
          "fd_compared_coordinates": int(ok.sum()), "fd_unresolved_coordinates": int((np.isfinite(dpos) & ~flip & ~resolved).sum()), "nan_tangents": int((~np.isfinite(dpos)).sum())})


el, edges = S.make_linkage(100000, seed=4)
prog = P.Program(el, edges)
assert prog.rc == 0, prog.error
d = prog.describe()
emit({"sketch": "configs[3] 100k linkage", "leaves": d["leaves"], "waves": d["waves"], "values": d["values"]})
own = P.sketch_values(edges)[None, :]
for T in (1, 8, 32):
    measure("configs[3] K=1", prog, own, T)
del prog

el, edges = S.make_linkage(20000, seed=6)
prog = P.Program(el, edges)
d = prog.describe()
emit({"sketch": "20k linkage", "leaves": d["leaves"], "waves": d["waves"], "values": d["values"]})
base = P.sketch_values(edges)
vals = base * (1.0 + 1e-3 * np.random.default_rng(64).uniform(-1.0, 1.0, size=(64, len(base))))
vals[0] = base
measure("20k K=64", prog, vals, 8)

if len(sys.argv) > 1:
    os.makedirs(sys.argv[1], exist_ok=True)
    with open(os.path.join(sys.argv[1], "sketch_program_tangents_bench.jsonl"), "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")
