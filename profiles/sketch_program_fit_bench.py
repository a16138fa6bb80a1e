"""Sketch-program fits (SketchProgram::fit) against the same fit driven from the host:
  1. configs[3] (the 100k-point linkage) at K = 1 with n_free = 8;
  2. the 20k linkage at K = 64 with n_free = 8.
Targets are the positions at the sketch's own values, observed at up to 48 coordinates that depend
on the free values; starts move the free values by 1e-3 .. 1e-2 relative.  The device fit reports its
device time (events), host clock, iterations and launches.  The host-driven loop runs the same number of
iterations of runTangents (T = n_free, the selector as directions) plus a numpy damped Gauss-Newton
step, and reports its host clock per iteration.  Every shape is warmed up; medians of 5.  Prints the
card and its power limit first, then one JSON line per measurement; with an output directory argument
also writes them there (sketch_program_fit_bench.jsonl).
Usage: python profiles/sketch_program_fit_bench.py [out_dir]"""
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
gcs = importlib.import_module("2d_geometry_constraint_solver_b200")
gcs.capi.init([0])
import program_fit_lib as F  # noqa: E402
import sketch_gen as S  # noqa: E402
from program_restate import Arrays  # noqa: E402
from program_restate_fit import Fit  # noqa: E402

lines = []


def emit(d):
    print(json.dumps(d), flush=True)
    lines.append(d)


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
emit({"card": card.splitlines()[0] if card else "unknown", "library": gcs.capi.load().gcs_b200_version().decode()})


def case(name, n, seed, K, n_free, reps=5):
    el, edges = S.make_linkage(n, seed=seed)
    prog = F.Program(el, edges)
    v = F.sketch_values(edges)
    p = Arrays.from_desc(prog.desc())
    angle = p.value_is_angle.astype(bool)
    cv = np.where(angle, np.cos(v), v)[None]
    free, os_, oc, _ = F.problem(p, cv, n_free, seed=5)
    rc, pos, _, _ = prog.run(v[None])
    rng = np.random.default_rng(1)
    start = np.repeat(v[None], K, axis=0)
    start[:, free] *= 1.0 + rng.uniform(1e-3, 1e-2, (K, n_free)) * rng.choice([-1.0, 1.0], (K, n_free))
    targets = np.repeat(pos[:, os_, oc], K, axis=0)
    fit = Fit(free, os_, oc, max_iterations=30)
    runs = []
    for r in range(reps + 1):
        t0 = time.perf_counter()
        rc, vals, _, _, res, st = prog.fit(start, targets, fit)
        wall = time.perf_counter() - t0
        assert rc == 0
        if r:
            runs.append((st["device_us"], wall, st["launches"]))
    iters = max(x["iterations"] for x in res)
    dev = float(np.median([x[0] for x in runs])) / 1e3
    emit({"case": name, "path": "device fit", "K": K, "n_free": n_free, "n_obs": len(os_), "iterations": iters,
          "statuses": sorted(set(x["status"] for x in res)), "device_ms": dev, "host_ms": float(np.median([x[1] for x in runs])) * 1e3,
          "device_ms_per_iteration": dev / iters, "launches": runs[0][2],
          "max_rel_err": float((np.abs(vals[:, free] - v[free]) / np.abs(v[free])).max())})
    # the same number of iterations driven from the host: runTangents + a numpy damped step
    sel = np.zeros((K, len(v), n_free))
    sel[:, free, np.arange(n_free)] = 1.0
    x = start.copy()
    for r in range(2):
        prog.run_tangents(x, sel)
    per = []
    for r in range(reps):
        x = start.copy()
        t0 = time.perf_counter()
        for _ in range(iters):
            rc, ps, dps, nc, _ = prog.run_tangents(x, sel)
            res_ = ps[:, os_, oc] - targets
            J = dps[:, os_, oc, :]
            A = np.einsum("koi,koj->kij", J, J)
            g = np.einsum("koi,ko->ki", J, res_)
            A += 1e-3 * np.einsum("kii->ki", A)[:, :, None] * np.eye(n_free)
            x[:, free] += np.linalg.solve(A, -g[:, :, None])[:, :, 0]
        per.append((time.perf_counter() - t0) / iters)
    emit({"case": name, "path": "host-driven runTangents + numpy step", "K": K, "n_free": n_free, "iterations": iters,
          "host_ms_per_iteration": float(np.median(per)) * 1e3, "host_ms": float(np.median(per)) * 1e3 * iters})


case("configs[3] 100k linkage", 100000, 4, 1, 8)
case("20k linkage", 20000, 6, 64, 8)
if len(sys.argv) > 1:
    os.makedirs(sys.argv[1], exist_ok=True)
    with open(os.path.join(sys.argv[1], "sketch_program_fit_bench.jsonl"), "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")
