"""Sketch programs (gcs/b200/sketch_program.hpp) against the wave solver, in one process:
  1. the 100k-point linkage (configs[3]) at K = 1: compile time and run time (device events and the
     host clock to completion) next to gcs_host_system_solve_ex's solve_us, outputs bit for bit;
  2. the 20k and 100k linkages at K = 16 / 128 / 1024: leaf solves per second (K x leaves / run time)
     and launches per run, next to K = 16 sequential host-path solves.
Prints the card and its power limit first, then one JSON line per measurement; with an output
directory argument also writes them there (sketch_program_bench.jsonl).
Usage: python profiles/sketch_program_bench.py [out_dir]"""
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
import host_lib as H  # noqa: E402
import program_lib as P  # noqa: E402
import sketch_gen as S  # noqa: E402

lines = []


def emit(d):
    print(json.dumps(d), flush=True)
    lines.append(d)


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
emit({"card": card.splitlines()[0] if card else "unknown"})


def values_for(edges, K, seed):
    base = P.sketch_values(edges)
    u = np.random.default_rng(seed).uniform(-1.0, 1.0, size=(K, len(base)))
    v = base * (1.0 + 1e-3 * u)
    v[0] = base
    return v


def with_values(edges, vals):
    out, it = [], iter(vals)
    for e in edges:
        e = dict(e)
        if e["type"] != S.VIRT:
            e["value"] = float(next(it))
        out.append(e)
    return out


def median(xs):
    return float(np.median(np.asarray(xs, dtype=np.float64)))


sketches = {n: S.make_linkage(n, seed=4 if n == 100000 else 6) for n in (20000, 100000)}

# ---- 1. configs[3] at K = 1 ----
el, edges = sketches[100000]
t0 = time.perf_counter()
prog = P.Program(el, edges)
create_s = time.perf_counter() - t0
assert prog.rc == 0, prog.error
d = prog.describe()
own = P.sketch_values(edges)[None, :]
for _ in range(3):  # warm-up: module load, device tables, pinned staging
    rc, pos, nc, st = prog.run(own)
    H.system_solve_ex(el, edges)
runs, host = [], []
for _ in range(7):  # the two paths alternate
    rc, pos, nc, st = prog.run(own)
    assert rc == 0, H.last_error()
    runs.append(st)
    rc2, out, hs = H.system_solve_ex(el, edges)
    assert rc2 == 0, H.last_error()
    host.append(hs)
xy = np.ascontiguousarray(pos[0, :, :2])
same = bool(np.array_equal(xy.view(np.uint64), np.array([e["pos"] for e in out]).view(np.uint64)))
emit({"measurement": "configs[3] K=1", "leaves": d["leaves"], "waves": d["waves"], "rows": d["rows"],
      "create_incl_decomposition_ms": create_s * 1e3, "compile_ms": runs[0]["compile_us"] / 1e3,
      "program_run_ms_host_clock": median([s["run_us"] for s in runs]) / 1e3,
      "program_device_ms_events": median([s["device_us"] for s in runs]) / 1e3,
      "program_upload_ms": median([s["upload_us"] for s in runs]) / 1e3, "program_download_ms": median([s["download_us"] for s in runs]) / 1e3,
      "launches_per_run": runs[0]["launches"],
      "host_path_solve_ms": median([h["solve_us"] for h in host]) / 1e3,
      "host_path_pack_ms": median([h["pack_us"] for h in host]) / 1e3, "host_path_device_ms": median([h["device_us"] for h in host]) / 1e3,
      "host_path_apply_ms": median([h["apply_us"] for h in host]) / 1e3, "host_path_launches": host[0]["launches"],
      "bit_identical": same})

# ---- 2. sweeps ----
for n, (el, edges) in sketches.items():
    prog = P.Program(el, edges)
    d = prog.describe()
    seq = None
    for K in (16, 128, 1024):
        vals = values_for(edges, K, seed=K)
        prog.run(vals)  # warm-up at this K (grows the device tables and the staging once)
        res = []
        for _ in range(3):
            rc, pos, nc, st = prog.run(vals)
            assert rc == 0, H.last_error()
            res.append(st)
        run_s = median([s["run_us"] for s in res]) * 1e-6
        dev_s = median([s["device_us"] for s in res]) * 1e-6
        row = {"measurement": f"sweep n={n} K={K}", "leaves": d["leaves"], "waves": d["waves"], "launches_per_run": res[0]["launches"],
               "run_ms_host_clock": run_s * 1e3, "device_ms_events": dev_s * 1e3,
               "upload_ms": median([s["upload_us"] for s in res]) / 1e3, "download_ms": median([s["download_us"] for s in res]) / 1e3,
               "leaf_solves_per_s_host_clock": K * d["leaves"] / run_s, "leaf_solves_per_s_device": K * d["leaves"] / dev_s,
               "nonconverged_instances": int((nc > 0).sum())}
        if K == 16:
            t0 = time.perf_counter()
            solve_us = 0
            for k in range(K):
                rc, out, hs = H.system_solve_ex(el, with_values(edges, vals[k]))
                assert rc == 0
                solve_us += hs["solve_us"]
                if k == K - 1:
                    last = np.array([e["pos"] for e in out])
            seq = {"host_path_16_solve_ms": solve_us / 1e3, "host_path_16_wall_ms": (time.perf_counter() - t0) * 1e3,
                   "host_path_leaf_solves_per_s": K * d["leaves"] / (solve_us * 1e-6),
                   "last_instance_bit_identical": bool(np.array_equal(np.ascontiguousarray(pos[K - 1, :, :2]).view(np.uint64), last.view(np.uint64)))}
            row.update(seq)
        emit(row)
        del pos, vals

if len(sys.argv) > 1:
    os.makedirs(sys.argv[1], exist_ok=True)
    with open(os.path.join(sys.argv[1], "sketch_program_bench.jsonl"), "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")
