"""Fused sketch-program runs (gcs_b200_program_run_fused: every wave in one cooperative launch) against
the wave-by-wave run (gcs_b200_program_run, GCS_VARIANT_DEFAULT), in one process:
  1. configs[3] (the 100 k-point linkage) and the 20 k linkage at K = 1, 4, 16, 64, 256, 1024: device
     time (CUDA events around the device entry point on one stream) of the two, alternated after a
     warm-up of every shape, medians of 21 repetitions (7 at K >= 256); outputs compared bit for bit;
  2. tangent runs (gcs_b200_program_run_tangents against run_fused) at T = 1, 8, 32 for K = 1, 16;
  3. the host clock of SketchProgram::run against SketchProgram::runFused at K = 1 (pageable host
     tables in and out, one device);
  4. the fused kernel's registers (cuobjdump), and from them the blocks per SM and the grid of every K
     (grid_derived: what fused_on's rule gives for these registers, min(blocks per SM x SMs, blocks the
     largest wave needs); derived here, not read from the launch).
Prints the card and its power limit and the library's source hash first, then one JSON line per
measurement; with an output directory argument also writes them there (sketch_program_fused_bench.jsonl).
Usage: python profiles/sketch_program_fused_bench.py [out_dir]"""
import ctypes as C
import importlib
import json
import os
import re
import shutil
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
gcs = importlib.import_module("2d_geometry_constraint_solver_b200")
gcs.capi.init([0])
import host_lib as H  # noqa: E402
import program_restate as R  # noqa: E402
import program_tangents_lib as P  # noqa: E402
import sketch_gen as S  # noqa: E402
from util import bits  # noqa: E402

lib = gcs.capi.load()
lines = []
THREADS = 128  # kFusedThreads of csrc/sketch_program.cu


def emit(d):
    print(json.dumps(d), flush=True)
    lines.append(d)


card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
emit({"card": card.splitlines()[0] if card else "unknown", "library": lib.gcs_b200_version().decode()})

# registers of program_fused_kernel and the blocks of 128 threads that fit an SM by registers
regs = None
cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
if os.path.exists(cuobjdump):
    out = subprocess.run([cuobjdump, "--dump-resource-usage", gcs.capi.LIB_PATH], capture_output=True, text=True).stdout
    m = re.search(r"program_fused_kernel.*?\n.*?REG:(\d+)\s+STACK:(\d+)", out)
    if m:
        regs = int(m.group(1))
        emit({"kernel": "program_fused_kernel", "registers": regs, "stack": int(m.group(2))})
sms = torch.cuda.get_device_properties(0).multi_processor_count
per_sm = min(2048 // THREADS, 65536 // (-(-regs * 32 // 256) * 256 * (THREADS // 32))) if regs else None
emit({"sms": sms, "blocks_per_sm_by_registers": per_sm})


def same(a, b):
    return a.shape == b.shape and bool(((bits(a) == bits(b)) | (np.isnan(a) & np.isnan(b))).all())


def median(xs):
    return float(np.median(np.asarray(xs, dtype=np.float64)))


def values(p, base, K, seed):
    angle = p.value_is_angle.astype(bool)
    u = np.random.default_rng(seed).uniform(-1.0, 1.0, size=(K, len(base)))
    v = np.where(angle, base + 1e-2 * u, base * (1.0 + 1e-3 * u))
    v[0] = base
    return np.where(angle, np.cos(v), v)


class Dev:
    """device tables of one program at one (K, T) and the two entry points on one stream"""

    def __init__(self, h, p, vals, T, seed):
        dev = torch.device("cuda", 0)
        K = vals.shape[0]
        self.h, self.K, self.T = h, K, T
        self.v = torch.from_numpy(vals).to(dev)
        self.dv = torch.from_numpy(np.random.default_rng(seed).standard_normal((K, p.n_values, T))).to(dev) if T else None
        self.out = {}
        for path in ("waves", "fused"):
            self.out[path] = (torch.empty((K, p.n_slots, 4), dtype=torch.float64, device=dev), torch.empty(K, dtype=torch.int32, device=dev),
                              torch.empty((K, p.n_slots, 4, T), dtype=torch.float64, device=dev) if T else None)
        self.stream = torch.cuda.Stream(device=0)

    def enqueue(self, path):
        pos, nc, dpos = self.out[path]
        s = self.stream.cuda_stream
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        if path == "fused":
            rc = lib.gcs_b200_program_run_fused(self.h, self.K, ptr(self.v), ptr(pos), ptr(nc), self.T, ptr(self.dv), ptr(dpos), s)
        elif self.T:
            rc = lib.gcs_b200_program_run_tangents(self.h, self.K, ptr(self.v), ptr(pos), ptr(nc), self.T, ptr(self.dv), ptr(dpos), 0, s)
        else:
            rc = lib.gcs_b200_program_run(self.h, self.K, ptr(self.v), ptr(pos), ptr(nc), 0, s)
        assert rc == 0, lib.gcs_b200_last_error()

    def time(self, path):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(self.stream)
        before = lib.gcs_b200_launch_count()
        self.enqueue(path)
        launches = lib.gcs_b200_launch_count() - before
        b.record(self.stream)
        b.synchronize()
        return a.elapsed_time(b), launches

    def equal(self):
        (p0, n0, d0), (p1, n1, d1) = self.out["waves"], self.out["fused"]
        torch.cuda.synchronize()
        ok = same(p0.cpu().numpy(), p1.cpu().numpy()) and torch.equal(n0, n1)
        return ok and (d0 is None or same(d0.cpu().numpy(), d1.cpu().numpy()))


def compare(name, h, p, vals, T, widest):
    d = Dev(h, p, vals, T, seed=T)
    for _ in range(3):  # warm-up of the shape, both paths
        d.time("waves"), d.time("fused")
    reps = 21 if d.K < 256 else 7
    t = {"waves": [], "fused": []}
    launches = {}
    for _ in range(reps):
        for path in ("waves", "fused"):
            ms, n = d.time(path)
            t[path].append(ms)
            launches[path] = n
    K = d.K
    # derived from the registers and fused_on's rule, not read from the launch
    grid = max(1, min(per_sm * sms, -(-widest * K // THREADS))) if per_sm else None
    emit({"case": name, "K": K, "T": T, "reps": reps, "waves_ms": median(t["waves"]), "fused_ms": median(t["fused"]),
          "waves_min_ms": min(t["waves"]), "fused_min_ms": min(t["fused"]), "speedup": median(t["waves"]) / median(t["fused"]),
          "launches": launches, "grid_derived": grid, "bitwise_equal": d.equal()})


def host_fused_api(hl):
    hl.gcs_host_program_run_fused.argtypes = [C.c_void_p, C.c_int64, C.POINTER(C.c_double), C.c_int, C.POINTER(C.c_double),
                                              C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_uint32), C.c_int,
                                              C.POINTER(C.c_int64)]
    return hl


for name, n, seed in (("configs[3] linkage100k", 100000, 4), ("linkage20k", 20000, 6)):
    el, edges = S.make_linkage(n, seed=seed)
    prog = P.Program(el, edges)
    assert prog.rc == 0, prog.error
    p = R.Arrays.from_desc(prog.desc())
    base = P.sketch_values(edges)
    widest = max(int(p.offsets[R.KINDS * (w + 1)] - p.offsets[R.KINDS * w]) for w in range(p.n_waves))
    emit({"case": name, "waves": p.n_waves, "rows": int(p.n_rows), "slots": p.n_slots, "widest_wave": widest})
    h = C.c_void_p()
    assert lib.gcs_b200_program_create(C.byref(p.desc()), 0, C.byref(h)) == 0, lib.gcs_b200_last_error()
    for K in (1, 4, 16, 64, 256, 1024):
        compare(name, h, p, values(p, base, K, seed=K), 0, widest)
    for K in (1, 16):
        for T in (1, 8, 32):
            compare(name, h, p, values(p, base, K, seed=K), T, widest)
    lib.gcs_b200_program_destroy(h)
    # the host clock of SketchProgram::run against runFused at K = 1 (radians, pageable tables)
    hl = host_fused_api(H.load())
    vals = base[None, :].copy()
    pos, dpos = np.zeros((1, p.n_slots, 4)), np.zeros((1, p.n_slots, 4, 1))
    nc, stats = np.zeros(1, dtype=np.uint32), np.zeros(7, dtype=np.int64)
    clock = {"run": [], "runFused": []}
    for i in range(23):
        for path in ("run", "runFused"):
            t0 = time.perf_counter()
            if path == "run":
                rc, want, wnc, _ = prog.run(vals)
            else:
                rc = hl.gcs_host_program_run_fused(prog.handle, 1, H._dp(vals), 0, None, H._dp(pos), H._dp(dpos),
                                                   nc.ctypes.data_as(C.POINTER(C.c_uint32)), 1, stats.ctypes.data_as(C.POINTER(C.c_int64)))
            dt = time.perf_counter() - t0
            assert rc == 0, H.last_error()
            if i >= 3:
                clock[path].append(dt * 1e3)
    emit({"case": name, "K": 1, "host_clock": True, "run_ms": median(clock["run"]), "runFused_ms": median(clock["runFused"]),
          "bitwise_equal": same(pos, want) and bool(np.array_equal(nc, wnc))})

if len(sys.argv) > 1:
    os.makedirs(sys.argv[1], exist_ok=True)
    with open(os.path.join(sys.argv[1], "sketch_program_fused_bench.jsonl"), "w") as f:
        for d in lines:
            f.write(json.dumps(d) + "\n")
