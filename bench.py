#!/usr/bin/env python
"""bench.py — sub-system Newton solves/sec on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
  python bench.py --gpus 1 --steps K --dump-outputs DIR    # + the outputs of the last timed step as DIR/*.npy
  python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path, host cores

Workload of the line (config.workload): BASELINE.json configs[1] — 2^20 independent synthetic
triangle clusters per GPU, half K1 (distance+distance: ZeroFixedPoints / TwoFixedPointsDistance
shapes), half K5 (angle + unit normal), one solve2D-equivalent each (2 seeds, reference defaults) +
root selection (+ line reconstruction for K5).  A step = one pass over that batch = one K1 launch +
one K5 launch.  Weak scaling: rank r owns instances [r*2^19, (r+1)*2^19) of each kind's index
space; no data-path collective (NCCL only carries the barrier and the max-over-ranks of the time).

`value`   whole-job solves/s with the batch resident in HBM; a step is one gcs_b200_solve_many call
          (both launches as one job), CUDA events around it on the launching stream, summed over
          the steps, max over ranks; L2 flushed between steps.  `sequential_launches` = the two
          launches one after the other, each between its own events (what `roofline` is quoted on).
          Kernel class: config.variant (the opt-in contracted kernels by default; the library
          default = bit-identical kernels is timed beside it under `bit_identical`).
`e2e`     the same metric through the host-buffer C-ABI calls (gcs_b200_solve_host_async per batch
          + gcs_b200_wait): pinned HOST inputs and outputs, H2D + kernels + D2H inside the region;
          batches in the shape the packer emits them (anchor columns of the zero-fixed solvers
          NULL); `e2e.pcie` = copy-only ceiling of the same byte counts, probed in the same run.
`roofline` the dominant kernel (K1): algorithmic FP64 flops (work model of DESIGN.md section 3,
          from the MEASURED iteration counts) / its event-timed duration, against the DFMA peak
          measured live by gcs_b200_fp64_probe (MEASURED_PEAKS.json has no FP64 figure); the HBM
          side is reported beside it against MEASURED_PEAKS.json.
`configs` the other BASELINE configs, each measured in this run: multistart8 (configs[2]),
          sweep64m (configs[4]: 2^26 instances sharded over the N ranks, strong scaling), kinds
          (K2 / K3 / K4 kernel lines; K4 is the HBM-bound kind), sketch100k (configs[3] through
          GeometricConstraintSystem), sharded (N > 1: gcs_b200_solve_sharded in ONE process over
          the N devices, checked against one device).
`cpu_baseline` / `--impl reference`  the reference's own solve2D + primitives + heuristics sources
          (oracle/_ref, built from /root/reference against stand-in Eigen/autodiff headers) where
          that library is present, else the restated C oracle; all host threads.
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib
import json
import os
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_PER_GPU = 1 << 20
METRIC = "subsystem Newton solves/sec"
UNIT = "solves/s"
WORKLOAD = ("configs[1]: 2^20 synthetic triangle clusters per GPU (2^19 K1 distance-distance + 2^19 K5 "
            "angle-normal), 2 seeds each, FP64")
VARIANT_NAMES = {0: "default", 1: "static", 2: "refill", 3: "sorted", 4: "pair", 5: "contracted", 6: "contracted-static",
                 7: "contracted-sorted"}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--variant", type=int, default=5,
                    help="5 (default) contracted arithmetic: discrete outputs identical to the reference, coordinates to 1e-9 "
                         "(6 static / 7 sorted); 0 the library default = bit-identical kernels (1 static, 2 refill, "
                         "3 sorted, 4 pair).  With a contracted variant the bit-identical default is timed beside it.")
    ap.add_argument("--n", type=int, default=N_PER_GPU, help="solves per GPU (default 2^20)")
    ap.add_argument("--cpu-seconds", type=float, default=8.0, help="CPU time of the cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="only the configs[1] line (skip the `configs` key)")
    ap.add_argument("--workload", default="configs1", choices=["configs1", "multistart8", "sweep64m"],
                    help="configs1 = the bench line (BASELINE configs[1], with the other configs under `configs`); "
                         "multistart8 / sweep64m: that config alone as the line")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the line's timed path returned in its last step as DIR/<name>.npy "
                         "(float64 coordinates, float32 roots / update counts / flags; rank 0's batches; at most 64 MB, a fixed "
                         "seeded sample of instances beyond that), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "configs1"):
        ap.error("--dump-outputs writes the outputs of the configs1 line of the b200 arm")
    return args


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def load_traffic(lib):
    """Per-launch DRAM bytes / executed flops of the dominant kernel from the last committed
    `ncu --set full` capture (profiles/traffic.json).  The capture names the source hash of the
    library it was taken from; `stale` says whether the library running now is another build."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        t = json.load(open(p))
    except Exception:
        return {}, None
    now = lib.gcs_b200_version().decode()
    stale = None
    if t.get("_src_hash"):
        stale = t["_src_hash"] not in now
    return t, stale


class ClockSampler:
    """Polls NVML for SM clock + throttle reasons while a region runs."""

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self.period = float(os.environ.get("GCS_BENCH_CLOCK_PERIOD", "0.001"))
        self._stop = threading.Event()
        self._in_region = False
        self.region = []
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None
        self.t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self.nv
        names = {}
        if nv:
            for k in dir(nv):
                if k.startswith("nvmlClocksEventReason") or k.startswith("nvmlClocksThrottleReason"):
                    v = getattr(nv, k)
                    if isinstance(v, int) and v not in (0,):
                        names.setdefault(v, k.replace("nvmlClocksEventReason", "").replace("nvmlClocksThrottleReason", ""))
        while not self._stop.is_set():
            if nv:
                try:
                    mhz = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
                    try:
                        r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                    except Exception:
                        r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                    self.samples.append(mhz)
                    if self._in_region:
                        self.region.append(mhz)
                        for bit, nm in names.items():
                            if r & bit and nm not in ("GpuIdle", "None", "All"):
                                self.reasons.add(nm)
                except Exception:
                    pass
            time.sleep(self.period)

    def start(self):
        self.t.start()

    def enter(self):
        self._in_region = True

    def leave(self):
        self._in_region = False

    def stop(self):
        self._stop.set()
        self.t.join(timeout=1.0)
        src = self.region if self.region else self.samples
        return {
            "sm_mhz": float(np.median(src)) if src else None,
            "sm_max_mhz": self.max_mhz,
            "reasons": sorted(self.reasons),
            "samples_in_timed_region": len(self.region),
        }


def make_batches(synth, n, rank):
    half = n // 2
    first = rank * half
    return [synth.make_pp(half, first=first), synth.make_ang(half, first=first)]


DUMP_LIMIT = 60 * 10**6  # bytes of array data: with the .npy headers a dump stays under 64 MB
OUT_NAMES = {1: ("x", "y"), 5: ("p1x", "p1y", "p2x", "p2y")}  # include/gcs_b200.h: point kinds x,y; line kinds p1, p2


def dump_outputs(path, dbs):
    """Writes the outputs of the device batches `dbs` as path/k<kind>_<name>.npy: the solved coordinates
    (float64), the chosen root and, per seed, the update count and the convergence flag (float32, [n_seeds][n]).
    Where all of it would exceed DUMP_LIMIT, every array of a kind keeps the same fixed seeded sample of
    instances, whose indices are written as k<kind>_index.npy (float64)."""
    total = sum(d.n * (8 * len(d.out) + 4 + 8 * d.n_seeds) for d in dbs)
    # the share of every kind's instances kept, the 8-byte index of each kept instance included
    keep = DUMP_LIMIT / (total + 8 * sum(d.n for d in dbs)) if total > DUMP_LIMIT else None
    os.makedirs(path, exist_ok=True)
    written = 0
    for d in dbs:
        idx = None
        if keep is not None:
            idx = np.sort(np.random.default_rng(d.kind).choice(d.n, int(d.n * keep), replace=False))
        arrays = {name: col.cpu().numpy() for name, col in zip(OUT_NAMES[d.kind], d.out)}
        arrays["root_index"] = d.root_index.cpu().numpy().astype(np.float32)
        arrays["iters"] = d.iters.cpu().numpy().astype(np.float32)
        arrays["converged"] = d.converged.cpu().numpy().astype(np.float32)
        for name, a in arrays.items():
            a = a if idx is None else a[..., idx]
            np.save(os.path.join(path, f"k{d.kind}_{name}.npy"), np.ascontiguousarray(a))
            written += a.nbytes
        if idx is not None:
            np.save(os.path.join(path, f"k{d.kind}_index.npy"), idx.astype(np.float64))
            written += 8 * idx.size
    assert written <= DUMP_LIMIT, written


def base_config(args):
    """`config` is built from the command line alone, so both arms print the same dict (the driver
    compares them); what a run found out about itself goes under `run`."""
    v = args.variant
    return {"workload": WORKLOAD, "solves_per_gpu": args.n, "kinds": "K1 x n/2 + K5 x n/2", "seeds": 2, "dtype": "f64",
            "l2": "GPU arm: 256 MiB flush write between timed steps; CPU arm: a step's 113 MB of columns exceed the host caches",
            "gpu_kernel_class": (f"{VARIANT_NAMES.get(v, v)}: the opt-in GCS_VARIANT_CONTRACTED kernels (iteration counts, flags, roots "
                                 "identical to the reference, coordinates to 1e-9) - NOT the library default; the default bit-identical "
                                 "kernels are timed in the same run under `bit_identical`" if v >= 5 else
                                 f"{VARIANT_NAMES.get(v, v)}: bit-identical to the reference arithmetic")}


# --------------------------------------------------------------------------------------------
# CPU leg: the reference's own sources where oracle/_ref exists, else the restated oracle
# --------------------------------------------------------------------------------------------
def cpu_backend():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import __graft_entry__ as g
    g.build_oracle()
    try:
        import ref_lib as R
        if R.available():
            R.load()
            return ("reference", lambda b, t: R.solve_batch(b, count_iters=False, threads=t), R.load().gcs_ref_max_threads(),
                    "the reference's solve2D / equation primitives / heuristics sources compiled from /root/reference "
                    "(oracle/_ref; Eigen and autodiff are the stand-in headers of oracle/ref_shim)")
    except Exception:
        pass
    import oracle_lib as O
    return ("port", lambda b, t: O.solve(b, t), O.max_threads(),
            "restated C oracle (oracle/gcs_oracle.c): oracle/_ref is not present on this box")


def host_threads():
    # every core this process may run on (torchrun exports OMP_NUM_THREADS=1; the CPU arm is meant
    # to use the whole host)
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_rate(gcs, seconds, threads=0):
    """Solves/s of the CPU path on a bounded sample of the same workload (same generators, same
    K1/K5 mix), repeated until about `seconds` of wall time have been spent."""
    synth = gcs.synth
    kind, solve, cores, what = cpu_backend()
    if threads < 1:
        threads = host_threads()
    cores = threads
    m = 1 << 15
    bs = [synth.make_pp(m).alloc_outputs(), synth.make_ang(m).alloc_outputs()]
    for b in bs:  # warm the threads and the pages
        solve(b, threads)
    done, t_total, reps = 0, 0.0, 0
    while t_total < seconds or reps < 2:
        t0 = time.perf_counter()
        for b in bs:
            solve(b, threads)
        t_total += time.perf_counter() - t0
        done += 2 * m
        reps += 1
    sample = f"{reps} x ({m} K1 + {m} K5) solves of the bench generators, {cores} threads, {t_total:.1f} s; {what}"
    return done / t_total, cores, kind, sample


def faithful_rate(n_leaves=8192):
    """The reference's REAL per-leaf path: classifyAndSolve on ConstraintGraphs of shared_ptr
    elements (matches() probes, role assignment, solve2D through autodiff, heuristics, write-back,
    the two std::cerr prints per leaf, here sent to /dev/null), one thread as in the reference.
    n_leaves zero-fixed triangles (K1) + n_leaves zero-fixed line-line-point angle leaves (K5);
    the timed call also builds each leaf's 3-node graph.  None where oracle/_ref is absent."""
    try:
        import ref_lib as R
        if not R.available():
            return None
        import math
        rng = np.random.default_rng(5)
        el, lv = [], []
        for i in range(n_leaves):
            d = rng.uniform(10, 500)
            px, py = rng.uniform(-300, 800), rng.uniform(5, 500) * (1 if rng.random() < 0.5 else -1)
            pts = [(0.0, 0.0), (d, 0.0), (px, py)]
            b = len(el)
            el += [{"type": 0, "canvas": [float(x + 500), float(y + 500)]} for x, y in pts]
            lv.append({"elems": [b, b + 1, b + 2], "edges": [
                {"a": b, "b": b + 1, "type": 0, "value": float(d)},
                {"a": b, "b": b + 2, "type": 0, "value": float(math.hypot(px, py))},
                {"a": b + 1, "b": b + 2, "type": 0, "value": float(math.hypot(px - d, py))}]})
        for i in range(n_leaves):
            l1 = rng.uniform(50, 500)
            ang = rng.uniform(math.radians(5), math.radians(175))
            l2 = rng.uniform(50, 500)
            ox, oy = rng.uniform(-100, 100), rng.uniform(-100, 100)
            line1 = [0.0, 0.0, l1, 0.0]
            line2 = [ox, oy, ox + l2 * math.cos(ang), oy + l2 * math.sin(ang)]
            p = (rng.uniform(-200, 200), rng.uniform(20, 300))
            ex, ey = line2[2] - line2[0], line2[3] - line2[1]
            d2 = abs(ex * (p[1] - line2[1]) - ey * (p[0] - line2[0])) / math.hypot(ex, ey)
            b = len(el)
            el += [{"type": 1, "canvas": [float(v + 500) for v in line1]}, {"type": 1, "canvas": [float(v + 500) for v in line2]},
                   {"type": 0, "canvas": [float(p[0] + 500), float(p[1] + 500)]}]
            lv.append({"elems": [b, b + 1, b + 2], "edges": [
                {"a": b, "b": b + 1, "type": 1, "value": float(ang), "flip": False},
                {"a": b + 2, "b": b, "type": 0, "value": float(abs(p[1]))},
                {"a": b + 2, "b": b + 1, "type": 0, "value": float(d2)}]})
        devnull = os.open(os.devnull, os.O_WRONLY)
        saved = os.dup(2)
        sys.stderr.flush()
        os.dup2(devnull, 2)
        try:
            R.leaves_solve(el[:30], lv[:10])  # warm
            t0 = time.perf_counter()
            rc, status, _ = R.leaves_solve(el, lv)
            dt = time.perf_counter() - t0
        finally:
            os.dup2(saved, 2)
            os.close(devnull)
            os.close(saved)
        # the ctypes marshalling of the element / edge arrays happens inside leaves_solve too: time it alone and subtract
        t1 = time.perf_counter()
        import host_lib as H
        H.to_c(el, [], R.RefElement, R.RefEdge)
        H.to_c([], [e for lf in lv for e in lf["edges"]], R.RefElement, R.RefEdge)
        H.from_c(el, H.to_c(el, [], R.RefElement, R.RefEdge)[0])
        marshal = time.perf_counter() - t1
        solve_s = max(dt - marshal, 1e-9)
        ok = int(sum(1 for s in status if s == 0))
        return {"value": 2 * n_leaves / solve_s, "unit": UNIT, "cores": 1, "kind": "reference",
                "sample": f"{n_leaves} ZeroFixedPointsTriangle + {n_leaves} ZeroFixedLLPAngleTriangle leaves through the reference's own "
                          f"classifyAndSolve on ConstraintGraphs (its per-leaf std::cerr prints to /dev/null), single thread as the "
                          f"reference runs; {solve_s:.2f} s after subtracting {marshal:.2f} s of Python marshalling; {ok} of "
                          f"{2 * n_leaves} leaves returned Success; includes building each leaf's 3-node graph"}
    except Exception as ex:  # pragma: no cover - diagnostic leg only
        return {"error": repr(ex)[:200]}


def run_reference(args, rank):
    """--impl reference: the CPU path on the box's host cores, rank 0 only.  A step = the FULL
    configs[1] batch (n/2 K1 + n/2 K5 solves) on all host threads; ms_per_step is measured."""
    if rank != 0:
        return
    gcs = importlib.import_module("2d_geometry_constraint_solver_b200")
    kind, solve, _, what = cpu_backend()
    threads = host_threads()
    n = args.n
    bs = [b.alloc_outputs() for b in make_batches(gcs.synth, n, 0)]
    for b in bs:
        b.want_cand = False
    ts = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        for b in bs:
            solve(b, threads)
        dt = time.perf_counter() - t0
        if i >= args.warmup:
            ts.append(dt)
    total = float(np.sum(ts))
    v = n * len(ts) / total
    sample = f"{len(ts)} steps x ({n // 2} K1 + {n // 2} K5) solves = the full configs[1] batch per step, {threads} threads; {what}"
    out = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": total / len(ts) * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": base_config(args),
        "note": "CPU path on the box's host cores, rank 0 only (one host serves all N GPUs: the value does not scale with N)",
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": threads, "kind": kind, "sample": sample},
        "cpu_baseline_faithful": faithful_rate(),
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(out), flush=True)


# --------------------------------------------------------------------------------------------
# shared measurement helpers (GPU arm)
# --------------------------------------------------------------------------------------------
class Ctx:
    def __init__(self, args, rank, local_rank, world):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.args, self.rank, self.local_rank, self.world = args, rank, local_rank, world
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.gloo = None
        if world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
            self.gloo = dist.new_group(backend="gloo")  # host-side waits that must not occupy the GPUs
        self.gcs = importlib.import_module("2d_geometry_constraint_solver_b200")
        self.capi, self.synth = self.gcs.capi, self.gcs.synth
        self.capi.init([local_rank])
        self.lib = self.capi.load()
        self.stream = torch.cuda.current_stream(self.dev)
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)  # > 126 MB L2
        self.warmup = max(args.warmup, 3)
        self._dfma = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize(self.dev)

    def host_barrier(self):
        if self.world > 1:
            self.dist.barrier(group=self.gloo)

    def max_over_ranks(self, v):
        t = self.torch.tensor([float(v)], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def all_ok(self, ok):
        t = self.torch.tensor([1 if ok else 0], device=self.dev, dtype=self.torch.int32)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return int(t.item()) == 1

    def dfma_peak(self):
        if self._dfma is None:
            self._dfma = self.lib.gcs_b200_fp64_probe(self.local_rank, 0)
        return self._dfma

    def time_launches(self, dbs, steps, warmup=3):
        """`steps` passes over the device-resident batches `dbs`, L2 flushed between passes, CUDA
        events around every launch on the launching stream.  Returns ms[len(dbs)][steps]."""
        torch = self.torch
        for _ in range(warmup):
            self.flush.fill_(1)
            for d in dbs:
                d.solve()
        self.barrier()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(len(dbs) + 1)] for _ in range(steps)]
        for k in range(steps):
            self.flush.fill_(k & 0xFF)  # evict the batch from L2 between timed steps (outside the events)
            evs[k][0].record(self.stream)
            for j, d in enumerate(dbs):
                d.solve()
                evs[k][j + 1].record(self.stream)
        self.barrier()
        return np.array([[e[j].elapsed_time(e[j + 1]) for e in evs] for j in range(len(dbs))])

    def contract_check(self, a, b):
        """Contracted batch `a` against bit-identical batch `b` (same inputs), on the device."""
        torch = self.torch
        same = bool(torch.equal(a.iters, b.iters)) and bool(torch.equal(a.converged, b.converged)) \
            and bool(torch.equal(a.root_index, b.root_index))
        cols = [c.abs() for c in a.cols if c is not None]
        scale = torch.clamp(torch.stack(cols).max(dim=0).values, min=1.0)
        worst = 0.0
        for x, y in zip(a.out, b.out):
            worst = max(worst, float(((x - y).abs() / torch.maximum(scale, y.abs())).max().item()))
        return same, worst

    def rerun_stats(self, dbs):
        st = (C.c_uint64 * 8)()
        self.lib.gcs_b200_contracted_stats_ex(self.local_rank, st, 1)
        for d in dbs:
            d.solve()
        self.lib.gcs_b200_contracted_stats_ex(self.local_rank, st, 1)
        return {"runs_per_step": int(sum(d.n * d.n_seeds for d in dbs)), "conditioning": int(st[0]), "selection": int(st[1]),
                "bounce": int(st[2]), "band": int(st[3]), "cap": int(st[4]), "non_finite": int(st[5])}


def pinned_batch(ctx, h, want_flags):
    """`h` (HostBatch, possibly with NULL anchor columns) re-homed in page-locked memory from the
    library's own allocator: one [present columns][n] slab up, one [out columns][n] slab down."""
    capi = ctx.capi
    keep = []
    pres = [c for c, col in enumerate(h.cols) if col is not None]
    slab = capi.PinnedArray((len(pres), h.n)); keep.append(slab)
    for j, c in enumerate(pres):
        slab.array[j] = h.cols[c]
    cols = [None] * len(h.cols)
    for j, c in enumerate(pres):
        cols[c] = slab.array[j]
    code = capi.PinnedArray(h.n, np.uint8); keep.append(code)
    code.array[...] = h.code
    hb = capi.HostBatch(h.kind, h.n_seeds, cols, code.array, None, h.variant, want_cand=False)
    oslab = capi.PinnedArray((capi.OUT_COLS[h.kind], h.n)); keep.append(oslab)
    hb.out = [oslab.array[c] for c in range(oslab.array.shape[0])]
    root = capi.PinnedArray(h.n, np.uint8); keep.append(root)
    hb.root_index = root.array
    hb.cand = None
    if want_flags:
        it = capi.PinnedArray((h.n_seeds, h.n), np.int16); keep.append(it)
        cv = capi.PinnedArray((h.n_seeds, h.n), np.uint8); keep.append(cv)
        hb.iters, hb.converged = it.array, cv.array
    else:
        hb.iters = hb.converged = None
    hb._keep = keep
    return hb


def batch_d2h_bytes(capi, b):
    return capi.OUT_COLS[b.kind] * 8 * b.n + (b.n if b.root_index is not None else 0) \
        + (b.n_seeds * 2 * b.n if b.iters is not None else 0) + (b.n_seeds * b.n if b.converged is not None else 0)


def time_e2e(ctx, batches, steps):
    """Wall-clock solves/s of `steps` passes: gcs_b200_solve_host_async per batch + gcs_b200_wait."""
    capi = ctx.capi
    # the C descriptors are built once (a caller in C has them on its stack): the loop below is the
    # C-ABI calls and nothing else
    lib, dev = ctx.lib, ctx.local_rank
    for b in batches:
        if not b.out:
            b.alloc_outputs()
    descs = [b.cbatch() for b in batches]
    refs = [C.byref(d) for d in descs]

    def one():
        for r in refs:
            rc = lib.gcs_b200_solve_host_async(r, dev)
            if rc:
                capi.check(rc, "gcs_b200_solve_host_async")
        capi.check(lib.gcs_b200_wait(dev), "gcs_b200_wait")

    for _ in range(3):
        one()
    l1 = ctx.lib.gcs_b200_launch_count()
    ctx.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        one()
    ctx.barrier()
    dt = time.perf_counter() - t0
    launches = ctx.lib.gcs_b200_launch_count() - l1
    return ctx.max_over_ranks(dt), dt, int(launches)


# --------------------------------------------------------------------------------------------
# the other BASELINE configs (each also runnable alone with --workload)
# --------------------------------------------------------------------------------------------
def bench_multistart(ctx, steps):
    """configs[2]: 2^20 K1 clusters per GPU x 8 initial guesses, orientation-based root selection."""
    capi, synth, args = ctx.capi, ctx.synth, ctx.args
    n = 1 << 20
    hb = synth.make_pp(n, first=ctx.rank * n, n_seeds=8)
    hb.variant = args.variant
    db = capi.DeviceBatch(hb, ctx.dev, want_cand=False, variant=args.variant)
    l0 = ctx.lib.gcs_b200_launch_count()
    ms = ctx.time_launches([db], steps)[0]
    launches = ctx.lib.gcs_b200_launch_count() - l0
    total_ms = ctx.max_over_ranks(float(ms.sum()))
    out = _extra_line(ctx, db, ms, total_ms, n * ctx.world, n, "weak",
                      "configs[2]: 2^20 K1 clusters per GPU x 8 initial guesses, orientation-based root selection", 8, launches, steps)
    contract = None
    if args.variant >= 5:
        db0 = capi.DeviceBatch(hb, ctx.dev, want_cand=False, variant=0)
        ms0 = ctx.time_launches([db0], max(2, steps // 2), warmup=1)[0]
        same, worst = ctx.contract_check(db, db0)
        contract = {"iters_flags_roots_equal": same, "max_rel_coordinate_error": worst, "tolerance": 1e-9, "solves_compared": n,
                    "bit_identical_launch_ms": float(ms0.mean())}
        del db0
    out["contract_check_rank0"] = contract
    # end to end: pinned host columns -> results in pinned host memory
    pb = pinned_batch(ctx, hb, want_flags=False)
    e2e_steps = 4
    t_max, _, _ = time_e2e(ctx, [pb], e2e_steps)
    out["e2e"] = {"value": n * ctx.world * e2e_steps / t_max, "unit": UNIT, "h2d_bytes_per_step": pb.input_bytes(),
                  "d2h_bytes_per_step": batch_d2h_bytes(capi, pb), "api": "gcs_b200_solve_host_async + gcs_b200_wait (pinned)"}
    return out


def bench_sweep(ctx, steps):
    """configs[4]: 2^26 perturbed K1 instances generated on the device, sharded by index over the ranks."""
    capi, synth, args = ctx.capi, ctx.synth, ctx.args
    torch = ctx.torch
    shard = importlib.import_module("2d_geometry_constraint_solver_b200.shard")
    n_total = 1 << 26
    lo, hi = shard.shard_range(n_total, ctx.rank, ctx.world)
    n = hi - lo
    db = capi.DeviceBatch.empty(capi.KIND_PP, 2, n, ctx.dev, variant=args.variant)
    ptrs = (C.c_void_p * 6)(*[c.data_ptr() for c in db.cols])

    def gen():
        capi.check(ctx.lib.gcs_b200_synth_pp(ctx.local_rank, C.c_void_p(ctx.stream.cuda_stream), synth.BASE_SEED, lo, n, 4096, ptrs,
                                             C.c_void_p(db.code.data_ptr())), "gcs_b200_synth_pp")
    gen()
    l0 = ctx.lib.gcs_b200_launch_count()
    ms = ctx.time_launches([db], steps, warmup=2)[0]
    launches = ctx.lib.gcs_b200_launch_count() - l0
    total_ms = ctx.max_over_ranks(float(ms.sum()))
    out = _extra_line(ctx, db, ms, total_ms, n_total, n, "strong",
                      "configs[4]: parametric sweep, 2^26 K1 instances = 4096 base clusters x 16384 perturbations (+-5% on ra, rb, d), "
                      "generated on the device, sharded by index over the ranks", 2, launches, steps)
    contract = None
    if args.variant >= 5:
        db0 = capi.DeviceBatch.empty(capi.KIND_PP, 2, n, ctx.dev, variant=0)
        for dst, src in zip(db0.cols, db.cols):
            dst.copy_(src)
        db0.code.copy_(db.code)
        db0.solve()
        torch.cuda.synchronize(ctx.dev)
        same, worst = ctx.contract_check(db, db0)
        contract = {"iters_flags_roots_equal": same, "max_rel_coordinate_error": worst, "tolerance": 1e-9, "solves_compared": int(n)}
        del db0
    out["contract_check_rank0"] = contract
    # end to end: generation + solve + (x, y, root) to pinned host memory
    outs = [torch.empty(n, dtype=torch.float64, pin_memory=True) for _ in range(2)]
    roots = torch.empty(n, dtype=torch.uint8, pin_memory=True)

    def e2e_step():
        gen()
        db.solve()
        for o, dcol in zip(outs, db.out):
            o.copy_(dcol, non_blocking=True)
        roots.copy_(db.root_index, non_blocking=True)
        torch.cuda.synchronize(ctx.dev)
    e2e_step()
    ctx.barrier()
    t0 = time.perf_counter()
    e2e_steps = 2
    for _ in range(e2e_steps):
        e2e_step()
    ctx.barrier()
    t_max = ctx.max_over_ranks(time.perf_counter() - t0)
    out["e2e"] = {"value": n_total * e2e_steps / t_max, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 17 * n,
                  "api": "gcs_b200_synth_pp + gcs_b200_solve + D2H of (x, y, root) to pinned memory"}
    return out


def _extra_line(ctx, db, ms, total_ms, n_total, n_rank, scaling, name, n_seeds, launches, steps):
    synth = ctx.synth
    torch = ctx.torch
    it = db.iters
    w = float((it.to(torch.int64) + 1).sum().item()) * synth.F_EVAL[1] + n_rank * synth.F_SELECT[1]
    ach = w / (float(ms.mean()) * 1e-3) / 1e12
    dfma = ctx.dfma_peak()
    return {
        "metric": METRIC, "value": n_total * steps / (total_ms * 1e-3), "unit": UNIT, "n_gpus": ctx.world, "steps": steps,
        "ms_per_step": total_ms / steps, "scaling": scaling,
        "config": {"workload": name, "solves_total": n_total, "solves_rank0": int(n_rank), "l2": "256 MiB flush write between timed steps",
                   "converged_fraction_rank0": float(db.converged.to(torch.float32).mean().item()),
                   "mean_iters_per_seed_rank0": float(it.to(torch.float32).mean().item()),
                   "variant": VARIANT_NAMES[ctx.args.variant]},
        "gpu_launches": int(launches),
        "roofline": {"kernel": ctx.lib.gcs_b200_kernel_name(1, n_seeds, ctx.args.variant).decode(), "bound": "fp64",
                     "achieved": ach, "peak": dfma, "unit": "TFLOP/s", "frac": ach / dfma if dfma > 0 else None, "traffic": None,
                     "launch_ms_rank0": float(ms.mean()), "algorithmic_flops_per_launch_rank0": w},
    }


def bench_kinds(ctx, steps=10):
    """K2 / K3 / K4 kernel lines (2^19 sub-systems each, device-resident, L2 flushed): launch time,
    algorithmic flops and bytes against the FP64 and HBM peaks, for the kernel class of the line and
    for the bit-identical default.  K4 (two linear equations: two updates per seed) is the
    HBM-leaning kind; its batch has no parallel line pairs (those never converge and run to the cap)."""
    capi, synth, args = ctx.capi, ctx.synth, ctx.args
    peaks, _ = load_peaks()
    n = 1 << 19
    out = {}
    for kind in (2, 3, 4):
        hb = synth.make_pll(n, parallel_every=0) if kind == 4 else synth.make(kind, n)
        row = {"n": n}
        dbs = {}
        for label, variant in ([("line_variant", args.variant)] + ([("bit_identical", 0)] if args.variant >= 5 else [])):
            db = dbs[label] = capi.DeviceBatch(hb, ctx.dev, want_cand=False, variant=variant)
            ms = ctx.time_launches([db], steps, warmup=2)[0]
            it = db.iters.cpu().numpy()
            w = synth.algorithmic_flops(kind, it)
            b = db.algorithmic_bytes()
            t = float(np.mean(ms)) * 1e-3
            dfma = ctx.dfma_peak()
            row[label] = {"kernel": ctx.lib.gcs_b200_kernel_name(kind, 2, variant).decode(), "launch_ms": t * 1e3,
                          "fp64_tflops": w / t / 1e12, "fp64_frac": w / t / 1e12 / dfma if dfma > 0 else None,
                          "hbm_gbs": b / t / 1e9, "hbm_frac": b / t / 1e9 / peaks.get("hbm_gbs", 6650.0),
                          "algorithmic_flops_per_launch": w, "algorithmic_bytes_per_launch": b,
                          "mean_iters_per_seed": float(it.mean())}
        if "bit_identical" in dbs:
            same, worst = ctx.contract_check(dbs["line_variant"], dbs["bit_identical"])
            row["contract_check"] = {"iters_flags_roots_equal": same, "max_rel_coordinate_error": worst}
        if kind == 4:  # the HBM-bound kind at a size where the launch's fixed cost no longer shows
            del dbs, db
            n4 = 1 << 22
            db4 = capi.DeviceBatch(synth.make_pll(n4, parallel_every=0), ctx.dev, want_cand=False, variant=args.variant)
            t4 = float(np.mean(ctx.time_launches([db4], steps, warmup=2)[0])) * 1e-3
            b4 = db4.algorithmic_bytes()
            row["at_4m"] = {"n": n4, "kernel": ctx.lib.gcs_b200_kernel_name(kind, 2, args.variant).decode(), "launch_ms": t4 * 1e3,
                            "hbm_gbs": b4 / t4 / 1e9, "hbm_frac": b4 / t4 / 1e9 / peaks.get("hbm_gbs", 6650.0),
                            "algorithmic_bytes_per_launch": b4}
            del db4
        row["bound"] = "hbm" if kind == 4 else "fp64"
        out[f"K{kind}"] = row
    return out


def bench_sketch(ctx, n_points=100000):
    """configs[3]: one rigidly well-constrained linkage of n_points points through the host mirror
    (GeometricConstraintSystem -> decomposition -> wave-batched solveGcs on the device)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import host_lib as H
    import sketch_gen as S
    el, edges = S.make_linkage(n_points, seed=4)
    H.system_solve_ex(el[:2000], [e for e in edges if max(e["a"], e["b"]) < 2000])  # warm-up (context, arena)
    best = None
    for _ in range(4):  # the first full-size call grows the host mirror's pooled buffers
        t0 = time.perf_counter()
        rc, got, stats = H.system_solve_ex(el, edges)
        wall = time.perf_counter() - t0
        if rc != 0:
            return {"error": H.last_error()}
        if best is None or stats["solve_us"] < best["solve_us"]:
            best = dict(stats, wall_s_incl_python_marshalling=wall)
    # every distance constraint of the sketch must hold in the result
    pos = np.array([g["pos"][:2] for g in got])
    a = np.array([e["a"] for e in edges]); b = np.array([e["b"] for e in edges]); v = np.array([e["value"] for e in edges])
    resid = np.abs(np.hypot(*(pos[a] - pos[b]).T) - v)
    return {"workload": f"configs[3]: linkage of {n_points} points, {len(edges)} distance constraints, through "
                        "GeometricConstraintSystem::solveGeometricConstraintSystem", **best,
            "leaves_per_s_solve": best["leaves"] / (best["solve_us"] * 1e-6),
            "device_share_of_solve": best["device_us"] / max(best["solve_us"], 1),
            "constraints_satisfied_to_1e-6": int((resid <= 1e-6 * np.maximum(1.0, v)).sum()), "constraints": len(edges),
            "max_constraint_residual": float(resid.max())}


def bench_sharded(ctx):
    """N > 1: gcs_b200_solve_sharded inside ONE process (rank 0) over the N devices of the box, checked
    bit for bit against the same batch on one device; the other ranks wait at a host-side barrier."""
    if ctx.world == 1:
        return None
    out = None
    ctx.barrier()
    if ctx.rank == 0:
        capi, synth = ctx.capi, ctx.synth
        try:
            capi.init(list(range(ctx.world)))
            n = 1 << 20
            res = {}
            for kind in (1, 5):
                a = synth.make(kind, n)
                a.variant = ctx.args.variant
                a.want_cand = False
                pa = pinned_batch(ctx, a, want_flags=True)
                capi.solve_sharded(pa, ctx.world)  # warm (arenas on every device)
                t0 = time.perf_counter()
                capi.solve_sharded(pa, ctx.world)
                dt = time.perf_counter() - t0
                b = synth.make(kind, n)
                b.variant = ctx.args.variant
                b.want_cand = False
                pb = pinned_batch(ctx, b, want_flags=True)
                capi.solve_host(pb, ctx.local_rank)
                same = all(np.array_equal(x.view(np.uint64), y.view(np.uint64)) for x, y in zip(pa.out, pb.out)) \
                    and np.array_equal(pa.iters, pb.iters) and np.array_equal(pa.converged, pb.converged) \
                    and np.array_equal(pa.root_index, pb.root_index)
                res[f"K{kind}"] = {"n": n, "devices": ctx.world, "identical_to_one_device": bool(same), "ms": dt * 1e3,
                                   "solves_per_s": n / dt}
            out = res
        except Exception as ex:
            out = {"error": repr(ex)[:300]}
        finally:
            capi.init([ctx.local_rank])
    ctx.host_barrier()
    return out


# --------------------------------------------------------------------------------------------
def _quiet_stdout():
    """Library chatter on file descriptor 1 (NCCL prints its version there on some boxes) goes to
    stderr; the JSON line is the only thing written to the real stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real, "w", buffering=1)


def main():
    args = parse()
    args0 = argparse.Namespace(**vars(args))  # as given on the command line (args.variant changes if the contract check fails)
    _quiet_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    ctx = Ctx(args, rank, local_rank, world)
    dist = ctx.dist
    if args.workload != "configs1":
        line = bench_multistart(ctx, args.steps) if args.workload == "multistart8" else bench_sweep(ctx, args.steps)
        if rank == 0:
            line.update({"warmup": ctx.warmup, "higher_is_better": True, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                         "cpu_baseline": None})
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    capi, synth, lib, dev, stream = ctx.capi, ctx.synth, ctx.lib, ctx.dev, ctx.stream
    n = args.n
    warmup = ctx.warmup
    host = make_batches(synth, n, rank)
    for h in host:
        h.variant = args.variant
    devb = [capi.DeviceBatch(h, dev, want_cand=False, variant=args.variant) for h in host]
    flush = ctx.flush
    barrier = ctx.barrier

    # A step = the whole batch as ONE job through gcs_b200_solve_many (the library runs the K1 and
    # the K5 launch concurrently on its own streams, stream-ordered as a whole on the caller's
    # stream); CUDA events around the call on the launching stream.
    def timed_jobs(dbs, steps, warm):
        for _ in range(warm):
            flush.fill_(1)
            capi.solve_many(dbs)
        barrier()
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(steps)]
        l0 = lib.gcs_b200_launch_count()
        t0 = time.perf_counter()
        for k in range(steps):
            flush.fill_(k & 0xFF)  # evict the batch from L2 between timed steps (outside the events)
            evs[k][0].record(stream)
            capi.solve_many(dbs)
            evs[k][1].record(stream)
        barrier()
        wall = time.perf_counter() - t0
        ms = np.array([e[0].elapsed_time(e[1]) for e in evs])
        return ms, lib.gcs_b200_launch_count() - l0, wall

    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.enter()
    ms_job, launches, t_wall = timed_jobs(devb, args.steps, warmup)
    total_ms = ctx.max_over_ranks(float(ms_job.sum()))
    value = (n * world * args.steps) / (total_ms * 1e-3)

    # ---- the same launches one after the other on one stream, each between its own events: the
    #      per-kernel durations the roofline is quoted on ----
    ms_seq = ctx.time_launches(devb, args.steps, warmup)
    ms_k1, ms_k5 = ms_seq[0], ms_seq[1]
    seq_ms = ctx.max_over_ranks(float((ms_k1 + ms_k5).sum()))
    sequential = {"value": (n * world * args.steps) / (seq_ms * 1e-3), "unit": UNIT, "ms_per_step": seq_ms / args.steps,
                  "note": "the two launches of a step one after the other on one stream (gcs_b200_solve x2), sum of the per-launch event times"}

    # ---- the bit-identical kernels on the same batches, timed the same two ways, and the contract
    #      between the two checked on the full batch (contracted variants only) ----
    bit_identical = None
    violation = None
    if args.variant >= 5:
        devb0 = [capi.DeviceBatch(h, dev, want_cand=False, variant=0) for h in host]
        ms0_job, launches0, _ = timed_jobs(devb0, args.steps, warmup)
        t0_job = ctx.max_over_ranks(float(ms0_job.sum()))
        ms0 = ctx.time_launches(devb0, args.steps, warmup)
        ms0_k1, ms0_k5 = ms0[0], ms0[1]
        t0_sum = ctx.max_over_ranks(float((ms0_k1 + ms0_k5).sum()))
        same, worst = True, 0.0
        for a, b in zip(devb, devb0):
            s_, w_ = ctx.contract_check(a, b)
            same, worst = same and s_, max(worst, w_)
        if os.environ.get("GCS_BENCH_TEST_VIOLATION"):  # exercises the fallback below
            same = False
        if not ctx.all_ok(same and worst <= 1e-9):
            # Never report a number from results that failed their check: the line falls back to the
            # bit-identical kernels (timed above, on the same batches) and says so.
            print(f"[bench] CONTRACT VIOLATED by variant {args.variant} on rank {rank}'s view (discrete outputs equal = {same}, "
                  f"max relative error = {worst:.3e}); reporting the bit-identical kernels instead", file=sys.stderr, flush=True)
            violation = {"variant": args.variant, "iters_flags_roots_equal_rank": same, "max_rel_coordinate_error_rank": worst}
            args.variant = 0
            devb, ms_k1, ms_k5, launches = devb0, ms0_k1, ms0_k5, launches0
            total_ms = t0_job
            value = (n * world * args.steps) / (total_ms * 1e-3)
            sequential["value"], sequential["ms_per_step"] = (n * world * args.steps) / (t0_sum * 1e-3), t0_sum / args.steps
            for h in host:
                h.variant = 0
        bit_identical = {
            "variant": "default (newton_sorted_kernel, literal Householder QR, no contraction): what GCS_VARIANT_DEFAULT and the host mirror run",
            "value": (n * world * args.steps) / (t0_job * 1e-3), "unit": UNIT, "ms_per_step": t0_job / args.steps,
            "sequential_launches": {"value": (n * world * args.steps) / (t0_sum * 1e-3), "ms_per_step": t0_sum / args.steps},
            "k1_launch_ms": float(ms0_k1.mean()), "k5_launch_ms": float(ms0_k5.mean()),
            "contract_check_rank0": {"iters_flags_roots_equal": same, "max_rel_coordinate_error": worst, "tolerance": 1e-9,
                                     "solves_compared": int(sum(d.n for d in devb))},
        }
        if violation is None:
            del devb0

    # devb are the batches `value` was timed on, holding the outputs of their last timed launch (every
    # timed launch of a batch recomputes the same outputs from the same inputs)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, devb)

    # ---- iteration histogram -> algorithmic work of the dominant kernel ----
    it1 = devb[0].iters.cpu().numpy()
    it5 = devb[1].iters.cpu().numpy()
    w_k1 = synth.algorithmic_flops(1, it1)
    w_k5 = synth.algorithmic_flops(5, it5)
    k1_ms = float(np.mean(ms_k1))
    k5_ms = float(np.mean(ms_k5))
    b_k1 = devb[0].algorithmic_bytes()
    b_k5 = devb[1].algorithmic_bytes()

    # ---- end to end through the host-buffer C-ABI calls, pinned host memory.  Batches as the
    #      packer emits them: the zero-fixed (anchored) shapes and the general shapes are different
    #      solvers, hence different batches; the anchor columns are NULL (not stored, not copied).
    #      What comes back is what the reference's solvers produce: the solved coordinates and the
    #      chosen root (solve2D returns no iteration counts / flags, newton_raphson.hpp:97-101). ----
    e2e_batches = []
    for h in host:
        even = np.arange(0, h.n, 2)
        odd = np.arange(1, h.n, 2)
        for part in (h.take(even).anchored(), h.take(odd)):
            part.variant = args.variant
            e2e_batches.append(pinned_batch(ctx, part, want_flags=False))
    # the larger uploads first: what trails the last upload is then the smallest batch's last range
    e2e_batches.sort(key=lambda b: -b.input_bytes())
    h2d = sum(b.input_bytes() for b in e2e_batches)
    d2h = sum(batch_d2h_bytes(capi, b) for b in e2e_batches)
    e2e_steps = max(3, min(args.steps, 20))
    e2e_t, e2e_s, e2e_launches = time_e2e(ctx, e2e_batches, e2e_steps)
    e2e_value = n * world * e2e_steps / e2e_t
    # the e2e results must equal the device-resident ones (same inputs, same kernels)
    for b in e2e_batches:
        src = devb[0] if b.kind == 1 else devb[1]
        sel = slice(0, None, 2) if any(c is None for c in b.cols) else slice(1, None, 2)
        assert np.array_equal(b.out[0], src.out[0].cpu().numpy()[sel]), "e2e coordinates differ from the device-resident run"
        assert np.array_equal(b.root_index, src.root_index.cpu().numpy()[sel]), "e2e roots differ from the device-resident run"
    # the same step in the round-1 wire format (dense 6 / 13 columns, iteration counts and flags
    # downloaded too), for continuity
    dense = [pinned_batch(ctx, h, want_flags=True) for h in host]
    dense_t, _, _ = time_e2e(ctx, dense, max(3, e2e_steps // 2))
    dense_line = {"value": n * world * max(3, e2e_steps // 2) / dense_t, "unit": UNIT,
                  "h2d_bytes_per_step": sum(b.input_bytes() for b in dense), "d2h_bytes_per_step": sum(batch_d2h_bytes(capi, b) for b in dense),
                  "note": "round-1 wire format: anchor columns shipped as zeros, iteration counts and flags downloaded"}
    del dense
    # copy-only ceiling of the same byte counts, all ranks at once (one contiguous copy per direction
    # and the pipeline's own granularity), on the library's copy streams
    barrier()
    probe1 = capi.pcie_probe(local_rank, h2d, d2h, 1, False, 9)
    barrier()
    probe_p = capi.pcie_probe(local_rank, h2d, d2h, 16, False, 9)
    e2e_ms = e2e_t / e2e_steps * 1e3
    best_ms = ctx.max_over_ranks(min(probe1["both_ms_best"], probe_p["both_ms_best"]))
    typical_ms = ctx.max_over_ranks(min(probe1["both_ms_median"], probe_p["both_ms_median"]))
    pcie = {"h2d_gbs_rank0": probe1["h2d_gbs"], "d2h_gbs_rank0": probe1["d2h_gbs"],
            "ceiling_ms_per_step": best_ms, "ceiling_solves_per_s": n * world / (best_ms * 1e-3), "frac_of_ceiling": best_ms / e2e_ms,
            "typical_copy_only_ms_per_step": typical_ms, "frac_of_typical_copy_only": typical_ms / e2e_ms,
            "aggregate_gbs_at_ceiling": (h2d + d2h) * world / (best_ms * 1e-3) / 1e9,
            "how": "gcs_b200_pcie_probe: the step's H2D and D2H byte counts from / to pinned memory, both directions at once, every rank "
                   "at the same time, as one contiguous copy per direction and as 16 pieces (the faster of the two); ceiling = the best of "
                   "9 repetitions, typical = their median (under contention between ranks the two differ by 1.6x); max over ranks. "
                   "Standalone sweep: profiles/r2_pcie_probe.md"}
    sampler.leave()
    clocks = sampler.stop()

    # ---- peaks (after the timed regions: the probe heats the chip) ----
    dfma_peak = ctx.dfma_peak()
    mix_peak = lib.gcs_b200_fp64_probe(local_rank, 1)
    peaks, peak_src = load_peaks()
    ach_tf = w_k1 / (k1_ms * 1e-3) / 1e12
    traffic, traffic_stale = load_traffic(lib)
    vname = VARIANT_NAMES[args.variant]
    rerun_stats = ctx.rerun_stats(devb) if args.variant >= 5 else None
    kernel_name = lib.gcs_b200_kernel_name(1, 2, args.variant).decode()
    fma_kernel = args.variant >= 5
    roofline = {
        "kernel": kernel_name,
        "bound": "fp64",
        "bound_note": "FP64 CUDA-core pipe (no tensor-core work on this path); the HBM side is under 'hbm'",
        "achieved": ach_tf, "peak": dfma_peak, "unit": "TFLOP/s", "frac": ach_tf / dfma_peak if dfma_peak > 0 else None,
        "peak_source": "measured live: gcs_b200_fp64_probe DFMA micro-benchmark (FMA = 2 flops); MEASURED_PEAKS.json has no FP64 entry",
        "traffic": traffic.get(kernel_name, {}).get("dram_bytes_per_launch"),
        "traffic_source": traffic.get(kernel_name, {}).get("source"),
        "traffic_capture_is_of_another_build": traffic_stale,
        "algorithmic_flops_per_launch": w_k1,
        "algorithmic_flops_note": ("SURVEY.md 8d work model: (iters+1) * 64 flops per seed + selection, from the measured iteration "
                                   "counts - the reference algorithm's work (Householder QR counted at 44 flops per update).  The "
                                   "contracted kernels reach the same iterates with a closed-form landing and the scalar Newton map along the "
                                   "constraint line (8 FP64 instructions per update), so for them `achieved` is a rate of "
                                   "reference-algorithm work, not of executed flops; see "
                                   "executed_*" if fma_kernel else
                                   "SURVEY.md 8d work model from the measured iteration counts"),
        "executed_flops_per_launch": traffic.get(kernel_name, {}).get("executed_flops_per_launch"),
        "flops_per_solve": w_k1 / devb[0].n,
        "mean_iters_per_seed": float(it1.mean()),
        "launch_ms": k1_ms,
        "share_of_step": k1_ms / (k1_ms + k5_ms),
        "hbm": {"achieved": b_k1 / (k1_ms * 1e-3) / 1e9, "peak": peaks.get("hbm_gbs"), "unit": "GB/s",
                "frac": b_k1 / (k1_ms * 1e-3) / 1e9 / peaks.get("hbm_gbs", 1.0), "peak_source": peak_src,
                "algorithmic_bytes_per_launch": b_k1},
        "second_kernel": {"kernel": "K5", "launch_ms": k5_ms, "achieved_tflops": w_k5 / (k5_ms * 1e-3) / 1e12,
                          "hbm_gbs": b_k5 / (k5_ms * 1e-3) / 1e9, "mean_iters_per_seed": float(it5.mean()),
                          "algorithmic_flops_per_launch": w_k5, "algorithmic_bytes_per_launch": b_k5},
    }
    ex = roofline["executed_flops_per_launch"]
    if ex:
        roofline["executed_tflops"] = ex / (k1_ms * 1e-3) / 1e12
        roofline["executed_frac"] = ex / (k1_ms * 1e-3) / 1e12 / dfma_peak if dfma_peak > 0 else None
    if not fma_kernel:
        roofline["non_fma_peak"] = mix_peak
        roofline["frac_of_non_fma_peak"] = ach_tf / mix_peak if mix_peak > 0 else None

    # ---- the other BASELINE configs, measured in this run ----
    configs = None
    if not args.no_extras:
        configs = {}
        t_extra = time.perf_counter()
        for name, fn in (("multistart8", lambda: bench_multistart(ctx, 5)), ("sweep64m", lambda: bench_sweep(ctx, 3)),
                         ("kinds", lambda: bench_kinds(ctx))):
            try:
                configs[name] = fn()
            except Exception as ex_:  # an extra may not take the line down
                if world > 1:
                    raise
                configs[name] = {"error": repr(ex_)[:300]}
        if rank == 0:
            try:
                configs["sketch100k"] = bench_sketch(ctx)
            except Exception as ex_:
                configs["sketch100k"] = {"error": repr(ex_)[:300]}
        ctx.host_barrier()
        configs["sharded"] = bench_sharded(ctx)
        configs["seconds"] = time.perf_counter() - t_extra

    cpu = faithful = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, cores, kind, desc = cpu_rate(ctx.gcs, args.cpu_seconds)
        cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": kind, "sample": desc}
        faithful = faithful_rate()

    if rank == 0:
        cfg = base_config(args0)
        run = {"variant": vname,
               "parity_class": ("contract: iteration counts, convergence flags and root indices identical to the reference, "
                                "coordinates within 1e-9 relative (checked in this run against the bit-identical kernels)"
                                if fma_kernel else "bit-identical to the reference arithmetic"),
               "literal_reruns": rerun_stats,
               "contract_violation": violation,
               "timing": "CUDA events around each step's gcs_b200_solve_many call on the launching stream, sum over steps, max over ranks",
               "wall_s_timed_region_incl_flush": t_wall,
               "library": lib.gcs_b200_version().decode()}
        out = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "run": run,
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "steps": e2e_steps, "ms_per_step": e2e_ms, "gpu_launches": int(e2e_launches),
                    "api": "gcs_b200_solve_host_async x4 + gcs_b200_wait (pinned host buffers, wall clock incl. copies)",
                    "device_api_of_value": "gcs_b200_solve_many([K1 batch, K5 batch]) per step",
                    "wire_format": "one batch per solver shape (anchored K1 / general K1 / anchored K5 / general K5), anchor columns NULL; "
                                   "down: solved coordinates + chosen root",
                    "pcie": pcie, "dense_round1_format": dense_line},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "sequential_launches": sequential,
            "bit_identical": bit_identical,
            "configs": configs,
            "cpu_baseline": cpu,
            "cpu_baseline_faithful": faithful,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
