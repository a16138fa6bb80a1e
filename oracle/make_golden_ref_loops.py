#!/usr/bin/env python
"""Golden vectors for the tests that compared live with the reference build (oracle/_ref) on seeded inputs:
tests/test_gpu_host.py (three whole sketches, the 100k-point linkage, the unchecked linkage),
tests/test_golden.py (20k instances per kind) and tests/test_merge3.py (fresh Merge3 rows, the PPP
enumeration loop).  Needs a GPU:

    python oracle/make_golden_ref_loops.py        ->  tests/golden/ref_loops.npz

The reference build cannot be made from the repository, so the values are this project's outputs on the
inputs those tests generate.  They are the reference's: at commit 75a1834, whose package, include/,
oracle/ and tests/ are identical to those of commit 110631d where this file was made, the GPU tests ran
against the reference build and passed, positions and merged poses bit for bit.  The 20k-per-kind rows
are the CPU oracle's, which that test compared with the reference the same way (candidates bit for bit,
iteration counts where not capped).  Large outputs are stored as a digest (tests/util.py digest; the
100k-point linkage with a fixed sample beside it), which compares bit for bit, NaN with NaN."""
import importlib
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import __graft_entry__ as entry  # noqa: E402
import host_lib as H  # noqa: E402
import oracle_lib as O  # noqa: E402
import sketch_gen as S  # noqa: E402
import test_gpu_host as TH  # noqa: E402
import test_merge3 as TM  # noqa: E402
from util import digest, positions  # noqa: E402


def main(path=os.path.join(ROOT, "tests", "golden", "ref_loops.npz")):
    entry.build_cuda()
    entry.build_oracle()
    entry.build_host()
    gcs = importlib.import_module("2d_geometry_constraint_solver_b200")
    gcs.capi.init([0])
    out = {}
    for seed, first, n in TH.WHOLE_SKETCHES:
        el, lv = S.make_sketch(n, seed=seed, first_shape=first)
        rc, got, _ = H.system_solve_ex(el, S.sketch_graph(el, lv))
        assert rc == 0, H.last_error()
        pos, out[f"sketch{seed}_set"] = positions(got)
        out[f"sketch{seed}_pos_sha256"] = np.array(digest(pos))
    el, edges = S.make_linkage_unchecked(6000, seed=4)
    rc, got, _ = H.system_solve_ex(el, edges)
    assert rc == 0, H.last_error()
    pos, out["unchecked_set"] = positions(got)
    out["unchecked_pos_sha256"] = np.array(digest(pos))
    el, edges = S.make_linkage(100000, seed=4)
    rc, got, _ = H.system_solve_ex(el, edges)
    assert rc == 0, H.last_error()
    xy = np.array([e["pos"] for e in got])
    out["config4_xy_sha256"], out["config4_xy_sample"] = np.array(digest(xy)), xy[TH.config4_sample(len(xy))]
    for kind in (1, 2, 3, 4, 5):
        a = O.solve(gcs.synth.make(kind, 20000, seed=77 + kind).alloc_outputs())
        out[f"scale_k{kind}_sha256"] = np.array([digest(a.cand), digest(np.minimum(a.iters, 999)), digest(a.root_index)])
    for kase, rows in TM.fresh_rows():
        rc, res, ok, _ = H.m3_solve(kase, rows, mode=1)
        assert rc == 0, H.last_error()
        out[f"m3fresh_k{kase}_out_sha256"], out[f"m3fresh_k{kase}_ok"] = np.array(digest(res[ok == 1])), ok
    merges = [H.m3_ppp_merge(*sc) for sc in TM.ppp_scenarios()]
    assert all(m[0] >= 0 for m in merges), H.last_error()
    out["ppp_n"] = np.array([m[0] for m in merges], dtype=np.int32)
    out["ppp_ids"] = np.concatenate([m[1] for m in merges]).astype(np.int32)
    out["ppp_pose4"] = np.concatenate([np.asarray(m[2]).reshape(-1, 4) for m in merges])
    np.savez_compressed(path, **out)
    print(f"{path}: {os.path.getsize(path)} bytes")


if __name__ == "__main__":
    main(*sys.argv[1:])
