#!/usr/bin/env python
"""Timing of the surface-sampled distance (``distance.surface_distance``, csrc/distance.cu) on the 1M-face case.

  python scripts/bench_surface_distance.py --out <dir>        -> <dir>/bench_surface_distance.json

Case: ``synth.make_case(224)`` (1,003,520 faces, 501,762 vertices); A = the noisy mesh, B = the clean one.  For each
sample count per side (default 1M, 4M, 16M) every stage is timed with CUDA events around ``--reps`` calls after
``--warmup`` calls; the JSON holds the median and the spread (min, max) in milliseconds:

  prefix (face weights, their max, quantised weights and their prefix, on B), sample (one side), query A->B and B->A
  of the samples, angles (one side), stats (one vector of n values, including its read to the host), and
  ``surface_distance(a, b_tree)`` end to end as a training loop would call it: B's tree (and its prefix) reused, A
  given as float32 positions on the device, so A's tree and prefix are built in every call.

For comparison the same run times the vertex query A->B (501,762 points) and ``hausdorff(a, b_tree)``.  Peak device
memory of one ``surface_distance`` call above what was allocated before it is read with
``torch.cuda.max_memory_allocated``; it holds the sample buffers and A's tree and prefix.  The device name, power
limit and max SM clock are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

from scripts.bench_mesh_distance import gpu_info, timed  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=224, help="icosphere frequency (F = 20 n^2)")
    ap.add_argument("--samples", default="1048576,4194304,16777216", help="comma-separated samples per side")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_surface_distance.py needs a CUDA device")

    from dual_dmp_b200 import synth
    from dual_dmp_b200._lib import lib, ptr, stream_ptr
    from dual_dmp_b200.distance import MeshBVH, _normal_angles, distance_stats, hausdorff, surface_distance

    dev = torch.device("cuda:0")
    case = synth.make_case(args.n)
    faces = case.faces
    V, F = len(case.gt_vs), len(faces)
    res = {"case": f"synth.make_case({args.n})", "V": V, "F": F, **gpu_info(), "warmup": args.warmup,
           "reps": args.reps}
    tb = MeshBVH(case.gt_vs, faces, dev)           # B: clean
    ta = MeshBVH(case.noise_vs, faces, dev)        # A: noisy
    st = stream_ptr(dev)
    ws = torch.empty(int(lib.query("ddmp_surface_prefix_workspace_bytes", F)) // 8, dtype=torch.int64, device=dev)
    prefix = torch.empty(F, dtype=torch.int64, device=dev)

    def prefix_stage():
        lib.call("ddmp_surface_prefix", ptr(tb.vs), ptr(tb.faces), F, ptr(prefix), ptr(ws), st)

    pos = ta.vs.float()                            # network output: float32 positions on the device
    faces_dev = tb.faces
    res["prefix"] = timed(prefix_stage, args.warmup, args.reps)
    torch.cuda.synchronize()
    tb.sample_surface(1)                           # builds and keeps B's prefix
    assert torch.equal(prefix, tb._prefix)
    res["vertex_query_a_to_b"] = timed(lambda: tb.query(ta.vs), args.warmup, args.reps)
    res["hausdorff_training_loop"] = timed(lambda: hausdorff((pos, faces_dev), tb), args.warmup, args.reps)
    res["by_samples"] = {}
    for n in (int(x) for x in args.samples.split(",")):
        pa, fa = ta.sample_surface(n, 0, 0)
        pb, fb = tb.sample_surface(n, 0, 1)
        d_ab, g_ab = tb.query(pa)
        stages = {
            "sample": timed(lambda: tb.sample_surface(n, 0, 1), args.warmup, args.reps),
            "query_a_to_b": timed(lambda: tb.query(pa), args.warmup, args.reps),
            "query_b_to_a": timed(lambda: ta.query(pb), args.warmup, args.reps),
            "angles": timed(lambda: _normal_angles(ta, fa, tb, g_ab), args.warmup, args.reps),
            "stats": timed(lambda: distance_stats(d_ab), args.warmup, args.reps),
            "surface_distance_training_loop": timed(lambda: surface_distance((pos, faces_dev), tb, n),
                                                    args.warmup, args.reps),
        }
        del pa, fa, pb, fb, d_ab, g_ab
        torch.cuda.synchronize()
        base = torch.cuda.memory_allocated(dev)
        torch.cuda.reset_peak_memory_stats(dev)
        rep = surface_distance((pos, faces_dev), tb, n)
        torch.cuda.synchronize()
        peak = torch.cuda.max_memory_allocated(dev) - base
        q_ns = {k: stages[k]["median_ms"] * 1e6 / n for k in ("query_a_to_b", "query_b_to_a")}
        res["by_samples"][str(n)] = {
            "stages": stages, "query_ns_per_point": q_ns,
            "vertex_query_ns_per_point": res["vertex_query_a_to_b"]["median_ms"] * 1e6 / V,
            "peak_bytes_above_baseline": peak, "peak_bytes_per_sample_per_side": peak / (2 * n),
            "report": rep}
        print(n, json.dumps({k: v["median_ms"] for k, v in stages.items()}), "peak MB", peak / 2 ** 20, flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_surface_distance.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k]["median_ms"] for k in ("prefix", "vertex_query_a_to_b", "hausdorff_training_loop")}))
    print("wrote", path)


if __name__ == "__main__":
    main()
