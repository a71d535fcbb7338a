#!/usr/bin/env python
"""Timing of the GPU point-to-mesh distance (csrc/distance.cu) on the synthetic 1M-face case.

  python scripts/bench_mesh_distance.py --out <dir>        -> <dir>/bench_mesh_distance.json

Case: ``synth.make_case(224)`` (1,003,520 faces, 501,762 vertices); A = the noisy vertices, B = the clean ones, over
the shared faces, both directions.  Every stage is timed with CUDA events around ``--reps`` launches after
``--warmup`` launches; the JSON holds the median and the spread (min, max) in milliseconds:

  keys (scene box + Morton codes), sort (torch.sort, stable), build (topology + refit), query A->B, query B->A,
  stats (one direction), two-sided ``hausdorff`` from host arrays (uploads and both trees included) and in the form a
  training loop uses (B's tree built once, A's positions already on the device).

The exhaustive kernel is timed on a seeded 4,096-point subset for the speed-up of the BVH query.  The working set of
one direction (64-byte nodes + 16-byte leaves per face, float64 vertices) is about 100 MB, within the 126 MB L2 of a
B200, so the repeated queries read it mostly from L2 after the first pass; that is also the situation of an
evaluation run every few epochs right after a step.  The device name and power limit are read in the same run.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402


def timed(fn, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    ms = np.asarray(ms)
    return {"median_ms": float(np.median(ms)), "min_ms": float(ms.min()), "max_ms": float(ms.max()), "reps": reps}


def gpu_info():
    out = {"device": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        out["power_limit_and_max_sm_clock"] = q
    except (OSError, subprocess.SubprocessError) as e:
        out["power_limit_and_max_sm_clock"] = f"unavailable: {e}"
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--n", type=int, default=224, help="icosphere frequency (F = 20 n^2)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--reps", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_mesh_distance.py needs a CUDA device")

    from dual_dmp_b200 import synth
    from dual_dmp_b200._lib import lib, ptr, stream_ptr
    from dual_dmp_b200.distance import MeshBVH, distance_stats, hausdorff

    dev = torch.device("cuda:0")
    t0 = time.time()
    case = synth.make_case(args.n)
    setup_s = time.time() - t0
    faces = case.faces
    V, F = len(case.gt_vs), len(faces)
    res = {"case": f"synth.make_case({args.n})", "V": V, "F": F, **gpu_info(), "case_setup_s": setup_s}

    tb = MeshBVH(case.gt_vs, faces, dev)           # B: clean
    ta = MeshBVH(case.noise_vs, faces, dev)        # A: noisy
    st = stream_ptr(dev)
    scratch = torch.zeros(int(lib.query("ddmp_prep_scratch_bytes")) // 8 + 1, dtype=torch.float64, device=dev)
    bbox = torch.empty(6, dtype=torch.float64, device=dev)
    keys = torch.empty(F, dtype=torch.int64, device=dev)
    nodes = torch.empty_like(tb.nodes)
    leaves = torch.empty_like(tb.leaves)
    parent = torch.empty(2 * F - 1, dtype=torch.int32, device=dev)
    counters = torch.zeros(F - 1, dtype=torch.int32, device=dev)

    def keys_stage():
        lib.call("ddmp_prep_bbox", ptr(tb.vs), ptr(bbox), ptr(scratch), V, st)
        lib.call("ddmp_bvh_keys", ptr(tb.vs), ptr(tb.faces), ptr(bbox), ptr(keys), F, st)

    keys_stage()
    sorted_keys, order = torch.sort(keys, stable=True)

    def build_stage():
        lib.call("ddmp_bvh_build", ptr(tb.vs), ptr(tb.faces), ptr(sorted_keys), ptr(order), ptr(nodes), ptr(leaves),
                 ptr(parent), ptr(counters), F, st)

    build_stage()
    torch.cuda.synchronize()
    assert torch.equal(leaves, tb.leaves) and int(counters.abs().sum()) == 0

    d_ab, _ = tb.query(ta.vs)
    stages = {
        "keys": timed(keys_stage, args.warmup, args.reps),
        "sort": timed(lambda: torch.sort(keys, stable=True), args.warmup, args.reps),
        "build": timed(build_stage, args.warmup, args.reps),
        "query_a_to_b": timed(lambda: tb.query(ta.vs), args.warmup, args.reps),
        "query_b_to_a": timed(lambda: ta.query(tb.vs), args.warmup, args.reps),
        "stats": timed(lambda: distance_stats(d_ab), args.warmup, args.reps),
        "hausdorff_from_host_arrays": timed(lambda: hausdorff((case.noise_vs, faces), (case.gt_vs, faces), dev),
                                            args.warmup, args.reps),
    }
    pos = ta.vs.float()                                  # network output: float32 positions on the device
    faces_dev = tb.faces
    stages["hausdorff_training_loop"] = timed(lambda: hausdorff((pos, faces_dev), tb), args.warmup, args.reps)

    rng = np.random.default_rng(0)
    sub = torch.from_numpy(case.noise_vs[rng.choice(V, 4096, replace=False)]).to(dev)
    stages["exhaustive_4096"] = timed(lambda: tb._query_exhaustive(sub), 1, max(3, args.reps // 10))
    stages["bvh_4096"] = timed(lambda: tb.query(sub), args.warmup, args.reps)
    d1, f1 = tb.query(sub)
    d2, f2 = tb._query_exhaustive(sub)
    res["exhaustive_equal_bitwise"] = bool(torch.equal(d1, d2) and torch.equal(f1, f2))
    res["speedup_bvh_over_exhaustive_4096"] = stages["exhaustive_4096"]["median_ms"] / stages["bvh_4096"]["median_ms"]
    per_point_ms = stages["exhaustive_4096"]["median_ms"] / 4096
    res["exhaustive_full_a_to_b_estimate_ms"] = per_point_ms * V
    res["stages"] = stages
    res["report"] = hausdorff((case.noise_vs, faces), (case.gt_vs, faces), dev)
    res["working_set_bytes_one_direction"] = {"nodes": 64 * (F - 1), "leaves": 16 * F, "target_vertices": 24 * V,
                                              "query_points": 24 * V, "outputs": 12 * V}
    res["training_step_ms_reference"] = 57.6
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_mesh_distance.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: (v["median_ms"] if isinstance(v, dict) else v) for k, v in stages.items()}))
    print("wrote", path)


if __name__ == "__main__":
    main()
