"""Cost of evaluating a batch of fits: the per-fit host evaluation fit_many used to run against
``distance.BatchEvaluator`` on the device, alone and inside the fit_many loop, in one process.

    python scripts/bench_fit_eval.py --out profiles/bench_fit_eval_r3.json

1. Evaluation alone.  host: per fit, positions to the host, numpy face normals + vertex normals, ``Loss.mad``,
   ``hausdorff(o1, gt_tree)`` (the clean tree built once, the output tree per call).  device: ``evaluate`` + one read
   of the numbers.  B in {1, 4, 16, 64} at 12,500 faces, {1, 8} at 200K faces, 1 at 1M faces.
2. The fit_many loop, 300 iterations (30 evaluations, 3 OBJ snapshots), old and new loop alternated, three rounds
   each, against the bare ``MultiDualStep`` step rate: 12,500 faces with the CAD weights (k = 3,0,3,4,2, bnfloop 5),
   B = 16; 200K faces with the default weights, B = 8.
3. Tree quality after refit: query time of the refit output tree against a fresh build at the last evaluation.

Synthetic icospheres (synth.make_case; positions = clean + noise); every fit of a batch has its own networks.
"""
from __future__ import annotations

import argparse
import copy
import json
import os
import sys
import tempfile
import time
import types

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from scripts.bench_multi_fit import _nets, card  # noqa: E402

EVAL_CASES = [(25, (1, 4, 16, 64)), (100, (1, 8)), (224, (1,))]
LOOP_CASES = {"cad_12k": dict(n=25, k=(3.0, 0.0, 3.0, 4.0, 2.0), bnfloop=5, B=16),
              "default_200k": dict(n=100, k=(3.0, 4.0, 4.0, 4.0, 1.0), bnfloop=1, B=8)}


def _mesh(vs, faces):
    from dual_dmp_b200.util.mesh import Mesh
    m = types.SimpleNamespace(vs=np.asarray(vs, dtype=np.float64), faces=np.asarray(faces))
    Mesh.compute_face_normals(m)
    return m


def _sync_ms(fn, reps):
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return 1000.0 * (time.perf_counter() - t) / reps


def host_eval(pos, o1s, gts, gt_trees):
    """fit_many's evaluation before BatchEvaluator, per fit"""
    import dual_dmp_b200.util.loss as Loss
    from dual_dmp_b200.distance import hausdorff
    from dual_dmp_b200.util.mesh import Mesh
    out = []
    for p, o1, gt, tree in zip(pos, o1s, gts, gt_trees):
        o1.vs = p.to("cpu").numpy().copy()
        Mesh.compute_face_normals(o1)
        Mesh.compute_vert_normals(o1)
        out.append((Loss.mad(o1.fn, gt.fn), hausdorff((o1.vs, o1.faces), tree)["hausdorff"]))
    return out


def bench_eval(dev, reps):
    from dual_dmp_b200 import synth
    from dual_dmp_b200.distance import BatchEvaluator, MeshBVH
    rows = []
    for n, batches in EVAL_CASES:
        vs, faces = synth.icosphere(n)
        gt = _mesh(vs, faces)
        noisy = _mesh(vs + np.random.RandomState(0).normal(0, 0.2 / n, vs.shape), faces)
        for B in batches:
            pos = [torch.from_numpy(noisy.vs + np.random.RandomState(i).normal(0, 0.05 / n, vs.shape)).float().to(dev)
                   for i in range(B)]
            gts = [gt] * B
            gt_trees = [MeshBVH(gt.vs, gt.faces, dev) for _ in range(B)]
            o1s = [types.SimpleNamespace(vs=None, faces=faces) for _ in range(B)]
            ev = BatchEvaluator([noisy] * B, gts, dev)
            dev_fn = lambda: ev.evaluate(pos)["hausdorff_rel"].tolist()          # noqa: E731
            host_fn = lambda: host_eval(pos, o1s, gts, gt_trees)                 # noqa: E731
            dev_fn(), host_fn()
            r = max(1, reps // max(1, B * len(faces) // 200_000))
            t_dev = [_sync_ms(dev_fn, r) for _ in range(3)]
            t_host = [_sync_ms(host_fn, r) for _ in range(3)]
            got, ref = ev.evaluate(pos), host_fn()
            mad_err = max(abs(a - b[0]) / abs(b[0]) for a, b in zip(got["mad"].tolist(), ref))
            h_same = all(a == b[1] for a, b in zip(got["hausdorff"].tolist(), ref))
            row = {"faces_per_fit": len(faces), "B": B, "host_ms": [round(x, 3) for x in t_host],
                   "device_ms": [round(x, 3) for x in t_dev], "speedup_best": round(min(t_host) / min(t_dev), 1),
                   "mad_max_rel_diff": mad_err, "hausdorff_bitwise_equal": h_same}
            print(json.dumps({"eval": row}), flush=True)
            rows.append(row)
            del ev, gt_trees
            torch.cuda.empty_cache()
    return rows


def old_loop(step, meta, iters, out_dir):
    import dual_dmp_b200.util.loss as Loss
    from dual_dmp_b200.util.mesh import Mesh
    for epoch in range(1, iters + 1):
        step.step(epoch)
        if epoch % 10 == 0:
            for i, m in enumerate(meta):
                m["o1"].vs = step.pos[i].to("cpu").numpy().copy()
                Mesh.compute_face_normals(m["o1"])
                Mesh.compute_vert_normals(m["o1"])
                m["mad"] = Loss.mad(m["o1"].fn, m["gt"].fn)
        if epoch % 100 == 0:
            for i, m in enumerate(meta):
                Mesh.save(m["o1"], os.path.join(out_dir, "{}_{}_ddmp={:.3f}.obj".format(i, epoch, m["mad"])))


def new_loop(step, meta, iters, out_dir, evaluator, writer_cls, dev):
    side = torch.cuda.Stream(dev)
    writer = writer_cls()
    report = None
    try:
        for epoch in range(1, iters + 1):
            step.step(epoch)
            if epoch % 10 == 0:
                report = evaluator.evaluate(step.pos)
            if epoch % 100 == 0:
                mads = report["mad"].tolist()
                cur = torch.cuda.current_stream(dev)
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    host = [torch.empty(p.shape, dtype=p.dtype, pin_memory=True).copy_(p, non_blocking=True)
                            for p in step.pos]
                    done = torch.cuda.Event()
                    done.record(side)
                cur.wait_stream(side)
                writer.put(done, [(os.path.join(out_dir, "{}_{}_ddmp={:.3f}.obj".format(i, epoch, mads[i])), h,
                                   meta[i]["o1"].faces) for i, h in enumerate(host)])
    finally:
        writer.close()
    return report


def bare_loop(step, iters):
    for epoch in range(1, iters + 1):
        step.step(epoch)


def _fit_many():
    import importlib.util
    spec = importlib.util.spec_from_file_location("fit_many", os.path.join(ROOT, "scripts", "fit_many.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def _query_ms(tree, pts, reps=20):
    tree.query(pts)
    return _sync_ms(lambda: tree.query(pts), reps)


def bench_loop(name, cfg, dev, iters, rounds):
    from bench import build_case
    from dual_dmp_b200 import synth
    from dual_dmp_b200.distance import BatchEvaluator, MeshBVH
    from dual_dmp_b200.step import MultiDualStep
    n_mesh, s_mesh, ds = build_case(cfg["n"])
    case = synth.make_case(cfg["n"])
    gt = _mesh(case.gt_vs, case.faces)
    B = cfg["B"]
    fits = [dict(zip(("posnet", "normnet"), _nets(dev, i)), dataset=ds, n_mesh=n_mesh, k=cfg["k"]) for i in range(B)]
    step = MultiDualStep(fits, bnfloop=cfg["bnfloop"])
    meta = [dict(o1=copy.copy(n_mesh), gt=gt, mad=None) for _ in range(B)]
    evaluator = BatchEvaluator([n_mesh] * B, [gt] * B, dev)
    writer_cls = _fit_many().SnapshotWriter
    for epoch in (1, 2, 3, 4, 101, 102, 103, 104):   # eager passes and both phases' captures
        step.step(epoch)
    t = {"bare": [], "old": [], "new": []}
    with tempfile.TemporaryDirectory() as out_dir:
        for _ in range(rounds):
            for arm in ("bare", "old", "new"):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if arm == "bare":
                    bare_loop(step, iters)
                elif arm == "old":
                    old_loop(step, meta, iters, out_dir)
                else:
                    new_loop(step, meta, iters, out_dir, evaluator, writer_cls, dev)
                torch.cuda.synchronize()
                t[arm].append(time.perf_counter() - t0)
    rate = {arm: [round(B * iters / x, 1) for x in v] for arm, v in t.items()}
    # tree quality at the last evaluation: refit output tree against a fresh build on the same positions
    gt_vs = torch.from_numpy(gt.vs).to(dev)
    refit_ms = _query_ms(evaluator.out[0], gt_vs)
    fresh_ms = _query_ms(MeshBVH(step.pos[0], n_mesh.faces, dev), gt_vs)
    row = {"workload": f"icosphere n={cfg['n']}: {len(n_mesh.faces)} faces per fit, k={list(cfg['k'])}, "
                       f"bnfloop={cfg['bnfloop']}", "B": B, "iterations": iters,
           "seconds": {k: [round(x, 3) for x in v] for k, v in t.items()}, "fit_iters_per_s": rate,
           "new_over_old_best": round(min(t["old"]) / min(t["new"]), 3),
           "new_over_bare_best": round(min(t["bare"]) / min(t["new"]), 3),
           "tree_query_ms": {"refit_output_tree": round(refit_ms, 3), "fresh_build": round(fresh_ms, 3),
                             "points": len(gt.vs)}}
    print(json.dumps({name: row}), flush=True)
    del step, evaluator, fits
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    return row


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="write the JSON record here")
    ap.add_argument("--iters", type=int, default=300)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--reps", type=int, default=20, help="evaluations per timing at 12,500 faces x B = 1")
    ap.add_argument("--skip-eval", action="store_true")
    ap.add_argument("--loops", nargs="*", default=list(LOOP_CASES), choices=list(LOOP_CASES))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_fit_eval: needs a CUDA device")
    dev = torch.device("cuda:0")
    out = {"card": card(dev), "started": time.strftime("%Y-%m-%d %H:%M:%S")}
    if not args.skip_eval:
        out["evaluation"] = bench_eval(dev, args.reps)
    out["fit_many_loop"] = {name: bench_loop(name, LOOP_CASES[name], dev, args.iters, args.rounds)
                            for name in args.loops}
    out["card_after"] = card(dev)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
