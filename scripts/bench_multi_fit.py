"""Throughput of a batch of fits on one GPU: MultiDualStep over B fits against the same B fits as graph-replayed
DualSteps run one after another, alternated in one process, three repeats each.

    python scripts/bench_multi_fit.py --out profiles/bench_multi_fit_r3.json

Cases: synth.make_case(25) (12,500 faces) with the CAD loss weights (k = 3,0,3,4,2, bnfloop 5), B in 1..64, and
make_case(100) (200K faces) with the default weights and bnfloop 1, B in 1..32.  Every fit has its own networks and
dataset (the same mesh, so the separate arm's per-fit cost is one mesh's).  The 200K separate arm keeps at most
--max-separate DualSteps alive (their captured graphs hold the activations) and replays them round-robin, B
replays per pass.  Library launches per step are counted on an eager pass (replays launch nothing from the host).
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

import torch  # noqa: E402

CASES = {
    "cad_12k": dict(n=25, k=(3.0, 0.0, 3.0, 4.0, 2.0), bnfloop=5, batches=(1, 2, 4, 8, 16, 32, 64), steps=40),
    "default_200k": dict(n=100, k=(3.0, 4.0, 4.0, 4.0, 1.0), bnfloop=1, batches=(1, 2, 4, 8, 16, 32), steps=6),
}


def card(dev) -> dict:
    q = subprocess.run(["nvidia-smi", "-i", str(dev.index or 0), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(dev), "nvidia_smi": q.stdout.strip()}


def _nets(dev, seed):
    from dual_dmp_b200.util.networks import NormalNet, PosNet
    torch.manual_seed(seed)
    return PosNet(dev).to(dev), NormalNet(dev).to(dev)


def _time(fn, reps: int) -> float:
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run_case(name, cfg, dev, repeats, max_separate, only=None):
    sys.path.insert(0, ROOT)
    from bench import build_case
    from dual_dmp_b200._lib import lib
    from dual_dmp_b200.step import DualStep, MultiDualStep
    n_mesh, s_mesh, ds = build_case(cfg["n"])
    k, loop, steps = cfg["k"], cfg["bnfloop"], cfg["steps"]
    rows = []
    for B in cfg["batches"]:
        if only and B not in only:
            continue
        fits = []
        for i in range(B):
            p, q = _nets(dev, i)
            fits.append(dict(posnet=p, normnet=q, dataset=ds, n_mesh=n_mesh, k=k))
        multi = MultiDualStep(fits, bnfloop=loop)
        n_sep = min(B, max_separate)
        seps = [DualStep(*_nets(dev, 1000 + i), ds, n_mesh, k=k, bnfloop=loop) for i in range(n_sep)]
        ep = {"m": 101}

        def multi_step():
            multi.step(ep["m"])
            ep["m"] += 1

        def sep_pass(state={"e": 101}):
            for j in range(B):
                seps[j % n_sep].step(state["e"])
                if j % n_sep == n_sep - 1 or j == B - 1:
                    state["e"] += 1

        # eager passes (the first three steps of each phase), counting library launches, then capture
        for _ in range(2):
            multi_step()
        torch.cuda.synchronize()
        l0 = lib.query("ddmp_launch_count")
        multi_step()
        torch.cuda.synchronize()
        multi_launches = lib.query("ddmp_launch_count") - l0
        for _ in range(2):
            seps[0].step(101 + _)
        torch.cuda.synchronize()
        l0 = lib.query("ddmp_launch_count")
        seps[0].step(103)
        torch.cuda.synchronize()
        single_launches = lib.query("ddmp_launch_count") - l0
        for s in seps[1:]:
            for e in (101, 102, 103):
                s.step(e)
        sep_pass({"e": 104})
        for _ in range(2):
            multi_step()
        t_multi, t_sep = [], []
        for _ in range(repeats):
            t_multi.append(_time(multi_step, steps))
            t_sep.append(_time(lambda: sep_pass(), steps))
        bm, bs = min(t_multi), min(t_sep)
        row = {"B": B, "faces_per_fit": len(n_mesh.faces),
               "batched_ms_per_step": [round(x, 3) for x in t_multi],
               "separate_ms_per_B_steps": [round(x, 3) for x in t_sep],
               "batched_fit_iters_per_s": round(1000.0 * B / bm, 1),
               "separate_fit_iters_per_s": round(1000.0 * B / bs, 1),
               "speedup_best_of_3": round(bs / bm, 3),
               "separate_dualsteps_alive": n_sep,
               "library_launches_per_step_eager": {"batched": int(multi_launches), "separate_B_steps":
                                                   int(single_launches) * B},
               "peak_mem_GB": round(torch.cuda.max_memory_allocated(dev) / 1e9, 1)}
        print(json.dumps({name: row}), flush=True)
        rows.append(row)
        del multi, seps, fits
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        torch.cuda.reset_peak_memory_stats(dev)
    return {"workload": f"icosphere n={cfg['n']}: {len(n_mesh.faces)} faces per fit, k={list(k)}, bnfloop={loop}",
            "steps_per_timing": steps, "rows": rows}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--out", default=None, help="write the JSON record here")
    ap.add_argument("--cases", nargs="*", default=list(CASES), choices=list(CASES))
    ap.add_argument("--batches", type=int, nargs="*", default=None, help="only these B")
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--max-separate", type=int, default=8,
                    help="DualSteps kept alive for the separate arm of the 200K case")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("bench_multi_fit: needs a CUDA device")
    dev = torch.device("cuda:0")
    import __graft_entry__  # noqa: F401  (puts the repository on sys.path)
    out = {"card": card(dev), "started": time.strftime("%Y-%m-%d %H:%M:%S"), "cases": {}}
    for name in args.cases:
        cap = args.max_separate if name == "default_200k" else 1 << 30
        out["cases"][name] = run_case(name, CASES[name], dev, args.repeats, cap, args.batches)
    out["card_after"] = card(dev)
    text = json.dumps(out, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
