"""A/B of the dense transforms' single-product mode (dense_precision="f16x1", DDMP_GEMM_F16X1) against the default
3-term fp16 split, alternated in one process:

  1. per shape: X.W^T (with the fused BatchNorm + LeakyReLU prologue), dH.W and dH^T.act(X) of every trunk layer on
     the fp16-split kernels, at N = 501,762 (PosNet, vertices of the 1M-face mesh) and 1,003,520 rows (NormalNet,
     faces); the L2 is overwritten before every timed call; median of --reps;
  2. graph-replayed DualStep ms/step at 1M faces (icosphere 224) and 200K faces (icosphere 100): one DualStep per mode
     from one state_dict, blocks of --steps replays alternated --rounds times;
  3. the MAD gap of one 200K-face fit run --fit-iters iterations in both modes from one state_dict (reported, not a
     pass/fail criterion).

    python scripts/bench_dense_precision.py --out profiles/bench_dense_precision_r3.json

The card's name, power limit and max SM clock are read in the same run.  A text summary goes next to the JSON.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

SHAPES = [(64, 128), (128, 256), (256, 256), (256, 512), (512, 512), (512, 256), (256, 128), (128, 64)]
MODES = ("fp32", "f16x1")


def card() -> dict:
    q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def per_shape(rows_list, reps, log):
    from dual_dmp_b200 import functional as F_
    dev = torch.device("cuda:0")
    flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)          # 256 MB > the 126 MB L2
    out = []
    for n in rows_list:
        for cin, cout in SHAPES:
            g = torch.Generator(device="cpu").manual_seed(cin * 1000 + cout)
            X = torch.randn(n, cin, generator=g).to(dev)
            W = (torch.randn(cout, cin, generator=g) / cin ** 0.5).to(dev)
            dH = (torch.randn(n, cout, generator=g) * 1e-3).to(dev)
            sc = (torch.rand(cin, generator=g) + 0.5).to(dev)
            sh = torch.randn(cin, generator=g).to(dev)
            bx = (torch.nn.functional.leaky_relu(X[:65536] * sc + sh, 0.01).abs().amax(0) * 1.5).contiguous()
            bd = dH[:65536].abs().amax(0).mul(1.5).contiguous()
            H, G = torch.empty(n, cout, device=dev), torch.empty(n, cin, device=dev)
            calls = {
                "xw": lambda m: F_.gemm_xw(X, W, scale=sc, shift=sh, amax=bx, out=H, dense_precision=m),
                "dx": lambda m: F_.gemm_dx(dH, W, amax=bd, out=G, dense_precision=m),
                "dw": lambda m: F_.gemm_dw(dH, X, cin, scale=sc, shift=sh, amax_dh=bd, amax_x=bx, dense_precision=m),
            }
            for name, fn in calls.items():
                times = {m: [] for m in MODES}
                for m in MODES:
                    fn(m)
                torch.cuda.synchronize()
                for _ in range(reps):
                    for m in MODES:
                        flush.zero_()
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                        fn(m)
                        e1.record()
                        torch.cuda.synchronize()
                        times[m].append(e0.elapsed_time(e1))
                med = {m: statistics.median(times[m]) for m in MODES}
                row = {"op": name, "rows": n, "cin": cin, "cout": cout,
                       "ms": {m: {"median": med[m], "min": min(times[m]), "max": max(times[m])} for m in MODES},
                       "speedup": med["fp32"] / med["f16x1"]}
                out.append(row)
                log(f"{name} {cin:3d}->{cout:3d} rows={n:8d}  fp32 {med['fp32']:.3f} ms  f16x1 {med['f16x1']:.3f} ms  "
                    f"x{row['speedup']:.2f}")
            del X, W, dH, H, G
            torch.cuda.empty_cache()
    return out


def _nets(dev, seed):
    from dual_dmp_b200.util.networks import NormalNet, PosNet
    torch.manual_seed(seed)
    return PosNet(dev).to(dev), NormalNet(dev).to(dev)


def _steppers(case, dev, k=(3.0, 4.0, 4.0, 4.0, 1.0), bnfloop=1):
    from dual_dmp_b200.step import DualStep
    n_mesh, ds = case
    pos0, nrm0 = _nets(dev, 0)
    out = {}
    for m in MODES:
        p, q = _nets(dev, 1)
        p.load_state_dict(pos0.state_dict())
        q.load_state_dict(nrm0.state_dict())
        out[m] = DualStep(p, q, ds, n_mesh, k=k, bnfloop=bnfloop, dense_precision=m)
    return out


def step_ab(name, case, dev, steps, rounds, log):
    st = _steppers(case, dev)
    ep = {m: 101 for m in MODES}
    for m in MODES:                                   # warm-up and capture (epoch > 100: the BNF phase)
        for _ in range(5):
            st[m].step(ep[m]); ep[m] += 1
    torch.cuda.synchronize()
    times = {m: [] for m in MODES}
    for _ in range(rounds):
        for m in MODES:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                st[m].step(ep[m]); ep[m] += 1
            e1.record()
            torch.cuda.synchronize()
            times[m].append(e0.elapsed_time(e1) / steps)
    med = {m: statistics.median(times[m]) for m in MODES}
    log(f"DualStep {name}: fp32 {med['fp32']:.3f} ms/step  f16x1 {med['f16x1']:.3f} ms/step  "
        f"({100 * (med['fp32'] - med['f16x1']) / med['fp32']:+.1f} %)  rounds fp32 {['%.3f' % t for t in times['fp32']]} "
        f"f16x1 {['%.3f' % t for t in times['f16x1']]}")
    del st
    torch.cuda.empty_cache()
    return {"case": name, "ms_per_step": {m: {"median": med[m], "rounds": times[m]} for m in MODES},
            "steps_per_round": steps, "rounds": rounds, "gain_percent": 100 * (med["fp32"] - med["f16x1"]) / med["fp32"]}


def mad_gap(n_ico, iters, dev, log):
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import e2e_mad
    from dual_dmp_b200 import synth
    from dual_dmp_b200.util.datamaker import dataset_from_meshes
    from dual_dmp_b200.util.mesh import Mesh
    from types import SimpleNamespace
    case = synth.make_case(n_ico)
    n_mesh = Mesh(vs=case.noise_vs, faces=case.faces)
    gt = Mesh(vs=case.gt_vs, faces=case.faces)
    ds = dataset_from_meshes(n_mesh, SimpleNamespace(vs=case.smooth_vs))
    st = _steppers((n_mesh, ds), dev)
    curves = {m: [] for m in MODES}
    t0 = time.perf_counter()
    for m in MODES:
        for epoch in range(1, iters + 1):
            st[m].step(epoch)
            if epoch % 50 == 0:
                curves[m].append(e2e_mad.eval_mad(st[m].pos, n_mesh.faces, gt.fn))
    initial = e2e_mad.numpy_mad(n_mesh.fn, gt.fn)
    fin = {m: curves[m][-1] for m in MODES}
    gap = (fin["f16x1"] - fin["fp32"]) / fin["fp32"]
    log(f"MAD gap, {len(n_mesh.faces)} faces, {iters} iterations from one state_dict: initial {initial:.4f}, "
        f"fp32 {fin['fp32']:.4f}, f16x1 {fin['f16x1']:.4f} ({100 * gap:+.2f} %) [{time.perf_counter() - t0:.0f} s]")
    del st
    torch.cuda.empty_cache()
    return {"faces": int(len(n_mesh.faces)), "iters": iters, "initial_mad": initial, "mad_every_50": curves,
            "final": fin, "relative_gap": gap}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--fit-iters", type=int, default=300)
    ap.add_argument("--skip", nargs="*", default=[], choices=["shapes", "step1m", "step200k", "mad"])
    args = ap.parse_args()
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    dev = torch.device("cuda:0")
    sys.path.insert(0, ROOT)
    from bench import build_case
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    res = {"card": card(), "options": {"reps": args.reps, "steps": args.steps, "rounds": args.rounds,
                                       "fit_iters": args.fit_iters, "skip": args.skip}}
    log(f"{res['card']['device']} | {res['card']['nvidia_smi']}")
    if "shapes" not in args.skip:
        res["per_shape"] = per_shape([501762, 1003520], args.reps, log)
    if "step1m" not in args.skip:
        n_mesh, _, ds = build_case(224)
        res["step_1m"] = step_ab(f"{len(n_mesh.faces)} faces", (n_mesh, ds), dev, args.steps, args.rounds, log)
        del n_mesh, ds
    if "step200k" not in args.skip:
        n_mesh, _, ds = build_case(100)
        res["step_200k"] = step_ab(f"{len(n_mesh.faces)} faces", (n_mesh, ds), dev, 4 * args.steps, args.rounds, log)
        del n_mesh, ds
    if "mad" not in args.skip:
        res["mad_200k"] = mad_gap(100, args.fit_iters, dev, log)
    res["card_after"] = card()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    with open(os.path.splitext(args.out)[0] + ".txt", "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
