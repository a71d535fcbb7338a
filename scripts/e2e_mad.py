#!/usr/bin/env python
"""End-to-end parity run (north_star: "MAD after the reference iteration count within 2 % relative").

Trains the CPU oracle (oracle/: restated PyG path + reference losses) and the product (libddmp_b200 CUDA path) from
ONE state_dict on ONE noisy mesh for the reference iteration count (reference main.py:21, --iter 1000), evaluates
MAD against the clean mesh every 10 epochs exactly like reference main.py:117-123 (pos -> host numpy -> float64 face
normals -> Loss.mad), and writes both curves as JSON.

  python scripts/e2e_mad.py --arm oracle  --config default --out tests/golden/e2e_mad_default.json   (CPU, here)
  python scripts/e2e_mad.py --arm product --config cad --path dualstep --out gpurun_out/...          (GPU box)
  python scripts/e2e_mad.py --arm both ...                                                           (GPU box)

Weight sets: "default" = reference main.py:22-28 (k=3,4,4,4,1, bnfloop=1); "cad" = reference README.md:57 /
main4real.py:18-24 (k=3,0,3,4,2, bnfloop=5).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

CONFIGS = {"default": ((3.0, 4.0, 4.0, 4.0, 1.0), 1), "cad": ((3.0, 0.0, 3.0, 4.0, 2.0), 5)}


def numpy_mad(n1, n2):
    """reference util/loss.py:261-272"""
    inner = np.sum(n1 * n2, 1)
    sad = np.rad2deg(np.arccos(np.clip(inner, -1.0, 1.0)))
    return float(np.sum(sad) / len(sad))


def face_normals64(vs, faces):
    """reference util/mesh.py:87-92"""
    fn = np.cross(vs[faces[:, 1]] - vs[faces[:, 0]], vs[faces[:, 2]] - vs[faces[:, 0]])
    return fn / (np.linalg.norm(fn, axis=1, keepdims=True) + 1e-24)


def eval_mad(pos, faces, gt_fn):
    """reference main.py:118-123: network output -> host numpy -> Mesh.compute_face_normals -> Loss.mad"""
    new_pos = pos.to("cpu").detach().numpy().copy()
    return numpy_mad(face_normals64(new_pos.astype(np.float64), faces), gt_fn)


def initial_state(seed):
    from oracle.networks_ref import NormalNetRef, PosNetRef
    torch.manual_seed(seed)
    return PosNetRef(), NormalNetRef()


def run_oracle(case, k, bnfloop, iters, seed, threads, log):
    from oracle import step_ref
    n_mesh, s_mesh, gt_mesh = case
    torch.set_num_threads(threads)
    posnet, normnet = initial_state(seed)
    ds = step_ref.make_dataset(n_mesh, s_mesh)
    opt_pos = torch.optim.Adam(posnet.parameters(), lr=0.01)
    opt_norm = torch.optim.Adam(normnet.parameters(), lr=0.01)
    curve, norm_curve, losses = [], [], []
    t0 = time.perf_counter()
    for epoch in range(1, iters + 1):
        total, _, pos, norm = step_ref.train_step(posnet, normnet, opt_pos, opt_norm, ds, n_mesh, k, bnfloop, epoch)
        if epoch % 10 == 0:
            curve.append(eval_mad(pos, n_mesh.faces, gt_mesh.fn))
            norm_curve.append(numpy_mad(norm.double().numpy(), gt_mesh.fn))
            losses.append(float(total))
            if epoch % 100 == 0:
                log(f"oracle  epoch {epoch:4d} loss {float(total):.6f} MAD {curve[-1]:.4f} "
                    f"normnet-MAD {norm_curve[-1]:.4f} ({time.perf_counter() - t0:.0f} s)")
    return {"mad": curve, "normnet_mad": norm_curve, "loss": losses, "threads": threads,
            "seconds": time.perf_counter() - t0}


def run_product(case, k, bnfloop, iters, seed, path, log, perturb=0, dense_precision="fp32"):
    """``dense_precision``: the networks' dense-transform accuracy contract ("fp32" | "f16x1", util.networks).
    ``perturb`` > 0: every initial weight is multiplied by (1 + 1e-7 * N(0,1)) drawn with that seed -- a rounding-level
    perturbation, like the reduction-order changes that distinguish the oracle's own runs; the chaotic fit turns it into
    an independent trajectory, which gives the (otherwise bitwise deterministic) product an ensemble"""
    from dual_dmp_b200.step import DualStep
    from dual_dmp_b200.util import loss as L
    from dual_dmp_b200.util.datamaker import dataset_from_meshes
    from dual_dmp_b200.util.networks import NormalNet, PosNet
    assert torch.cuda.is_available(), "the product arm needs a CUDA device (no CPU fallback)"
    n_mesh, s_mesh, gt_mesh = case
    dev = torch.device("cuda:0")
    pos_ref, nrm_ref = initial_state(seed)
    posnet, normnet = PosNet(dev).to(dev), NormalNet(dev).to(dev)
    posnet.load_state_dict(pos_ref.state_dict())
    normnet.load_state_dict(nrm_ref.state_dict())
    posnet.dense_precision = normnet.dense_precision = dense_precision
    if perturb:
        g = torch.Generator(device="cpu").manual_seed(1000 + int(perturb))
        with torch.no_grad():
            for net in (posnet, normnet):
                for p_ in net.parameters():
                    p_.mul_((1.0 + 1e-7 * torch.randn(p_.shape, generator=g)).to(dev))
    ds = dataset_from_meshes(n_mesh, s_mesh)
    curve, norm_curve, losses = [], [], []
    t0 = time.perf_counter()
    if path == "dualstep":
        stepper = DualStep(posnet, normnet, ds, n_mesh, k=k, bnfloop=bnfloop)
        for epoch in range(1, iters + 1):
            loss = stepper.step(epoch)
            if epoch % 10 == 0:
                curve.append(eval_mad(stepper.pos, n_mesh.faces, gt_mesh.fn))
                norm_curve.append(numpy_mad(stepper.norm.double().cpu().numpy(), gt_mesh.fn))
                losses.append(float(loss))
                if epoch % 100 == 0:
                    log(f"product epoch {epoch:4d} loss {float(loss):.6f} MAD {curve[-1]:.4f} "
                        f"normnet-MAD {norm_curve[-1]:.4f} ({time.perf_counter() - t0:.0f} s)")
    else:   # the reference's loop body verbatim over the drop-in modules (main.py:88-110)
        opt_pos = torch.optim.Adam(posnet.parameters(), lr=0.01)
        opt_norm = torch.optim.Adam(normnet.parameters(), lr=0.01)
        for epoch in range(1, iters + 1):
            posnet.train(); normnet.train()
            opt_pos.zero_grad(); opt_norm.zero_grad()
            pos = posnet(ds)
            l1 = L.pos_rec_loss(pos, n_mesh.vs)
            l2 = L.mesh_laplacian_loss(pos, n_mesh)
            norm = normnet(ds)
            l3 = L.norm_rec_loss(norm, n_mesh.fn)
            l4, _ = L.fn_bnf_loss(pos, norm, n_mesh, loop=bnfloop)
            if epoch <= 100:
                l4 = l4 * 0.0
            l5 = L.pos_norm_loss(pos, norm, n_mesh)
            loss = k[0] * l1 + k[1] * l2 + k[2] * l3 + k[3] * l4 + k[4] * l5
            loss.backward()
            torch.nn.utils.clip_grad_norm_(normnet.parameters(), 0.8)
            opt_pos.step(); opt_norm.step()
            if epoch % 10 == 0:
                curve.append(eval_mad(pos, n_mesh.faces, gt_mesh.fn))
                norm_curve.append(numpy_mad(norm.detach().double().cpu().numpy(), gt_mesh.fn))
                losses.append(float(loss))
                if epoch % 100 == 0:
                    log(f"product epoch {epoch:4d} loss {float(loss):.6f} MAD {curve[-1]:.4f} "
                        f"normnet-MAD {norm_curve[-1]:.4f} ({time.perf_counter() - t0:.0f} s)")
    return {"mad": curve, "normnet_mad": norm_curve, "loss": losses, "path": path, "dense_precision": dense_precision,
            "seconds": time.perf_counter() - t0}


def compare(a, b, tail=10):
    """relative MAD difference at the final evaluation and averaged over the last ``tail`` evaluations"""
    fa, fb = a["mad"][-1], b["mad"][-1]
    ta, tb = float(np.mean(a["mad"][-tail:])), float(np.mean(b["mad"][-tail:]))
    return {"final": [fa, fb], "final_rel_diff": abs(fa - fb) / fb, "tail_mean": [ta, tb],
            "tail_rel_diff": abs(ta - tb) / tb, "tail_evals": tail,
            "max_rel_diff_over_curve": float(np.max(np.abs(np.array(a["mad"]) - np.array(b["mad"])) / np.array(b["mad"])))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--arm", default="both", choices=["oracle", "product", "both"])
    ap.add_argument("--config", default="default", choices=list(CONFIGS))
    ap.add_argument("--n", type=int, default=9, help="icosphere frequency (F = 20 n^2; 9 -> 1,620 faces)")
    ap.add_argument("--iters", type=int, default=1000)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--threads", type=int, default=min(8, os.cpu_count() or 1))
    ap.add_argument("--path", default="dualstep", choices=["dualstep", "dropin"])
    ap.add_argument("--out", default=None)
    ap.add_argument("--dense-precision", default="fp32", choices=["fp32", "f16x1"],
                    help="product arm: accuracy contract of the dense transforms (DESIGN.md 4.2)")
    args = ap.parse_args()
    from tests.helpers import small_case
    case = small_case("ico", args.n)
    k, bnfloop = CONFIGS[args.config]
    log = lambda s: print(s, file=sys.stderr, flush=True)   # noqa: E731
    out = {"config": args.config, "k": k, "bnfloop": bnfloop, "n": args.n, "faces": int(len(case[0].faces)),
           "iters": args.iters, "seed": args.seed, "initial_mad": numpy_mad(case[0].fn, case[2].fn),
           "eval": "reference main.py:117-123 every 10 epochs"}
    if args.arm in ("oracle", "both"):
        out["oracle"] = run_oracle(case, k, bnfloop, args.iters, args.seed, args.threads, log)
    if args.arm in ("product", "both"):
        out["product"] = run_product(case, k, bnfloop, args.iters, args.seed, args.path, log,
                                     dense_precision=args.dense_precision)
    if args.arm == "both":
        out["compare"] = compare(out["product"], out["oracle"])
        log(json.dumps(out["compare"]))
    text = json.dumps(out)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        open(args.out, "w").write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
