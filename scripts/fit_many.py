"""Fit many meshes at once: the loop of the Dual-DMP training driver (tests/drivers/main.py) over a list of dataset
directories, with up to ``--batch`` fits sharing one GPU as one ``MultiDualStep`` iteration.

    python scripts/fit_many.py data/mesh_a data/mesh_b ... --iter 1000 --batch 8
    torchrun --nproc_per_node 8 scripts/fit_many.py data/* --batch 8      # directories sharded over the GPUs

Each directory holds ``*_noise.obj`` and ``*_smooth.obj`` (and optionally ``*_gt.obj``), as for the single-mesh driver.
Every 10 epochs the MAD against ``*_gt.obj`` is evaluated when it exists; every 100 epochs the current mesh is saved to
``<input>/output/<epoch>_ddmp=<mad>.obj``.  At the end one JSON line per mesh is printed.
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH_HELP = ("fits per GPU batch (the list is run in chunks of this size).  Memory bounds it: the saved activations "
              "of one fit come to about 15 GB per 1M faces, so about 3 GB per 200K-face mesh; a 180 GB B200 holds a "
              "batch of about 50 such fits, fewer with other work on the card.")


def get_parser() -> argparse.ArgumentParser:
    p = argparse.ArgumentParser(description="Dual Deep Mesh Prior, many meshes per GPU")
    p.add_argument("inputs", nargs="+", help="dataset directories (a directory without *_noise.obj is searched one "
                                             "level down for dataset directories)")
    p.add_argument("--pos_lr", type=float, default=0.01)
    p.add_argument("--norm_lr", type=float, default=0.01)
    p.add_argument("--iter", type=int, default=1000)
    p.add_argument("--k1", type=float, default=3.0)
    p.add_argument("--k2", type=float, default=4.0)
    p.add_argument("--k3", type=float, default=4.0)
    p.add_argument("--k4", type=float, default=4.0)
    p.add_argument("--k5", type=float, default=1.0)
    p.add_argument("--grad_crip", type=float, default=0.8)
    p.add_argument("--bnfloop", type=int, default=1)
    p.add_argument("--batch", type=int, default=8, help=BATCH_HELP)
    return p


def parse_args(argv=None) -> argparse.Namespace:
    args = get_parser().parse_args(argv)
    if args.iter < 1:
        raise SystemExit("fit_many: --iter must be at least 1")
    if args.batch < 1:
        raise SystemExit("fit_many: --batch must be at least 1")
    if args.bnfloop < 0:
        raise SystemExit("fit_many: --bnfloop must not be negative")
    return args


def is_dataset(path: str) -> bool:
    return bool(glob.glob(os.path.join(path, "*_noise.obj"))) and bool(glob.glob(os.path.join(path, "*_smooth.obj")))


def discover(inputs) -> list:
    """dataset directories in the order given; a directory that is not one contributes its sorted sub-directories
    that are"""
    out = []
    for p in inputs:
        p = os.path.normpath(p)
        if is_dataset(p):
            out.append(p)
        elif os.path.isdir(p):
            out += [d for d in sorted(glob.glob(os.path.join(p, "*"))) if os.path.isdir(d) and is_dataset(d)]
        else:
            raise SystemExit(f"fit_many: {p} is not a directory")
    if not out:
        raise SystemExit("fit_many: no dataset directory (with *_noise.obj and *_smooth.obj) found")
    return out


def chunks(items, size: int):
    return [items[i: i + size] for i in range(0, len(items), size)]


def fit_batch(dirs, args, device) -> list:
    import torch

    import dual_dmp_b200.util.datamaker as Datamaker
    import dual_dmp_b200.util.loss as Loss
    from dual_dmp_b200.step import MultiDualStep
    from dual_dmp_b200.util.mesh import Mesh
    from dual_dmp_b200.util.networks import NormalNet, PosNet

    k = (args.k1, args.k2, args.k3, args.k4, args.k5)
    fits, meta = [], []
    for d in dirs:
        mesh_dic, dataset = Datamaker.create_dataset(d)
        gt, n_mesh, o1 = mesh_dic["gt_mesh"], mesh_dic["n_mesh"], mesh_dic["o1_mesh"]
        out_dir = os.path.join(d, "output")
        os.makedirs(out_dir, exist_ok=True)
        fits.append(dict(posnet=PosNet(device).to(device), normnet=NormalNet(device).to(device), dataset=dataset,
                         n_mesh=n_mesh, k=k, pos_lr=args.pos_lr, norm_lr=args.norm_lr, grad_clip=args.grad_crip))
        mad = Loss.mad(n_mesh.fn, gt.fn) if gt is not None else None
        meta.append(dict(input=d, out_dir=out_dir, gt=gt, o1=o1, initial_mad=mad, mad=mad))
    step = MultiDualStep(fits, bnfloop=args.bnfloop)
    loss = None
    for epoch in range(1, args.iter + 1):
        loss = step.step(epoch)
        if epoch % 10 == 0:
            for i, m in enumerate(meta):
                m["o1"].vs = step.pos[i].to("cpu").numpy().copy()
                Mesh.compute_face_normals(m["o1"])
                Mesh.compute_vert_normals(m["o1"])
                if m["gt"] is not None:
                    m["mad"] = Loss.mad(m["o1"].fn, m["gt"].fn)
        if epoch % 100 == 0:
            for m in meta:
                mad = m["mad"] if m["mad"] is not None else float("nan")
                Mesh.save(m["o1"], os.path.join(m["out_dir"], "{}_ddmp={:.3f}.obj".format(epoch, mad)))
    final = loss.to("cpu").tolist()
    return [dict(input=m["input"], iters=args.iter, final_loss=final[i], initial_mad=m["initial_mad"],
                 final_mad=m["mad"]) for i, m in enumerate(meta)]


def main(argv=None) -> None:
    args = parse_args(argv)
    import torch

    from dual_dmp_b200 import dist
    rank, local_rank, world = dist.env_rank_world()
    device = torch.device("cuda", local_rank)
    torch.cuda.set_device(device)
    dist.init(device=device)
    dirs = discover(args.inputs)
    mine = [dirs[i] for i in dist.shard_items(len(dirs), rank, world)]
    results = []
    for batch in chunks(mine, args.batch):
        results += fit_batch(batch, args, device)
    for r in results:
        print(json.dumps(dict(r, rank=rank)), flush=True)


if __name__ == "__main__":
    main()
