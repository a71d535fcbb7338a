"""Fit many meshes at once: the loop of the Dual-DMP training driver (tests/drivers/main.py) over a list of dataset
directories, with up to ``--batch`` fits sharing one GPU as one ``MultiDualStep`` iteration.

    python scripts/fit_many.py data/mesh_a data/mesh_b ... --iter 1000 --batch 8
    torchrun --nproc_per_node 8 scripts/fit_many.py data/* --batch 8      # directories sharded over the GPUs

Each directory holds ``*_noise.obj`` and ``*_smooth.obj`` (and optionally ``*_gt.obj``), as for the single-mesh driver.
Every 10 epochs the fits with a ``*_gt.obj`` are evaluated on the GPU (``distance.BatchEvaluator``: MAD and the
two-sided distance to the clean mesh, all fits of the batch in a few launches, no host synchronisation); every 100
epochs the current mesh is saved to ``<input>/output/<epoch>_ddmp=<mad>.obj`` by a writer thread while training goes on.
At the end one JSON line per mesh is printed; fits with a clean mesh also report ``final_hausdorff``,
``final_hausdorff_rel`` and ``final_mean_rel`` of the last evaluation (None before the first).
"""
from __future__ import annotations

import argparse
import glob
import json
import os
import queue
import sys
import threading

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
    p.add_argument("--dense-precision", default="fp32", choices=["fp32", "f16x1"],
                   help="accuracy contract of the networks' dense transforms: fp32 (default) or f16x1 (one fp16 product "
                        "on the tensor-core layers; DESIGN.md 4.2)")
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


class SnapshotWriter:
    """One thread that writes OBJ snapshots (``synth.write_obj``, the format of ``Mesh.save``) off the training thread.
    ``put(event, jobs)``: once ``event`` (the device-to-host copies of the positions) has completed, write each
    ``(path, vs, faces)``.  ``close()`` waits for every write and re-raises the first error."""

    def __init__(self):
        self._q: queue.Queue = queue.Queue()
        self._error = None
        self._thread = threading.Thread(target=self._run, name="fit_many-snapshots", daemon=True)
        self._thread.start()

    def _run(self) -> None:
        from dual_dmp_b200.synth import write_obj
        while True:
            item = self._q.get()
            if item is None:
                return
            event, jobs = item
            if self._error is not None:
                continue
            try:
                if event is not None:
                    event.synchronize()
                for path, vs, faces in jobs:
                    write_obj(path, vs.numpy() if hasattr(vs, "numpy") else vs, faces)
            except BaseException as e:      # re-raised on the training thread by close()
                self._error = e

    def put(self, event, jobs) -> None:
        if self._error is not None:
            raise self._error
        self._q.put((event, jobs))

    def close(self) -> None:
        self._q.put(None)
        self._thread.join()
        if self._error is not None:
            raise self._error


def fit_batch(dirs, args, device) -> list:
    import torch

    import dual_dmp_b200.util.datamaker as Datamaker
    import dual_dmp_b200.util.loss as Loss
    from dual_dmp_b200.distance import BatchEvaluator
    from dual_dmp_b200.step import MultiDualStep
    from dual_dmp_b200.util.networks import NormalNet, PosNet

    k = (args.k1, args.k2, args.k3, args.k4, args.k5)
    fits, meta = [], []
    for d in dirs:
        mesh_dic, dataset = Datamaker.create_dataset(d)
        gt, n_mesh, o1 = mesh_dic["gt_mesh"], mesh_dic["n_mesh"], mesh_dic["o1_mesh"]
        out_dir = os.path.join(d, "output")
        os.makedirs(out_dir, exist_ok=True)
        fits.append(dict(posnet=PosNet(device).to(device), normnet=NormalNet(device).to(device), dataset=dataset,
                         n_mesh=n_mesh, k=k, pos_lr=args.pos_lr, norm_lr=args.norm_lr, grad_clip=args.grad_crip,
                         dense_precision=args.dense_precision))
        mad = Loss.mad(n_mesh.fn, gt.fn) if gt is not None else None
        meta.append(dict(input=d, out_dir=out_dir, gt=gt, o1=o1, initial_mad=mad, mad=mad))
    step = MultiDualStep(fits, bnfloop=args.bnfloop)
    with_gt = [i for i, m in enumerate(meta) if m["gt"] is not None]
    evaluator = BatchEvaluator([meta[i]["o1"] for i in with_gt], [meta[i]["gt"] for i in with_gt], device) \
        if with_gt else None
    side = torch.cuda.Stream(device)
    writer = SnapshotWriter()
    loss = report = None
    try:
        for epoch in range(1, args.iter + 1):
            loss = step.step(epoch)
            if epoch % 10 == 0 and evaluator is not None:
                report = evaluator.evaluate([step.pos[i] for i in with_gt])
            if epoch % 100 == 0:
                if report is not None:       # the file names need the MADs: one read for the batch
                    for i, mad in zip(with_gt, report["mad"].tolist()):
                        meta[i]["mad"] = mad
                # positions to pinned host buffers on a side stream; the next step waits for the copies only
                cur = torch.cuda.current_stream(device)
                side.wait_stream(cur)
                with torch.cuda.stream(side):
                    host = [torch.empty(p.shape, dtype=p.dtype, pin_memory=True).copy_(p, non_blocking=True)
                            for p in step.pos]
                    done = torch.cuda.Event()
                    done.record(side)
                cur.wait_stream(side)
                writer.put(done, [(os.path.join(m["out_dir"], "{}_ddmp={:.3f}.obj".format(
                    epoch, m["mad"] if m["mad"] is not None else float("nan"))), h, m["o1"].faces)
                    for m, h in zip(meta, host)])
    finally:
        writer.close()
    final = loss.to("cpu").tolist()
    finals = {}
    if report is not None:
        mads, h, hr, mr = (report[k].tolist() for k in ("mad", "hausdorff", "hausdorff_rel", "mean_rel"))
        for j, i in enumerate(with_gt):
            meta[i]["mad"] = mads[j]
            finals[i] = dict(final_hausdorff=h[j], final_hausdorff_rel=hr[j], final_mean_rel=mr[j])
    out = []
    for i, m in enumerate(meta):
        r = dict(input=m["input"], iters=args.iter, final_loss=final[i], initial_mad=m["initial_mad"],
                 final_mad=m["mad"])
        if m["gt"] is not None:
            r.update(finals.get(i, dict(final_hausdorff=None, final_hausdorff_rel=None, final_mean_rel=None)))
        out.append(r)
    return out


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
