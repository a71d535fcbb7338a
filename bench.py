#!/usr/bin/env python
"""Benchmark of the Dual-DMP training hot path (BASELINE.json metric: train iters/s of the dual GCN step —
PosNet + NormalNet forward, five losses, backward, clip, Adam; reference main.py:88-110 — at 1M faces).

  python bench.py --gpus N --steps K --warmup W            our arm   (libddmp_b200 CUDA kernels)
        N = 1: one 1M-face mesh on one GPU (BASELINE.json configs[2], the metric's configuration).
        N > 1: ONE mesh of N x 1M faces (icosphere n = round(224 sqrt N)) range-partitioned over the N GPUs with NCCL
               halo exchange + BatchNorm / gradient all-reduce (configs[4]'s mechanism, weak scaling); value is in
               1M-face-equivalent iters/s so the N = 1 point is the same quantity.  --mode independent = one mesh fit
               per GPU (configs[3]'s mechanism), --mode partition --freq n = strong scaling on a fixed mesh.
  python bench.py --impl reference --gpus N ...            reference arm: the CPU oracle port of the reference's
                                                           PyG path on the host cores, timed on the SAME 1M-face mesh
                                                           (as many whole steps as fit the time budget)

One JSON line on stdout (rank 0).  See DESIGN.md "Measurement" for every field.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _claim_stdout():
    """stdout must carry the one JSON line only, but libraries write to file descriptor 1 behind Python's back (NCCL
    prints its version banner there).  Keep a private duplicate of the real stdout for the result line and point
    descriptor 1 at stderr for everything else."""
    sys.stdout.flush()
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return real


RESULT_OUT = _claim_stdout() if __name__ == "__main__" else sys.stdout

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "train iters/s (dual GCN fwd+bwd+loss+clip+Adam)"
WIDTHS_POS = [16, 32, 64, 128, 256, 256, 512, 512, 256, 256, 128, 64, 32]
WIDTHS_NORM = [7, 32, 64, 128, 256, 256, 512, 512, 256, 256, 128, 64, 32]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", "--freq", dest="n", type=int, default=224,
                    help="icosphere frequency: F = 20 n^2 (224 -> 1,003,520 faces); use --freq under torchrun")
    ap.add_argument("--bnfloop", type=int, default=1)
    ap.add_argument("--k", type=float, nargs=5, default=[3.0, 4.0, 4.0, 4.0, 1.0])
    ap.add_argument("--cpu-n", type=int, default=None,
                    help="icosphere frequency of the CPU arm's mesh (default: the benchmark mesh itself when host RAM "
                         "allows, else the largest that fits, flagged as extrapolated)")
    ap.add_argument("--cpu-budget-s", type=float, default=240.0, help="wall-clock budget of the reference arm's steps")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="run PosNet and NormalNet on one stream")
    ap.add_argument("--no-graph", action="store_true", help="time the eager drop-in step instead of the CUDA-graph one")
    ap.add_argument("--mode", default="auto", choices=["auto", "independent", "partition", "partition-weak"],
                    help="auto: N=1 -> one mesh on one GPU; N>1 -> 'partition-weak' (one mesh of N x 1M faces "
                         "range-partitioned over the GPUs, NCCL halo exchange; weak scaling).  'independent' = one mesh "
                         "fit per GPU, no data-path collective.  'partition' = strong scaling on the --freq mesh")
    ap.add_argument("--no-mode-a", action="store_true", help="N>1: skip the independent-replica side measurement")
    ap.add_argument("--no-small", action="store_true", help="N=1: skip the fandisk-sized CAD-weights side measurement")
    ap.add_argument("--detail", default=None, help="write a per-kernel-group timing table (JSON) to this path")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="write what the last timed step computed (loss, PosNet / NormalNet outputs, updated "
                         "parameters) as DIR/<name>.npy, so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# ---------------------------------------------------------------------------------------------------------------------
def build_case(n, device=None):
    """synthetic case with the reference's data conventions (SURVEY.md §8d).  ``device``: run the preprocessing (rescale,
    noise along the vertex normal, 30 smoothing sweeps) with the float64 device kernels of dual_dmp_b200.preprocess
    instead of numpy -- used for the multi-million-face meshes of the partitioned mode"""
    from dual_dmp_b200 import synth
    from dual_dmp_b200.util.datamaker import dataset_from_meshes
    from dual_dmp_b200.util.mesh import Mesh
    from types import SimpleNamespace
    if device is not None:
        from dual_dmp_b200 import preprocess
        case = preprocess.make_case_device(n, device)
    else:
        case = synth.make_case(n)
    n_mesh = Mesh(vs=case.noise_vs, faces=case.faces)
    s_mesh = SimpleNamespace(vs=case.smooth_vs)      # only the smoothed vertices are read (reference datamaker.py:87)
    return n_mesh, s_mesh, dataset_from_meshes(n_mesh, s_mesh)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, loss, pos, norm, posnet, normnet):
    """Write the results of one step as float32 / float64 .npy files.  The mesh, its noise and the initial weights are
    seeded, so the same arguments give the same inputs on every run.  Meshes so large that the files would exceed
    DUMP_LIMIT_BYTES keep a fixed, seeded sample of the rows of ``pos`` and ``norm`` (sorted row indices, seed 0)."""
    flat = lambda net: torch.cat([p.detach().reshape(-1) for p in net.parameters()]).cpu().numpy()   # noqa: E731
    fixed = {"loss": np.asarray([loss.item()], dtype=np.float64),
             "posnet_params": flat(posnet), "normnet_params": flat(normnet)}
    rows = {"pos": pos.detach().float().cpu().numpy(), "norm": norm.detach().float().cpu().numpy()}
    budget = DUMP_LIMIT_BYTES - 4096 - sum(a.nbytes for a in fixed.values())      # 4096: room for the .npy headers
    total = sum(a.nbytes for a in rows.values())
    if total > budget:
        rng = np.random.default_rng(0)
        rows = {k_: a[np.sort(rng.choice(len(a), int(len(a) * budget / total), replace=False))]
                for k_, a in rows.items()}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in {**fixed, **rows}.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def spmm_bytes(n_nodes, nnz, C):
    """SURVEY.md §8d: rowptr + col + w + read H once + write Y once."""
    return 4 * ((n_nodes + 1) + 2 * nnz + 2 * n_nodes * C)


def _sha256(path):
    import hashlib
    return hashlib.sha256(open(path, "rb").read()).hexdigest()


def spmm_traffic(args, n_sp, sp_bytes):
    """DRAM traffic per SpMM launch (dram__bytes_read.sum + dram__bytes_write.sum, average over the 48 launches of a
    step) from the committed ncu capture -- reported only when that capture was taken on the spmm.cu that is being
    benchmarked (sha256 of the kernel sources recorded by scripts/spmm_traffic.py) and on the benchmark mesh; else null."""
    path = os.path.join(ROOT, "profiles", "spmm_dram_traffic_r2.json")
    try:
        tj = json.load(open(path))
    except Exception:
        return None, "no ncu capture for this build (profiles/spmm_dram_traffic_r2.json missing)"
    import hashlib
    srcs = [os.path.join(ROOT, "dual_dmp_b200", "csrc", f) for f in ("spmm.cu", "spmm_tile.cu")]
    sha = hashlib.sha256(b"".join(open(p_, "rb").read() for p_ in srcs)).hexdigest()
    if tj.get("spmm_sources_sha256") != sha:
        return None, "ncu capture is of older aggregation kernels (sha256 of spmm.cu + spmm_tile.cu differs): not reported"
    if args.n != tj.get("n") or not n_sp:
        return None, "ncu capture is of another mesh"
    return tj["dram_bytes_per_launch_avg"], (
        "dram__bytes_read.sum + dram__bytes_write.sum, average per launch over the %d launches of a step, ncu capture "
        "%s of this spmm.cu; algorithmic average per launch = %.0f" % (tj.get("launches"), tj.get("source"),
                                                                      sp_bytes / n_sp))


def loss_bytes(V, F, E, bnfloop):
    """SURVEY.md §8d algorithmic bytes of the loss phase, forward + backward (fp32 values, int32 indices)"""
    fwd = (24 * V                              # pos_rec
           + 24 * F                            # norm_rec
           + 4 * (V + 1) + 4 * 2 * E + 24 * V  # uniform Laplacian over the vertex CSR
           + 12 * F + 12 * V + 12 * F          # pos_norm: faces + pos + normals
           + 12 * F + 12 * V + 16 * F          # face geometry of the BNF setup: read faces + pos, write fc | fa
           + bnfloop * 48 * F)                 # BNF iterations: f2f + read n + write n + wc*fa
    return 2 * fwd


def loss_phase_roofline(stepper, n_mesh, args, peak, reps=20):
    """The five losses, forward + backward down to d(loss)/d(pos) and d(loss)/d(norm), captured as one CUDA graph and
    replayed between CUDA events; L2 is flushed (256 MB memset) before every replay because in the real step the loss
    kernels run after >10 GB of activation traffic, i.e. on cold index tables."""
    from dual_dmp_b200._lib import lib
    from dual_dmp_b200.util import loss as L
    dev = stepper.device
    k = args.k
    pos = stepper.pos.detach().clone().requires_grad_(True)
    nrm = stepper.norm.detach().clone().requires_grad_(True)
    tgt_vs, tgt_fn = stepper.tgt_vs, stepper.tgt_fn

    def body():
        pos.grad = None
        nrm.grad = None
        if stepper.fused_loss:          # what DualStep runs: one cooperative kernel (ddmp_dual_loss) + two scalings
            loss, _ = L.dual_loss(pos, nrm, n_mesh, tgt_vs, tgt_fn, k, args.bnfloop, 1.0)
        else:
            l1 = L.pos_rec_loss(pos, tgt_vs)
            l2 = L.mesh_laplacian_loss(pos, n_mesh)
            l3 = L.norm_rec_loss(nrm, tgt_fn)
            l4, _ = L.fn_bnf_loss(pos, nrm, n_mesh, loop=args.bnfloop)
            l5 = L.pos_norm_loss(pos, nrm, n_mesh)
            loss = k[0] * l1 + k[1] * l2 + k[2] * l3 + k[3] * l4 + k[4] * l5
        loss.backward()
        return loss.detach()

    side = torch.cuda.Stream(dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for _ in range(2):
            body()
        l0 = lib.query("ddmp_launch_count")
        body()
        launches = lib.query("ddmp_launch_count") - l0
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        body()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    ms = []
    for i in range(reps + 2):
        flush.zero_()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        g.replay()
        e.record()
        torch.cuda.synchronize()
        if i >= 2:
            ms.append(s.elapsed_time(e))
    V, F, E = len(n_mesh.vs), len(n_mesh.faces), len(n_mesh.edges)
    nbytes = loss_bytes(V, F, E, args.bnfloop)
    t = sum(ms) / len(ms)
    ach = nbytes / (t * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": ("dual_loss_kernel (one cooperative launch): " if stepper.fused_loss else "loss phase: ")
                                      + "pos_rec + laplacian + norm_rec + bnf (setup, %d iteration(s)) + pos_norm, "
                                        "forward and backward to d/dpos, d/dnorm" % args.bnfloop,
            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "frac_of_nominal_8000": ach / 8000.0,
            "algorithmic_bytes": nbytes, "ms": t, "library_launches": int(launches),
            "timed_in": "CUDA-graph replay of the loss phase alone, %d replays, L2 flushed before each (cold index "
                        "tables, as inside the step); the working set (~%d MB) fits L2, so values above the HBM peak "
                        "would mean cache residency" % (reps, nbytes // 2 // (1 << 20))}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for i, nm in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


# ---------------------------------------------------------------------------------------------------------------------
def run_ours(args):
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    assert torch.cuda.is_available(), "bench.py (our arm) needs a CUDA device; there is no CPU fallback"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)

    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200._lib import lib
    from dual_dmp_b200.util import loss as L
    from dual_dmp_b200.util.networks import NormalNet, PosNet

    # mode A (SURVEY.md §8e): every rank fits its own mesh, no data-path collective -> weak scaling
    n_mesh, s_mesh, ds = build_case(args.n)
    V, F = len(n_mesh.vs), len(n_mesh.faces)
    torch.manual_seed(0)
    posnet, normnet = PosNet(dev).to(dev), NormalNet(dev).to(dev)
    opt_pos = torch.optim.Adam(posnet.parameters(), lr=0.01)
    opt_norm = torch.optim.Adam(normnet.parameters(), lr=0.01)
    k = args.k

    def step(ds_, tgt_vs, tgt_fn, epoch, sync_loss):
        posnet.train(); normnet.train()
        opt_pos.zero_grad(); opt_norm.zero_grad()
        pos = posnet(ds_)
        l1 = L.pos_rec_loss(pos, tgt_vs)
        l2 = L.mesh_laplacian_loss(pos, n_mesh)
        nrm = normnet(ds_)
        l3 = L.norm_rec_loss(nrm, tgt_fn)
        l4, _ = L.fn_bnf_loss(pos, nrm, n_mesh, loop=args.bnfloop)
        if epoch <= 100:
            l4 = l4 * 0.0
        l5 = L.pos_norm_loss(pos, nrm, n_mesh)
        loss = k[0] * l1 + k[1] * l2 + k[2] * l3 + k[3] * l4 + k[4] * l5
        loss.backward()
        torch.nn.utils.clip_grad_norm_(normnet.parameters(), 0.8)
        opt_pos.step(); opt_norm.step()
        return loss.item() if sync_loss else loss

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
            torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = lib.query("ddmp_launch_count")
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if dist is not None:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), lib.query("ddmp_launch_count") - launches0

    # ---- resident arm: inputs and targets already in HBM -----------------------------------------------------------
    # dual_dmp_b200.step.DualStep = the same loop body (same autograd Functions, same kernels), inputs resident,
    # replayed as a CUDA graph.  --no-graph times the eager drop-in step instead.
    import copy
    from dual_dmp_b200.step import DualStep
    stepper = DualStep(posnet, normnet, ds, n_mesh, k=k, bnfloop=args.bnfloop, capture=not args.no_graph,
                       overlap=not args.no_overlap)
    ds_dev, tgt_vs, tgt_fn = stepper.dataset, stepper.tgt_vs, stepper.tgt_fn
    opt_pos, opt_norm = stepper.opt_pos, stepper.opt_norm
    epoch0 = 101   # past the reference's 100-iteration BNF warm-up, so every loss term is live

    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(max(args.warmup, 5)):            # 3 eager warm-up calls, then capture, then replays
        stepper.step(epoch0 + i)
    last_loss = [None]

    def timed_step(i):
        last_loss[0] = stepper.step(epoch0 + i)

    ms, _ = timed(timed_step, args.steps, 0)
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:             # before the passes below move the parameters on
        dump_outputs(args.dump_outputs, last_loss[0], stepper.pos, stepper.norm, posnet, normnet)
    ms_per_step = ms / args.steps
    value = world * 1000.0 / ms_per_step

    # ---- roofline pass: the same K steps eagerly, every SpMM launch bracketed by CUDA events on its stream ----------
    spmm_events = []
    orig_spmm = F_.spmm_gcn

    def spmm_timed(graph, H, *a, **kw):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        out = orig_spmm(graph, H, *a, **kw)
        e.record()
        spmm_events.append((s, e, spmm_bytes(graph.n, graph.nnz, H.shape[1]), H.shape[1], graph.n))
        return out

    # ... and every dense feature transform (X.W^T, dH.W, dH^T.X) the same way, for the tensor-pipe roofline
    gemm_events = []
    orig_gemms = (F_.gemm_xw, F_.gemm_dx, F_.gemm_dw)

    def timed_gemm(fn, kind):
        def wrapped(*a, **kw):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = fn(*a, **kw)
            e.record()
            if kind == "xw":
                W = a[1]; rows = kw.get("n") or a[0].shape[0]; cout, cin = W.shape
            elif kind == "dx":
                W = a[1]; rows = a[0].shape[0]; cout, cin = W.shape
            else:
                rows, cout = a[0].shape; cin = a[2]
            # which split the library picks for this launch (mirrors csrc/gemm_tc.cu): fp16 pieces when the caller
            # supplied operand bounds, else 3xTF32
            if kind == "dw":
                f16 = kw.get("amax_dh") is not None and kw.get("amax_x") is not None
            else:
                f16 = kw.get("amax") is not None
            gemm_events.append((s, e, 2.0 * rows * cin * cout, min(cin, cout) >= 64, f16))
            return out
        return wrapped

    F_.spmm_gcn = spmm_timed
    F_.gemm_xw, F_.gemm_dx, F_.gemm_dw = (timed_gemm(orig_gemms[0], "xw"), timed_gemm(orig_gemms[1], "dx"),
                                          timed_gemm(orig_gemms[2], "dw"))
    pt = PhaseTimer()
    pt.patch(F_, "bn_bwd_spmm_tile", "BatchNorm backward + backward aggregation (reduce, finalize, fused tile kernel)")
    pt.patch(F_, "bn_lrelu_backward", "BatchNorm backward (reduce, finalize, apply)")
    pt.patch(F_, "bn_stats_finalize", "BatchNorm statistics finalize")
    pt.patch(L, "dual_loss", "losses forward+backward (dual_loss_kernel)")
    pt.patch(stepper.opt_pos, "step", "clip + Adam")
    pt.patch(stepper.opt_norm, "step", "clip + Adam")
    was_overlap, stepper.overlap = stepper.overlap, False      # one stream: per-launch events must not time-slice
    # Per-launch events are only meaningful while the GPU, not the host, is the bottleneck: an event pair around a
    # launch also covers the time the GPU waits for that launch to arrive.  Two untimed eager steps absorb one-time
    # costs (allocator growth after the graph capture), and every step starts with a ~30 ms spin kernel so the host
    # is a full step ahead when the short kernels of the narrow layers are issued; the spin time is measured with
    # its own events and subtracted from the eager step time.
    spin_events = []

    def eager_step(i):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        torch.cuda._sleep(60_000_000)
        e.record()
        spin_events.append((s, e))
        return stepper._body(False)

    for i in range(2):
        stepper._body(False)
    spmm_events.clear()
    gemm_events.clear()
    ms_eager, launches = timed(eager_step, args.steps, 0)
    ms_eager -= sum(s.elapsed_time(e) for s, e in spin_events)
    launches -= 0                                               # the spin kernel is torch's, not counted by the library
    stepper.overlap = was_overlap
    F_.spmm_gcn = orig_spmm
    F_.gemm_xw, F_.gemm_dx, F_.gemm_dw = orig_gemms
    pt.restore()
    torch.cuda.synchronize()
    phases = {k_: v / args.steps for k_, v in pt.totals_ms().items()}
    tc_ms = sum(s.elapsed_time(e) for s, e, _, tc, _ in gemm_events if tc)
    tc_flop = sum(f for _, _, f, tc, _ in gemm_events if tc)
    tc16_ms = sum(s.elapsed_time(e) for s, e, _, tc, f16 in gemm_events if tc and f16)
    tc16_flop = sum(f for _, _, f, tc, f16 in gemm_events if tc and f16)
    ff_ms = sum(s.elapsed_time(e) for s, e, _, tc, _ in gemm_events if not tc)
    ff_flop = sum(f for _, _, f, tc, _ in gemm_events if not tc)
    n_tc = sum(1 for ev in gemm_events if ev[3])
    gemm_events.clear()
    sp_ms = sum(s.elapsed_time(e) for s, e, _, _, _ in spmm_events)
    sp_bytes = sum(b for _, _, b, _, _ in spmm_events)
    n_sp = len(spmm_events)
    by_width = {}
    for s, e, b, C, nn in spmm_events:
        d = by_width.setdefault(f"n={nn},C={C}", [0.0, 0, 0])
        d[0] += s.elapsed_time(e); d[1] += b; d[2] += 1
    spmm_events.clear()

    # ---- end-to-end arm: host buffers, H2D of the step's inputs and D2H of the loss inside the timed region ---------
    e2e = None
    if not args.no_e2e:
        ds_host = copy.copy(ds).pin_memory()
        vs_host = torch.from_numpy(n_mesh.vs).pin_memory()       # float64 targets, uploaded every step like the
        fn_host = torch.from_numpy(n_mesh.fn).pin_memory()       # reference's loss calls do (util/loss.py:10,52)
        h2d = sum(t.numel() * t.element_size() for t in (ds_host.z1, ds_host.z2, ds_host.x_pos, vs_host, fn_host))

        # (1) DualStep with streamed inputs: every step uploads its inputs from pinned host memory (on a copy stream,
        #     one step ahead, overlapping the running iteration) and reads its loss back to the host
        def streamed(i):
            loss = stepper.step(epoch0 + i)
            stepper.prefetch(ds_host, vs_host, fn_host)           # inputs of the next step
            return loss.item()

        stepper.prefetch(ds_host, vs_host, fn_host)               # inputs of the first warm-up step
        ms_s, _ = timed(streamed, args.steps, args.warmup)
        torch.cuda.synchronize()

        # (2) the reference's own loop body over the drop-in modules (eager, torch.optim.Adam, synchronous uploads)
        opt_pos = torch.optim.Adam(posnet.parameters(), lr=0.01)
        opt_norm = torch.optim.Adam(normnet.parameters(), lr=0.01)
        ms_e, _ = timed(lambda i: step(ds_host, n_mesh.vs, n_mesh.fn, epoch0 + i, True), args.steps, args.warmup)
        e2e = {"value": world * 1000.0 * args.steps / ms_s, "unit": "iters/s", "h2d_bytes_per_step": int(h2d),
               "d2h_bytes_per_step": 8,
               "path": "DualStep.prefetch + DualStep.step + loss.item(): per-step upload of z1/z2/x_pos/targets from "
                       "pinned host memory on a copy stream (one step ahead), graph replay, loss read back",
               "dropin_loop_value": world * 1000.0 * args.steps / ms_e,
               "dropin_loop": "reference main.py:88-110 verbatim over dual_dmp_b200.util modules (eager, synchronous "
                              "uploads, torch.optim.Adam)"}

    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    loss_roof = loss_phase_roofline(stepper, n_mesh, args, peak)
    achieved = sp_bytes / (sp_ms * 1e-3) / 1e9 if sp_ms > 0 else 0.0
    traffic, traffic_note = spmm_traffic(args, n_sp, sp_bytes)
    out = {
        "metric": METRIC, "value": value, "unit": "iters/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"synthetic icosphere n={args.n}: {F} faces / {V} vertices, Gaussian noise 0.2, "
                               f"k={args.k}, bnfloop={args.bnfloop}, one independent mesh fit per GPU",
                   "faces": F, "vertices": V, "l2_policy": "working set (>=10 GB of saved activations) exceeds L2",
                   "optimizer": "clip + Adam (reference main.py:108-110): library kernels ddmp_grad_norm + "
                                "ddmp_adam_step_dev over flat buffers in the resident arm, torch.optim.Adam in the e2e arm",
                   "step": "eager drop-in modules" if args.no_graph else
                           "dual_dmp_b200.step.DualStep: same kernels, replayed as a CUDA graph"},
        "e2e": e2e, "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "spmm_gcn_kernel (all GCN aggregation launches, fwd+bwd)",
                     "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "peak_source": "MEASURED_PEAKS.json hbm_gbs (measured copy)" if peaks else "fallback 6650",
                     "frac_of_nominal_8000": achieved / 8000.0, "traffic": traffic, "traffic_source": traffic_note,
                     "launches_per_step": n_sp // max(args.steps, 1), "share_of_step": sp_ms / ms_eager,
                     "timed_in": "eager pass of the same steps right after the timed region (CUDA events cannot be "
                                 "read back from inside a replayed graph), single stream; eager ms/step = %.3f"
                                 % (ms_eager / args.steps),
                     "algorithmic_bytes_per_step": sp_bytes // max(args.steps, 1)},
        "clocks": sampler.summary(),
    }
    bf16_sus = float(peaks.get("bf16_tflops_sustained", 1400.0))
    tc_tflops = tc_flop / (tc_ms * 1e-3) / 1e12 if tc_ms > 0 else 0.0
    out["roofline"]["by_width_GBps"] = {k_: round(v[1] / (v[0] * 1e-3) / 1e9, 1) for k_, v in by_width.items() if v[0] > 0}
    out["roofline"]["tensor"] = {
        "bound": "tensor", "kernel": "tc_gemm_nt16x2/nt16 (tcgen05 kind::f16, fp32 emulated with 3 fp16 MMAs: X.W^T and "
                                     "dH.W; tc_gemm_tn16x2/tn16: dH^T.X); all dense transforms of width >= 64",
        "achieved": tc_tflops, "unit": "TFLOP/s", "peak": bf16_sus, "frac": tc_tflops / bf16_sus,
        "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (cuBLAS bf16, kernel timed inside a long step)",
        "achieved_counts": "ALGORITHMIC fp32 flops 2*rows*Cin*Cout; an fp32 product costs 3 MMAs, so the ceiling "
                           "against this peak is 1/3 for the fp16-split launches (fp16 issues at the bf16 rate) and "
                           "1/6 for the 3xTF32 launches (half rate)",
        "fp16_split": {"tflops": tc16_flop / (tc16_ms * 1e-3) / 1e12 if tc16_ms > 0 else None,
                       "share_of_tc_time": tc16_ms / tc_ms if tc_ms > 0 else None,
                       "frac_of_ceiling": (3.0 * tc16_flop / (tc16_ms * 1e-3) / 1e12 / bf16_sus) if tc16_ms > 0 else None},
        "tf32_split": {"tflops": (tc_flop - tc16_flop) / ((tc_ms - tc16_ms) * 1e-3) / 1e12 if tc_ms > tc16_ms else None,
                       "frac_of_ceiling": (6.0 * (tc_flop - tc16_flop) / ((tc_ms - tc16_ms) * 1e-3) / 1e12 / bf16_sus)
                       if tc_ms > tc16_ms else None},
        "frac_of_split_ceiling": ((3.0 * tc16_flop + 6.0 * (tc_flop - tc16_flop)) / (tc_ms * 1e-3) / 1e12 / bf16_sus)
                                 if tc_ms > 0 else None,
        "launches_per_step": n_tc // max(args.steps, 1), "share_of_step": tc_ms / ms_eager,
        "algorithmic_flop_per_step": tc_flop / max(args.steps, 1),
        "ffma_small_width": {"tflops": ff_flop / (ff_ms * 1e-3) / 1e12 if ff_ms > 0 else None,
                             "share_of_step": ff_ms / ms_eager}}
    out["roofline"]["loss"] = loss_roof
    phases["GCN aggregation, forward (+ backward when unfused)"] = sp_ms / args.steps
    phases["dense transforms, tensor cores"] = tc_ms / args.steps
    phases["dense transforms, FFMA (width < 64)"] = ff_ms / args.steps
    phases["whole eager step"] = ms_eager / args.steps
    out["config"]["phases_ms_per_step"] = {k_: round(v, 3) for k_, v in sorted(phases.items())}
    if args.detail:
        os.makedirs(os.path.dirname(os.path.abspath(args.detail)), exist_ok=True)
        json.dump({k_: {"ms_total": v[0], "GBps": v[1] / (v[0] * 1e-3) / 1e9 if v[0] > 0 else None, "launches": v[2]}
                   for k_, v in by_width.items()}, open(args.detail, "w"), indent=1)
    if world == 1 and not args.no_small:
        out["config"]["cad_small_mesh"] = small_cad_line(dev)
    if not args.no_cpu_baseline and world == 1:
        torch.cuda.empty_cache()
        out["cpu_baseline"] = cpu_reference(args, max_steps=1, warmup=1, budget_s=120.0, case=(n_mesh, s_mesh))
    print(json.dumps(out), file=RESULT_OUT, flush=True)
    if dist is not None:
        dist.destroy_process_group()


# ---------------------------------------------------------------------------------------------------------------------
ORACLE_BYTES_PER_FACE = 135_000     # resident set of one oracle step (PyG-style saved edge messages), measured: 122-130 KB


def small_cad_line(dev, n=25, steps=200):
    """side measurement (not the headline): a fandisk-sized mesh (BASELINE.json configs[0]: 12,946 faces there, 12,500
    here) with the CAD loss weights of reference README.md:57 (k=3,0,3,4,2, bnfloop=5) -- the regime where launch count,
    not bandwidth, limits the step: CUDA-graph replay of DualStep against the eager drop-in loop"""
    from dual_dmp_b200._lib import lib
    from dual_dmp_b200.step import DualStep
    from dual_dmp_b200.util.networks import NormalNet, PosNet
    n_mesh, s_mesh, ds = build_case(n)
    k, loop = (3.0, 0.0, 3.0, 4.0, 2.0), 5
    res = {"workload": f"icosphere n={n}: {len(n_mesh.faces)} faces, k={list(k)}, bnfloop={loop}"}
    for label, capture in (("graph_replay", True), ("eager", False)):
        torch.manual_seed(0)
        p, q = PosNet(dev).to(dev), NormalNet(dev).to(dev)
        st = DualStep(p, q, ds, n_mesh, k=k, bnfloop=loop, capture=capture)
        for i in range(6):
            st.step(101 + i)
        torch.cuda.synchronize()
        l0 = lib.query("ddmp_launch_count")
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            st.step(107 + i)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        res[label] = {"ms_per_step": round(ms, 4), "iters_per_s": round(1000.0 / ms, 1)}
        if not capture:
            res[label]["library_launches_per_step"] = int((lib.query("ddmp_launch_count") - l0) // steps)
    return res


def _pick_cpu_mesh(args):
    """the benchmark mesh itself when the host has the RAM for the oracle's saved edge messages, else the largest
    smaller icosphere that fits (the result is then flagged as extrapolated)"""
    if args.cpu_n is not None:
        return args.cpu_n
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64 << 30
    for n in (args.n, 160, 128, 100, 64, 40):
        if n <= args.n and 20 * n * n * ORACLE_BYTES_PER_FACE * 1.15 < avail:
            return n
    return 20


def _cpu_threads():
    """thread count for the oracle: quick calibration (one warm + one timed step on a 32,000-face mesh per candidate)"""
    from oracle import step_ref
    from oracle.networks_ref import NormalNetRef, PosNetRef
    ncpu = os.cpu_count() or 1
    cands = sorted({min(8, ncpu), min(16, ncpu), ncpu})
    if len(cands) == 1:
        return cands[0], {}
    n_mesh, s_mesh, _ = build_case(40)
    ds = step_ref.make_dataset(n_mesh, s_mesh)
    seen = {}
    for th in cands:
        torch.set_num_threads(th)
        torch.manual_seed(0)
        nets = PosNetRef(), NormalNetRef()
        opts = [torch.optim.Adam(m.parameters(), lr=0.01) for m in nets]
        step_ref.train_step(nets[0], nets[1], opts[0], opts[1], ds, n_mesh, epoch=101)
        t0 = time.perf_counter()
        step_ref.train_step(nets[0], nets[1], opts[0], opts[1], ds, n_mesh, epoch=102)
        seen[th] = time.perf_counter() - t0
    return min(seen, key=seen.get), seen


def cpu_reference(args, max_steps, warmup, budget_s, case=None):
    """The oracle port of the reference's PyG CPU path (oracle/step_ref.py = reference main.py:88-110) timed on the
    host cores ON THE BENCHMARK MESH: ``warmup`` untimed steps, then whole steps until ``max_steps`` or the time
    budget is reached.  kind="port": torch_geometric is not installable here.  Nothing is extrapolated unless the
    host cannot hold the oracle's working set (then the largest mesh that fits is timed and the result is scaled
    linearly in faces, with ``extrapolated: true``)."""
    from oracle import step_ref
    from oracle.networks_ref import NormalNetRef, PosNetRef
    threads, calib = _cpu_threads()
    n = _pick_cpu_mesh(args)
    if case is not None and n == args.n:
        n_mesh, s_mesh = case
    else:
        n_mesh, s_mesh, _ = build_case(n)
    ds = step_ref.make_dataset(n_mesh, s_mesh)
    F = len(n_mesh.faces)
    target_faces = 20 * args.n * args.n
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    posnet, normnet = PosNetRef(), NormalNetRef()
    opt_pos = torch.optim.Adam(posnet.parameters(), lr=0.01)
    opt_norm = torch.optim.Adam(normnet.parameters(), lr=0.01)
    t_start = time.perf_counter()
    for i in range(warmup):
        step_ref.train_step(posnet, normnet, opt_pos, opt_norm, ds, n_mesh, tuple(args.k), args.bnfloop, 101 + i)
    times = []
    while len(times) < max_steps:
        t0 = time.perf_counter()
        step_ref.train_step(posnet, normnet, opt_pos, opt_norm, ds, n_mesh, tuple(args.k), args.bnfloop,
                            101 + warmup + len(times))
        times.append(time.perf_counter() - t0)
        if time.perf_counter() - t_start + times[-1] > budget_s:
            break
    dt = sum(times) / len(times)
    extrapolated = F != target_faces
    out = {"value": (1.0 / dt) * (F / float(target_faces)), "unit": "iters/s", "cores": threads, "kind": "port",
           "sample": f"{len(times)} whole step(s) after {warmup} warm-up of the oracle (reference main.py:88-110 restated, "
                     f"PyG-style GCNConv) on the icosphere n={n} mesh ({F} faces), {threads} threads: {dt:.2f} s/iter"
                     + ("" if not extrapolated else f"; host RAM too small for {target_faces} faces, scaled linearly"),
           "extrapolated": extrapolated, "steps_timed": len(times), "warmup_run": warmup,
           "measured_s_per_iter": dt, "sample_faces": F, "thread_calibration_s_per_iter_at_32000_faces": calib}
    return out


def run_reference(args):
    """reference arm: rank 0 alone times the CPU oracle on the benchmark mesh; steps / warmup in the line are the ones
    actually run (a 1M-face oracle step takes tens of seconds, so the time budget, not --steps, ends the loop)"""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    F_target = 20 * args.n * args.n
    base = cpu_reference(args, max_steps=max(1, args.steps), warmup=1, budget_s=args.cpu_budget_s)
    out = {"impl": "reference", "metric": METRIC, "value": base["value"], "unit": "iters/s",
           "n_gpus": int(os.environ.get("WORLD_SIZE", "1")), "steps": base["steps_timed"], "warmup": base["warmup_run"],
           "ms_per_step": 1000.0 * base["measured_s_per_iter"], "higher_is_better": True, "scaling": "weak",
           "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"synthetic icosphere n={args.n}: {F_target} faces / {10 * args.n * args.n + 2} vertices, "
                                  f"Gaussian noise 0.2, k={args.k}, bnfloop={args.bnfloop}; CPU oracle timed on "
                                  f"{base['sample_faces']} faces",
                      "faces": base["sample_faces"], "requested_steps": args.steps, "requested_warmup": args.warmup,
                      "extrapolated": base["extrapolated"]},
           "cpu_baseline": base,
           "e2e": {"value": base["value"], "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), file=RESULT_OUT, flush=True)


class PhaseTimer:
    """CUDA-event brackets around host-side calls (events on the current stream), summed per label"""

    def __init__(self):
        self.events, self.patches = {}, []

    def patch(self, obj, name, label):
        fn = getattr(obj, name)
        timer = self

        def wrapped(*a, **kw):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            out = fn(*a, **kw)
            e.record()
            timer.events.setdefault(label, []).append((s, e))
            return out
        setattr(obj, name, wrapped)
        self.patches.append((obj, name, fn))

    def restore(self):
        for obj, name, fn in reversed(self.patches):
            setattr(obj, name, fn)
        self.patches.clear()

    def totals_ms(self):
        return {k_: sum(s.elapsed_time(e) for s, e in v) for k_, v in self.events.items()}


def weak_freq(world, base=224):
    """icosphere frequency whose face count is closest to world x (20 base^2)"""
    import math
    return int(round(base * math.sqrt(world)))


def run_partitioned(args, weak):
    """mode B (SURVEY.md §8e): ONE mesh range-partitioned over all ranks, per-layer NCCL halo exchange, BatchNorm /
    gradient all-reduce.  weak: the mesh has world x 1M faces and value is in 1M-face-equivalent iters/s (N = 1 is
    then exactly the single-GPU benchmark); strong (--mode partition): the --freq mesh, value = iters/s of that fit."""
    import torch.distributed as dist
    from dual_dmp_b200 import dist as D
    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200._lib import lib
    from dual_dmp_b200.partition import PartitionedGraph, PartitionedNet
    from dual_dmp_b200.step import DualStep
    from dual_dmp_b200.util import loss as L
    from dual_dmp_b200.util.networks import NormalNet, PosNet
    rank, local_rank, world = D.env_rank_world()
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    n = weak_freq(world, args.n) if weak else args.n
    t_setup = time.perf_counter()
    n_mesh, s_mesh, ds = build_case(n, device=dev if n > 256 else None)
    V, F = len(n_mesh.vs), len(n_mesh.faces)
    F_base = 20 * args.n * args.n
    torch.manual_seed(0)
    posnet, normnet = PosNet(dev).to(dev), NormalNet(dev).to(dev)
    overlap = world > 1 and not args.no_overlap
    if world > 1:
        # one NCCL communicator per network: PosNet and NormalNet run on two compute streams (DualStep overlap), so the
        # halo exchange / BatchNorm all-reduce latency of one network is hidden behind the kernels of the other; the
        # collectives of one communicator stay in program order on every rank
        g_pos = dist.new_group(list(range(world))) if overlap else None
        g_nrm = dist.new_group(list(range(world))) if overlap else None
        ppos, pnrm = PartitionedNet(posnet, rank, world, group=g_pos), PartitionedNet(normnet, rank, world, group=g_nrm)
    else:
        ppos, pnrm = posnet, normnet
    # the reference loop body as one object; eager (no graph capture across NCCL calls)
    stepper = DualStep(ppos, pnrm, ds, n_mesh, k=args.k, bnfloop=args.bnfloop, capture=False, overlap=overlap)
    epoch0 = 101
    sampler = ClockSampler(local_rank)
    sampler.start()
    for i in range(max(args.warmup, 3)):
        stepper.step(epoch0 + i)
    setup_s = time.perf_counter() - t_setup

    def timed(fn, steps):
        D.barrier(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.query("ddmp_launch_count")
        e0.record()
        for i in range(steps):
            out = fn(i)
        e1.record()
        D.barrier(dev)
        return D.max_over_ranks(e0.elapsed_time(e1), dev), lib.query("ddmp_launch_count") - l0, out

    ms, launches, loss = timed(lambda i: stepper.step(epoch0 + 3 + i), args.steps)
    sampler.stop_flag = True
    ms_per_step = ms / args.steps
    scale = (F / float(F_base)) if weak else 1.0
    value = scale * 1000.0 / ms_per_step

    # ---- per-phase pass: the same steps with event brackets around every communication / kernel group ---------------
    pt = PhaseTimer()
    if world > 1:
        pt.patch(PartitionedGraph, "pack", "halo pack (ddmp_gather_rows)")
        pt.patch(PartitionedGraph, "all_to_all", "halo all_to_all (NCCL)")
        pt.patch(PartitionedGraph, "allreduce_", "all_reduce: BatchNorm sums + weight gradients (NCCL)")
        pt.patch(PartitionedGraph, "gather_outputs", "all_gather of the network outputs")
    pt.patch(F_, "spmm_gcn", "SpMM")
    pt.patch(F_, "bn_stats_finalize_peer", "BatchNorm statistics: reduce + all-reduce over NVLink peer memory + finalize (one kernel)")
    pt.patch(F_, "bn_lrelu_backward", "BatchNorm backward (reduce, peer-memory all-reduce + finalize, apply)")
    for nm in ("gemm_xw", "gemm_dx", "gemm_dw"):
        pt.patch(F_, nm, "dense transforms")
    pt.patch(L, "dual_loss", "losses forward + backward (dual_loss_kernel, replicated over the whole mesh)")
    pt.patch(stepper.opt_pos, "step", "clip + Adam")
    pt.patch(stepper.opt_norm, "step", "clip + Adam")
    sp_bytes = [0]
    orig_spmm = F_.spmm_gcn

    def spmm_counted(graph, H, *a, **kw):
        sp_bytes[0] += spmm_bytes(graph.n, graph.nnz, H.shape[1])
        return orig_spmm(graph, H, *a, **kw)
    F_.spmm_gcn = spmm_counted
    was_overlap, stepper.overlap = stepper.overlap, False      # one stream: per-phase events must not time-slice
    # two untimed steps first: the single-stream configuration allocates from its own (still empty) allocator pool, and
    # the cudaMalloc calls of its first step would be billed to whichever phase happened to allocate
    for i in range(2):
        stepper.step(epoch0 + 3 + args.steps + i)
    torch.cuda.synchronize()
    pt.events.clear()
    sp_bytes[0] = 0
    ms_ph, _, _ = timed(lambda i: stepper.step(epoch0 + 5 + args.steps + i), args.steps)
    stepper.overlap = was_overlap
    F_.spmm_gcn = orig_spmm
    pt.restore()
    torch.cuda.synchronize()
    phases = {k_: v / args.steps for k_, v in pt.totals_ms().items()}
    phases["whole step (this pass)"] = ms_ph / args.steps
    sp_ms = pt.totals_ms().get("SpMM", 0.0)

    # ---- e2e: this rank's slice of the inputs + the (replicated) float64 targets from pinned host memory every step,
    #      loss read back
    e2e = None
    if not args.no_e2e:
        if world > 1:
            pg_p, pg_n = posnet.last_graph, normnet.last_graph
            ids_p, ids_n = pg_p.own_ids.cpu(), pg_n.own_ids.cpu()
            host = {"z1": ds.z1.detach()[ids_p].contiguous().pin_memory(),
                    "x_pos": ds.x_pos.detach()[ids_p].contiguous().pin_memory(),
                    "z2": ds.z2.detach()[ids_n].contiguous().pin_memory()}
            dst = {"z1": ppos._cache[3], "x_pos": ppos._cache[4], "z2": pnrm._cache[3]}
        else:
            host = {"z1": ds.z1.detach().pin_memory(), "x_pos": ds.x_pos.detach().pin_memory(),
                    "z2": ds.z2.detach().pin_memory()}
            dst = {"z1": stepper.dataset.z1, "x_pos": stepper.dataset.x_pos, "z2": stepper.dataset.z2}
        host["tgt_vs"] = torch.from_numpy(n_mesh.vs).pin_memory()
        host["tgt_fn"] = torch.from_numpy(n_mesh.fn).pin_memory()
        dst["tgt_vs"], dst["tgt_fn"] = stepper.tgt_vs, stepper.tgt_fn
        h2d = sum(t.numel() * t.element_size() for t in host.values())

        def e2e_step(i):
            with torch.no_grad():
                for k_, t in host.items():
                    dst[k_].copy_(t, non_blocking=True)
            return stepper.step(epoch0 + 3 + 2 * args.steps + i).item()

        e2e_step(0)
        ms_e, _, _ = timed(e2e_step, args.steps)
        e2e = {"value": scale * 1000.0 * args.steps / ms_e, "unit": "iters/s", "h2d_bytes_per_step": int(h2d) * world,
               "d2h_bytes_per_step": 8 * world,
               "path": "every step: each rank uploads its slice of z1/z2/x_pos and the float64 targets from pinned host "
                       "memory, runs DualStep.step over the PartitionedNets, reads the loss back (.item())"}

    halo = {}
    peer_errors, peer_used = 0, False
    if world > 1:
        for name, net in (("vertex_graph", posnet), ("face_graph", normnet)):
            g = net.last_graph
            halo[name] = {"owned_rows": g.n, "halo_rows": g.n_halo, "sent_rows": g.n_send}
            if g.peer is not None:
                peer_used = True
                peer_errors += g.peer.error()
    mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30

    # ---- side measurement: mode A (one independent 1M-face fit per GPU, no data-path collective) ---------------------
    mode_a = None
    if weak and world > 1 and not args.no_mode_a:
        del stepper, ppos, pnrm
        torch.cuda.empty_cache()
        n_mesh1, s_mesh1, ds1 = build_case(args.n)
        torch.manual_seed(0)
        p1, q1 = PosNet(dev).to(dev), NormalNet(dev).to(dev)
        st1 = DualStep(p1, q1, ds1, n_mesh1, k=args.k, bnfloop=args.bnfloop)
        for i in range(5):
            st1.step(epoch0 + i)
        ms_a, _, _ = timed(lambda i: st1.step(epoch0 + 5 + i), args.steps)
        mode_a = {"value": world * 1000.0 * args.steps / ms_a, "unit": "iters/s", "ms_per_step": ms_a / args.steps,
                  "what": "one independent 1M-face fit per GPU (BASELINE configs[3] mechanism), CUDA-graph DualStep, no "
                          "data-path collective"}

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        ach = sp_bytes[0] / (sp_ms * 1e-3) / 1e9 if sp_ms > 0 else 0.0
        limiter = max(((k_, v) for k_, v in phases.items() if "NCCL" in k_ or "all_gather" in k_ or "pack" in k_
                       or "replicated" in k_), key=lambda kv: kv[1], default=(None, 0.0))
        out = {"metric": METRIC, "value": value, "unit": "iters/s", "n_gpus": world, "steps": args.steps,
               "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
               "scaling": "weak" if weak else "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
               "config": {"workload": (f"ONE synthetic icosphere n={n}: {F} faces / {V} vertices = {world} x ~1M faces, "
                                       f"Morton range-partitioned over {world} GPU(s), per-layer NCCL halo exchange, "
                                       f"BatchNorm-statistic and weight-gradient all-reduce, replicated losses; value = "
                                       f"(faces / {F_base}) x iters/s (1M-face-equivalent iterations per second)")
                          if weak else
                          (f"ONE synthetic icosphere n={n}: {F} faces / {V} vertices, Morton range-partitioned over "
                           f"{world} GPU(s) (strong scaling), per-layer NCCL halo exchange"),
                          "faces": F, "vertices": V, "mode": "partition-weak" if weak else "partition",
                          "iters_per_s_of_this_mesh": 1000.0 / ms_per_step, "rank0_partition": halo,
                          "rank0_peak_mem_GiB": round(mem, 2), "setup_s": round(setup_s, 1),
                          "l2_policy": "working set (>=10 GB of saved activations per rank) exceeds L2",
                          "batchnorm_allreduce": ("fused into the statistics / backward-sum kernels: one-shot exchange over NVLink "
                                                  "peer memory (csrc/comm.cu), %d bounded-wait errors" % peer_errors)
                                                 if peer_used else "NCCL all_reduce",
                          "streams": "PosNet / NormalNet on two compute streams, one NCCL communicator each" if overlap
                                     else "one compute stream",
                          "phases_ms_per_step_rank0": {k_: round(v, 3) for k_, v in sorted(phases.items())},
                          "phases_note": "per-phase pass runs on ONE stream (no overlap), so the phases add up to its "
                                         "step time, not to ms_per_step",
                          "largest_non_compute_phase": limiter[0],
                          "mode_a_replicas": mode_a},
               "e2e": e2e, "gpu_launches": int(launches), "loss": float(loss.detach()),
               "roofline": {"bound": "hbm", "kernel": "spmm_gcn_kernel (rank 0's aggregation launches over its owned rows)",
                            "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak if peak else None,
                            "traffic": None, "timed_in": "per-phase pass (event brackets, same steps)"},
               "clocks": sampler.summary()}
        print(json.dumps(out), file=RESULT_OUT, flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse_args()
    world_ = int(os.environ.get("WORLD_SIZE", "1"))
    if a.dump_outputs and (a.impl == "reference" or a.mode.startswith("partition")
                           or (a.mode == "auto" and world_ > 1)):
        sys.exit("--dump-outputs is implemented for our arm's one-mesh-per-GPU run (--mode auto on one GPU, "
                 "or --mode independent)")
    if a.impl == "reference":
        run_reference(a)
    elif a.mode == "partition":
        run_partitioned(a, weak=False)
    elif a.mode == "partition-weak" or (a.mode == "auto" and world_ > 1):
        run_partitioned(a, weak=True)
    else:
        run_ours(a)
