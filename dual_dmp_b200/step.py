"""The training iteration of the reference drivers as one object (SURVEY.md §8f, N1).

``DualStep.step(epoch)`` is reference main.py:88-110 / main4real.py:53-70: zero_grad, PosNet and NormalNet forward, the
five losses (``loss_norm2 *= 0`` while epoch <= 100), weighted sum, backward, ``clip_grad_norm_`` on NormalNet, two
Adam steps.  Inputs and targets are kept resident on the device (the reference re-uploads ~100 MB per step at 1M
faces), nothing synchronises the host, and the whole iteration is captured into CUDA graphs (one for the BNF warm-up
phase, one for the rest, sharing a memory pool) so a step is a single graph launch: at fandisk size the eager step
is bound by ~700 Python-side launches (8.5 ms), the replayed one by the GPU.

The numerics are those of the eager drop-in path: the same autograd Functions and kernels are what gets captured.
"""
from __future__ import annotations

import copy

import numpy as np
import torch

from .util import loss as L


class DualStep:
    def __init__(self, posnet, normnet, dataset, n_mesh, k=(3.0, 4.0, 4.0, 4.0, 1.0), bnfloop=1, pos_lr=0.01,
                 norm_lr=0.01, grad_clip=0.8, bnf_warmup_epochs=100, capture=True, overlap=True,
                 fused_optimizer=True, fused_loss=True, dense_precision=None):
        """``dense_precision``: None keeps each network's ``dense_precision`` attribute; "fp32" or "f16x1" sets it on
        both (util.networks: the accuracy contract of the dense transforms' tensor-core kernels)."""
        dev = torch.device(posnet.device)
        if dev.type != "cuda":
            raise RuntimeError("DualStep runs on CUDA only (dual_dmp_b200 has no CPU path)")
        set_dense_precision((posnet, normnet), dense_precision)
        self.device = dev
        self.posnet, self.normnet, self.mesh = posnet, normnet, n_mesh
        self.k, self.bnfloop, self.grad_clip = tuple(float(x) for x in k), int(bnfloop), float(grad_clip)
        self.bnf_warmup_epochs = int(bnf_warmup_epochs)
        self.dataset = copy.copy(dataset).to(dev)                       # resident inputs
        self.tgt_vs = torch.from_numpy(n_mesh.vs).to(dev)               # float64 targets, like the reference
        self.tgt_fn = torch.from_numpy(n_mesh.fn).to(dev)
        self.capture = bool(capture)
        # PosNet and NormalNet are independent until the losses: run them on two streams so the memory-bound
        # kernels of one network (SpMM, BatchNorm) overlap the tensor-core GEMMs of the other; autograd runs each
        # network's backward on the stream of its forward
        self.overlap = bool(overlap)
        self._streams = (torch.cuda.Stream(dev), torch.cuda.Stream(dev)) if self.overlap else None
        self.fused_optimizer = bool(fused_optimizer)
        # the five loss calls + weighted sum + their backward as one cooperative kernel (util.loss.dual_loss)
        self.fused_loss = bool(fused_loss)
        if self.fused_optimizer:       # clip + Adam as two library kernels per network over flat buffers
            self.opt_pos = FusedAdam(posnet, lr=pos_lr)
            self.opt_norm = FusedAdam(normnet, lr=norm_lr, max_norm=self.grad_clip)
        else:
            self.opt_pos = torch.optim.Adam(posnet.parameters(), lr=pos_lr, capturable=self.capture)
            self.opt_norm = torch.optim.Adam(normnet.parameters(), lr=norm_lr, capturable=self.capture)
        self._graphs: dict = {}
        self._static_loss: dict = {}
        # streaming inputs (prefetch): staging copies of the per-step inputs, filled by a copy stream
        self._stage = None
        self._copy_stream = None
        self._stage_ready = None
        self._stage_free = None
        self._pending = False
        self._eager_calls = 0
        self.pos = None      # outputs of the most recent step (static tensors when captured)
        self.norm = None

    # ---- the loop body (reference main.py:88-110) ------------------------------------------------------------------
    def _body(self, bnf_off: bool) -> torch.Tensor:
        k = self.k
        self.posnet.train()
        self.normnet.train()
        self.opt_pos.zero_grad(set_to_none=True)
        self.opt_norm.zero_grad(set_to_none=True)
        if self.overlap:
            cur = torch.cuda.current_stream(self.device)
            s_pos, s_nrm = self._streams
            s_pos.wait_stream(cur)
            s_nrm.wait_stream(cur)
            with torch.cuda.stream(s_nrm):           # the larger network first
                nrm = self.normnet(self.dataset)
            with torch.cuda.stream(s_pos):
                pos = self.posnet(self.dataset)
            cur.wait_stream(s_pos)
            cur.wait_stream(s_nrm)
            pos.record_stream(cur)
            nrm.record_stream(cur)
        else:
            pos = self.posnet(self.dataset)
            nrm = self.normnet(self.dataset)
        if self.fused_loss:
            loss, self.parts = L.dual_loss(pos, nrm, self.mesh, self.tgt_vs, self.tgt_fn, k, self.bnfloop,
                                           0.0 if bnf_off else 1.0)
        else:
            l1 = L.pos_rec_loss(pos, self.tgt_vs)
            l2 = L.mesh_laplacian_loss(pos, self.mesh)
            l3 = L.norm_rec_loss(nrm, self.tgt_fn)
            l4, _ = L.fn_bnf_loss(pos, nrm, self.mesh, loop=self.bnfloop)
            if bnf_off:
                l4 = l4 * 0.0               # still computed and back-propagated, exactly like the reference (:101-102)
            l5 = L.pos_norm_loss(pos, nrm, self.mesh)
            loss = k[0] * l1 + k[1] * l2 + k[2] * l3 + k[3] * l4 + k[4] * l5
        loss.backward()
        if not self.fused_optimizer:
            torch.nn.utils.clip_grad_norm_(self.normnet.parameters(), self.grad_clip)
        self.opt_pos.step()
        self.opt_norm.step()
        self.pos, self.norm = pos.detach(), nrm.detach()
        return loss.detach()

    def _capture(self, bnf_off: bool) -> None:
        g = torch.cuda.CUDAGraph()
        pool = next(iter(self._graphs.values())).pool() if self._graphs else None
        with torch.cuda.graph(g, pool=pool):
            self._static_loss[bnf_off] = self._body(bnf_off)
        self._graphs[bnf_off] = g

    # ---- streaming inputs: host -> staging on a copy stream, overlapped with the running step ----------------------
    def _static_inputs(self):
        return {"z1": self.dataset.z1, "z2": self.dataset.z2, "x_pos": self.dataset.x_pos,
                "tgt_vs": self.tgt_vs, "tgt_fn": self.tgt_fn}

    def prefetch(self, dataset_host, tgt_vs_host, tgt_fn_host) -> int:
        """Start uploading the inputs of the NEXT ``step`` (the tensors the reference loop moves to the device every
        iteration: ``z1``, ``z2``, ``x_pos`` and the float64 targets) from pinned host memory.  The copies run on a
        dedicated stream into staging buffers, so they overlap the iteration that is executing; the next ``step``
        waits for them, moves staging -> static inputs (device-to-device) and runs.  Returns the bytes enqueued."""
        host = {"z1": dataset_host.z1, "z2": dataset_host.z2, "x_pos": dataset_host.x_pos,
                "tgt_vs": tgt_vs_host, "tgt_fn": tgt_fn_host}
        static = self._static_inputs()
        if self._stage is None:
            self._stage = {k: torch.empty_like(v) for k, v in static.items()}
            self._copy_stream = torch.cuda.Stream(self.device)
            self._stage_ready = torch.cuda.Event()
            self._stage_free = torch.cuda.Event()
            self._stage_free.record(torch.cuda.current_stream(self.device))
        nbytes = 0
        self._copy_stream.wait_event(self._stage_free)       # the previous staging -> static move has been issued
        with torch.no_grad(), torch.cuda.stream(self._copy_stream):
            for k, dst in self._stage.items():
                src = host[k]
                if src.shape != dst.shape or src.dtype != dst.dtype:
                    raise ValueError(f"prefetch: {k} is {tuple(src.shape)} {src.dtype}, expected "
                                     f"{tuple(dst.shape)} {dst.dtype}")
                dst.copy_(src, non_blocking=True)
                nbytes += src.numel() * src.element_size()
            self._stage_ready.record(self._copy_stream)
        self._pending = True
        return nbytes

    def _consume_prefetch(self) -> None:
        cur = torch.cuda.current_stream(self.device)
        cur.wait_event(self._stage_ready)
        with torch.no_grad():
            for k, dst in self._static_inputs().items():
                dst.copy_(self._stage[k], non_blocking=True)
        self._stage_free.record(cur)
        self._pending = False

    def step(self, epoch: int) -> torch.Tensor:
        """one training iteration; returns the (device, float64) loss without synchronising"""
        bnf_off = epoch <= self.bnf_warmup_epochs
        if self._pending:
            self._consume_prefetch()
        if not self.capture:
            return self._body(bnf_off)
        if bnf_off not in self._graphs:
            if self._eager_calls < 3:
                # warm-up on a side stream (graph/index caches, optimizer state, allocator) before capturing
                self._eager_calls += 1
                s = torch.cuda.Stream(self.device)
                s.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(s):
                    loss = self._body(bnf_off)
                torch.cuda.current_stream(self.device).wait_stream(s)
                return loss
            self._capture(bnf_off)
        self._graphs[bnf_off].replay()
        return self._static_loss[bnf_off]


def set_dense_precision(nets, dense_precision) -> None:
    """set ``dense_precision`` ("fp32" | "f16x1") on every network; None leaves them as they are"""
    if dense_precision is None:
        return
    from .functional import check_dense_precision
    check_dense_precision(dense_precision)
    for net in nets:
        net.dense_precision = dense_precision


class FusedAdam:
    """``clip_grad_norm_`` + ``torch.optim.Adam`` of one network as two library kernels over flat buffers
    (reference main.py:108-110; SURVEY.md §8f N1).  The parameters of ``module`` are re-pointed at views of one flat
    buffer, so ``module.parameters()`` / ``state_dict()`` keep working; the step count lives on the device, which
    makes ``step()`` CUDA-graph capturable."""

    def __init__(self, module, lr=0.01, betas=(0.9, 0.999), eps=1e-8, max_norm=None):
        from ._lib import lib
        self.params = [p for p in module.parameters() if p.requires_grad]
        dev = self.params[0].device
        if dev.type != "cuda":
            raise RuntimeError("FusedAdam runs on CUDA only (dual_dmp_b200 has no CPU path)")
        n = sum(p.numel() for p in self.params)
        self.flat = torch.empty(n, dtype=torch.float32, device=dev)
        off = 0
        for p in self.params:
            k = p.numel()
            self.flat[off: off + k].copy_(p.detach().reshape(-1))
            p.data = self.flat[off: off + k].view_as(p)
            off += k
        import ctypes
        counts = [p.numel() for p in self.params]
        offsets = [sum(counts[:i]) for i in range(len(counts))]
        self._counts = (ctypes.c_int64 * len(counts))(*counts)
        self._offsets = (ctypes.c_int64 * len(counts))(*offsets)
        self.gflat = torch.empty_like(self.flat)           # flat gradient, filled by ddmp_gather_flat every step
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.step_count = torch.zeros((), dtype=torch.int64, device=dev)
        self.norm = torch.zeros((), dtype=torch.float32, device=dev)
        self.scratch = torch.zeros(lib.query("ddmp_loss_scratch_bytes") // 8 + 1, dtype=torch.float64, device=dev)
        self.lr, self.betas, self.eps, self.max_norm = float(lr), betas, float(eps), max_norm
        self.device = dev

    def zero_grad(self, set_to_none=True):
        for p in self.params:
            p.grad = None

    def step(self):
        from ._lib import lib, ptr, set_device, stream_ptr
        set_device(self.device)
        st = stream_ptr(self.device)
        import ctypes
        grads = [p.grad if p.grad.is_contiguous() else p.grad.contiguous() for p in self.params]
        srcs = (ctypes.c_void_p * len(grads))(*[t.data_ptr() for t in grads])
        g = self.gflat                                                   # flat gradient: one library launch
        lib.call("ddmp_gather_flat", srcs, self._offsets, self._counts, len(grads), ptr(g), st)
        clip = None
        if self.max_norm is not None:
            lib.call("ddmp_grad_norm", ptr(g), ptr(self.norm), ptr(self.scratch), g.numel(), st)
            clip = self.norm
        lib.call("ddmp_adam_step_dev", ptr(self.flat), ptr(g), ptr(self.exp_avg), ptr(self.exp_avg_sq), ptr(clip),
                 float(self.max_norm or 0.0), self.lr, self.betas[0], self.betas[1], self.eps, ptr(self.step_count),
                 g.numel(), st)


class GroupFusedAdam:
    """``FusedAdam`` of many networks over ONE flat buffer: gather, clip norms and Adam are one library launch each for
    all of them (``ddmp_gather_table``, ``ddmp_grad_norm_segments``, ``ddmp_adam_segments``), with a per-network lr and
    clip.  Network ``i`` is segment ``i``; its results equal a ``FusedAdam`` of that network bit for bit.  Parameters are
    re-pointed at views of the flat buffer, so ``parameters()`` / ``state_dict()`` keep working."""

    def __init__(self, modules, lrs, max_norms, betas=(0.9, 0.999), eps=1e-8):
        from ._lib import lib
        from . import multi
        self.params = [[p for p in m.parameters() if p.requires_grad] for m in modules]
        flat_params = [p for ps in self.params for p in ps]
        dev = flat_params[0].device
        if dev.type != "cuda":
            raise RuntimeError("GroupFusedAdam runs on CUDA only (dual_dmp_b200 has no CPU path)")
        if any(p.device != dev for p in flat_params):
            raise ValueError("GroupFusedAdam: every network must be on one device")
        self.counts = [sum(p.numel() for p in ps) for ps in self.params]
        self.offsets, total = multi.segment_offsets(self.counts)
        self.flat = torch.zeros(total, dtype=torch.float32, device=dev)
        gather = []
        for ps, off in zip(self.params, self.offsets):
            for p in ps:
                k = p.numel()
                self.flat[off: off + k].copy_(p.detach().reshape(-1))
                p.data = self.flat[off: off + k].view_as(p)
                gather.append((off, k))
                off += k
        self._gather_rows = np.array(gather, dtype=np.int64)
        self._longest_param = max(k for _, k in gather)
        self.gflat = torch.zeros_like(self.flat)
        self.exp_avg = torch.zeros_like(self.flat)
        self.exp_avg_sq = torch.zeros_like(self.flat)
        self.step_count = torch.zeros((), dtype=torch.int64, device=dev)
        n = len(self.params)
        clip = [m is not None for m in max_norms]
        seg = multi.segment_table(self.counts, clip, lrs, [m or 0.0 for m in max_norms])
        self.segments = torch.from_numpy(seg).to(dev)          # no addresses in it: written once
        self.clips = any(clip)
        self.norms = torch.zeros(n, dtype=torch.float32, device=dev)
        self.scratch = torch.zeros(n * int(lib.query("ddmp_loss_scratch_bytes")) // 8 + 1, dtype=torch.float64,
                                   device=dev)
        self.betas, self.eps, self.device = betas, float(eps), dev

    def segment(self, i: int) -> slice:
        """the slice of network ``i`` in ``flat`` / ``exp_avg`` / ``exp_avg_sq``"""
        return slice(self.offsets[i], self.offsets[i] + self.counts[i])

    def zero_grad(self, set_to_none=True):
        for ps in self.params:
            for p in ps:
                p.grad = None

    def step(self, tables):
        """``tables``: the ``multi.DeviceTables`` that holds the gradient-address table of this iteration"""
        from ._lib import lib, ptr, set_device, stream_ptr
        set_device(self.device)
        st = stream_ptr(self.device)
        grads = [p.grad if p.grad.is_contiguous() else p.grad.contiguous() for ps in self.params for p in ps]
        rows = np.concatenate([np.array([[g.data_ptr()] for g in grads], dtype=np.int64), self._gather_rows], axis=1)
        table = tables.put("grads", rows)
        lib.call("ddmp_gather_table", ptr(table), len(grads), self._longest_param, ptr(self.gflat), st)
        n, longest = len(self.counts), max(self.counts)
        if self.clips:
            lib.call("ddmp_grad_norm_segments", ptr(self.gflat), ptr(self.segments), n, longest, ptr(self.norms),
                     ptr(self.scratch), st)
        lib.call("ddmp_adam_segments", ptr(self.flat), ptr(self.gflat), ptr(self.exp_avg), ptr(self.exp_avg_sq),
                 ptr(self.segments), n, longest, ptr(self.norms), self.betas[0], self.betas[1], self.eps,
                 ptr(self.step_count), st)


class MultiDualStep(DualStep):
    """``DualStep`` of B independent fits on one GPU as one iteration: each fit's PosNet and NormalNet forward on a
    stream pair of its own, one batched loss phase (``multi.DualLossMulti``), the backward passes (autograd runs each
    network's on the stream of its forward) and one batched optimizer (``GroupFusedAdam``); captured into one CUDA graph
    per phase like ``DualStep``.  Every fit's numbers equal those of its own ``DualStep`` bit for bit.

    ``fits``: one dict per mesh with ``posnet``, ``normnet``, ``dataset``, ``n_mesh`` and optionally ``k``, ``pos_lr``,
    ``norm_lr``, ``grad_clip``, ``bnfloop`` and ``dense_precision`` (the defaults of ``DualStep``; fits may differ in
    ``dense_precision``).  All fits share ``bnfloop``: a batch that
    mixes values is rejected, run it as two batches.  ``step(epoch)`` returns the per-fit totals ``[B]`` (float64);
    ``.pos[i]``, ``.norm[i]``, ``.parts[i]`` are fit ``i``'s outputs."""

    def __init__(self, fits, bnfloop=1, bnf_warmup_epochs=100, capture=True):
        from . import multi
        fits = [dict(f) for f in fits]
        if not fits:
            raise ValueError("MultiDualStep: no fits")
        loops = {int(f.get("bnfloop", bnfloop)) for f in fits}
        if len(loops) != 1:
            raise ValueError(f"MultiDualStep: the fits mix bnfloop values {sorted(loops)}; run one batch per value")
        devs = {torch.device(n.device) for f in fits for n in (f["posnet"], f["normnet"])}
        if any(d.type != "cuda" for d in devs):
            raise RuntimeError("MultiDualStep runs on CUDA only (dual_dmp_b200 has no CPU path)")
        if len(devs) != 1:
            raise ValueError(f"MultiDualStep: the fits are on several devices {sorted(map(str, devs))}; one batch "
                             "runs on one device")
        dev = devs.pop()
        for f in fits:
            set_dense_precision((f["posnet"], f["normnet"]), f.get("dense_precision"))
        self.device = dev
        self.bnfloop = loops.pop()
        self.bnf_warmup_epochs = int(bnf_warmup_epochs)
        self.capture = bool(capture)
        self.fits = fits
        self.ks = [tuple(float(x) for x in f.get("k", (3.0, 4.0, 4.0, 4.0, 1.0))) for f in fits]
        self.datasets = [copy.copy(f["dataset"]).to(dev) for f in fits]
        self.tgt_vs = [torch.from_numpy(f["n_mesh"].vs).to(dev) for f in fits]
        self.tgt_fn = [torch.from_numpy(f["n_mesh"].fn).to(dev) for f in fits]
        self._streams = [(torch.cuda.Stream(dev), torch.cuda.Stream(dev)) for _ in fits]
        nets = [n for f in fits for n in (f["posnet"], f["normnet"])]
        self.opt = GroupFusedAdam(
            nets, [lr for f in fits for lr in (f.get("pos_lr", 0.01), f.get("norm_lr", 0.01))],
            [m for f in fits for m in (None, float(f.get("grad_clip", 0.8)))])
        self._tables = multi.DeviceTables(dev)
        self._pinned = None
        self._graphs: dict = {}
        self._static_loss: dict = {}
        self._pending = False
        self._eager_calls = 0
        self.pos = self.norm = self.parts = None

    def prefetch(self, *args, **kwargs):
        raise NotImplementedError("MultiDualStep keeps its inputs resident; streamed inputs are a DualStep feature")

    def _body(self, bnf_off: bool) -> torch.Tensor:
        from . import multi
        from .graph import pin_graphs, topology_for
        self._tables.phase = bnf_off
        self.opt.zero_grad(set_to_none=True)
        cur = torch.cuda.current_stream(self.device)
        poss, nrms = [], []
        for f, ds, (s_pos, s_nrm) in zip(self.fits, self.datasets, self._streams):
            f["posnet"].train()
            f["normnet"].train()
            s_pos.wait_stream(cur)
            s_nrm.wait_stream(cur)
            with torch.cuda.stream(s_nrm):           # the larger network first
                nrms.append(f["normnet"](ds))
            with torch.cuda.stream(s_pos):
                poss.append(f["posnet"](ds))
        for (s_pos, s_nrm), pos, nrm in zip(self._streams, poss, nrms):
            cur.wait_stream(s_pos)
            cur.wait_stream(s_nrm)
            pos.record_stream(cur)
            nrm.record_stream(cur)
        if self._pinned is None:      # B > 32 fits outgrow graph_for's cache: keep every fit's graphs reachable
            import weakref
            pairs = [(ds.edge_index, f["posnet"].last_graph) for f, ds in zip(self.fits, self.datasets)]
            pairs += [(ds.face_index, f["normnet"].last_graph) for f, ds in zip(self.fits, self.datasets)]
            self._pinned = pin_graphs(pairs)
            from .graph import unpin_graphs
            weakref.finalize(self, unpin_graphs, list(self._pinned))
        topos = [topology_for(f["n_mesh"], self.device) for f in self.fits]
        totals, self.parts = multi.DualLossMulti.apply(self._tables, topos, self.tgt_vs, self.tgt_fn, self.ks,
                                                       self.bnfloop, 0.0 if bnf_off else 1.0, *poss, *nrms)
        totals.sum().backward()
        self.opt.step(self._tables)
        self.pos = [p.detach() for p in poss]
        self.norm = [n.detach() for n in nrms]
        return totals.detach()

    def _capture(self, bnf_off: bool) -> None:
        self._tables.prepare(bnf_off)
        super()._capture(bnf_off)
        self._tables.flush()
