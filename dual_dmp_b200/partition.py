"""Partitioned mode (SURVEY.md §8e, mode B): ONE very large mesh over G GPUs of a box.

Nodes (vertices for PosNet, faces for NormalNet) are sorted along the Morton curve and split into G contiguous ranges
of equal size; rank r owns range r.  GCN aggregation only touches 1-ring neighbours, so per layer each rank needs the
feature rows of the nodes just outside its range (the halo, O(sqrt(N/G)) rows for a surface mesh):

    GEMM on owned rows -> pack boundary rows (ddmp_gather_rows) -> NCCL all-to-all (variable splits) straight into the
    tail of the feature buffer -> SpMM over owned rows reading [owned | halo] -> BatchNorm partial sums -> all-reduce.

Backward uses the same exchange on dY (A_hat is symmetric, so every rank computes its own rows of A_hat dY; no
reverse scatter-add), all-reduces the two BatchNorm-backward sums per layer, and all-reduces the weight gradients
once per network at the end.  Weights, optimiser state and the (cheap, < 2 % of a step) losses are replicated: the
network outputs are all-gathered and every rank evaluates the five losses on the whole mesh, then back-propagates
the slice of d(loss)/d(output) that belongs to its rows.

The index logic is plain numpy and is tested without GPUs (tests/test_partition_cpu.py, gloo world_size 2).
"""
from __future__ import annotations

from typing import List

import numpy as np
import torch
import torch.distributed as dist

from ._lib import lib, ptr, set_device, stream_ptr
from .graph import sfc_order


def split_bounds(n: int, world: int) -> np.ndarray:
    """range r = [bounds[r], bounds[r+1]) of the Morton-ordered nodes"""
    return np.array([(r * n) // world for r in range(world + 1)], dtype=np.int64)


class PartitionPlan:
    """Host-side (numpy) description of every rank's part of one graph.  Built identically on every rank from the
    global graph; rank-local pieces are extracted with ``local(rank)``."""

    def __init__(self, edge_index, num_nodes: int, coords, world: int):
        ei = edge_index.detach().cpu().numpy() if isinstance(edge_index, torch.Tensor) else np.asarray(edge_index)
        ei = ei.astype(np.int64, copy=False)
        n = int(num_nodes)
        c = coords.detach().cpu().numpy() if isinstance(coords, torch.Tensor) else np.asarray(coords)
        self.n, self.world = n, int(world)
        self.perm = sfc_order(c[:, :3])                     # new -> old
        inv = np.empty(n, dtype=np.int64)
        inv[self.perm] = np.arange(n, dtype=np.int64)
        self.inv = inv
        self.bounds = split_bounds(n, world)
        src, dst = ei[0], ei[1]
        keep = src != dst
        loops = np.arange(n, dtype=np.int64)
        s = np.concatenate([inv[src[keep]], loops])
        d = np.concatenate([inv[dst[keep]], loops])
        order = np.lexsort((s, d))
        self.row = d[order]
        self.col = s[order]
        self.rowptr = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(np.bincount(self.row, minlength=n), out=self.rowptr[1:])
        deg = np.diff(self.rowptr).astype(np.float32)
        dis = (np.float32(1.0) / np.sqrt(deg)).astype(np.float32)
        self.w = (dis[self.row] * dis[self.col]).astype(np.float32)
        # symmetric adjacency is what lets the backward pass reuse the forward exchange
        order_t = np.lexsort((d, s))
        if not (np.array_equal(s[order_t], self.row) and np.array_equal(d[order_t], self.col)):
            raise ValueError("partitioned mode needs a symmetric graph (mesh adjacency)")
        self.owner_of_col = np.searchsorted(self.bounds, self.col, side="right") - 1
        self.owner_of_row = np.searchsorted(self.bounds, self.row, side="right") - 1

    def local(self, rank: int) -> dict:
        lo, hi = int(self.bounds[rank]), int(self.bounds[rank + 1])
        e0, e1 = int(self.rowptr[lo]), int(self.rowptr[hi])
        col = self.col[e0:e1]
        own = (col >= lo) & (col < hi)
        halo = np.unique(col[~own])                          # ascending global id => grouped by owner rank
        halo_owner = np.searchsorted(self.bounds, halo, side="right") - 1
        recv_counts = np.bincount(halo_owner, minlength=self.world).astype(np.int64)
        lcol = np.empty(col.shape[0], dtype=np.int64)
        lcol[own] = col[own] - lo
        lcol[~own] = (hi - lo) + np.searchsorted(halo, col[~own])
        # rows this rank must send: for every other rank q, my nodes that appear as columns of q's rows
        cross = (self.owner_of_col == rank) & (self.owner_of_row != rank)
        q = self.owner_of_row[cross]
        i = self.col[cross]
        key = np.unique(q * np.int64(self.n) + i)            # sorted by destination rank, then global id
        send_rank, send_node = key // self.n, key % self.n
        send_counts = np.bincount(send_rank, minlength=self.world).astype(np.int64)
        return dict(lo=lo, hi=hi, n_own=hi - lo, n_halo=int(halo.size),
                    rowptr=(self.rowptr[lo:hi + 1] - e0).astype(np.int32), col=lcol.astype(np.int32),
                    w=self.w[e0:e1].copy(), halo=halo, send_idx=(send_node - lo).astype(np.int32),
                    send_counts=send_counts, recv_counts=recv_counts)


class PeerComm:
    """One exchange buffer per rank, mapped by every peer of the box through CUDA IPC: the transport of the fused
    "reduce + all-reduce + finalize" BatchNorm kernels (csrc/comm.cu; ddmp_bn_stats_finalize_peer /
    ddmp_bn_bwd_finalize_peer), which replace an NCCL all-reduce between two small kernels by one kernel that exchanges its
    2*C sums with P2P stores over NVLink.  One instance per partitioned network (PosNet and NormalNet run on two streams:
    each needs its own buffer and sequence counter).  ``DDMP_PEER_ALLREDUCE=0`` keeps the NCCL route."""

    def __init__(self, rank: int, world: int, device, group=None):
        import ctypes
        self.rank, self.world, self.device = int(rank), int(world), torch.device(device)
        self.seq = 0
        set_device(self.device)
        local = ctypes.c_void_p()
        lib.call("ddmp_comm_alloc", ctypes.byref(local))
        self.local = local.value
        handle = ctypes.create_string_buffer(64)
        lib.call("ddmp_comm_ipc_handle", self.local, handle)
        handles = [None] * self.world
        dist.all_gather_object(handles, bytes(handle.raw), group=group)
        self._opened = []
        ptrs = (ctypes.c_void_p * self.world)()
        for r, h in enumerate(handles):
            if r == self.rank:
                ptrs[r] = self.local
            else:
                out = ctypes.c_void_p()
                lib.call("ddmp_comm_ipc_open", ctypes.create_string_buffer(h, 64), ctypes.byref(out))
                self._opened.append(out.value)
                ptrs[r] = out.value
        self.ptrs = ptrs
        dist.barrier(group=group)                  # every rank has mapped every buffer before the first exchange

    def next_seq(self) -> int:
        self.seq += 1
        return self.seq

    def error(self) -> int:
        import ctypes
        e = ctypes.c_int32(0)
        lib.call("ddmp_comm_error", self.local, ctypes.byref(e))
        return int(e.value)

    def close(self):
        for p_ in self._opened:
            lib.call("ddmp_comm_ipc_close", p_)
        self._opened = []
        if self.local:
            lib.call("ddmp_comm_free", self.local)
            self.local = None


class PartitionedGraph:
    """Device-resident part of rank ``rank``; duck-types the GcnGraph fields the SpMM wrapper reads."""

    def __init__(self, plan: PartitionPlan, rank: int, device, group=None):
        p = plan.local(rank)
        dev = torch.device(device)
        self.plan, self.rank, self.world, self.device, self.group = plan, rank, plan.world, dev, group
        self.n = p["n_own"]                                  # rows this rank computes
        self.n_halo = p["n_halo"]
        self.n_ext = self.n + self.n_halo
        self.n_global = plan.n
        self.lo, self.hi = p["lo"], p["hi"]
        self.rowptr = torch.from_numpy(p["rowptr"]).to(dev)
        self.col = torch.from_numpy(p["col"]).to(dev)
        self.w = torch.from_numpy(p["w"]).to(dev)
        self.rowptr_t, self.col_t, self.w_t = self.rowptr, self.col, self.w
        self.nnz = int(p["col"].shape[0])
        self.identity, self.perm = False, None
        self.send_idx = torch.from_numpy(p["send_idx"]).to(dev)
        self.send_counts: List[int] = [int(x) for x in p["send_counts"]]
        self.recv_counts: List[int] = [int(x) for x in p["recv_counts"]]
        self.n_send = int(sum(self.send_counts))
        # caller numbering of the rows this rank owns (for slicing inputs / assembling outputs)
        self.own_ids = torch.from_numpy(plan.perm[self.lo:self.hi].copy()).to(dev)
        self.perm_all = torch.from_numpy(plan.perm.copy()).to(dev)
        self._send_bufs: dict = {}                           # width -> persistent packed-rows buffer
        self.peer = None                                     # PeerComm (NVLink peer-memory BatchNorm reductions) or None

    # ---- collectives (NCCL on GPUs; enqueued on the current stream, no host synchronisation) -----------------------
    def exchange(self, X_ext: torch.Tensor) -> None:
        """fill the halo rows X_ext[n_own:] with the owners' current rows of X_ext[:n_own] (all ranks call this)"""
        self.all_to_all(X_ext, self.pack(X_ext))

    def pack(self, X_ext: torch.Tensor) -> torch.Tensor:
        """boundary rows every peer needs, grouped by destination rank, in a persistent buffer per width"""
        C = X_ext.shape[1]
        send = self._send_bufs.get(C)
        if send is None:
            send = self._send_bufs[C] = torch.empty(self.n_send, C, dtype=torch.float32, device=self.device)
        if self.n_send:
            lib.call("ddmp_gather_rows", ptr(X_ext), ptr(self.send_idx), ptr(send), self.n_send, C,
                     stream_ptr(self.device))
        return send

    def all_to_all(self, X_ext: torch.Tensor, send: torch.Tensor) -> None:
        dist.all_to_all_single(X_ext[self.n:], send, output_split_sizes=self.recv_counts,
                               input_split_sizes=self.send_counts, group=self.group)

    def allreduce_(self, t: torch.Tensor) -> torch.Tensor:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=self.group)
        return t

    def all_gather_equal(self, mine: torch.Tensor) -> List[torch.Tensor]:
        """rank-ordered list of every rank's (equally shaped) tensor"""
        parts = [torch.empty_like(mine) for _ in range(self.world)]
        dist.all_gather(parts, mine, group=self.group)
        return parts

    def gather_outputs(self, out_own: torch.Tensor) -> torch.Tensor:
        """[n_own, k] rows of every rank -> [N, k] in the CALLER's numbering (same on all ranks)"""
        return _AllGatherRows.apply(out_own, self)


class _AllGatherRows(torch.autograd.Function):
    @staticmethod
    def forward(ctx, out_own, pg: PartitionedGraph):
        k = out_own.shape[1]
        sizes = [int(pg.plan.bounds[r + 1] - pg.plan.bounds[r]) for r in range(pg.world)]
        m = max(sizes)                                        # ranges differ by at most one row: pad to equal size
        mine = torch.zeros(m, k, dtype=out_own.dtype, device=out_own.device)
        mine[: out_own.shape[0]] = out_own
        parts = pg.all_gather_equal(mine)
        full_sorted = torch.cat([p[:s] for p, s in zip(parts, sizes)], dim=0)     # Morton order
        full = torch.empty_like(full_sorted)
        full[pg.perm_all] = full_sorted                      # caller's numbering
        ctx.pg = pg
        return full

    @staticmethod
    def backward(ctx, g_full):
        pg = ctx.pg
        # the losses are evaluated identically on every rank, so d(loss)/d(own rows) is just this rank's slice
        return g_full.index_select(0, pg.own_ids).contiguous(), None


class PartitionedNet(torch.nn.Module):
    """Runs a ``PosNet`` / ``NormalNet`` (dual_dmp_b200.util.networks) on this rank's part of the mesh.

    ``forward(data)`` takes the same ``data`` object on every rank and returns the FULL ``[N, 3]`` output in the
    caller's numbering on every rank (all-gathered), so the reference's loss calls work unchanged.  Parameters are the
    wrapped module's own (replicated; identical on all ranks as long as every rank applies the same optimiser step to
    the all-reduced gradients)."""

    def __init__(self, net, rank: int, world: int, group=None):
        super().__init__()
        self.net, self.rank, self.world, self.group = net, int(rank), int(world), group
        self._cache = None

    @property
    def device(self):
        return self.net.device

    def _prepare(self, data):
        from . import functional as F_
        net = self.net
        dev = torch.device(net.device)
        is_pos = net.KIND == F_.HEAD_POS
        edge_index = data.edge_index if is_pos else data.face_index
        feats = data.z1 if is_pos else data.z2
        if self._cache is not None and self._cache[0] is edge_index and self._cache[1] is feats:
            return self._cache[2:]
        coords = data.x_pos if is_pos else data.z2.detach()[:, :3]
        plan = PartitionPlan(edge_index, feats.shape[0], coords, self.world)
        pg = PartitionedGraph(plan, self.rank, dev, self.group)
        import os
        if self.world > 1 and dev.type == "cuda" and os.environ.get("DDMP_PEER_ALLREDUCE", "1") != "0" \
                and dist.get_backend(self.group) == "nccl":
            pg.peer = PeerComm(self.rank, self.world, dev, self.group)
        ids = pg.own_ids.cpu()
        x_own = feats.detach().cpu()[ids].contiguous().to(dev)                   # static inputs: sliced once
        xpos_own = data.x_pos.detach().cpu()[ids].contiguous().to(dev) if is_pos else None
        self._cache = (edge_index, feats, pg, x_own, xpos_own)
        return pg, x_own, xpos_own

    def forward(self, data):
        from . import functional as F_
        net = self.net
        pg, x_own, xpos_own = self._prepare(data)
        bns = [getattr(net, f"bn{i}") for i in range(1, 13)]
        buffers = [(bn.running_mean, bn.running_var) for bn in bns]
        out_own = F_.GcnNetFunction.apply(pg, net.KIND, net.training, buffers, net.taps, x_own, xpos_own,
                                          *net._params(), F_.check_dense_precision(net.dense_precision))
        net.last_graph = pg
        if net.training:
            torch._foreach_add_([bn.num_batches_tracked for bn in bns], 1)
        return pg.gather_outputs(out_own)
