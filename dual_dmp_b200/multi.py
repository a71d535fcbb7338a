"""Pieces of a batch of independent fits sharing one GPU (``step.MultiDualStep``): the launch packing and the batched
loss phase over the library's ``ddmp_dual_loss_multi``, and the device tables the batched kernels read.

The per-mesh inputs of the batched kernels are device addresses.  Those of a CUDA-graph-captured iteration are only
known once the capture has allocated them, and they stay the same at every replay, so ``DeviceTables`` writes a table
right away outside capture and, for a capture, once it has ended: a replay reads a table whose contents never change
and copies nothing.
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from ._lib import lib, ptr, require_cuda, set_device, stream_ptr

LOSS_THREADS = 256
DESC_WORDS = 22          # DDMP_DUAL_LOSS_DESC_WORDS, include/ddmp_b200.h
SEGMENT_WORDS = 5        # DDMP_SEGMENT_WORDS


def loss_blocks(V: int, F: int, grid: int) -> int:
    """blocks of a mesh's loss phase: those of its stand-alone ``ddmp_dual_loss`` launch on a grid of ``grid`` blocks"""
    return min(int(grid), -(-max(int(V), int(F)) // LOSS_THREADS))


def pack_launches(blocks, capacity: int):
    """Split meshes with ``blocks[i]`` blocks each into consecutive cooperative launches, in caller order, each with at
    most ``capacity`` blocks.  Returns ``[(start, stop, batched)]``: ``batched`` False marks a mesh that exceeds
    ``capacity`` on its own and runs through the stand-alone kernel."""
    out, start, used = [], 0, 0
    for i, b in enumerate(blocks):
        b = int(b)
        if b < 1 or capacity < 1:
            raise ValueError("pack_launches: block counts and capacity must be positive")
        if b > capacity:
            if i > start:
                out.append((start, i, True))
            out.append((i, i + 1, False))
            start, used = i + 1, 0
            continue
        if used + b > capacity:
            out.append((start, i, True))
            start, used = i, 0
        used += b
    if start < len(blocks):
        out.append((start, len(blocks), True))
    return out


def f32_words(x) -> np.ndarray:
    """float32 values as int64 table words: the IEEE bits in the low 4 bytes, upper 4 bytes zero"""
    return np.asarray(x, dtype=np.float32).view(np.uint32).astype(np.int64)


def loss_descriptor(pos, nrm, tgt_vs, tgt_fn, topo, ws, gpos, gnrm, losses, k) -> np.ndarray:
    """one row of the ``ddmp_dual_loss_multi`` table (layout: include/ddmp_b200.h)"""
    row = np.zeros(DESC_WORDS, dtype=np.int64)
    row[:15] = [ptr(t) for t in (pos, nrm, tgt_vs, tgt_fn, topo.faces, topo.f2f, topo.rslot, topo.lap_rowptr,
                                 topo.lap_col, topo.corner_ptr, topo.corner_slot, ws, gpos, gnrm, losses)]
    row[15], row[16] = topo.V, topo.F
    row[17:22] = f32_words(k)
    return row


SEGMENT_ALIGN = 128      # floats: every network's parameters start 512-byte aligned, as in an allocation of their own
                         # (the GEMMs read weights by TMA and 16-byte vector loads)


def segment_offsets(counts) -> list:
    """start of each segment in the flat buffers (aligned to SEGMENT_ALIGN elements) and the buffers' length"""
    out, off = [], 0
    for c in counts:
        out.append(off)
        off += -(-int(c) // SEGMENT_ALIGN) * SEGMENT_ALIGN
    return out, off


def segment_table(counts, clip, lrs, max_norms) -> np.ndarray:
    """rows (offset, count, clip, lr, max_norm) of the ``ddmp_*_segments`` table, at ``segment_offsets(counts)``"""
    n = len(counts)
    t = np.zeros((n, SEGMENT_WORDS), dtype=np.int64)
    t[:, 1] = counts
    t[:, 0] = segment_offsets(counts)[0]
    t[:, 2] = [1 if c else 0 for c in clip]
    t[:, 3] = f32_words(lrs)
    t[:, 4] = f32_words(max_norms)
    return t


class DeviceTables:
    """int64 device tables, one per (phase, name): the tables a captured graph reads stay its own.

    A table is never allocated inside a capture: a block the capture hands out may be one that an earlier kernel of the
    same graph uses, and every replay would then overwrite the table before the batched kernels read it.  ``prepare``
    allocates a phase's tables, with the shapes an eager pass gave them, before its capture begins."""

    def __init__(self, device):
        self.device = torch.device(device)
        self.phase = None
        self._tables: dict = {}
        self._pending: list = []

    def prepare(self, phase) -> None:
        for (_, name), t in list(self._tables.items()):
            if (phase, name) not in self._tables:
                self._tables[(phase, name)] = torch.empty_like(t)

    def put(self, name: str, host: np.ndarray) -> torch.Tensor:
        host = np.ascontiguousarray(host, dtype=np.int64)
        key = (self.phase, name)
        t = self._tables.get(key)
        if t is None or t.shape != host.shape:
            if torch.cuda.is_current_stream_capturing():
                raise RuntimeError(f"DeviceTables: table {name!r} of phase {self.phase!r} was not prepared before "
                                   "capture")
            t = torch.empty(host.shape, dtype=torch.int64, device=self.device)
            self._tables[key] = t
        if torch.cuda.is_current_stream_capturing():
            self._pending.append((t, host.copy()))
        else:
            t.copy_(torch.from_numpy(host).pin_memory(), non_blocking=True)
        return t

    def flush(self) -> None:
        """write the tables of a finished capture"""
        for t, host in self._pending:
            t.copy_(torch.from_numpy(host))
        self._pending.clear()


class DualLossMulti(torch.autograd.Function):
    """``functional.DualLoss`` of B meshes in one batched launch (or as few consecutive ones as capacity allows):
    returns the per-mesh totals ``[B]`` (float64) and parts ``[B,5]``, each equal bit for bit to a stand-alone call."""

    @staticmethod
    def forward(ctx, tables, topos, tgts_vs, tgts_fn, ks, loop, bnf_scale, *tensors):
        B = len(topos)
        poss, nrms = tensors[:B], tensors[B:]
        dev = poss[0].device
        set_device(dev)
        g_single = int(lib.query("ddmp_dual_loss_grid", 0))
        capacity = int(lib.query("ddmp_dual_loss_grid", 1))
        losses = torch.empty(B, 6, dtype=torch.float64, device=dev)
        nbytes = [-(-int(lib.query("ddmp_dual_loss_workspace_bytes", t.V, t.F, int(loop))) // 256) * 256
                  for t in topos]
        ws = torch.empty(sum(nbytes) // 4, dtype=torch.float32, device=dev)
        offs = np.concatenate([[0], np.cumsum(nbytes)[:-1]]) // 4
        rows, gposs, gnrms = [], [], []
        for i, topo in enumerate(topos):
            pos = require_cuda(poss[i], torch.float32, "dual_loss_multi pos")
            nrm = require_cuda(nrms[i], torch.float32, "dual_loss_multi norm")
            tv = require_cuda(tgts_vs[i], torch.float64, "dual_loss_multi target positions")
            tf = require_cuda(tgts_fn[i], torch.float64, "dual_loss_multi target normals")
            if any(t.device != dev for t in (pos, nrm, tv, tf, topo.faces)):
                raise ValueError("dual_loss_multi: every tensor of the batch must be on one device")
            if pos.shape != (topo.V, 3) or nrm.shape != (topo.F, 3) or tv.shape != pos.shape or tf.shape != nrm.shape:
                raise RuntimeError(f"dual_loss_multi: shapes of mesh {i} do not match the mesh")
            gpos, gnrm = torch.empty_like(pos), torch.empty_like(nrm)
            gposs.append(gpos)
            gnrms.append(gnrm)
            rows.append(loss_descriptor(pos, nrm, tv, tf, topo, ws[int(offs[i]):], gpos, gnrm, losses[i], ks[i]))
        table = tables.put("loss", np.stack(rows))
        vf = np.array([[t.V, t.F] for t in topos], dtype=np.int64)
        blocks = [loss_blocks(t.V, t.F, g_single) for t in topos]
        st = stream_ptr(dev)
        for start, stop, batched in pack_launches(blocks, capacity):
            if batched:
                n = stop - start
                lib.call("ddmp_dual_loss_multi", table.data_ptr() + start * DESC_WORDS * 8,
                         vf[start:stop].ctypes.data_as(ctypes.c_void_p), n, float(bnf_scale), int(loop), st)
            else:
                r, topo = rows[start], topos[start]
                lib.call("ddmp_dual_loss", *[int(x) for x in r[:11]], *[float(x) for x in ks[start]],
                         float(bnf_scale), int(loop), int(r[11]), nbytes[start], int(r[12]), int(r[13]), int(r[14]),
                         topo.V, topo.F, st)
        ctx.save_for_backward(*gposs, *gnrms)
        parts = losses[:, :5]
        ctx.mark_non_differentiable(parts)
        return losses[:, 5], parts

    @staticmethod
    def backward(ctx, gout, _gparts):
        saved = ctx.saved_tensors
        B = len(saved) // 2
        g = gout.to(torch.float32)
        return (None,) * 7 + tuple(saved[i] * g[i] for i in range(B)) + tuple(saved[B + i] * g[i] for i in range(B))
