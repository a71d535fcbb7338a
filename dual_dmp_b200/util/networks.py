"""Drop-in for reference ``util/networks.py``: ``PosNet(device)``, ``NormalNet(device)``, ``forward(data)``.

Same module tree and parameter names as the reference (conv1..conv12 with ``.lin.weight [Cout,Cin]`` / ``.bias``,
bn1..bn12 = ``nn.BatchNorm1d``, linear1, linear2, l_relu; reference util/networks.py:13-44,74-105), so a
``state_dict`` moves freely between the reference/oracle and this implementation.  ``forward`` runs the whole
network as one ``torch.autograd.Function`` over the libddmp_b200 CUDA kernels — no torch_geometric, no Triton, no
CPU fallback (a CPU ``device`` raises).

``GCNConv`` is also usable on its own, ``conv(x, edge_index)``, as a replacement of torch_geometric.nn.GCNConv
with the defaults the reference uses (add_self_loops, symmetric normalisation, bias).
"""
from __future__ import annotations

import math

import torch
import torch.nn as nn

from .. import functional as F_
from ..graph import graph_for

POS_WIDTHS = [16, 32, 64, 128, 256, 256, 512, 512, 256, 256, 128, 64, 32, 16, 3]
NORM_WIDTHS = [7, 32, 64, 128, 256, 256, 512, 512, 256, 256, 128, 64, 32, 16, 3]


class _Lin(nn.Module):
    """``GCNConv.lin``: bias-free linear map, weight [out, in], glorot-uniform init (PyG ``inits.glorot``)."""

    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.weight = nn.Parameter(torch.empty(out_channels, in_channels))
        a = math.sqrt(6.0 / (in_channels + out_channels))
        with torch.no_grad():
            self.weight.uniform_(-a, a)


class GCNConv(nn.Module):
    def __init__(self, in_channels: int, out_channels: int):
        super().__init__()
        self.in_channels, self.out_channels = in_channels, out_channels
        self.lin = _Lin(in_channels, out_channels)
        self.bias = nn.Parameter(torch.zeros(out_channels))

    def forward(self, x: torch.Tensor, edge_index: torch.Tensor) -> torch.Tensor:
        graph = graph_for(edge_index, x.shape[0], x.device, coords=None, reorder=False)
        return F_.GCNConvFunction.apply(x, self.lin.weight, self.bias, graph)


class _Net(nn.Module):
    KIND = F_.HEAD_POS
    WIDTHS = POS_WIDTHS

    def __init__(self, device):
        super().__init__()
        self.device = device
        h = self.WIDTHS
        for i in range(12):
            setattr(self, f"conv{i + 1}", GCNConv(h[i], h[i + 1]))
        self.linear1 = nn.Linear(h[12], h[13])
        self.linear2 = nn.Linear(h[13], h[14])
        for i in range(12):
            setattr(self, f"bn{i + 1}", nn.BatchNorm1d(h[i + 1]))
        self.l_relu = nn.LeakyReLU()
        self.reorder = True          # Morton-sort the graph (set False to keep the caller's numbering)
        self.taps = None             # set to a list to collect (Y_l, stats_l) of every layer (parity tests)
        self.last_graph = None       # GcnGraph used by the most recent forward (holds the row permutation)
        # accuracy contract of the trunk's dense transforms: "fp32" (default; fp32-accurate products) or "f16x1" (one
        # fp16 product on the tensor-core layers with operand bounds, DDMP_GEMM_F16X1 in include/ddmp_b200.h)
        self.dense_precision = "fp32"

    def _params(self):
        p = []
        for i in range(1, 13):
            conv, bn = getattr(self, f"conv{i}"), getattr(self, f"bn{i}")
            p += [conv.lin.weight, conv.bias, bn.weight, bn.bias]
        return p + [self.linear1.weight, self.linear1.bias, self.linear2.weight, self.linear2.bias]

    def _run(self, x_in, x_pos, edge_index, coords):
        dev = torch.device(self.device)
        if dev.type != "cuda":
            raise RuntimeError("dual_dmp_b200 networks run on CUDA only (no CPU fallback); got device %s" % dev)
        graph = graph_for(edge_index, x_in.shape[0], dev, coords=coords if self.reorder else None,
                          reorder=self.reorder)
        self.last_graph = graph
        bns = [getattr(self, f"bn{i}") for i in range(1, 13)]
        buffers = [(bn.running_mean, bn.running_var) for bn in bns]
        out = F_.GcnNetFunction.apply(graph, self.KIND, self.training, buffers, self.taps, x_in.detach(), x_pos,
                                      *self._params(), F_.check_dense_precision(self.dense_precision))
        if self.training:
            torch._foreach_add_([bn.num_batches_tracked for bn in bns], 1)
        return out


class PosNet(_Net):
    """reference util/networks.py:8-67."""
    KIND = F_.HEAD_POS
    WIDTHS = POS_WIDTHS

    def forward(self, data):
        dev = self.device
        z1 = data.z1.to(dev, non_blocking=True)
        x_pos = data.x_pos.to(dev, non_blocking=True)
        # the reference also draws an unused randn(V,3) here (:50); it has no effect on the result and is skipped
        return self._run(z1, x_pos, data.edge_index, coords=data.x_pos)


class NormalNet(_Net):
    """reference util/networks.py:69-129."""
    KIND = F_.HEAD_NORM
    WIDTHS = NORM_WIDTHS

    def forward(self, data):
        dev = self.device
        z2 = data.z2.to(dev, non_blocking=True)
        # z2 = [centroid | normal | area] (reference util/datamaker.py:80-81): its first three columns place the
        # faces on the space-filling curve
        return self._run(z2, None, data.face_index, coords=data.z2.detach()[:, :3])
