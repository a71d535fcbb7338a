"""Graph builder of the hot path: reordered CSR with precomputed GCN weights, and the index tables of the losses.

Replaces the per-call ``gcn_norm`` of torch_geometric (recomputed 24x per step through reference
util/networks.py:51-62,112-123) by a one-off build:

* nodes are sorted along a Morton (Z-order) space-filling curve of their 3-D coordinates, so the rows a CTA
  gathers in the SpMM are close in memory (L1/L2 reuse);
* CSR rows are TARGET nodes, one self loop per node appended (``add_remaining_self_loops``), columns ascending;
* ``w = deg^-1/2[row] * deg^-1/2[col]`` is computed once on the device (``ddmp_gcn_edge_weights``).

The integer part is exact: ``to_edge_list()`` returns the directed edge multiset in the caller's numbering and is
tested bit-exact against the input ``edge_index`` plus self loops.
"""
from __future__ import annotations

import numpy as np
import torch

from ._lib import lib, ptr, set_device, stream_ptr


def _part1by2(x: np.ndarray) -> np.ndarray:
    x = x.astype(np.uint64) & np.uint64(0x1FFFFF)
    x = (x | (x << np.uint64(32))) & np.uint64(0x1F00000000FFFF)
    x = (x | (x << np.uint64(16))) & np.uint64(0x1F0000FF0000FF)
    x = (x | (x << np.uint64(8))) & np.uint64(0x100F00F00F00F00F)
    x = (x | (x << np.uint64(4))) & np.uint64(0x10C30C30C30C30C3)
    x = (x | (x << np.uint64(2))) & np.uint64(0x1249249249249249)
    return x


def morton_order(coords: np.ndarray) -> np.ndarray:
    """Permutation (new -> old) that sorts points along a 63-bit Morton curve; ties broken by original id."""
    c = np.asarray(coords, dtype=np.float64)
    lo, hi = c.min(axis=0), c.max(axis=0)
    span = np.where(hi > lo, hi - lo, 1.0)
    q = np.floor((c - lo) / span * float((1 << 21) - 1)).astype(np.uint64)
    code = _part1by2(q[:, 0]) | (_part1by2(q[:, 1]) << np.uint64(1)) | (_part1by2(q[:, 2]) << np.uint64(2))
    return np.argsort(code, kind="stable").astype(np.int64)


def hilbert_order(coords: np.ndarray, bits: int = 20) -> np.ndarray:
    """Permutation (new -> old) that sorts points along a 3-D Hilbert curve (``bits`` bits per axis, Skilling's
    axes-to-transpose construction, vectorised); ties broken by original id.  Consecutive cells of a Hilbert curve are
    always face-adjacent, so a run of consecutive rows is one connected patch -- a Morton run falls apart into distant
    pieces wherever it crosses a high-order cell boundary, and the rows gathered across such a break miss L2."""
    c = np.asarray(coords, dtype=np.float64)
    lo, hi = c.min(axis=0), c.max(axis=0)
    span = np.where(hi > lo, hi - lo, 1.0)
    q = np.floor((c - lo) / span * float((1 << bits) - 1)).astype(np.uint64)
    X = [q[:, 0].copy(), q[:, 1].copy(), q[:, 2].copy()]
    one = np.uint64(1)
    Q = one << np.uint64(bits - 1)
    while Q > one:                                   # inverse undo
        P = Q - one
        for i in range(3):
            hit = (X[i] & Q) != 0
            t = np.where(hit, np.uint64(0), (X[0] ^ X[i]) & P)
            X[0] = np.where(hit, X[0] ^ P, X[0] ^ t)
            X[i] = X[i] ^ t
        Q >>= one
    X[1] ^= X[0]                                     # Gray encode
    X[2] ^= X[1]
    t = np.zeros_like(X[0])
    Q = one << np.uint64(bits - 1)
    while Q > one:
        t = np.where((X[2] & Q) != 0, t ^ (Q - one), t)
        Q >>= one
    code = (_part1by2(X[0] ^ t) << np.uint64(2)) | (_part1by2(X[1] ^ t) << np.uint64(1)) | _part1by2(X[2] ^ t)
    return np.argsort(code, kind="stable").astype(np.int64)


def sfc_order(coords: np.ndarray) -> np.ndarray:
    """Row order of the reordered graphs: Morton curve; ``DDMP_SFC=hilbert`` selects the Hilbert curve.  On the 1M-face
    benchmark graphs the two are equivalent for the aggregation kernels (out-of-block references 14.8 / 15.1 % face,
    18.0 / 18.3 % vertex graph; 4,036 vs 4,044 GB/s step-weighted, profiles/spmm_slice_ab_r2.txt), so the cheaper key
    stays the default."""
    import os
    if os.environ.get("DDMP_SFC", "morton").lower() == "hilbert":
        return hilbert_order(coords)
    return morton_order(coords)


class GcnGraph:
    """Device-resident normalised adjacency of one graph (vertex graph or face-adjacency graph)."""

    def __init__(self, edge_index, num_nodes: int, device, coords=None, reorder: bool = True):
        ei = edge_index.detach().cpu().numpy() if isinstance(edge_index, torch.Tensor) else np.asarray(edge_index)
        ei = ei.astype(np.int64, copy=False)
        n = int(num_nodes)
        if ei.size and (ei.min() < 0 or ei.max() >= n):
            raise ValueError("edge_index out of range")
        self.n = n
        self.device = torch.device(device)
        if reorder and coords is not None:
            c = coords.detach().cpu().numpy() if isinstance(coords, torch.Tensor) else np.asarray(coords)
            perm = sfc_order(c[:, :3])
        else:
            perm = np.arange(n, dtype=np.int64)
        inv = np.empty(n, dtype=np.int64)
        inv[perm] = np.arange(n, dtype=np.int64)
        self.identity = bool((perm == np.arange(n)).all())

        src, dst = ei[0], ei[1]
        keep = src != dst                               # add_remaining_self_loops: drop loops, append (i, i)
        loops = np.arange(n, dtype=np.int64)
        s = np.concatenate([inv[src[keep]], loops])
        d = np.concatenate([inv[dst[keep]], loops])
        rowptr, col = self._csr(d, s, n)
        # symmetric <=> the transposed edge set gives the same CSR
        rowptr_t, col_t = self._csr(s, d, n)
        self.symmetric = bool(np.array_equal(rowptr, rowptr_t) and np.array_equal(col, col_t))
        if rowptr[-1] >= 2 ** 31:
            raise ValueError("graph too large for int32 indices")

        dev = self.device
        self.perm_host = perm
        self.perm = None if self.identity else torch.from_numpy(perm.astype(np.int32)).to(dev)
        self.rowptr = torch.from_numpy(rowptr.astype(np.int32)).to(dev)
        self.col = torch.from_numpy(col.astype(np.int32)).to(dev)
        self.nnz = int(rowptr[-1])
        self.w = torch.empty(self.nnz, dtype=torch.float32, device=dev)
        set_device(dev)
        lib.call("ddmp_gcn_edge_weights", ptr(self.rowptr), ptr(self.col), ptr(self.w), n, stream_ptr(dev))
        if self.symmetric:
            self.rowptr_t, self.col_t, self.w_t = self.rowptr, self.col, self.w
        else:
            # directed graph (operator-level use only): backward aggregates over the transposed edges with the SAME
            # per-edge weights deg_in^-1/2[src] * deg_in^-1/2[dst]
            deg = np.diff(rowptr).astype(np.float32)
            dis = (1.0 / np.sqrt(deg)).astype(np.float32)
            order = np.lexsort((d, s))
            w_t = (dis[s[order]] * dis[d[order]]).astype(np.float32)
            self.rowptr_t = torch.from_numpy(rowptr_t.astype(np.int32)).to(dev)
            self.col_t = torch.from_numpy(col_t.astype(np.int32)).to(dev)
            self.w_t = torch.from_numpy(w_t).to(dev)

    @staticmethod
    def _csr(rows: np.ndarray, cols: np.ndarray, n: int):
        order = np.lexsort((cols, rows))
        rowptr = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(np.bincount(rows, minlength=n), out=rowptr[1:])
        return rowptr, cols[order]

    def to_edge_list(self) -> np.ndarray:
        """Directed (src, dst) pairs in the caller's numbering, self loops included, lexicographically sorted."""
        rowptr = self.rowptr.cpu().numpy().astype(np.int64)
        col = self.col.cpu().numpy().astype(np.int64)
        dst = np.repeat(np.arange(self.n, dtype=np.int64), np.diff(rowptr))
        p = self.perm_host
        pairs = np.stack([p[col], p[dst]])
        return pairs[:, np.lexsort((pairs[1], pairs[0]))]


_graph_cache: dict = {}
# graphs a caller holds on to (pin_graphs): looked up after the cache, never evicted by it.  A batch of fits asks for
# more graphs than the cache keeps, and rebuilding one inside CUDA-graph capture would fail.
_pinned: dict = {}


def graph_for(edge_index: torch.Tensor, num_nodes: int, device, coords=None, reorder: bool = True) -> GcnGraph:
    """Cache keyed on the identity of the caller's ``edge_index`` tensor (the reference passes the same tensor at
    every step, util/networks.py:49,110)."""
    key = (edge_index.data_ptr(), tuple(edge_index.shape), int(num_nodes), str(torch.device(device)), bool(reorder),
           coords is not None)
    hit = _graph_cache.get(key)
    if hit is not None and hit[0] is edge_index:
        return hit[1]
    hit = _pinned.get(key)
    if hit is not None and hit[0] is edge_index:
        return hit[1]
    g = GcnGraph(edge_index, num_nodes, device, coords=coords, reorder=reorder)
    g.cache_key = key
    if len(_graph_cache) > 64:
        _graph_cache.clear()
    _graph_cache[key] = (edge_index, g)
    return g


def pin_graphs(pairs) -> list:
    """Keep each (edge_index, graph) -- a graph as ``graph_for(edge_index, ...)`` returned it -- reachable by
    ``graph_for`` until ``unpin_graphs`` of the returned keys."""
    keys = []
    for edge_index, g in pairs:
        _pinned[g.cache_key] = (edge_index, g)
        keys.append(g.cache_key)
    return keys


def unpin_graphs(keys) -> None:
    for k in keys:
        _pinned.pop(k, None)


class MeshTopology:
    """Device index tables the loss kernels need, in the caller's numbering (built once per Mesh and device):
    faces, f2f and its reverse-slot map, the unweighted vertex adjacency CSR (Laplacian loss) and the corner CSR
    (vertex <- incident face corners) that turns every scatter-add backward into a gather."""

    def __init__(self, mesh, device):
        dev = torch.device(device)
        faces = np.asarray(mesh.faces, dtype=np.int64)
        V, F = len(mesh.vs), len(faces)
        self.V, self.F, self.device = V, F, dev
        self.faces = torch.from_numpy(faces.astype(np.int32)).to(dev)
        f2f = np.asarray(mesh.f2f, dtype=np.int64)
        nb = np.where(f2f < 0, 0, f2f)
        back = f2f[nb]                                           # [F,3,3] rows of the neighbours
        match = back == np.arange(F, dtype=np.int64)[:, None, None]
        rslot = match.argmax(axis=2)
        if not (match.any(axis=2) | (f2f < 0)).all():
            raise ValueError("f2f is not symmetric")
        self.f2f = torch.from_numpy(f2f.astype(np.int32)).to(dev)
        self.rslot = torch.from_numpy(rslot.astype(np.int32)).to(dev)
        # vertex adjacency without self loops (reference util/mesh.py:189-197), rows ascending
        e = np.asarray(mesh.edges, dtype=np.int64)
        rows = np.concatenate([e[:, 0], e[:, 1]])
        cols = np.concatenate([e[:, 1], e[:, 0]])
        rp, cl = GcnGraph._csr(rows, cols, V)
        self.lap_rowptr = torch.from_numpy(rp.astype(np.int32)).to(dev)
        self.lap_col = torch.from_numpy(cl.astype(np.int32)).to(dev)
        # corner CSR: slots 3*f+k grouped by vertex
        flat = faces.reshape(-1)
        order = np.argsort(flat, kind="stable")
        cp = np.zeros(V + 1, dtype=np.int64)
        np.cumsum(np.bincount(flat, minlength=V), out=cp[1:])
        self.corner_ptr = torch.from_numpy(cp.astype(np.int32)).to(dev)
        self.corner_slot = torch.from_numpy(order.astype(np.int32)).to(dev)
        self.scratch = torch.zeros(lib.query("ddmp_loss_scratch_bytes") // 8 + 1, dtype=torch.float64, device=dev)


def topology_for(mesh, device) -> MeshTopology:
    dev = torch.device(device)
    cache = mesh.__dict__.setdefault("_ddmp_topology", {})
    key = (str(dev), id(mesh.faces), id(mesh.f2f))
    topo = cache.get(key)
    if topo is None:
        cache.clear()
        topo = MeshTopology(mesh, dev)
        cache[key] = topo
    return topo
