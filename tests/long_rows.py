"""Meshes and graphs whose CSR rows are long: hub vertices, fan caps and dense graph rows (plain numpy).

Every kernel that walks a CSR row has a second code path for rows longer than its chunk, batch or shared-memory
budget: the aggregation kernels reload (col, w) every G = min(32, C/4) entries, the tile-staged kernels read (col, w)
from global memory once a row block holds more than 9 entries per row, and the loss kernels gather neighbours in
batches of 8.  Icospheres have a maximum valence of 6 and never get there; UV spheres, fan discs and cylinders with
fan caps (CAD meshes) have poles of valence 20 to 1000+.
"""
from __future__ import annotations

import numpy as np

# pole / hub valences the tests cover: both sides of every chunk (8, 16, 32) and two far past them
POLE_VALENCES = (7, 8, 9, 15, 16, 17, 31, 32, 33, 64, 1000, 4096)
# aggregation row lengths around every chunk G in {8, 16, 32}: G-1, G, G+1, 2G, 2G+1; and 1, 2, 3 around the unroll U
BOUNDARY_ROWS = tuple(sorted({x for g in (8, 16, 32) for x in (g - 1, g, g + 1, 2 * g, 2 * g + 1)}))
SHORT_ROWS = (1, 2, 3)
# (kind, hub valence, rings) of the GPU tests: losses against the CPU oracle (<= 130k faces), geometry, preprocessing
LOSS_MESHES = [("uv", 4096, 14), ("fan", 1000, 6), ("cyl", 33, 8), ("uv", 9, 6), ("fan", 17, 5), ("cyl", 64, 4)]
GEOM_MESHES = [("uv", 4096, 14), ("uv", 1000, 3), ("fan", 33, 4), ("cyl", 17, 4)]
PREP_MESHES = [("uv", 4096, 14), ("fan", 1000, 6), ("cyl", 64, 4)]
META_PER_ROW = 9          # (col, w) entries per row the tile-staged kernels keep in shared memory (csrc/spmm_tile.cu)


# ---------------------------------------------------------------------------------------------------------------------
# meshes
# ---------------------------------------------------------------------------------------------------------------------
def _ring_faces(m: int, n_rings: int, hub_a: bool, hub_b: bool) -> np.ndarray:
    """Faces of `n_rings` rings of `m` vertices (ring r, slot j -> vertex base + r*m + j), consecutive rings joined by
    quads split along one diagonal, optional fans to hub A (vertex 0, before ring 0) and hub B (last vertex, after the
    last ring).  Consistently oriented."""
    base = 1 if hub_a else 0
    j = np.arange(m)
    jn = (j + 1) % m
    out = []
    if hub_a:
        out.append(np.stack([np.zeros(m, np.int64), base + jn, base + j], axis=1))
    for r in range(n_rings - 1):
        a, b = base + r * m, base + (r + 1) * m
        out.append(np.stack([a + j, a + jn, b + jn], axis=1))
        out.append(np.stack([a + j, b + jn, b + j], axis=1))
    if hub_b:
        last = base + (n_rings - 1) * m
        hb = base + n_rings * m
        out.append(np.stack([np.full(m, hb, np.int64), last + j, last + jn], axis=1))
    return np.concatenate(out).astype(np.int64)


def _unit_mean_edge(vs: np.ndarray, faces: np.ndarray) -> np.ndarray:
    """scale to mean edge length 1 (the reference's data convention, synth.make_case)"""
    from dual_dmp_b200 import synth
    e = synth.unique_edges(faces, len(vs))
    return vs / np.linalg.norm(vs[e[:, 0]] - vs[e[:, 1]], axis=1).mean()


def _orient_outward(vs: np.ndarray, faces: np.ndarray) -> np.ndarray:
    """flip every face if the signed volume of the closed surface is negative"""
    p0, p1, p2 = vs[faces[:, 0]], vs[faces[:, 1]], vs[faces[:, 2]]
    vol = np.einsum("ij,ij->i", p0, np.cross(p1, p2)).sum()
    return faces if vol > 0 else faces[:, [0, 2, 1]].copy()


def uv_sphere(m: int, rings: int):
    """Closed UV sphere: two poles of valence `m`, `rings` latitude rings of `m` vertices (valence 5-6).  The faces next
    to the poles are slivers once m is large.  Returns (vs [V,3] float64, faces [F,3] int64), F = 2*m*rings."""
    assert m >= 3 and rings >= 1
    theta = np.pi * np.arange(1, rings + 1) / (rings + 1)
    phi = 2.0 * np.pi * np.arange(m) / m
    ring = np.stack([np.sin(theta)[:, None] * np.cos(phi)[None, :], np.sin(theta)[:, None] * np.sin(phi)[None, :],
                     np.repeat(np.cos(theta)[:, None], m, axis=1)], axis=2).reshape(-1, 3)
    vs = np.concatenate([[[0.0, 0.0, 1.0]], ring, [[0.0, 0.0, -1.0]]])
    faces = _orient_outward(vs, _ring_faces(m, rings, True, True))
    return _unit_mean_edge(vs, faces), faces


def fan_disc(K: int, rings: int):
    """Open disc: one centre of valence `K`, `rings` concentric rings of `K` vertices; the outer ring is the boundary,
    so `f2f` has -1 entries.  A shallow dome (normals up).  F = K*(2*rings - 1)."""
    assert K >= 3 and rings >= 1
    rad = np.arange(1, rings + 1, dtype=np.float64)
    phi = 2.0 * np.pi * np.arange(K) / K
    ring = np.stack([rad[:, None] * np.cos(phi)[None, :], rad[:, None] * np.sin(phi)[None, :],
                     np.repeat((-0.05 * rad ** 2)[:, None], K, axis=1)], axis=2).reshape(-1, 3)
    vs = np.concatenate([[[0.0, 0.0, 0.0]], ring])
    faces = _ring_faces(K, rings, True, False)
    p0, p1, p2 = vs[faces[:, 0]], vs[faces[:, 1]], vs[faces[:, 2]]
    if np.cross(p1 - p0, p2 - p0)[:, 2].sum() < 0:
        faces = faces[:, [0, 2, 1]].copy()
    return _unit_mean_edge(vs, faces), faces


def cylinder(m: int, rings: int):
    """Closed cylinder with fan caps (CAD-like): `rings` >= 2 rings of `m` vertices on the side, each cap a flat fan
    around a hub of valence `m`.  F = 2*m*rings."""
    assert m >= 3 and rings >= 2
    phi = 2.0 * np.pi * np.arange(m) / m
    z = np.linspace(0.0, 2.0, rings)
    ring = np.stack([np.tile(np.cos(phi), rings), np.tile(np.sin(phi), rings), np.repeat(z, m)], axis=1)
    vs = np.concatenate([[[0.0, 0.0, 0.0]], ring, [[0.0, 0.0, 2.0]]])
    faces = _orient_outward(vs, _ring_faces(m, rings, True, True))
    return _unit_mean_edge(vs, faces), faces


MESHES = {"uv": uv_sphere, "fan": fan_disc, "cyl": cylinder}


def make_mesh(kind: str, m: int, rings: int):
    return MESHES[kind](m, rings)


def valences(faces: np.ndarray, n_verts: int) -> np.ndarray:
    from dual_dmp_b200 import synth
    return np.bincount(synth.unique_edges(faces, n_verts).reshape(-1), minlength=n_verts)


# ---------------------------------------------------------------------------------------------------------------------
# graphs for the aggregation
# ---------------------------------------------------------------------------------------------------------------------
def _preferential_attachment(n: int, k: int, rng) -> list:
    """Barabasi-Albert graph (power-law degrees), edges (a, b) with a != b, unique"""
    edges, targets = set(), list(range(k))
    repeated = []
    for v in range(k, n):
        chosen = set()
        while len(chosen) < k:
            chosen.add(int(targets[rng.integers(len(targets))]) if repeated else int(rng.integers(v)))
        for t in chosen:
            edges.add((min(v, t), max(v, t)))
            repeated += [v, t]
        targets = repeated
    return sorted(edges)


def aggregation_graph(seed: int = 0):
    """A symmetric non-mesh graph for the GCN aggregation: a star of 4096 leaves, a clique of 40 nodes, a seeded power-law
    graph, three hubs of every row length in BOUNDARY_ROWS (row length = degree + the self loop), paths (rows of 3) and
    isolated nodes (rows of 1).  Caller order is block-heavy: the first 512 nodes hold the star's centre, the clique and
    one hub of each boundary length, interleaved with leaves, so the row blocks there exceed META_PER_ROW entries per
    row and the others do not.  Returns (edge_index [2, 2E] int64 with both directions, n, coords [n, 3] float64)."""
    rng = np.random.default_rng(seed)
    edges = []
    nxt = [0]

    def new(k):
        ids = np.arange(nxt[0], nxt[0] + k)
        nxt[0] += k
        return ids

    dense, sparse = [], []

    def star(k, where):
        c = new(1)[0]
        leaves = new(k)
        edges.extend((c, int(x)) for x in leaves)
        where.append(c)
        # a few leaves next to their hub, the rest spread over the sparse part
        where.extend(leaves[:3].tolist())
        sparse.extend(leaves[3:].tolist())

    star(4096, dense)
    cl = new(40)
    edges.extend((int(a), int(b)) for i, a in enumerate(cl) for b in cl[i + 1:])
    dense.extend(cl.tolist())
    for L in BOUNDARY_ROWS:
        for copy in range(3):
            star(L - 1, dense if copy == 0 else sparse)
    for _ in range(30):                               # a - b - c: b has a row of 3
        a, b, c = new(3)
        edges += [(int(a), int(b)), (int(b), int(c))]
        sparse.extend([int(a), int(b), int(c)])
    sparse.extend(new(53).tolist())                   # isolated: the self loop only
    pl = new(2000)
    edges.extend((int(pl[a]), int(pl[b])) for a, b in _preferential_attachment(2000, 2, rng))
    sparse.extend(pl.tolist())
    n = nxt[0]
    # caller order: the dense part first (shuffled, so long and short rows alternate), then the sparse part, shuffled
    dense = np.array(dense)[rng.permutation(len(dense))]
    n_fill = 512 - len(dense)
    sparse = np.array(sparse)[rng.permutation(len(sparse))]
    order = np.concatenate([dense, sparse[:n_fill]])
    order = np.concatenate([order[rng.permutation(len(order))], sparse[n_fill:]])
    assert len(order) == n and len(np.unique(order)) == n
    new_id = np.empty(n, np.int64)
    new_id[order] = np.arange(n)
    e = new_id[np.asarray(edges, dtype=np.int64)]
    ei = np.concatenate([e.T, e.T[[1, 0]]], axis=1)
    coords = rng.random((n, 3))
    return ei, n, coords


def csr_row_lengths(edge_index: np.ndarray, n: int, perm: np.ndarray | None = None) -> np.ndarray:
    """row lengths of the GCN CSR (incoming edges + one self loop) in the row order `perm` (new -> old) if given"""
    ei = np.asarray(edge_index)
    keep = ei[0] != ei[1]
    lens = np.bincount(ei[1][keep], minlength=n) + 1
    return lens if perm is None else lens[perm]


def block_nnz(row_lengths: np.ndarray, R: int) -> np.ndarray:
    pad = (-len(row_lengths)) % R
    return np.concatenate([row_lengths, np.zeros(pad, row_lengths.dtype)]).reshape(-1, R).sum(axis=1)
