"""Point-to-surface distance and two-sided Hausdorff statistics on the GPU (csrc/distance.cu).

``MeshBVH(vs, faces)`` builds a linear BVH over a target mesh once; ``.query(points)`` returns, for every point, the
exact float64 distance to the nearest triangle and that triangle's id.  ``hausdorff(a, b)`` measures how far two
meshes are apart, sampled at their vertices, the quantity upstream Dual-DMP reports with MeshLab
(check/hausdorff_checker.py, util/loss.py distance_from_reference_mesh), which needs pymeshlab.  Typical use next to
``Loss.mad`` in a training loop::

    gt = MeshBVH(gt_mesh.vs, gt_mesh.faces)              # the reference mesh's tree, built once per fit
    report = hausdorff(o1_mesh, gt)                       # report["hausdorff_rel"], report["mean_rel"]

``surface_distance(a, b, samples)`` does the same on area-weighted surface samples of both meshes, so the result does
not depend on how either mesh is triangulated, and adds the normal error across the nearest-face correspondence, which
needs no shared faces.

Contract (DESIGN.md "Point-to-mesh distance"): float64 triangle tests; a zero-area face counts as the segment or point
it spans; ties go to the lowest face id; results are deterministic and equal bit for bit those of an exhaustive scan.
"""
from __future__ import annotations

import math

import numpy as np
import torch

from ._lib import lib, ptr, set_device, stream_ptr

_NODE_BYTES = 64


def _device(device, *arrays) -> torch.device:
    for a in arrays:
        if isinstance(a, torch.Tensor) and a.is_cuda:
            return a.device if device is None else torch.device(device)
    return torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)


def _coords(x, what: str) -> np.ndarray | torch.Tensor:
    """[N,3] float32/float64 numpy array or CUDA tensor, validated on the host side"""
    if isinstance(x, torch.Tensor):
        if not x.is_cuda:
            raise RuntimeError(f"{what}: expected a CUDA tensor or a numpy array (dual_dmp_b200 has no CPU path), "
                               f"got a tensor on {x.device}")
        if x.dtype not in (torch.float32, torch.float64):
            raise ValueError(f"{what}: expected float32 or float64, got {x.dtype}")
    else:
        x = np.asarray(x)
        if x.dtype not in (np.float32, np.float64):
            raise ValueError(f"{what}: expected float32 or float64, got {x.dtype}")
    if x.ndim != 2 or x.shape[1] != 3:
        raise ValueError(f"{what}: expected shape [N, 3], got {tuple(x.shape)}")
    return x


def _to64(x, dev: torch.device) -> torch.Tensor:
    t = x if isinstance(x, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(x))
    return t.to(device=dev, dtype=torch.float64).contiguous()


def _faces(faces, n_verts: int) -> np.ndarray | torch.Tensor:
    if isinstance(faces, torch.Tensor):
        if not faces.is_cuda:
            raise RuntimeError(f"faces: expected a CUDA tensor or a numpy array (dual_dmp_b200 has no CPU path), "
                               f"got a tensor on {faces.device}")
        if faces.dtype.is_floating_point or faces.dtype.is_complex or faces.dtype == torch.bool:
            raise ValueError(f"faces: expected an integer array, got {faces.dtype}")
    else:
        faces = np.asarray(faces)
        if faces.size and not np.issubdtype(faces.dtype, np.integer):
            raise ValueError(f"faces: expected an integer array, got {faces.dtype}")
    if faces.ndim != 2 or faces.shape[1] != 3:
        raise ValueError(f"faces: expected shape [F, 3], got {tuple(faces.shape)}")
    if faces.shape[0] == 0:
        raise ValueError("faces: the target mesh has no faces")
    if faces.shape[0] >= 1 << 30:
        raise ValueError(f"faces: at most 2^30 - 1 faces are supported, got {faces.shape[0]}")
    lo, hi = int(faces.min()), int(faces.max())
    if lo < 0 or hi >= n_verts:
        raise ValueError(f"faces: vertex ids must lie in [0, {n_verts}), got [{lo}, {hi}]")
    return faces


class MeshBVH:
    """Linear BVH over the triangles of (vs [V,3], faces [F,3]) on one CUDA device, built once at construction.

    ``vs`` may be a numpy array (uploaded) or a CUDA tensor, float32 or float64 (widened to float64); ``faces`` an
    integer numpy array or CUDA tensor.  ``.vs`` / ``.faces`` hold the device copies (float64 / int32), so a
    ``MeshBVH`` is itself a mesh for ``hausdorff``."""

    def __init__(self, vs, faces, device=None):
        vs = _coords(vs, "vs")
        faces = _faces(faces, vs.shape[0])
        self.device = dev = _device(device, vs, faces)
        if dev.type != "cuda":
            raise RuntimeError(f"MeshBVH runs on CUDA only (dual_dmp_b200 has no CPU path), got device {dev}")
        self.vs = _to64(vs, dev)
        fc = faces if isinstance(faces, torch.Tensor) else torch.from_numpy(np.ascontiguousarray(faces))
        self.faces = fc.to(device=dev, dtype=torch.int32).contiguous()
        self.V, self.F = int(self.vs.shape[0]), int(self.faces.shape[0])
        st = self._stream()
        self._scratch = torch.zeros(int(lib.query("ddmp_prep_scratch_bytes")) // 8 + 1, dtype=torch.float64, device=dev)
        self.bbox = torch.empty(6, dtype=torch.float64, device=dev)
        lib.call("ddmp_prep_bbox", ptr(self.vs), ptr(self.bbox), ptr(self._scratch), self.V, st)
        keys = torch.empty(self.F, dtype=torch.int64, device=dev)
        lib.call("ddmp_bvh_keys", ptr(self.vs), ptr(self.faces), ptr(self.bbox), ptr(keys), self.F, st)
        keys, order = torch.sort(keys, stable=True)
        n_int = max(self.F - 1, 1)
        self.nodes = torch.empty(n_int * _NODE_BYTES // 4, dtype=torch.int32, device=dev)
        self.leaves = torch.empty(self.F, 4, dtype=torch.int32, device=dev)
        self.parent = torch.empty(2 * self.F - 1, dtype=torch.int32, device=dev)
        self.counters = torch.zeros(n_int, dtype=torch.int32, device=dev)        # kept zeroed for refit
        lib.call("ddmp_bvh_build", ptr(self.vs), ptr(self.faces), ptr(keys), ptr(order), ptr(self.nodes),
                 ptr(self.leaves), ptr(self.parent), ptr(self.counters), self.F, st)
        self._prefix = None            # the sampler's face-weight prefix, built by the first sample_surface

    def refit(self, vs) -> None:
        """Move the tree to new positions ``vs`` [V,3] of the same mesh: ``.vs`` and ``.bbox`` take the new values and
        the node boxes are recomputed over the kept topology.  Queries stay exact; only their speed depends on how well
        the topology, built for the first positions, fits the new ones."""
        vs = _coords(vs, "vs")
        if vs.shape[0] != self.V:
            raise ValueError(f"refit: expected {self.V} vertices, got {vs.shape[0]}")
        self.vs.copy_(_to64(vs, self.device))
        self._prefix = None
        st = self._stream()
        lib.call("ddmp_prep_bbox", ptr(self.vs), ptr(self.bbox), ptr(self._scratch), self.V, st)
        lib.call("ddmp_bvh_refit", ptr(self.vs), ptr(self.leaves), ptr(self.nodes), ptr(self.parent),
                 ptr(self.counters), self.F, st)

    def _stream(self) -> int:
        set_device(self.device)
        return stream_ptr(self.device)

    def _points(self, points) -> torch.Tensor:
        return _to64(_coords(points, "points"), self.device)

    def query(self, points) -> tuple[torch.Tensor, torch.Tensor]:
        """(dist float64 [P], face int32 [P]) on the BVH's device: distance from every point to the nearest triangle
        and that triangle's id in the caller's face numbering (the lowest id on an exact tie)."""
        pts = self._points(points)
        P = int(pts.shape[0])
        dist = torch.empty(P, dtype=torch.float64, device=self.device)
        face = torch.empty(P, dtype=torch.int32, device=self.device)
        if P:
            lib.call("ddmp_point_mesh_distance", ptr(pts), P, ptr(self.vs), ptr(self.nodes), ptr(self.leaves), self.F,
                     ptr(dist), ptr(face), self._stream())
        return dist, face

    def _query_exhaustive(self, points) -> tuple[torch.Tensor, torch.Tensor]:
        """the same outputs by scanning all faces per point: the reference tests and benchmarks compare against"""
        pts = self._points(points)
        P = int(pts.shape[0])
        dist = torch.empty(P, dtype=torch.float64, device=self.device)
        face = torch.empty(P, dtype=torch.int32, device=self.device)
        if P:
            lib.call("ddmp_point_mesh_distance_exhaustive", ptr(pts), P, ptr(self.vs), ptr(self.faces), self.F,
                     ptr(dist), ptr(face), self._stream())
        return dist, face

    def sample_surface(self, n: int, seed: int = 0, side: int = 0) -> tuple[torch.Tensor, torch.Tensor]:
        """(points float64 [n,3], face int32 [n]) on the tree's device: ``n`` deterministic points on the surface,
        stratified by area (each face gets ``n`` times its share of the area in samples, to within less than 2), in face
        order, uniform inside each face.  ``(seed, side)`` select the random numbers; ``surface_distance`` draws mesh a
        with side 0 and mesh b with side 1.  The first call reads the total weight back from the device once and raises
        ``ValueError`` when the mesh has zero total area."""
        n = _check_int(n, "samples", 1, 1 << 31)
        seed = _check_int(seed, "seed", 0, 1 << 63)
        side = _check_int(side, "side", 0, 1 << 31)
        st = self._stream()
        if self._prefix is None:
            ws = torch.empty(int(lib.query("ddmp_surface_prefix_workspace_bytes", self.F)) // 8, dtype=torch.int64,
                             device=self.device)
            prefix = torch.empty(self.F, dtype=torch.int64, device=self.device)
            lib.call("ddmp_surface_prefix", ptr(self.vs), ptr(self.faces), self.F, ptr(prefix), ptr(ws), st)
            if int(prefix[-1]) == 0:
                raise ValueError("sample_surface: the mesh has zero total area (no surface to sample)")
            self._prefix = prefix
        pts = torch.empty(n, 3, dtype=torch.float64, device=self.device)
        face = torch.empty(n, dtype=torch.int32, device=self.device)
        lib.call("ddmp_surface_sample", ptr(self.vs), ptr(self.faces), ptr(self._prefix), self.F, n, seed, side,
                 ptr(pts), ptr(face), st)
        return pts, face


def _check_int(x, what: str, lo: int, hi: int | None = None) -> int:
    if isinstance(x, (bool, np.bool_)) or not isinstance(x, (int, np.integer)):
        raise ValueError(f"{what}: expected an int, got {type(x).__name__}")
    x = int(x)
    if x < lo or (hi is not None and x >= hi):
        raise ValueError(f"{what}: expected an int in [{lo}, {'inf' if hi is None else hi}), got {x}")
    return x


def distance_stats(dist: torch.Tensor) -> dict:
    """{min, max, mean, rms, n} of a CUDA float64 distance vector (fixed-order float64 reduction on the device)"""
    if not (isinstance(dist, torch.Tensor) and dist.is_cuda and dist.dtype == torch.float64 and dist.ndim == 1):
        raise RuntimeError("distance_stats: expected a 1-D float64 CUDA tensor (dual_dmp_b200 has no CPU path)")
    n = int(dist.shape[0])
    if n == 0:
        raise ValueError("distance_stats: no distances")
    dev = dist.device
    set_device(dev)
    scratch = torch.zeros(int(lib.query("ddmp_distance_scratch_bytes")) // 8 + 1, dtype=torch.float64, device=dev)
    out = torch.empty(4, dtype=torch.float64, device=dev)
    lib.call("ddmp_distance_stats", ptr(dist.contiguous()), n, ptr(out), ptr(scratch), stream_ptr(dev))
    lo, hi, s, s2 = out.tolist()
    return {"min": lo, "max": hi, "mean": s / n, "rms": math.sqrt(s2 / n), "n": n}


def _as_bvh(m, device) -> MeshBVH:
    if isinstance(m, MeshBVH):
        return m
    if isinstance(m, (tuple, list)) and len(m) == 2:
        return MeshBVH(m[0], m[1], device)
    if hasattr(m, "vs") and hasattr(m, "faces"):
        return MeshBVH(m.vs, m.faces, device)
    raise ValueError("hausdorff: expected a mesh (an object with .vs and .faces), a (vs, faces) pair or a MeshBVH")


def hausdorff(a, b, device=None) -> dict:
    """Two-sided distance between meshes ``a`` and ``b`` (each a ``Mesh``, anything with ``.vs`` / ``.faces``, a
    ``(vs, faces)`` pair, or a ``MeshBVH`` whose tree is then reused), sampled at the vertices of each:

    * ``a_to_b`` / ``b_to_a``: ``{min, max, mean, rms, n}`` of the distances from the vertices of one mesh to the
      surface of the other;
    * ``hausdorff = max(a_to_b.max, b_to_a.max)``, ``mean = (a_to_b.mean + b_to_a.mean) / 2``;
    * ``diag``: bounding-box diagonal of ``b`` (the reference mesh); ``hausdorff_rel`` / ``mean_rel`` are the two
      values divided by it, the figure upstream's MeshLab checker reports."""
    if device is None:
        device = next((m.device for m in (a, b) if isinstance(m, MeshBVH)), None)
    ta, tb = _as_bvh(a, device), _as_bvh(b, device)
    if ta.device != tb.device:
        raise ValueError(f"hausdorff: meshes on different devices ({ta.device}, {tb.device})")
    return _two_sided(distance_stats(tb.query(ta.vs)[0]), distance_stats(ta.query(tb.vs)[0]), tb)


def _two_sided(ab: dict, ba: dict, tb: MeshBVH) -> dict:
    """the report of ``hausdorff`` from the statistics of both directions; diag from b's box"""
    bb = tb.bbox.tolist()
    diag = math.sqrt(sum((bb[3 + k] - bb[k]) ** 2 for k in range(3)))
    h = max(ab["max"], ba["max"])
    mean = 0.5 * (ab["mean"] + ba["mean"])
    return {"a_to_b": ab, "b_to_a": ba, "hausdorff": h, "mean": mean, "diag": diag,
            "hausdorff_rel": h / diag if diag > 0 else float("nan"),
            "mean_rel": mean / diag if diag > 0 else float("nan")}


def _normal_angles(ta: MeshBVH, face_a: torch.Tensor, tb: MeshBVH, face_b: torch.Tensor) -> torch.Tensor:
    """degrees between the normal of ta's face face_a[i] and of tb's face face_b[i], float64 [n]"""
    n = int(face_a.shape[0])
    deg = torch.empty(n, dtype=torch.float64, device=ta.device)
    lib.call("ddmp_normal_angle", ptr(ta.vs), ptr(ta.faces), ptr(face_a), ptr(tb.vs), ptr(tb.faces), ptr(face_b), n,
             ptr(deg), ta._stream())
    return deg


def surface_distance(a, b, samples: int, seed: int = 0, device=None) -> dict:
    """Two-sided distance and normal error between meshes ``a`` and ``b`` of any topologies, sampled on their surfaces:
    ``samples`` area-weighted points per mesh (``MeshBVH.sample_surface``, a with side 0 and b with side 1, both with
    ``seed``), each queried against the other mesh's surface.  ``a`` and ``b`` take what ``hausdorff`` takes (a reused
    ``MeshBVH`` keeps its tree and its sampling prefix).  The report:

    * ``a_to_b`` / ``b_to_a``, ``hausdorff``, ``mean``, ``diag``, ``hausdorff_rel``, ``mean_rel``: as in ``hausdorff``,
      over the surface samples instead of the vertices, ``diag`` taken from b;
    * ``normal_a_to_b`` / ``normal_b_to_a``: ``{min, max, mean, rms, n}`` of the angle in degrees between the normal of
      a sample's face and the normal of its nearest face on the other mesh (``Loss.mad``'s angle, across that
      correspondence; a flipped face reads 180, a zero-area nearest face 90);
    * ``normal_mean = (normal_a_to_b.mean + normal_b_to_a.mean) / 2``; ``samples``, ``seed``.

    A mesh of zero total area raises ``ValueError``."""
    samples = _check_int(samples, "samples", 1, 1 << 31)
    seed = _check_int(seed, "seed", 0, 1 << 63)
    if device is None:
        device = next((m.device for m in (a, b) if isinstance(m, MeshBVH)), None)
    ta, tb = _as_bvh(a, device), _as_bvh(b, device)
    if ta.device != tb.device:
        raise ValueError(f"surface_distance: meshes on different devices ({ta.device}, {tb.device})")
    pa, fa = ta.sample_surface(samples, seed, 0)
    pb, fb = tb.sample_surface(samples, seed, 1)
    d_ab, g_ab = tb.query(pa)
    d_ba, g_ba = ta.query(pb)
    nab, nba = distance_stats(_normal_angles(ta, fa, tb, g_ab)), distance_stats(_normal_angles(tb, fb, ta, g_ba))
    return {**_two_sided(distance_stats(d_ab), distance_stats(d_ba), tb), "normal_a_to_b": nab, "normal_b_to_a": nba,
            "normal_mean": 0.5 * (nab["mean"] + nba["mean"]), "samples": samples, "seed": seed}


# batched evaluation (include/ddmp_b200.h, "Batched evaluation of many fits"): table widths and block counts
THREADS, MAX_BLOCKS = 256, 1024     # DDMP_DISTANCE_THREADS, DDMP_DISTANCE_MAX_BLOCKS
EVAL_WORDS = 10                     # DDMP_EVAL_DESC_WORDS
REFIT_WORDS = 8                     # DDMP_BVH_REFIT_DESC_WORDS
QUERY_WORDS = 10                    # DDMP_DISTANCE_DESC_WORDS
STATS_WORDS = 6                     # DDMP_DISTANCE_STATS_DESC_WORDS


def _blocks(n: int, capped: bool) -> int:
    b = -(-int(n) // THREADS)
    return min(b, MAX_BLOCKS) if capped else b


def block_table(rows, counts) -> tuple[np.ndarray, int]:
    """rows [n, W] (words 2.. filled in) with words 0 / 1 set to each row's first block and block count; the total"""
    t = np.array(rows, dtype=np.int64)
    counts = np.asarray(counts, dtype=np.int64)
    t[:, 1] = counts
    t[:, 0] = np.concatenate([[0], np.cumsum(counts)[:-1]])
    return t, int(counts.sum())


class BatchEvaluator:
    """Evaluation of B fits on one device in a fixed number of launches: per fit, the MAD of the current positions'
    face normals against the clean mesh's (``Loss.mad`` of ``Mesh.compute_face_normals`` on the float32 positions) and
    the two-sided distance of ``hausdorff(positions, clean)``.

    ``meshes[i]``: fit i's mesh (``.vs``, ``.faces``: topology and starting positions); ``gts[i]``: its clean mesh
    (``.vs``, ``.faces``, ``.fn`` float64 unit face normals, the same faces as ``meshes[i]``).  The clean meshes' trees
    are built once; each fit's output tree is built once on its starting positions and refit at every evaluation.
    ``evaluate`` needs no host synchronisation and does no per-fit host work beyond writing a table when the
    positions' addresses change."""

    def __init__(self, meshes, gts, device=None):
        from .multi import DeviceTables
        if len(meshes) != len(gts) or not meshes:
            raise ValueError(f"BatchEvaluator: expected one clean mesh per fit, got {len(meshes)} fits and "
                             f"{len(gts)} clean meshes")
        self.device = dev = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError(f"BatchEvaluator runs on CUDA only (dual_dmp_b200 has no CPU path), got device {dev}")
        self.B = B = len(meshes)
        self.out = [MeshBVH(m.vs, m.faces, dev) for m in meshes]
        self.gt = [MeshBVH(g.vs, g.faces, dev) for g in gts]
        self.gt_fn = []
        for i, (o, g, gm) in enumerate(zip(self.out, self.gt, gts)):
            fn = np.asarray(gm.fn, dtype=np.float64)
            if o.F != g.F or fn.shape != (g.F, 3):
                raise ValueError(f"BatchEvaluator: fit {i} has {o.F} faces, its clean mesh {g.F} faces and "
                                 f"{fn.shape[0]} normals")
            self.gt_fn.append(torch.from_numpy(np.ascontiguousarray(fn)).to(dev))
        # diag as hausdorff() computes it, on the host once
        diag = []
        for g in self.gt:
            bb = g.bbox.tolist()
            diag.append(math.sqrt(sum((bb[3 + k] - bb[k]) ** 2 for k in range(3))))
        self.diag = torch.tensor(diag, dtype=torch.float64, device=dev)
        slot = int(lib.query("ddmp_distance_scratch_bytes"))
        slot = -(-slot // 256) * 256
        self._scratch = torch.zeros(3 * B * slot // 8, dtype=torch.float64, device=dev)   # B eval slots, 2B stats slots
        sc = lambda k: self._scratch.data_ptr() + k * slot                                 # noqa: E731
        self.mad = torch.empty(B, dtype=torch.float64, device=dev)
        self.stats = torch.empty(2 * B, 4, dtype=torch.float64, device=dev)     # rows 2i: a_to_b, 2i+1: b_to_a
        P = [n for o, g in zip(self.out, self.gt) for n in (o.V, g.V)]
        offs = np.concatenate([[0], np.cumsum(P)])
        self._dist = torch.empty(int(offs[-1]), dtype=torch.float64, device=dev)
        self._face = torch.empty(int(offs[-1]), dtype=torch.int32, device=dev)
        #: per fit (dist a_to_b, face a_to_b, dist b_to_a, face b_to_a) of the last evaluation
        self.distances = [(self._dist[offs[2 * i]:offs[2 * i + 1]], self._face[offs[2 * i]:offs[2 * i + 1]],
                           self._dist[offs[2 * i + 1]:offs[2 * i + 2]], self._face[offs[2 * i + 1]:offs[2 * i + 2]])
                          for i in range(B)]
        self.counts = torch.tensor(P, dtype=torch.float64, device=dev).view(B, 2)
        self._tables = DeviceTables(dev)
        refit, q, s = [], [], []
        for i, (o, g) in enumerate(zip(self.out, self.gt)):
            refit.append([0, 0, ptr(o.vs), ptr(o.leaves), ptr(o.nodes), ptr(o.parent), ptr(o.counters), o.F])
            d_ab, f_ab, d_ba, f_ba = self.distances[i]
            q.append([0, 0, ptr(o.vs), o.V, ptr(g.vs), ptr(g.nodes), ptr(g.leaves), g.F, ptr(d_ab), ptr(f_ab)])
            q.append([0, 0, ptr(g.vs), g.V, ptr(o.vs), ptr(o.nodes), ptr(o.leaves), o.F, ptr(d_ba), ptr(f_ba)])
            s.append([0, 0, ptr(d_ab), o.V, ptr(self.stats[2 * i]), sc(B + 2 * i)])
            s.append([0, 0, ptr(d_ba), g.V, ptr(self.stats[2 * i + 1]), sc(B + 2 * i + 1)])
        rows, self._refit_blocks = block_table(refit, [_blocks(o.F, False) if o.F > 1 else 0 for o in self.out])
        self._refit = self._tables.put("refit", rows)
        rows, self._query_blocks = block_table(q, [_blocks(n, False) for n in P])
        self._query = self._tables.put("query", rows)
        rows, self._stats_blocks = block_table(s, [_blocks(n, True) for n in P])
        self._stats_t = self._tables.put("stats", rows)
        self._eval_rows = [[0, 0, 0, ptr(o.faces), ptr(fn), ptr(o.vs), ptr(self.mad[i]), sc(i), o.V, o.F]
                           for i, (o, fn) in enumerate(zip(self.out, self.gt_fn))]
        self._eval_blocks = [_blocks(max(o.V, o.F), True) for o in self.out]
        self._eval_key = None

    def evaluate(self, positions) -> dict:
        """positions: B float32 CUDA tensors [V_i, 3] (e.g. ``MultiDualStep.pos``).  Returns device tensors [B]:
        ``mad``; ``a_to_b`` / ``b_to_a``, each ``{min, max, mean, rms}``; ``hausdorff``, ``mean``, ``diag``,
        ``hausdorff_rel``, ``mean_rel``, with the meanings of ``hausdorff(positions, clean)``."""
        if len(positions) != self.B:
            raise ValueError(f"evaluate: expected {self.B} position tensors, got {len(positions)}")
        for i, (p, o) in enumerate(zip(positions, self.out)):
            if not (isinstance(p, torch.Tensor) and p.is_cuda and p.dtype == torch.float32):
                raise RuntimeError(f"evaluate: positions {i} must be a float32 CUDA tensor (dual_dmp_b200 has no CPU "
                                   "path)")
            if p.device != self.device or tuple(p.shape) != (o.V, 3) or not p.is_contiguous():
                raise ValueError(f"evaluate: positions {i} must be a contiguous [{o.V}, 3] tensor on {self.device}, "
                                 f"got {tuple(p.shape)} on {p.device}")
        key = tuple(p.data_ptr() for p in positions)
        if key != self._eval_key:
            for row, k in zip(self._eval_rows, key):
                row[2] = k
            rows, self._eval_total = block_table(self._eval_rows, self._eval_blocks)
            self._eval = self._tables.put("eval", rows)
            self._eval_key = key
        set_device(self.device)
        st = stream_ptr(self.device)
        B = self.B
        lib.call("ddmp_eval_mad_multi", ptr(self._eval), B, self._eval_total, st)
        if self._refit_blocks:
            lib.call("ddmp_bvh_refit_multi", ptr(self._refit), B, self._refit_blocks, st)
        lib.call("ddmp_point_mesh_distance_multi", ptr(self._query), 2 * B, self._query_blocks, st)
        lib.call("ddmp_distance_stats_multi", ptr(self._stats_t), 2 * B, self._stats_blocks, st)
        s = self.stats.view(B, 2, 4)
        mean = s[:, :, 2] / self.counts
        rms = torch.sqrt(s[:, :, 3] / self.counts)
        side = [{"min": s[:, k, 0].clone(), "max": s[:, k, 1].clone(), "mean": mean[:, k], "rms": rms[:, k]}
                for k in range(2)]
        h = torch.maximum(side[0]["max"], side[1]["max"])
        m = 0.5 * (mean[:, 0] + mean[:, 1])
        ok = self.diag > 0
        nan = torch.full_like(h, float("nan"))
        return {"mad": self.mad.clone(), "a_to_b": side[0], "b_to_a": side[1], "hausdorff": h, "mean": m,
                "diag": self.diag.clone(), "hausdorff_rel": torch.where(ok, h / self.diag, nan),
                "mean_rel": torch.where(ok, m / self.diag, nan)}
