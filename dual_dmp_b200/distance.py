"""Point-to-surface distance and two-sided Hausdorff statistics on the GPU (csrc/distance.cu).

``MeshBVH(vs, faces)`` builds a linear BVH over a target mesh once; ``.query(points)`` returns, for every point, the
exact float64 distance to the nearest triangle and that triangle's id.  ``hausdorff(a, b)`` measures how far two
meshes are apart, sampled at their vertices, the quantity upstream Dual-DMP reports with MeshLab
(check/hausdorff_checker.py, util/loss.py distance_from_reference_mesh), which needs pymeshlab.  Typical use next to
``Loss.mad`` in a training loop::

    gt = MeshBVH(gt_mesh.vs, gt_mesh.faces)              # the reference mesh's tree, built once per fit
    report = hausdorff(o1_mesh, gt)                       # report["hausdorff_rel"], report["mean_rel"]

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
        parent = torch.empty(2 * self.F - 1, dtype=torch.int32, device=dev)
        counters = torch.zeros(n_int, dtype=torch.int32, device=dev)
        lib.call("ddmp_bvh_build", ptr(self.vs), ptr(self.faces), ptr(keys), ptr(order), ptr(self.nodes),
                 ptr(self.leaves), ptr(parent), ptr(counters), self.F, st)

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
    ab = distance_stats(tb.query(ta.vs)[0])
    ba = distance_stats(ta.query(tb.vs)[0])
    bb = tb.bbox.tolist()
    diag = math.sqrt(sum((bb[3 + k] - bb[k]) ** 2 for k in range(3)))
    h = max(ab["max"], ba["max"])
    mean = 0.5 * (ab["mean"] + ba["mean"])
    return {"a_to_b": ab, "b_to_a": ba, "hausdorff": h, "mean": mean, "diag": diag,
            "hausdorff_rel": h / diag if diag > 0 else float("nan"),
            "mean_rel": mean / diag if diag > 0 else float("nan")}
