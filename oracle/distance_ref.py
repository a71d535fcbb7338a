"""Oracle: point-to-triangle and point-to-mesh distance in float64 numpy, brute force.  TEST INFRASTRUCTURE.

Written independently of the kernel's Voronoi-region classification (csrc/distance.cu): the point is projected onto
the triangle's plane and kept when its barycentric signs are all non-negative; otherwise the distance is the smallest
of the distances to the three edge segments.  A face whose squared normal is at most 1e-20 |b-a|^2 |c-a|^2 (zero area:
collinear or coincident corners; the same threshold as the kernel's contract) is the union of its edges.
"""
from __future__ import annotations

import numpy as np


def _segment_d2(p, a, b):
    ab = b - a
    l2 = np.einsum("...i,...i->...", ab, ab)
    t = np.einsum("...i,...i->...", p - a, ab) / np.where(l2 > 0, l2, 1.0)
    t = np.clip(np.where(l2 > 0, t, 0.0), 0.0, 1.0)
    d = p - (a + t[..., None] * ab)
    return np.einsum("...i,...i->...", d, d)


def point_triangle_d2(p, a, b, c) -> np.ndarray:
    """squared distance from points p to triangles (a, b, c); all [..., 3], broadcast"""
    p, a, b, c = (np.asarray(x, dtype=np.float64) for x in (p, a, b, c))
    n = np.cross(b - a, c - a)
    nn = np.einsum("...i,...i->...", n, n)
    ab2 = np.einsum("...i,...i->...", b - a, b - a)
    ac2 = np.einsum("...i,...i->...", c - a, c - a)
    flat = ~(nn > 1e-20 * ab2 * ac2)
    nn_safe = np.where(flat, 1.0, nn)
    h = np.einsum("...i,...i->...", p - a, n)                    # signed height times |n|
    q = p - (h / nn_safe)[..., None] * n                         # projection onto the plane
    inside = ~flat
    for u, v in ((a, b), (b, c), (c, a)):
        inside = inside & (np.einsum("...i,...i->...", np.cross(v - u, q - u), n) >= 0)
    edges = np.minimum(np.minimum(_segment_d2(p, a, b), _segment_d2(p, b, c)), _segment_d2(p, c, a))
    return np.where(inside, h * h / nn_safe, edges)


def point_mesh_distance(points, vs, faces, chunk: int = 1 << 22):
    """(dist [P], face [P]): exact distance to the nearest face and its id (lowest id among equal squared distances)"""
    points = np.asarray(points, dtype=np.float64).reshape(-1, 3)
    tri = np.asarray(vs, dtype=np.float64)[np.asarray(faces, dtype=np.int64)]
    F = len(tri)
    step = max(1, chunk // max(F, 1))
    dist = np.empty(len(points))
    face = np.empty(len(points), dtype=np.int64)
    for s in range(0, len(points), step):
        p = points[s:s + step, None, :]
        d2 = point_triangle_d2(p, tri[None, :, 0], tri[None, :, 1], tri[None, :, 2])
        k = np.argmin(d2, axis=1)
        face[s:s + step] = k
        dist[s:s + step] = np.sqrt(d2[np.arange(len(k)), k])
    return dist, face
