"""Oracle: the area-weighted surface sampler and the normal angle of csrc/distance.cu in numpy.  TEST INFRASTRUCTURE.

Restates include/ddmp_b200.h "Area-weighted surface samples" step by step: float64 face weights with the kernel's
order of operations (numpy rounds each IEEE operation as the kernel does without multiply-add contraction), the
quantised int64 weights and their prefix, splitmix64 in numpy uint64 arithmetic, the stratified targets in Python
integers (exact, where the kernel uses 128-bit integers), the face search and the sample points.  So the samples equal
the kernel's bit for bit.  The angles use numpy's arccos, which may differ from the device's in the last bits.
"""
from __future__ import annotations

import numpy as np

G = np.uint64(0x9E3779B97F4A7C15)
_M1, _M2 = np.uint64(0xBF58476D1CE4E5B9), np.uint64(0x94D049BB133111EB)


def _cross(u, w):
    return np.stack([u[:, 1] * w[:, 2] - u[:, 2] * w[:, 1], u[:, 2] * w[:, 0] - u[:, 0] * w[:, 2],
                     u[:, 0] * w[:, 1] - u[:, 1] * w[:, 0]], axis=1)


def _face_cross(vs, faces):
    vs = np.asarray(vs, dtype=np.float64)
    faces = np.asarray(faces, dtype=np.int64)
    a = vs[faces[:, 0]]
    return _cross(vs[faces[:, 1]] - a, vs[faces[:, 2]] - a)


def _norm(n):
    return np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2])


def face_weights(vs, faces) -> np.ndarray:
    """w_f = |(b-a) x (c-a)|, float64"""
    return _norm(_face_cross(vs, faces))


def quantised_prefix(vs, faces) -> tuple[np.ndarray, np.ndarray]:
    """(q int64 [F], P int64 [F]): q_f = rint(w_f / w_max * 2^32), 0 where not positive; P its inclusive prefix"""
    w = face_weights(vs, faces)
    wm = np.max(np.where(np.isnan(w), 0.0, w))
    with np.errstate(invalid="ignore", divide="ignore"):
        x = np.rint(w / wm * 4294967296.0)
    q = np.where(x > 0, x, 0.0).astype(np.int64)
    return q, np.cumsum(q)


def mix(z) -> np.ndarray:
    """splitmix64's output function, uint64 (wrapping)"""
    z = np.asarray(z, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = (z ^ (z >> np.uint64(30))) * _M1
        z = (z ^ (z >> np.uint64(27))) * _M2
    return z ^ (z >> np.uint64(31))


def words(seed: int, side: int, n: int) -> np.ndarray:
    """[n, 3] uint64: word k of sample i = mix(key + (3i + k + 1) * G), key = mix(mix(seed + G) + (side + 1) * G)"""
    with np.errstate(over="ignore"):
        key = mix(mix(np.uint64(seed) + G) + np.uint64(side + 1) * G)
        ctr = np.arange(1, 3 * n + 1, dtype=np.uint64) * G + key
    return mix(ctr).reshape(n, 3)


def targets(u0: np.ndarray, Q: int, n: int) -> np.ndarray:
    """T_i = ((i * 2^32 + u0_i) * Q) div (n * 2^32), in Python integers"""
    x = np.arange(n, dtype=object) * (1 << 32) + u0.astype(object)
    return np.array((x * int(Q)) // (int(n) << 32), dtype=np.uint64)


def sample_surface(vs, faces, n: int, seed: int = 0, side: int = 0):
    """(points float64 [n,3], face int64 [n], weights float64 [n,3] = (wa, wb, wc)) as the kernel computes them"""
    vs = np.asarray(vs, dtype=np.float64)
    faces = np.asarray(faces, dtype=np.int64)
    _, P = quantised_prefix(vs, faces)
    Q = int(P[-1])
    if Q == 0:
        raise ValueError("zero total area")
    w = words(seed, side, n)
    u0 = w[:, 0] >> np.uint64(32)
    s = np.sqrt((w[:, 1] >> np.uint64(11)).astype(np.float64) * 2.0 ** -53)
    r2 = (w[:, 2] >> np.uint64(11)).astype(np.float64) * 2.0 ** -53
    face = np.searchsorted(P.astype(np.uint64), targets(u0, Q, n), side="right")
    wa, wb, wc = 1.0 - s, s * (1.0 - r2), s * r2
    a, b, c = (vs[faces[face, k]] for k in range(3))
    pts = (wa[:, None] * a + wb[:, None] * b) + wc[:, None] * c
    return pts, face, np.stack([wa, wb, wc], axis=1)


def unit_normals(vs, faces) -> np.ndarray:
    """cross / (|cross| + 1e-24), Mesh.compute_face_normals's float64 expression"""
    n = _face_cross(vs, faces)
    return n / (_norm(n) + 1e-24)[:, None]


def normal_angles(vs_a, faces_a, face_a, vs_b, faces_b, face_b) -> np.ndarray:
    """degrees between the normal of face_a[i] of mesh A and of face_b[i] of mesh B"""
    na = unit_normals(vs_a, faces_a)[np.asarray(face_a)]
    nb = unit_normals(vs_b, faces_b)[np.asarray(face_b)]
    c = (na[:, 0] * nb[:, 0] + na[:, 1] * nb[:, 1]) + na[:, 2] * nb[:, 2]
    return np.rad2deg(np.arccos(np.clip(c, -1.0, 1.0)))
