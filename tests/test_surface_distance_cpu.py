"""CPU checks of the area-weighted surface sampler's numpy oracle (oracle/surface_ref.py, the restatement the GPU
sampler is checked against bit for bit): the stratification bound, zero-weight faces, samples inside their triangles,
the centroid of a triangle's samples, seeds; and the argument validation of ``surface_distance`` that runs before any
device call."""
import os

import numpy as np
import pytest
import torch

from dual_dmp_b200 import distance as D
from dual_dmp_b200 import synth
from oracle import surface_ref as S
from oracle.distance_ref import point_triangle_d2

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

# The angle between two equal unit normals is not exactly 0: their float64 dot product can round to a few ulps below
# 1, and arccos is steep there (arccos(1 - 2^-52) = 1.2e-6 degrees, arccos(1 - 2^-51) = 1.7e-6 degrees).
ANGLE_ROUNDING_DEG = 2e-6


def degenerate_mesh():
    """icosphere(4) plus zero-area faces (repeated, collinear corners) and slivers down to 1e-12 of the largest face"""
    vs, faces = synth.icosphere(4)
    V = len(vs)
    extra_v = np.array([[2.0, 0, 0], [3.0, 0, 0], [4.0, 0, 0], [2.0, 1e-6, 0], [2.0, 1e-12, 0], [2.0, 1e-9, 1e-9]])
    extra_f = np.array([[V, V + 1, V + 2], [V, V, V + 1], [0, 0, 0], [V, V + 1, V + 3], [V, V + 1, V + 4],
                        [V, V + 2, V + 5]])
    return np.concatenate([vs, extra_v]), np.concatenate([faces, extra_f])


def meshes():
    out = {}
    for name in ("tetra", "strip2", "open4", "ico3"):
        g = np.load(os.path.join(GOLDEN, name + ".npz"))
        out[name] = (g["vs"], g["faces"])
    out["icosphere8"] = synth.icosphere(8)
    out["degenerate"] = degenerate_mesh()
    return out


@pytest.mark.parametrize("name", ["tetra", "strip2", "open4", "ico3", "icosphere8", "degenerate"])
@pytest.mark.parametrize("n", [1, 97, 20000])
def test_stratification_bound_and_zero_weight_faces(name, n):
    vs, faces = meshes()[name]
    q, P = S.quantised_prefix(vs, faces)
    Q = int(P[-1])
    assert 0 < Q < 1 << 62
    _, face, _ = S.sample_surface(vs, faces, n, seed=3, side=0)
    count = np.bincount(face, minlength=len(faces))
    assert np.all(np.abs(count - n * q.astype(np.float64) / Q) < 2)
    assert np.all(count[q == 0] == 0)
    assert np.all(np.diff(face) >= 0)                          # samples follow the face order


def test_degenerate_weights():
    vs, faces = degenerate_mesh()
    q, _ = S.quantised_prefix(vs, faces)
    F0 = len(faces) - 6
    assert np.all(q[:F0] > 0)
    assert list(q[F0:F0 + 3]) == [0, 0, 0]                     # collinear, coincident, one point
    assert q[F0 + 3] > 0 and q[F0 + 4] == 0                    # 1e-6 sliver kept, 1e-12 one (below 2^-33) dropped
    assert q.max() == 1 << 32


@pytest.mark.parametrize("name", ["tetra", "strip2", "open4", "ico3", "icosphere8", "degenerate"])
def test_samples_lie_in_their_triangles(name):
    vs, faces = meshes()[name]
    pts, face, w = S.sample_surface(vs, faces, 5000, seed=11, side=1)
    assert np.all(w >= 0) and np.all(w <= 1)
    assert np.abs(w.sum(axis=1) - 1).max() <= 1e-15
    tri = np.asarray(vs, dtype=np.float64)[np.asarray(faces)[face]]
    scale = np.abs(tri).max(axis=(1, 2))
    d = np.sqrt(point_triangle_d2(pts, tri[:, 0], tri[:, 1], tri[:, 2]))
    assert np.all(d <= 1e-15 * np.maximum(scale, 1.0))


def test_barycentric_weights_of_samples_in_one_triangle():
    tri = np.array([[0.1, 0.2, 0.3], [1.3, 0.1, -0.2], [0.4, 0.9, 0.5]])
    pts, _, _ = S.sample_surface(tri, [[0, 1, 2]], 20000, seed=5)
    # weights of b and c from the two edge vectors (least squares), a's weight the rest
    e = np.stack([tri[1] - tri[0], tri[2] - tri[0]], axis=1)
    wbc = np.linalg.lstsq(e, (pts - tri[0]).T, rcond=None)[0].T
    bary = np.concatenate([1 - wbc.sum(axis=1, keepdims=True), wbc], axis=1)
    assert bary.min() >= -1e-15 and bary.max() <= 1 + 1e-15


def test_mean_of_one_triangle_is_its_centroid():
    tri = np.array([[0.0, 0.0, 0.0], [2.0, 0.0, 0.0], [0.5, 1.5, 0.7]])
    n = 100000
    pts, face, _ = S.sample_surface(tri, [[0, 1, 2]], n, seed=1)
    assert np.all(face == 0)
    # a uniform point in a triangle has covariance (sum of c_i c_i^T over the corners about the centroid) / 12
    c = tri - tri.mean(axis=0)
    sigma = np.sqrt(np.diag(c.T @ c) / 12.0)
    assert np.all(np.abs(pts.mean(axis=0) - tri.mean(axis=0)) < 5 * sigma / np.sqrt(n))


def test_seeds_and_sides():
    vs, faces = synth.icosphere(4)
    a = S.sample_surface(vs, faces, 3000, seed=7, side=0)
    b = S.sample_surface(vs, faces, 3000, seed=7, side=0)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    for other in (S.sample_surface(vs, faces, 3000, seed=8, side=0), S.sample_surface(vs, faces, 3000, seed=7, side=1)):
        assert not np.array_equal(a[0], other[0])


def test_splitmix64_reference_values():
    # splitmix64 seeded with 0 (state += G, then the output function): the published first outputs
    out = S.mix(np.arange(1, 4, dtype=np.uint64) * S.G)
    assert [int(x) for x in out] == [0xE220A8397B1DCDAF, 0x6E789E6AA1B965F4, 0x06C45D188009454F]


def test_targets_are_exact():
    # T_i = floor((i + u0 / 2^32) * Q / n) near the top of the ranges, checked with Python integers and fractions
    from fractions import Fraction
    u0 = np.array([0, 1, 0xFFFFFFFF, 0x80000000], dtype=np.uint64)
    Q, n = (1 << 62) - 1, 4
    T = S.targets(u0, Q, n)
    for i in range(n):
        assert int(T[i]) == int((Fraction(i) + Fraction(int(u0[i]), 1 << 32)) * Q / n)
        assert int(T[i]) < Q


def test_normal_angles_oracle():
    vs, faces = synth.icosphere(2)
    f = np.arange(len(faces))
    assert S.normal_angles(vs, faces, f, vs, faces, f).max() <= ANGLE_ROUNDING_DEG
    flipped = faces[:, [0, 2, 1]]
    assert np.abs(S.normal_angles(vs, faces, f, vs, flipped, f) - 180.0).max() <= ANGLE_ROUNDING_DEG
    flat = np.array([[0.0, 0, 0], [1, 0, 0], [2, 0, 0]])
    assert S.normal_angles(vs, faces, [0], flat, [[0, 1, 2]], [0])[0] == 90.0


def test_surface_distance_rejects_bad_input_before_any_device_call():
    vs, faces = synth.icosphere(2)
    m = (vs, faces)
    for bad in (0, -1, 1 << 31, 1.5, "10", True, None):
        with pytest.raises(ValueError, match="samples"):
            D.surface_distance(m, m, bad)
    for bad in (-1, 1 << 63, 0.0, "1", False):
        with pytest.raises(ValueError, match="seed"):
            D.surface_distance(m, m, 10, seed=bad)
    with pytest.raises(RuntimeError, match="no CPU path"):
        D.surface_distance((torch.from_numpy(vs), faces), m, 10)
    with pytest.raises(RuntimeError, match="no CPU path"):
        D.surface_distance((vs, torch.from_numpy(faces)), (torch.from_numpy(vs), faces), 10)
    with pytest.raises(ValueError, match="expected a mesh"):
        D.surface_distance(object(), m, 10)
