"""CPU checks of point-to-mesh distance: the float64 numpy oracle against analytic answers, and the argument
validation of dual_dmp_b200.distance that runs before any device call."""
import numpy as np
import pytest
import torch

from dual_dmp_b200 import distance as D
from oracle.distance_ref import point_mesh_distance, point_triangle_d2

TRI = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.0]])

# (point, squared distance to TRI): one point in each of the seven Voronoi regions
VORONOI = [
    ((-1.0, -1.0, 0.5), 2.25),    # vertex a
    ((2.0, -1.0, 0.0), 2.0),      # vertex b
    ((-1.0, 2.0, 0.0), 2.0),      # vertex c
    ((0.5, -1.0, 2.0), 5.0),      # edge ab, closest (0.5, 0, 0)
    ((-1.0, 0.5, 0.0), 1.0),      # edge ca, closest (0, 0.5, 0)
    ((1.0, 1.0, 3.0), 9.5),       # edge bc, closest (0.5, 0.5, 0)
    ((0.25, 0.25, -2.0), 4.0),    # face
]

# (corners, point, squared distance): zero-area faces are the segment or point they span
DEGENERATE = [
    (((0, 0, 0), (1, 0, 0), (2, 0, 0)), (1.5, 1.0, 0.0), 1.0),      # collinear, inside the span
    (((0, 0, 0), (1, 0, 0), (2, 0, 0)), (3.0, 0.0, 0.0), 1.0),      # collinear, beyond the far end
    (((0, 0, 0), (2, 0, 0), (1, 0, 0)), (-1.0, 0.0, 2.0), 5.0),     # collinear, other corner order
    (((0, 0, 0), (0, 0, 0), (0, 0, 2)), (1.0, 0.0, 1.0), 1.0),      # two coincident corners
    (((1, 1, 1), (1, 1, 1), (1, 1, 1)), (1.0, 1.0, 3.0), 4.0),      # one point
]

# regular tetrahedron centred at the origin, faces outward; inradius 1/sqrt(3)
TETRA_V = np.array([[1.0, 1.0, 1.0], [1.0, -1.0, -1.0], [-1.0, 1.0, -1.0], [-1.0, -1.0, 1.0]])
TETRA_F = np.array([[0, 1, 2], [0, 3, 1], [0, 2, 3], [1, 3, 2]])


def test_oracle_voronoi_regions():
    for p, d2 in VORONOI:
        assert point_triangle_d2(np.array(p), *TRI) == pytest.approx(d2, rel=1e-14, abs=1e-15), p


def test_oracle_points_on_surface():
    rng = np.random.default_rng(1)
    tri = rng.normal(size=(3, 3))
    w = rng.dirichlet(np.ones(3), size=200)
    d2 = point_triangle_d2(w @ tri, *tri)
    assert np.all(d2 <= 1e-28)
    assert np.all(point_triangle_d2(tri, *tri) <= 1e-28)
    assert point_triangle_d2(np.array([0.2, 0.3, 0.0]), *TRI) == 0.0


def test_oracle_degenerate_faces():
    for corners, p, d2 in DEGENERATE:
        got = point_triangle_d2(np.array(p, dtype=np.float64), *np.array(corners, dtype=np.float64))
        assert np.isfinite(got) and got == pytest.approx(d2, rel=1e-14), (corners, p)


def test_oracle_tetrahedron():
    for f in range(4):
        a, b, c = TETRA_V[TETRA_F[f]]
        centre = (a + b + c) / 3.0
        n = np.cross(b - a, c - a)
        n /= np.linalg.norm(n)
        assert n @ centre > 0                                     # outward
        d, face = point_mesh_distance((centre + 0.5 * n)[None], TETRA_V, TETRA_F)
        assert d[0] == pytest.approx(0.5, rel=1e-14) and face[0] == f
    d, face = point_mesh_distance(np.zeros((1, 3)), TETRA_V, TETRA_F)
    assert d[0] == pytest.approx(1.0 / np.sqrt(3.0), rel=1e-14)


def test_oracle_mesh_is_min_over_faces():
    rng = np.random.default_rng(2)
    vs, faces = rng.normal(size=(30, 3)), rng.integers(0, 30, size=(40, 3))
    pts = rng.normal(size=(50, 3)) * 2
    d, face = point_mesh_distance(pts, vs, faces, chunk=97)
    full = np.sqrt(point_triangle_d2(pts[:, None], vs[faces][None, :, 0], vs[faces][None, :, 1], vs[faces][None, :, 2]))
    np.testing.assert_array_equal(d, full.min(axis=1))
    np.testing.assert_array_equal(full[np.arange(len(pts)), face], d)


def test_meshbvh_rejects_bad_input_before_any_device_call():
    vs, faces = TETRA_V, TETRA_F
    with pytest.raises(RuntimeError, match="no CPU path"):
        D.MeshBVH(torch.from_numpy(vs), faces)
    with pytest.raises(RuntimeError, match="no CPU path"):
        D.MeshBVH(vs, torch.from_numpy(faces))
    with pytest.raises(ValueError, match="vertex ids"):
        D.MeshBVH(vs, faces + 1)
    with pytest.raises(ValueError, match="vertex ids"):
        D.MeshBVH(vs, -faces - 1)
    with pytest.raises(ValueError, match="no faces"):
        D.MeshBVH(vs, np.zeros((0, 3), dtype=np.int64))
    with pytest.raises(ValueError, match="shape"):
        D.MeshBVH(vs[:, :2], faces)
    with pytest.raises(ValueError, match="shape"):
        D.MeshBVH(vs, faces[:, :2])
    with pytest.raises(ValueError, match="float32 or float64"):
        D.MeshBVH(vs.astype(np.int64), faces)
    with pytest.raises(ValueError, match="integer"):
        D.MeshBVH(vs, faces.astype(np.float64))
    with pytest.raises(ValueError, match="expected a mesh"):
        D.hausdorff(object(), (vs, faces))
    with pytest.raises(RuntimeError, match="no CPU path"):
        D.distance_stats(torch.zeros(3, dtype=torch.float64))
