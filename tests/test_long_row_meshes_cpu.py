"""The long-row meshes and graphs of tests/long_rows.py are well-formed and reach the kernels' long-row paths."""
import numpy as np
import pytest

from tests import long_rows as LR


def _check_mesh(vs, faces, closed):
    from dual_dmp_b200 import synth
    from dual_dmp_b200.graph import MeshTopology
    from dual_dmp_b200.util.mesh import Mesh
    mesh = Mesh(vs=vs, faces=faces)                            # raises on a non-manifold edge / face
    V, F = len(vs), len(faces)
    assert np.array_equal(np.unique(faces), np.arange(V))     # no unreferenced vertex
    E = len(mesh.edges)
    assert np.array_equal(np.sort(mesh.edges, axis=0), np.sort(synth.unique_edges(faces, V).astype(np.int32), axis=0))
    assert V - E + F == (2 if closed else 1)                  # sphere / disc
    assert mesh.f2f.shape == (F, 3)
    assert ((mesh.f2f == -1).any()) != closed
    assert np.abs(np.linalg.norm(mesh.fn, axis=1) - 1.0).max() < 1e-9     # no zero-area face
    MeshTopology(mesh, "cpu")                                 # f2f symmetry check
    return mesh


@pytest.mark.parametrize("m", LR.POLE_VALENCES)
@pytest.mark.parametrize("kind", ["uv", "fan", "cyl"])
def test_generator_is_manifold_with_intended_valence(kind, m):
    rings = 3 if m > 1000 else 4
    vs, faces = LR.make_mesh(kind, m, rings)
    mesh = _check_mesh(vs, faces, closed=kind != "fan")
    val = LR.valences(faces, len(vs))
    assert val.max() == m
    hubs = np.nonzero(val == m)[0]
    assert len(hubs) == (1 if kind == "fan" else 2)
    if kind == "uv":
        assert len(faces) == 2 * m * rings and set(np.unique(val[val != m]).tolist()) <= {5, 6}
    if kind == "fan":
        assert (mesh.f2f == -1).sum() == m                    # one boundary edge per outer face
    # the corner CSR row of a hub (faces around it) is as long as its Laplacian row
    assert np.bincount(faces.reshape(-1), minlength=len(vs))[hubs].tolist() == [m] * len(hubs)


def test_uv_sphere_orientation_and_slivers():
    vs, faces = LR.uv_sphere(4096, 15)
    fn = np.cross(vs[faces[:, 1]] - vs[faces[:, 0]], vs[faces[:, 2]] - vs[faces[:, 0]])
    fc = vs[faces].mean(axis=1)
    assert (np.einsum("ij,ij->i", fn, fc) > 0).all()          # outward
    e = np.stack([vs[faces[:, k]] - vs[faces[:, (k + 1) % 3]] for k in range(3)], axis=1)
    el = np.linalg.norm(e, axis=2)
    assert (el.max(axis=1) / el.min(axis=1)).max() > 100     # sliver faces next to the poles
    assert len(faces) <= 130_000


def test_aggregation_graph_reaches_every_long_row_path():
    from dual_dmp_b200.graph import morton_order
    ei, n, coords = LR.aggregation_graph()
    assert ei.shape[0] == 2 and (ei[0] != ei[1]).all()
    pairs = set(map(tuple, ei.T.tolist()))
    assert all((b, a) in pairs for a, b in pairs)             # symmetric
    assert len(pairs) == ei.shape[1]                          # no duplicate edge
    for perm in (None, morton_order(coords)):
        lens = LR.csr_row_lengths(ei, n, perm)
        present = set(lens.tolist())
        # rows of every boundary length around the chunks G = 8, 16, 32 and around the unroll
        assert set(LR.BOUNDARY_ROWS) <= present and set(LR.SHORT_ROWS) <= present
        assert lens.max() == 4097 and 40 in present
        for R in (64, 128, 256):                              # row blocks of the tile-staged kernels
            nnz = LR.block_nnz(lens, R)
            heavy = nnz > LR.META_PER_ROW * R
            assert heavy.any() and not heavy.all(), (R, nnz)
    lens = LR.csr_row_lengths(ei, n)
    for R in (128, 256):
        # caller order: a long row and short rows share one row block
        blk = lens[:R]
        assert blk.max() > 64 and (blk <= 3).sum() > R // 4
    assert n % 256 != 0                                       # ragged last block
    # power-law part: a heavy tail of degrees
    deg = np.bincount(ei[0], minlength=n)
    assert (deg >= 20).sum() >= 10


def test_long_row_graph_boundary_rows_are_interleaved_in_sparse_blocks():
    ei, n, _ = LR.aggregation_graph()
    lens = LR.csr_row_lengths(ei, n)
    nnz = LR.block_nnz(lens, 128)
    light = np.nonzero(nnz <= LR.META_PER_ROW * 128)[0]
    in_light = np.concatenate([lens[b * 128:(b + 1) * 128] for b in light])
    assert set(LR.BOUNDARY_ROWS) <= set(in_light.tolist())   # shared-memory (col, w) path with long rows
