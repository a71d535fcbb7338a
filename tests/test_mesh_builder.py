"""The product's vectorised ``Mesh`` (dual_dmp_b200/util/mesh.py) is bit-exact, in canonical form, against the REAL
reference's outputs (tests/golden) and against the loop oracle on other meshes; edge cases of the reference."""
import os

import numpy as np
import pytest

from dual_dmp_b200 import synth
from dual_dmp_b200.util.mesh import Mesh
from oracle.mesh_ref import MeshRef, canonical_f2f, canonical_pairs

CASES = ["ico3", "ico6", "open4", "tetra", "strip2"]


@pytest.mark.parametrize("name", CASES)
def test_against_reference_golden(golden_dir, name):
    g = dict(np.load(os.path.join(golden_dir, name + ".npz")))
    m = Mesh(vs=g["vs"], faces=g["faces"])
    assert np.array_equal(m.edges, g["edges"]) and m.edges.dtype == np.int32
    assert np.array_equal(canonical_f2f(m.f2f), g["f2f_canon"]) and m.f2f.dtype == np.int64
    assert np.array_equal(m.f2f, g["f2f_canon"])          # the product emits the canonical form directly
    assert np.array_equal(canonical_pairs(m.f_edges), g["f_edges_canon"])
    assert np.array_equal(m.v_dims.numpy(), g["v_dims"])
    for k in ("fn", "fa", "fc"):
        assert np.array_equal(getattr(m, k), g[k]), k
    assert np.allclose(m.vn, g["vn"], rtol=0, atol=1e-15)
    v2v = m.v2v_mat
    assert v2v._nnz() == 2 * len(g["edges"])
    assert np.array_equal(v2v._indices()[:, :len(g["edges"])].numpy(), g["edges"].T.astype(np.int64))


@pytest.mark.parametrize("maker", [lambda: synth.icosphere(9), lambda: synth.open_patch(7, 0.2),
                                   lambda: synth.open_patch(5, -0.3)])
def test_against_loop_oracle(maker):
    vs, faces = maker()
    rng = np.random.RandomState(0)
    perm = rng.permutation(len(faces))                     # shuffled face order exercises first-appearance logic
    faces = faces[perm]
    m, r = Mesh(vs=vs, faces=faces), MeshRef(vs, faces)
    assert np.array_equal(m.edges, r.edges)
    assert np.array_equal(m.f2f, r.f2f)
    assert np.array_equal(canonical_pairs(m.f_edges), canonical_pairs(r.f_edges))
    assert np.array_equal(m.v_dims.numpy(), r.v_dims)
    assert [sorted(s) for s in m.vf] == [sorted(s) for s in r.vf]


def test_obj_round_trip(tmp_path):
    vs, faces = synth.icosphere(2)
    p = tmp_path / "a.obj"
    synth.write_obj(str(p), vs, faces)
    m = Mesh(str(p))
    assert np.array_equal(m.faces, faces)
    assert np.allclose(m.vs, vs.astype(np.float32), atol=1e-8)
    m.save(str(tmp_path / "b.obj"))
    m2 = Mesh(str(tmp_path / "b.obj"))
    assert np.array_equal(m2.vs, m.vs)


def test_non_manifold_raises():
    vs = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1], [0, -1, 0]], dtype=np.float64)
    faces = np.array([[0, 1, 2], [0, 1, 3], [0, 1, 4]])    # three faces on edge (0,1); reference: IndexError
    with pytest.raises(ValueError):
        Mesh(vs=vs, faces=faces)


def test_icosphere_invariants():
    vs, faces = synth.icosphere(5)
    m = Mesh(vs=vs, faces=faces)
    deg = m.v_dims.numpy()
    assert (deg == 5).sum() == 12 and (deg == 6).sum() == len(vs) - 12
    assert (m.f2f >= 0).all()
    assert m.f_edges.shape == (2, 3 * len(faces))
    fwd = set(map(tuple, m.f_edges.T.tolist()))
    assert fwd == set((b, a) for a, b in fwd) and len(fwd) == m.f_edges.shape[1]


def test_save_as_ply_format(tmp_path):
    """Mesh.save_as_ply (reference util/mesh.py:287-318, used by check/mad_checker.py:48): header, 6-decimal float32
    vertices, '3 i j k r g b 255' faces with the colour truncated to 0..255 (checked byte-identical to the reference
    writer when the build container's /root/reference is importable: oracle/make_golden.py conventions)"""
    import numpy as np
    from dual_dmp_b200 import synth
    from dual_dmp_b200.util.mesh import Mesh
    vs, faces = synth.icosphere(1)
    m = Mesh(vs=vs, faces=faces)
    col = np.clip(np.abs(m.fn) * 1.2, 0, None)              # some channels above 1 -> clipped to 255
    path = tmp_path / "a.ply"
    m.save_as_ply(str(path), col)
    lines = path.read_text().split("\n")
    assert lines[:3] == ["ply", "format ascii 1.0", "element vertex 12"]
    assert lines[6] == "element face 20" and lines[12] == "end_header"
    v0 = np.float32(vs[0])
    assert lines[13] == "{0:.6f} {1:.6f} {2:.6f}".format(*v0.tolist())
    f0 = lines[13 + 12].split()
    assert f0[0] == "3" and [int(x) for x in f0[1:4]] == faces[0].tolist() and f0[7] == "255"
    assert [int(x) for x in f0[4:7]] == np.clip((255 * np.float32(col[0])).astype(int), 0, 255).tolist()
    assert len(lines) == 13 + 12 + 20 + 1


def test_reference_functions_outside_the_hot_path_refuse_loudly():
    import pytest
    from dual_dmp_b200.util import loss as L
    for name in ("weighted_norm_rec_loss", "weighted_pos_norm_loss", "bnf", "distance_from_reference_mesh"):
        with pytest.raises(NotImplementedError, match="outside the accelerated hot path"):
            getattr(L, name)(None, None)


def test_morton_order():
    """graph.morton_order (the row order of the reordered graphs): the Z-order key, a permutation with stable ties"""
    import numpy as np
    from dual_dmp_b200.graph import morton_order
    b = 3
    g = np.stack(np.meshgrid(*[np.arange(1 << b)] * 3, indexing="ij"), -1).reshape(-1, 3).astype(float)
    q = morton_order(g)
    assert sorted(q.tolist()) == list(range(len(g)))
    assert np.abs(np.diff(g[q], axis=0)).sum(1).max() > 1          # Z-order jumps between cells
    dup = np.concatenate([g[:5], g[:5]])
    assert morton_order(dup).tolist()[:2] == [0, 5]
