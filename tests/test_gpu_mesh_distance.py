"""GPU checks of point-to-mesh distance (csrc/distance.cu, dual_dmp_b200/distance.py): analytic cases, the float64
oracle on golden and synthetic meshes, bit-equality of the BVH query with the exhaustive scan, determinism, the
statistics of ``hausdorff`` and the command-line tool."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from dual_dmp_b200 import synth
from dual_dmp_b200.distance import MeshBVH, hausdorff
from dual_dmp_b200.util.mesh import Mesh
from oracle.distance_ref import point_mesh_distance, point_triangle_d2
from tests.helpers import small_case
from tests.test_mesh_distance_cpu import DEGENERATE, TETRA_F, TETRA_V, TRI, VORONOI

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _diag(vs):
    return float(np.linalg.norm(vs.max(axis=0) - vs.min(axis=0)))


def _check_against_oracle(vs, faces, pts, diag):
    d, f = MeshBVH(vs, faces).query(pts)
    d, f = d.cpu().numpy(), f.cpu().numpy().astype(np.int64)
    d_ref, _ = point_mesh_distance(pts, vs, faces)
    tol = 1e-9 * diag
    assert np.abs(d - d_ref).max() <= tol
    tri = np.asarray(vs, dtype=np.float64)[np.asarray(faces)[f]]
    d_face = np.sqrt(point_triangle_d2(pts, tri[:, 0], tri[:, 1], tri[:, 2]))
    assert np.abs(d_face - d_ref).max() <= tol          # the returned face attains the distance


def _bitwise_equal_to_exhaustive(bvh, pts):
    d, f = bvh.query(pts)
    de, fe = bvh._query_exhaustive(pts)
    assert torch.equal(d, de), (d - de).abs().max().item()
    assert torch.equal(f, fe), int((f != fe).sum())
    assert torch.isfinite(d).all()


def test_analytic_cases():
    bvh = MeshBVH(TRI, [[0, 1, 2]])
    d, f = bvh.query(np.array([p for p, _ in VORONOI]))
    np.testing.assert_allclose(d.cpu().numpy() ** 2, [d2 for _, d2 in VORONOI], rtol=1e-14, atol=1e-15)
    assert (f == 0).all()
    on = np.array([[0.2, 0.3, 0.0], [0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.5, 0.5, 0.0]])
    assert (MeshBVH(TRI, [[0, 1, 2]]).query(on)[0] <= 1e-15).all()      # 0 up to the rounding of the corner weights
    for corners, p, d2 in DEGENERATE:
        d, _ = MeshBVH(np.array(corners, dtype=np.float64), [[0, 1, 2]]).query(np.array([p]))
        assert torch.isfinite(d).all() and d.item() ** 2 == pytest.approx(d2, rel=1e-14), (corners, p)
    tet = MeshBVH(TETRA_V, TETRA_F)
    for k in range(4):
        a, b, c = TETRA_V[TETRA_F[k]]
        n = np.cross(b - a, c - a)
        d, f = tet.query(((a + b + c) / 3.0 + 0.5 * n / np.linalg.norm(n))[None])
        assert d.item() == pytest.approx(0.5, rel=1e-14) and f.item() == k


@pytest.mark.parametrize("name", ["tetra", "strip2", "open4", "ico3"])
def test_golden_meshes_against_oracle(name):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    vs, faces = g["vs"], g["faces"]
    lo, hi = vs.min(axis=0), vs.max(axis=0)
    centre, half = (lo + hi) / 2, np.maximum(hi - lo, 1e-3)           # "twice the box": +-1 half-extent x 2
    rng = np.random.default_rng(7)
    pts = np.concatenate([vs, centre + (rng.random((2000, 3)) - 0.5) * 2 * half])
    _check_against_oracle(vs, faces, pts, _diag(vs))


@pytest.mark.parametrize("n", [8, 16])
def test_noisy_against_clean_both_directions(n):
    noisy, _, gt = small_case("ico", n)
    _check_against_oracle(gt.vs, gt.faces, noisy.vs, _diag(gt.vs))
    _check_against_oracle(noisy.vs, noisy.faces, gt.vs, _diag(noisy.vs))


def test_bvh_equals_exhaustive_n64():
    case = synth.make_case(64)
    bvh = MeshBVH(case.gt_vs, case.faces)
    assert bvh.F == 81920
    _bitwise_equal_to_exhaustive(bvh, case.noise_vs)
    rng = np.random.default_rng(3)
    dirs = rng.normal(size=(512, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    far = np.concatenate([dirs * s for s in (1e2, 1e4, 1e7)])
    _bitwise_equal_to_exhaustive(bvh, np.concatenate([far, np.zeros((4, 3))]))   # the sphere's centre ties widely


def test_bvh_equals_exhaustive_duplicate_keys():
    # 4 centres x 300 triangles sharing one centroid each (equal Morton keys), plus exact copies of some of them
    rng = np.random.default_rng(4)
    tris = []
    for c in ([0, 0, 0], [1, 0, 0], [0, 3, 0], [0, 0, 5]):
        e1, e2 = rng.normal(size=(300, 3)), rng.normal(size=(300, 3))
        tris.append(np.stack([c + e1, c + e2, c - e1 - e2], axis=1))
    tris = np.concatenate(tris)
    tris = np.concatenate([tris, tris[::7]])
    vs, faces = tris.reshape(-1, 3), np.arange(3 * len(tris)).reshape(-1, 3)
    bvh = MeshBVH(vs, faces)
    pts = rng.normal(size=(4096, 3)) * 3
    _bitwise_equal_to_exhaustive(bvh, np.concatenate([pts, vs]))
    _, f = bvh.query(vs[3 * 1200:3 * 1210])          # corners of the copies: the original (lower id) wins the tie
    assert (f.cpu().numpy() < 1200).all()


def test_one_face_mesh():
    bvh = MeshBVH(TRI, [[0, 1, 2]])
    rng = np.random.default_rng(5)
    _bitwise_equal_to_exhaustive(bvh, rng.normal(size=(1000, 3)))


@pytest.fixture(scope="module")
def case224():
    return synth.make_case(224)


def test_bvh_equals_exhaustive_1m_sample(case224):
    bvh = MeshBVH(case224.gt_vs, case224.faces)
    idx = np.random.default_rng(6).choice(len(case224.noise_vs), 65536, replace=False)
    _bitwise_equal_to_exhaustive(bvh, case224.noise_vs[idx])


def test_determinism_and_face_permutation():
    noisy, _, gt = small_case("ico", 16)
    bvh = MeshBVH(gt.vs, gt.faces)
    d1, f1 = bvh.query(noisy.vs)
    d2, f2 = MeshBVH(gt.vs, gt.faces).query(noisy.vs)
    assert torch.equal(d1, d2) and torch.equal(f1, f2)
    perm = np.random.default_rng(8).permutation(len(gt.faces))
    dp, fp = MeshBVH(gt.vs, gt.faces[perm]).query(noisy.vs)
    assert torch.equal(dp, d1)          # face ids may differ where faces tie (a shared nearest vertex or edge)


def test_inputs_float32_tensors_and_empty():
    noisy, _, gt = small_case("ico", 8)
    dev = torch.device("cuda")
    ref = MeshBVH(gt.vs.astype(np.float32).astype(np.float64), gt.faces).query(noisy.vs.astype(np.float32))
    got = MeshBVH(torch.from_numpy(gt.vs).float().to(dev), torch.from_numpy(gt.faces).to(dev)).query(
        torch.from_numpy(noisy.vs).float().to(dev))
    assert torch.equal(ref[0], got[0]) and torch.equal(ref[1], got[1])
    assert got[0].dtype == torch.float64 and got[1].dtype == torch.int32 and got[0].is_cuda
    d, f = MeshBVH(gt.vs, gt.faces).query(np.zeros((0, 3)))
    assert d.shape == (0,) and f.shape == (0,)
    with pytest.raises(RuntimeError, match="no CPU path"):
        MeshBVH(gt.vs, gt.faces).query(torch.zeros(4, 3))
    with pytest.raises(ValueError, match="shape"):
        MeshBVH(gt.vs, gt.faces).query(np.zeros((4, 2)))


def test_hausdorff_statistics():
    noisy, _, gt = small_case("ico", 16)
    rep = hausdorff(noisy, gt)
    assert rep == hausdorff((noisy.vs, noisy.faces), (gt.vs, gt.faces))
    assert rep == hausdorff(noisy, MeshBVH(gt.vs, gt.faces))
    d_ab = MeshBVH(gt.vs, gt.faces).query(noisy.vs)[0].cpu().numpy()
    d_ba = MeshBVH(noisy.vs, noisy.faces).query(gt.vs)[0].cpu().numpy()
    for s, d in ((rep["a_to_b"], d_ab), (rep["b_to_a"], d_ba)):
        assert s["n"] == len(d) and s["min"] == d.min() and s["max"] == d.max()
        assert s["mean"] == pytest.approx(d.mean(), rel=1e-12)
        assert s["rms"] == pytest.approx(np.sqrt((d * d).mean()), rel=1e-12)
    assert rep["hausdorff"] == max(d_ab.max(), d_ba.max())
    assert rep["mean"] == pytest.approx(0.5 * (d_ab.mean() + d_ba.mean()), rel=1e-12)
    assert rep["diag"] == pytest.approx(_diag(gt.vs), rel=1e-15)
    assert rep["hausdorff_rel"] == rep["hausdorff"] / rep["diag"] and rep["mean_rel"] == rep["mean"] / rep["diag"]
    same = hausdorff(gt, gt)
    assert same["hausdorff"] == 0.0 and same["mean"] == 0.0


def test_cli_matches_hausdorff(tmp_path):
    case = synth.make_case(8)
    synth.write_case(str(tmp_path / "c"), case)
    gt, noise = str(tmp_path / "c" / "c_gt.obj"), str(tmp_path / "c" / "c_noise.obj")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "mesh_distance.py"), "--gt", gt, noise, gt],
                         capture_output=True, text=True, check=True, cwd=str(tmp_path)).stdout
    lines = [json.loads(x) for x in out.strip().splitlines()]
    assert [x["file"] for x in lines] == [noise, gt]
    m_gt, m_noise = Mesh(gt), Mesh(noise)
    want = hausdorff(m_noise, m_gt)
    for k in ("hausdorff", "mean", "diag", "hausdorff_rel", "mean_rel", "a_to_b", "b_to_a"):
        assert lines[0][k] == want[k], k
    from dual_dmp_b200.util import loss as L
    assert lines[0]["mad"] == pytest.approx(L.mad(m_noise.fn, m_gt.fn), rel=1e-12)
    assert lines[1]["hausdorff"] == 0.0 and lines[1]["mad"] == pytest.approx(0.0, abs=1e-5)
