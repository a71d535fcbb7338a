"""GPU checks of the area-weighted surface sampler and ``surface_distance`` (csrc/distance.cu, dual_dmp_b200/distance.py):
samples bit for bit against the numpy oracle, sample distances against the exhaustive scan and the float64 oracle,
analytic cases on meshes of different topologies, determinism, the report's statistics, the command-line tool and a
1M-face case."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from dual_dmp_b200 import synth
from dual_dmp_b200.distance import MeshBVH, distance_stats, hausdorff, surface_distance
from dual_dmp_b200.util.mesh import Mesh
from oracle import surface_ref as S
from oracle.distance_ref import point_mesh_distance
from tests.helpers import small_case
from tests.test_surface_distance_cpu import ANGLE_ROUNDING_DEG, degenerate_mesh, meshes

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _diag(vs):
    return float(np.linalg.norm(vs.max(axis=0) - vs.min(axis=0)))


def grid_square(k: int, z: float = 0.0):
    """the unit square [0,1]^2 at height z as a k x k grid of 2k^2 triangles, normals +z"""
    t = np.linspace(0.0, 1.0, k + 1)
    x, y = np.meshgrid(t, t, indexing="ij")
    vs = np.stack([x.ravel(), y.ravel(), np.full(x.size, z)], axis=1)
    idx = np.arange((k + 1) ** 2).reshape(k + 1, k + 1)
    a, b, c, d = idx[:-1, :-1].ravel(), idx[1:, :-1].ravel(), idx[1:, 1:].ravel(), idx[:-1, 1:].ravel()
    faces = np.concatenate([np.stack([a, b, c], axis=1), np.stack([a, c, d], axis=1)])
    return vs, faces


@pytest.mark.parametrize("name", ["tetra", "strip2", "open4", "ico3", "icosphere8", "degenerate"])
@pytest.mark.parametrize("seed,side", [(0, 0), (3, 1)])
def test_samples_equal_oracle_bitwise(name, seed, side):
    vs, faces = meshes()[name]
    bvh = MeshBVH(vs, faces)
    for n in (1, 1000, 20011):
        pts, face = bvh.sample_surface(n, seed, side)
        assert pts.dtype == torch.float64 and face.dtype == torch.int32 and pts.shape == (n, 3) and face.is_cuda
        want_pts, want_face, _ = S.sample_surface(vs, faces, n, seed, side)
        np.testing.assert_array_equal(face.cpu().numpy(), want_face)
        assert np.array_equal(pts.cpu().numpy(), want_pts), np.abs(pts.cpu().numpy() - want_pts).max()
    np.testing.assert_array_equal(bvh._prefix.cpu().numpy(), S.quantised_prefix(vs, faces)[1])


def test_sample_distances_equal_exhaustive_and_oracle():
    noisy, _, gt = small_case("ico", 16)
    ta, tb = MeshBVH(noisy.vs, noisy.faces), MeshBVH(gt.vs, gt.faces)
    pa, fa = ta.sample_surface(6000, seed=2)
    d, f = tb.query(pa)
    de, fe = tb._query_exhaustive(pa)
    assert torch.equal(d, de) and torch.equal(f, fe)
    d_ref, _ = point_mesh_distance(pa.cpu().numpy(), gt.vs, gt.faces)
    assert np.abs(d.cpu().numpy() - d_ref).max() <= 1e-9 * _diag(gt.vs)
    deg = S.normal_angles(noisy.vs, noisy.faces, fa.cpu().numpy(), gt.vs, gt.faces, f.cpu().numpy())
    rep = surface_distance(ta, tb, 6000, seed=2)
    assert rep["a_to_b"]["max"] == d.max().item()
    assert rep["normal_a_to_b"]["mean"] == pytest.approx(deg.mean(), rel=1e-12)
    assert rep["normal_a_to_b"]["max"] == pytest.approx(deg.max(), rel=1e-12)


def test_square_against_grid_at_height():
    h = 0.25
    a, b = grid_square(1), grid_square(8, h)
    assert len(a[1]) == 2 and len(b[1]) == 128
    rep = surface_distance(a, b, 20000, seed=4)
    for side in ("a_to_b", "b_to_a"):
        assert rep[side]["min"] == pytest.approx(h, rel=1e-14) and rep[side]["max"] == pytest.approx(h, rel=1e-14)
    for side in ("normal_a_to_b", "normal_b_to_a"):
        assert rep[side]["max"] <= 1e-6
    assert rep["hausdorff"] == pytest.approx(h, rel=1e-14)


@pytest.mark.parametrize("alpha_deg", [7.5, 30.0])
def test_tilted_grid_angle(alpha_deg):
    a = grid_square(1)
    vs, faces = grid_square(8)
    al = math.radians(alpha_deg)
    rot = np.array([[1, 0, 0], [0, math.cos(al), -math.sin(al)], [0, math.sin(al), math.cos(al)]])
    centre = np.array([0.5, 0.5, 0.0])
    b = ((vs - centre) @ rot.T + centre, faces)                  # tilted about the x axis through the centre
    s = surface_distance(a, b, 20000, seed=6)["normal_b_to_a"]
    assert s["min"] == pytest.approx(alpha_deg, abs=1e-6) and s["max"] == pytest.approx(alpha_deg, abs=1e-6)
    assert s["n"] == 20000


def test_coarse_against_fine_icosphere_within_sagitta():
    coarse, fine = synth.icosphere(4), synth.icosphere(16)
    vs, faces = coarse
    n = synth.face_normals_areas(vs, faces)[0]
    rho = np.abs(np.einsum("ij,ij->i", n, vs[faces[:, 0]])).min()  # the nearest face plane to the centre
    sagitta = 1.0 - rho
    rep = surface_distance(coarse, fine, 200000, seed=1)
    assert rep["a_to_b"]["max"] <= sagitta + 1e-12 and rep["b_to_a"]["max"] <= sagitta + 1e-12
    assert rep["a_to_b"]["mean"] > 0.05 * sagitta                  # the faces' interiors are sampled, not just corners
    vertex = hausdorff(coarse, fine)
    assert vertex["b_to_a"]["max"] <= sagitta + 1e-12


def test_same_mesh_gives_zero():
    noisy, _, _ = small_case("ico", 16)
    rep = surface_distance(noisy, noisy, 50000, seed=9)
    assert rep["hausdorff"] <= 1e-14 * rep["diag"]
    assert rep["normal_a_to_b"]["max"] <= ANGLE_ROUNDING_DEG and rep["normal_b_to_a"]["max"] <= ANGLE_ROUNDING_DEG


def test_reruns_are_bitwise_equal():
    noisy, _, gt = small_case("ico", 16)
    tb = MeshBVH(gt.vs, gt.faces)
    assert surface_distance(noisy, tb, 30000, seed=5) == surface_distance((noisy.vs, noisy.faces), tb, 30000, seed=5)
    p1, f1 = tb.sample_surface(30000, 5, 1)
    p2, f2 = MeshBVH(gt.vs, gt.faces).sample_surface(30000, 5, 1)
    assert torch.equal(p1, p2) and torch.equal(f1, f2)
    assert surface_distance(noisy, tb, 30000, seed=6) != surface_distance(noisy, tb, 30000, seed=5)


def test_report_statistics():
    noisy, _, gt = small_case("ico", 16)
    ta, tb = MeshBVH(noisy.vs, noisy.faces), MeshBVH(gt.vs, gt.faces)
    n = 40000
    rep = surface_distance(ta, tb, n, seed=3)
    pa, fa = ta.sample_surface(n, 3, 0)
    pb, fb = tb.sample_surface(n, 3, 1)
    d_ab, g_ab = tb.query(pa)
    d_ba, g_ba = ta.query(pb)
    ang_ab = S.normal_angles(noisy.vs, noisy.faces, fa.cpu().numpy(), gt.vs, gt.faces, g_ab.cpu().numpy())
    ang_ba = S.normal_angles(gt.vs, gt.faces, fb.cpu().numpy(), noisy.vs, noisy.faces, g_ba.cpu().numpy())
    for key, d in (("a_to_b", d_ab), ("b_to_a", d_ba)):
        assert rep[key] == distance_stats(d)
        d = d.cpu().numpy()
        assert rep[key]["n"] == n and rep[key]["min"] == d.min() and rep[key]["max"] == d.max()
        assert rep[key]["mean"] == pytest.approx(d.mean(), rel=1e-12)
        assert rep[key]["rms"] == pytest.approx(np.sqrt((d * d).mean()), rel=1e-12)
    for key, ang in (("normal_a_to_b", ang_ab), ("normal_b_to_a", ang_ba)):
        s = rep[key]
        assert s["n"] == n and s["min"] == pytest.approx(ang.min(), abs=1e-9)
        assert s["max"] == pytest.approx(ang.max(), rel=1e-12)
        assert s["mean"] == pytest.approx(ang.mean(), rel=1e-12)
        assert s["rms"] == pytest.approx(np.sqrt((ang * ang).mean()), rel=1e-12)
    assert rep["hausdorff"] == max(rep["a_to_b"]["max"], rep["b_to_a"]["max"])
    assert rep["mean"] == 0.5 * (rep["a_to_b"]["mean"] + rep["b_to_a"]["mean"])
    assert rep["normal_mean"] == 0.5 * (rep["normal_a_to_b"]["mean"] + rep["normal_b_to_a"]["mean"])
    assert rep["diag"] == hausdorff(ta, tb)["diag"]
    assert rep["hausdorff_rel"] == rep["hausdorff"] / rep["diag"] and rep["mean_rel"] == rep["mean"] / rep["diag"]
    assert rep["samples"] == n and rep["seed"] == 3


def test_zero_area_and_refit():
    flat = (np.array([[0.0, 0, 0], [1, 0, 0], [2, 0, 0]]), [[0, 1, 2]])
    with pytest.raises(ValueError, match="zero total area"):
        MeshBVH(*flat).sample_surface(10)
    with pytest.raises(ValueError, match="zero total area"):
        surface_distance(grid_square(2), flat, 10)
    vs, faces = degenerate_mesh()
    bvh = MeshBVH(vs, faces)
    bvh.sample_surface(1000)
    bvh.refit(vs * 2.0)                                            # new positions: the prefix is rebuilt
    p1, f1 = bvh.sample_surface(1000)
    want, want_f, _ = S.sample_surface(vs * 2.0, faces, 1000)
    assert np.array_equal(p1.cpu().numpy(), want) and np.array_equal(f1.cpu().numpy(), want_f)
    with pytest.raises(ValueError, match="samples"):
        bvh.sample_surface(0)
    with pytest.raises(ValueError, match="side"):
        bvh.sample_surface(10, side=-1)


def test_cli_with_and_without_samples(tmp_path):
    case = synth.make_case(8)
    synth.write_case(str(tmp_path / "c"), case)
    gt, noise = str(tmp_path / "c" / "c_gt.obj"), str(tmp_path / "c" / "c_noise.obj")
    coarse = str(tmp_path / "coarse.obj")
    vs4, f4 = synth.icosphere(4)
    synth.write_obj(coarse, vs4 * np.abs(case.gt_vs).max(), f4)                    # another face count
    script = os.path.join(ROOT, "scripts", "mesh_distance.py")
    run = lambda *extra: subprocess.run([sys.executable, script, "--gt", gt, *extra, noise, coarse],  # noqa: E731
                                        capture_output=True, text=True, check=True, cwd=str(tmp_path)).stdout
    plain = [json.loads(x) for x in run().strip().splitlines()]
    assert [x["file"] for x in plain] == [noise, coarse]
    assert "mad" in plain[0] and "mad" not in plain[1] and all("surface" not in x for x in plain)
    m_gt = Mesh(gt)
    assert plain[1]["hausdorff"] == hausdorff(Mesh(coarse), m_gt)["hausdorff"]
    lines = [json.loads(x) for x in run("--samples", "5000", "--seed", "2").strip().splitlines()]
    for x, p, path in zip(lines, plain, (noise, coarse)):
        assert x["surface"] == surface_distance(Mesh(path), m_gt, 5000, seed=2), path
        assert {k: v for k, v in x.items() if k != "surface"} == p
    bad = subprocess.run([sys.executable, script, "--gt", gt, "--samples", "0", noise], capture_output=True, text=True)
    assert bad.returncode != 0 and "--samples" in bad.stderr


def test_1m_faces_4m_samples():
    case = synth.make_case(224)
    ta, tb = MeshBVH(case.noise_vs, case.faces), MeshBVH(case.gt_vs, case.faces)
    assert tb.F == 1003520
    n = 4 << 20
    rep = surface_distance(ta, tb, n, seed=0)
    for key in ("a_to_b", "b_to_a", "normal_a_to_b", "normal_b_to_a"):
        assert rep[key]["n"] == n and math.isfinite(rep[key]["max"])
    assert rep["hausdorff"] > 0 and rep["normal_mean"] > 0
    # stratification on the device: |count_f - n q_f / Q| < 2 for every face
    pb, fb = tb.sample_surface(n, 0, 1)
    P = tb._prefix
    q = torch.diff(P, prepend=torch.zeros(1, dtype=P.dtype, device=P.device))
    count = torch.bincount(fb.long(), minlength=tb.F)
    assert ((count.double() - n * q.double() / float(P[-1])).abs() < 2).all()
    assert (count[q == 0] == 0).all() and (torch.diff(fb) >= 0).all()
    idx = torch.from_numpy(np.random.default_rng(0).choice(n, 4096, replace=False)).to(pb.device)
    d, f = ta.query(pb[idx])
    de, fe = ta._query_exhaustive(pb[idx])
    assert torch.equal(d, de) and torch.equal(f, fe)
