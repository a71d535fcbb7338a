"""GPU checks of the batched evaluation (distance.BatchEvaluator, MeshBVH.refit, the *_multi kernels of
csrc/distance.cu): MAD against the host evaluation of the training driver, independence from the batch, distances and
statistics bit for bit those of hausdorff() / MeshBVH.query, refit against fresh trees and the exhaustive scan, no
effect on a captured MultiDualStep, and fit_many end to end."""
import copy
import glob
import importlib.util
import json
import os
import types

import numpy as np
import pytest
import torch

import dual_dmp_b200.util.loss as Loss
from dual_dmp_b200 import synth
from dual_dmp_b200._lib import lib
from dual_dmp_b200.distance import BatchEvaluator, MeshBVH, hausdorff
from dual_dmp_b200.util.mesh import Mesh
from tests.helpers import small_case

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = sorted(glob.glob(os.path.join(ROOT, "tests", "golden", "*.npz")))


def host_mad(pos32, faces, gt_fn):
    """the training driver's evaluation (main.py:117-123): numpy face normals of the float32 positions, Loss.mad"""
    o1 = types.SimpleNamespace(vs=np.asarray(pos32, dtype=np.float32), faces=np.asarray(faces))
    Mesh.compute_face_normals(o1)
    return float(Loss.mad(o1.fn, gt_fn))


def _golden(path):
    z = np.load(path)
    gt = Mesh(vs=z["vs"], faces=z["faces"])
    noisy = z["vs"] + np.random.RandomState(1).normal(0, 0.05, z["vs"].shape)
    return Mesh(vs=noisy, faces=z["faces"]), gt


def _ico(n, seed=314):
    c = synth.make_case(n, seed=seed)
    return Mesh(vs=c.noise_vs, faces=c.faces), Mesh(vs=c.gt_vs, faces=c.faces)


def _light(vs, faces):
    """a mesh for BatchEvaluator without Mesh's graph tables (large cases)"""
    fn, _ = synth.face_normals_areas(vs, faces)
    m = types.SimpleNamespace(vs=np.asarray(vs, dtype=np.float64), faces=np.asarray(faces))
    o = types.SimpleNamespace(vs=m.vs, faces=m.faces)
    Mesh.compute_face_normals(o)
    m.fn = o.fn
    return m


def _cases():
    out = [_golden(p) for p in GOLDEN]
    out.append(_ico(64))                                     # 81,920 faces
    n, g = _ico(6, seed=7)
    vs = n.vs.copy()
    f = n.faces
    vs[f[:5, 1]] = vs[f[:5, 0]]                              # zero-area faces: coincident corners
    vs[f[7, 2]] = 0.5 * (vs[f[7, 0]] + vs[f[7, 1]])          # and a collinear one
    out.append((types.SimpleNamespace(vs=vs, faces=f), g))
    return out


def _positions(meshes, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return [(torch.from_numpy(m.vs).float() + 0.01 * torch.randn(m.vs.shape, generator=g)).to(DEV).contiguous()
            for m in meshes]


def test_mad_matches_host_evaluation():
    cases = _cases()
    ev = BatchEvaluator([m for m, _ in cases], [g for _, g in cases], DEV)
    pos = _positions([m for m, _ in cases], 0)
    pos[-1] = torch.from_numpy(cases[-1][0].vs).float().to(DEV)      # keep the degenerate faces degenerate
    got = ev.evaluate(pos)["mad"].tolist()
    for i, (m, g) in enumerate(cases):
        ref = host_mad(pos[i].cpu().numpy(), m.faces, g.fn)
        assert abs(got[i] - ref) <= 1e-12 * abs(ref), (i, got[i], ref)


def _mixed():
    tri = types.SimpleNamespace(vs=np.array([[0., 0, 0], [1, 0, 0], [0, 1, 0]]), faces=np.array([[0, 1, 2]]))
    tri.fn = np.array([[0., 0, 1]])
    big_vs, big_f = synth.icosphere(100)                               # 200,000 faces
    gt_big = _light(big_vs, big_f)
    noisy_big = _light(big_vs + np.random.RandomState(2).normal(0, 2e-3, big_vs.shape), big_f)
    pairs = [(tri, tri), _golden(GOLDEN[-1]), (noisy_big, gt_big), _ico(10), small_case("open", 12)[::2], _ico(3)]
    return [m for m, _ in pairs], [g for _, g in pairs]


def _host(r, i):
    return {k: (r[k][i].item() if not isinstance(r[k], dict) else {q: r[k][q][i].item() for q in r[k]}) for k in r}


def test_independent_of_the_batch_and_equal_to_hausdorff():
    meshes, gts = _mixed()
    pos = _positions(meshes, 1)
    ev = BatchEvaluator(meshes, gts, DEV)
    n0 = lib.query("ddmp_launch_count")
    r = ev.evaluate(pos)
    launches = lib.query("ddmp_launch_count") - n0
    assert launches == 4                      # geometry + MAD, refit, distances, statistics: whatever B is
    for i, (m, g) in enumerate(zip(meshes, gts)):
        one = BatchEvaluator([m], [g], DEV)
        n0 = lib.query("ddmp_launch_count")
        r1 = one.evaluate([pos[i]])
        assert lib.query("ddmp_launch_count") - n0 == (launches if m.faces.shape[0] > 1 else launches - 1)
        a, b = _host(r, i), _host(r1, 0)
        assert a == b, (i, a, b)
        for t, t1 in zip(ev.distances[i], one.distances[0]):
            assert torch.equal(t, t1)
        ta, tb = MeshBVH(pos[i], m.faces), MeshBVH(g.vs, g.faces)
        ref = hausdorff(ta, tb)
        for side in ("a_to_b", "b_to_a"):
            for q in ("min", "max", "mean", "rms"):
                assert a[side][q] == ref[side][q], (i, side, q)
        for q in ("hausdorff", "mean", "diag", "hausdorff_rel", "mean_rel"):
            assert a[q] == ref[q], (i, q)
        d_ab, f_ab, d_ba, f_ba = ev.distances[i]
        dq, fq = tb.query(ta.vs)
        assert torch.equal(d_ab, dq) and torch.equal(f_ab, fq)
        dq, fq = ta.query(tb.vs)
        assert torch.equal(d_ba, dq) and torch.equal(f_ba, fq)


@pytest.mark.parametrize("target", ["clean", "perturbed", "collapsed"])
def test_refit_equals_fresh_build_and_exhaustive(target):
    noisy, gt = _ico(64)
    vs = {"clean": gt.vs,
          "perturbed": gt.vs + np.random.RandomState(3).normal(0, 5.0, gt.vs.shape),
          "collapsed": np.tile(gt.vs[:1], (len(gt.vs), 1))}[target]
    tree = MeshBVH(noisy.vs, noisy.faces)
    tree.refit(vs)
    fresh = MeshBVH(vs, noisy.faces)
    assert torch.equal(tree.vs, fresh.vs) and torch.equal(tree.bbox, fresh.bbox)
    pts = np.concatenate([gt.vs, noisy.vs]) + np.random.RandomState(4).normal(0, 0.5, (2 * len(gt.vs), 3))
    d, f = tree.query(pts)
    df, ff = fresh.query(pts)
    assert torch.equal(d, df) and torch.equal(f, ff)
    sub = pts[np.random.RandomState(5).choice(len(pts), 4096, replace=False)]
    d, f = tree.query(sub)
    de, fe = tree._query_exhaustive(sub)
    assert torch.equal(d, de) and torch.equal(f, fe)
    nodes = tree.nodes.clone()
    for _ in range(3):                                         # repeated refits are bitwise stable
        tree.refit(vs)
        assert torch.equal(tree.nodes, nodes)
    assert int(tree.counters.abs().sum()) == 0


def test_multi_dual_step_unaffected_and_values_match_host():
    from dual_dmp_b200.step import MultiDualStep
    from tests.test_gpu_multi_fit import _three_fits
    fits = _three_fits()
    twins = [dict(f, posnet=copy.deepcopy(f["posnet"]), normnet=copy.deepcopy(f["normnet"])) for f in fits]
    gts = [small_case("ico", 10)[2], small_case("open", 12)[2], None]
    a, b = MultiDualStep(fits, bnfloop=3), MultiDualStep(twins, bnfloop=3)
    ev = BatchEvaluator([f["n_mesh"] for f in fits[:2]], gts[:2], DEV)
    for ep in range(1, 121):
        ta, tb = a.step(ep), b.step(ep)
        _eq_all = [torch.equal(ta, tb)] + [torch.equal(x, y) for x, y in zip(a.pos + a.norm, b.pos + b.norm)]
        assert all(_eq_all), ep
        if ep % 10 == 0:
            r = ev.evaluate(a.pos[:2])
            mads = r["mad"].tolist()
            h = r["hausdorff"].tolist()
            for i in range(2):
                p = a.pos[i].cpu().numpy()
                ref = host_mad(p, fits[i]["n_mesh"].faces, gts[i].fn)
                assert abs(mads[i] - ref) <= 1e-12 * abs(ref), (ep, i)
                assert h[i] == hausdorff((p, fits[i]["n_mesh"].faces), gts[i])["hausdorff"], (ep, i)
    torch.cuda.synchronize()
    for f, t in zip(fits, twins):
        for n in ("posnet", "normnet"):
            for x, y in zip(f[n].parameters(), t[n].parameters()):
                assert torch.equal(x, y)


def _fit_many():
    spec = importlib.util.spec_from_file_location("fit_many", os.path.join(ROOT, "scripts", "fit_many.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_fit_many_end_to_end(tmp_path, capsys, monkeypatch):
    import dual_dmp_b200.step as step_mod
    seen = {}

    class Recording(step_mod.MultiDualStep):
        def step(self, epoch):
            out = super().step(epoch)
            if epoch % 100 == 0:
                seen[epoch] = [p.cpu().numpy().copy() for p in self.pos]
            return out

    monkeypatch.setattr(step_mod, "MultiDualStep", Recording)
    dirs = [synth.write_case(str(tmp_path / f"m{k}"), synth.make_case(n, seed=10 + k)) for k, n in enumerate((6, 9, 12))]
    _fit_many().main(dirs + ["--iter", "200", "--batch", "3"])
    lines = [json.loads(x) for x in capsys.readouterr().out.splitlines() if x.startswith("{")]
    assert [r["input"] for r in lines] == dirs
    for i, r in enumerate(lines):
        gt = Mesh(glob.glob(os.path.join(dirs[i], "*_gt.obj"))[0])
        pos = seen[200][i]
        ref = host_mad(pos, gt.faces, gt.fn)
        assert abs(r["final_mad"] - ref) <= 1e-12 * abs(ref), (r["final_mad"], ref)
        h = hausdorff((pos, gt.faces), gt)
        assert (r["final_hausdorff"], r["final_hausdorff_rel"], r["final_mean_rel"]) == \
            (h["hausdorff"], h["hausdorff_rel"], h["mean_rel"])
        for ep in (100, 200):
            snap = glob.glob(os.path.join(dirs[i], "output", f"{ep}_ddmp=*.obj"))
            assert len(snap) == 1
            o1 = Mesh(vs=gt.vs, faces=gt.faces)
            o1.vs = seen[ep][i]
            want = str(tmp_path / f"want{i}_{ep}.obj")
            Mesh.save(o1, want)
            assert open(snap[0], "rb").read() == open(want, "rb").read(), (i, ep)
