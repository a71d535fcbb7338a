"""The reference drivers (reference main.py:39-149, main4real.py:33-85) executed over the drop-in ``util`` package
(dual_dmp_b200/dropin), on an OBJ dataset directory written to disk.

The upstream driver scripts are not part of this repository.  ``tests/drivers/`` holds restatements of them that make
the same calls through the same ``util`` modules, and the tests run those.  Where ``__graft_entry__.build()`` has
staged the UNMODIFIED upstream scripts into the git-ignored ``baseline/_ref/`` (only ``main.py`` / ``main4real.py``,
none of the reference's ``util/``), the tests run the staged scripts instead.  ``viser`` (the web viewer main.py
starts unconditionally) is replaced by tests/stubs/viser.

Exercises in situ what no other test does: ``create_dataset(dir)`` (OBJ ingest of three files), ``PosNet(device)
.to(device)`` / ``NormalNet`` over ``torch.optim.Adam``, the five ``Loss.*`` calls with numpy float64 targets,
``clip_grad_norm_``, ``Mesh.compute_face_normals(o1_mesh)`` / ``Mesh.compute_vert_normals(o1_mesh)`` /
``Mesh.save(o1_mesh, path)`` called through the class, numpy ``Loss.mad``.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "baseline", "_ref")             # unmodified upstream drivers, when build() staged them
STORED = os.path.join(ROOT, "tests", "drivers")           # restatements kept in the repository

RUNNER = (
    "import runpy, sys\n"
    "sys.argv = sys.argv[1:]\n"            # argv[1] = driver path, rest = its flags
    "runpy.run_path(sys.argv[0], run_name='__main__')\n"
)


def _run_driver(script, workdir, flags, timeout=600):
    path = os.path.join(REF, script)
    if not os.path.exists(path):
        path = os.path.join(STORED, script)
    env = dict(os.environ)
    env["PYTHONPATH"] = os.pathsep.join(
        [os.path.join(ROOT, "dual_dmp_b200", "dropin"), ROOT, os.path.join(ROOT, "tests", "stubs")])
    # -c (not the script path) keeps the driver's own directory off sys.path[0]; `import util.*` must resolve to the
    # drop-in package
    r = subprocess.run([sys.executable, "-c", RUNNER, path, *flags], cwd=workdir, env=env, capture_output=True,
                       text=True, timeout=timeout)
    assert r.returncode == 0, r.stdout[-2000:] + "\n" + r.stderr[-4000:]
    return r.stdout, r.stderr


def _dataset(tmp_path, n=6, name="ico"):
    from dual_dmp_b200 import synth
    synth.write_case(str(tmp_path / "datasets" / name), synth.make_case(n))
    return os.path.join("datasets", name)


def test_staged_drivers_are_the_reference_files():
    """the stored drivers reach the product only through the ``util`` drop-in modules, as the upstream drivers do; when
    an upstream checkout is visible the staged copies must be byte-identical to it"""
    import ast
    for f in ("main.py", "main4real.py"):
        tree = ast.parse(open(os.path.join(STORED, f)).read())
        mods = {a.name for n in ast.walk(tree) if isinstance(n, ast.Import) for a in n.names}
        mods |= {n.module for n in ast.walk(tree) if isinstance(n, ast.ImportFrom)}
        assert not {m for m in mods if m.split(".")[0] in ("dual_dmp_b200", "oracle", "tests")}, (f, mods)
        assert {"util.datamaker", "util.loss", "util.mesh", "util.networks"} <= mods, (f, mods)
    src = "/root/reference"
    if not os.path.isdir(src) or not os.path.isdir(REF):
        return
    for f in ("main.py", "main4real.py"):
        assert open(os.path.join(src, f), "rb").read() == open(os.path.join(REF, f), "rb").read()
    assert not os.path.exists(os.path.join(REF, "util")), "only the two driver scripts are staged"


@pytest.mark.gpu
def test_reference_main_py_runs_over_the_dropin(tmp_path):
    inp = _dataset(tmp_path)
    out, err = _run_driver("main.py", str(tmp_path), ["-i", inp, "--iter", "100", "--port", "0"])
    m0 = re.search(r"initial_mad: ([0-9.]+)", out)
    m1 = re.search(r"final_mad: ([0-9.]+)", out)
    assert m0 and m1, out[-2000:]
    init_mad, final_mad = float(m0.group(1)), float(m1.group(1))
    assert np.isfinite(final_mad) and 0.0 < final_mad < init_mad, (init_mad, final_mad)
    # epoch 100 writes datasets/<name>/output/100_ddmp=<mad>.obj through Mesh.save (reference main.py:125-127)
    outdir = tmp_path / "datasets" / "ico" / "output"
    objs = sorted(os.listdir(outdir))
    assert objs == ["100_ddmp={:.3f}.obj".format(final_mad)], objs
    from dual_dmp_b200.util.mesh import Mesh
    m = Mesh(str(outdir / objs[0]))
    ref = Mesh(str(tmp_path / "datasets" / "ico" / "ico_gt.obj"))
    assert m.faces.shape == ref.faces.shape and np.array_equal(m.faces, ref.faces)
    assert np.isfinite(m.vs).all() and np.abs(m.vs - ref.vs).max() < 1.0      # denoised sphere, mean edge length 1


@pytest.mark.gpu
def test_reference_main4real_py_runs_over_the_dropin(tmp_path):
    inp = _dataset(tmp_path, name="scan")
    os.remove(tmp_path / "datasets" / "scan" / "scan_gt.obj")        # real scans have no ground truth (:33-41)
    _run_driver("main4real.py", str(tmp_path), ["-i", inp, "--iter", "20"])
    objs = sorted(os.listdir(tmp_path / "datasets" / "scan" / "output"))
    assert objs == ["10_ddmp.obj", "20_ddmp.obj"], objs              # every 10 epochs (main4real.py:80-83)
