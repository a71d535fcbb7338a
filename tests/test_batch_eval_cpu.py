"""CPU checks of the batched evaluation: the descriptor layouts of dual_dmp_b200.distance against the header's
#defines, the block tables, and fit_many's snapshot writer (byte-identical files, errors re-raised)."""
import importlib.util
import os
import re

import numpy as np
import pytest

from dual_dmp_b200 import distance, synth
from dual_dmp_b200.util.mesh import Mesh

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _defines():
    text = open(os.path.join(ROOT, "include", "ddmp_b200.h")).read()
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+(DDMP_\w+)\s+(\d+)\s", text)}


def _fit_many():
    spec = importlib.util.spec_from_file_location("fit_many", os.path.join(ROOT, "scripts", "fit_many.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_descriptor_layouts_match_header():
    d = _defines()
    assert distance.THREADS == d["DDMP_DISTANCE_THREADS"]
    assert distance.MAX_BLOCKS == d["DDMP_DISTANCE_MAX_BLOCKS"]
    assert distance.EVAL_WORDS == d["DDMP_EVAL_DESC_WORDS"]
    assert distance.REFIT_WORDS == d["DDMP_BVH_REFIT_DESC_WORDS"]
    assert distance.QUERY_WORDS == d["DDMP_DISTANCE_DESC_WORDS"]
    assert distance.STATS_WORDS == d["DDMP_DISTANCE_STATS_DESC_WORDS"]


def test_block_table_and_counts():
    t, total = distance.block_table(np.zeros((4, 6), dtype=np.int64) + 7, [3, 0, 5, 1])
    assert t[:, 0].tolist() == [0, 3, 3, 8] and t[:, 1].tolist() == [3, 0, 5, 1] and total == 9
    assert (t[:, 2:] == 7).all()
    assert distance._blocks(1, True) == 1 and distance._blocks(257, False) == 2
    assert distance._blocks(10 ** 7, True) == distance.MAX_BLOCKS
    assert distance._blocks(10 ** 7, False) == -(-10 ** 7 // 256)


def test_snapshot_writer_matches_mesh_save(tmp_path):
    base, faces = synth.icosphere(2)
    rng = np.random.default_rng(0)
    nv = len(base)
    fm = _fit_many()
    w = fm.SnapshotWriter()
    jobs = []
    for k in range(3):
        vs = (rng.standard_normal((nv, 3)) * 10 ** k).astype(np.float32)
        jobs.append((str(tmp_path / f"w{k}.obj"), vs, faces))
        m = Mesh(vs=base, faces=faces)
        m.vs = vs                    # as fit_many did: the float32 positions read back from the device
        Mesh.save(m, str(tmp_path / f"m{k}.obj"))
    w.put(None, jobs[:2])
    w.put(None, jobs[2:])
    w.close()
    for k in range(3):
        assert (tmp_path / f"w{k}.obj").read_bytes() == (tmp_path / f"m{k}.obj").read_bytes()


def test_snapshot_writer_reraises(tmp_path):
    fm = _fit_many()
    w = fm.SnapshotWriter()
    w.put(None, [(str(tmp_path / "missing" / "x.obj"), np.zeros((3, 3), np.float32), np.array([[0, 1, 2]]))])
    with pytest.raises(FileNotFoundError):
        w.close()
