"""Host-side pieces of a batch of fits (no GPU): the packing of the batched loss phase into cooperative launches, the
layout of the descriptor and segment tables, the argument checks of step.MultiDualStep, and fit_many.py's dataset
discovery, sharding and arguments."""
import importlib.util
import os
import re

import numpy as np
import pytest
import torch

from dual_dmp_b200 import multi

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _fit_many():
    spec = importlib.util.spec_from_file_location("fit_many", os.path.join(ROOT, "scripts", "fit_many.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


def test_loss_blocks_follow_the_single_mesh_launch():
    assert multi.loss_blocks(642, 1280, 592) == 5
    assert multi.loss_blocks(256, 100, 592) == 1
    assert multi.loss_blocks(257, 100, 592) == 2
    assert multi.loss_blocks(100_002, 200_000, 592) == 592        # 782 wanted, capped at the grid


def test_pack_launches_order_and_capacity():
    blocks = [49, 49, 300, 200, 49, 592, 10]
    plan = multi.pack_launches(blocks, 592)
    assert plan == [(0, 3, True), (3, 5, True), (5, 6, True), (6, 7, True)]
    for start, stop, batched in plan:
        assert sum(blocks[start:stop]) <= 592
    assert [i for s, e, _ in plan for i in range(s, e)] == list(range(len(blocks)))


def test_pack_launches_single_mesh_and_exact_fit():
    assert multi.pack_launches([7], 592) == [(0, 1, True)]
    assert multi.pack_launches([296, 296, 296], 592) == [(0, 2, True), (2, 3, True)]
    assert multi.pack_launches([1] * 1000, 592) == [(0, 592, True), (592, 1000, True)]


def test_pack_launches_oversized_mesh_runs_alone_unbatched():
    # the batched kernel may hold fewer co-resident blocks than the stand-alone one
    plan = multi.pack_launches([10, 592, 20, 30], 444)
    assert plan == [(0, 1, True), (1, 2, False), (2, 4, True)]
    assert multi.pack_launches([592], 444) == [(0, 1, False)]
    with pytest.raises(ValueError):
        multi.pack_launches([0, 3], 10)


def _header_define(name):
    text = open(os.path.join(ROOT, "include", "ddmp_b200.h")).read()
    return int(re.search(r"#define\s+" + name + r"\s+(\d+)", text).group(1))


def test_table_widths_match_the_header():
    assert multi.DESC_WORDS == _header_define("DDMP_DUAL_LOSS_DESC_WORDS")
    assert multi.SEGMENT_WORDS == _header_define("DDMP_SEGMENT_WORDS")


class _T:
    def __init__(self, p):
        self.p = p

    def data_ptr(self):
        return self.p


def test_loss_descriptor_layout():
    topo = type("Topo", (), {})()
    for i, name in enumerate(["faces", "f2f", "rslot", "lap_rowptr", "lap_col", "corner_ptr", "corner_slot"]):
        setattr(topo, name, _T(0x5000 + 16 * i))
    topo.V, topo.F = 642, 1280
    row = multi.loss_descriptor(_T(0x1000), _T(0x2000), _T(0x3000), _T(0x4000), topo, _T(0x6000), _T(0x7000),
                                _T(0x8000), _T(0x9000), (3.0, 4.0, 4.0, 10.0, 1.0))
    assert row.dtype == np.int64 and row.shape == (22,)
    assert list(row[:4]) == [0x1000, 0x2000, 0x3000, 0x4000]
    assert list(row[4:11]) == [0x5000 + 16 * i for i in range(7)]
    assert list(row[11:15]) == [0x6000, 0x7000, 0x8000, 0x9000]
    assert (row[15], row[16]) == (642, 1280)
    k = (row[17:22] & 0xFFFFFFFF).astype(np.uint32).view(np.float32)
    assert list(k) == [3.0, 4.0, 4.0, 10.0, 1.0] and (row[17:22] >> 32 == 0).all()


def test_segment_table_layout():
    t = multi.segment_table([5, 7, 300], [False, True, True], [0.01, 0.02, 0.5], [0.0, 0.8, 1e-3])
    assert t.shape == (3, 5) and t.dtype == np.int64
    assert multi.segment_offsets([5, 7, 300]) == ([0, 128, 256], 640)       # 512-byte aligned starts
    assert list(t[:, 0]) == [0, 128, 256] and list(t[:, 1]) == [5, 7, 300] and list(t[:, 2]) == [0, 1, 1]
    assert list(t[:, 3].astype(np.uint32).view(np.float32)) == list(np.float32([0.01, 0.02, 0.5]))
    assert list(t[:, 4].astype(np.uint32).view(np.float32)) == list(np.float32([0.0, 0.8, 1e-3]))


class _Net:
    def __init__(self, device):
        self.device = device


def _fits(devices, loops=(None, None)):
    out = []
    for d, lp in zip(devices, loops):
        f = dict(posnet=_Net(d), normnet=_Net(d), dataset=None, n_mesh=None)
        if lp is not None:
            f["bnfloop"] = lp
        out.append(f)
    return out


def test_multi_step_rejections():
    from dual_dmp_b200.step import MultiDualStep
    with pytest.raises(ValueError, match="bnfloop"):
        MultiDualStep(_fits(["cuda:0", "cuda:0"], (1, 5)))
    with pytest.raises(ValueError, match="bnfloop"):
        MultiDualStep(_fits(["cuda:0", "cuda:0"], (None, 5)), bnfloop=1)
    with pytest.raises(RuntimeError, match="CUDA only"):
        MultiDualStep(_fits(["cpu", "cpu"]))
    with pytest.raises(ValueError, match="several devices"):
        MultiDualStep(_fits([torch.device("cuda:0"), torch.device("cuda:1")]))
    with pytest.raises(ValueError, match="no fits"):
        MultiDualStep([])


def _dataset(path, name, gt=True):
    os.makedirs(path, exist_ok=True)
    for kind in ["noise", "smooth"] + (["gt"] if gt else []):
        open(os.path.join(path, f"{name}_{kind}.obj"), "w").close()


def test_fit_many_discovery(tmp_path):
    fm = _fit_many()
    _dataset(tmp_path / "b", "b")
    _dataset(tmp_path / "a", "a", gt=False)
    (tmp_path / "not_a_dataset").mkdir()
    _dataset(tmp_path / "single", "s")
    got = fm.discover([str(tmp_path / "single"), str(tmp_path)])
    assert got == [str(tmp_path / "single"), str(tmp_path / "a"), str(tmp_path / "b"), str(tmp_path / "single")]
    with pytest.raises(SystemExit):
        fm.discover([str(tmp_path / "not_a_dataset")])
    with pytest.raises(SystemExit):
        fm.discover([str(tmp_path / "missing")])


def test_fit_many_sharding_and_chunks():
    from dual_dmp_b200 import dist
    fm = _fit_many()
    dirs = [f"d{i}" for i in range(64)]
    shards = [[dirs[i] for i in dist.shard_items(len(dirs), r, 8)] for r in range(8)]
    assert sorted(sum(shards, [])) == sorted(dirs) and all(len(s) == 8 for s in shards)
    assert [len(c) for c in fm.chunks(shards[0], 3)] == [3, 3, 2]
    assert fm.chunks(["x"], 8) == [["x"]]


def test_fit_many_arguments():
    fm = _fit_many()
    a = fm.parse_args(["d1", "d2", "--iter", "200", "--k4", "10", "--bnfloop", "5", "--grad_crip", "0.5",
                       "--batch", "4", "--pos_lr", "0.02", "--norm_lr", "0.03"])
    assert a.inputs == ["d1", "d2"] and a.iter == 200 and a.k4 == 10.0 and a.bnfloop == 5 and a.grad_crip == 0.5
    assert a.batch == 4 and a.pos_lr == 0.02 and a.norm_lr == 0.03 and (a.k1, a.k2, a.k3, a.k5) == (3, 4, 4, 1)
    assert fm.parse_args(["d"]).batch == 8
    for bad in (["d", "--batch", "0"], ["d", "--iter", "0"], ["d", "--bnfloop", "-1"], []):
        with pytest.raises(SystemExit):
            fm.parse_args(bad)
    assert "15 GB per 1M faces" in fm.BATCH_HELP          # the help text says what bounds --batch
