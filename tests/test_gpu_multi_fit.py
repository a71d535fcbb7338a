"""A batch of fits on one GPU (step.MultiDualStep and its batched kernels) against separate single-mesh runs, bit for
bit: the batched loss phase against ddmp_dual_loss per mesh, the batched optimizer against FusedAdam per network, and
whole iterations against DualStep, captured and eager, across the epoch-100 BNF switch."""
import copy

import numpy as np
import pytest
import torch

from dual_dmp_b200.util.mesh import Mesh
from tests import long_rows
from tests.helpers import small_case

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CAD_K = (3.0, 4.0, 4.0, 10.0, 1.0)


def _hub_case():
    vs, faces = long_rows.make_mesh("fan", 48, 3)            # open disc, centre vertex of valence 48
    noisy = vs + np.random.RandomState(5).normal(0, 0.05, size=vs.shape)
    return Mesh(vs=noisy, faces=faces), Mesh(vs=vs, faces=faces)


def _fit(n_mesh, s_mesh, seed, **kw):
    from dual_dmp_b200.util.datamaker import dataset_from_meshes
    from dual_dmp_b200.util.networks import NormalNet, PosNet
    torch.manual_seed(seed)
    posnet, normnet = PosNet(DEV).to(DEV), NormalNet(DEV).to(DEV)
    return dict(posnet=posnet, normnet=normnet, dataset=dataset_from_meshes(n_mesh, s_mesh), n_mesh=n_mesh, **kw)


def _three_fits():
    ico_n, ico_s, _ = small_case("ico", 10)
    open_n, open_s, _ = small_case("open", 12)
    hub_n, hub_s = _hub_case()
    return [_fit(ico_n, ico_s, 1), _fit(open_n, open_s, 2, k=CAD_K, norm_lr=0.02),
            _fit(hub_n, hub_s, 3, k=CAD_K, pos_lr=0.005, grad_clip=0.5)]


def _single(f, bnfloop, capture):
    from dual_dmp_b200.step import DualStep
    return DualStep(f["posnet"], f["normnet"], f["dataset"], f["n_mesh"], k=f.get("k", (3.0, 4.0, 4.0, 4.0, 1.0)),
                    bnfloop=bnfloop, pos_lr=f.get("pos_lr", 0.01), norm_lr=f.get("norm_lr", 0.01),
                    grad_clip=f.get("grad_clip", 0.8), capture=capture)


def _eq(a, b, what):
    assert a.shape == b.shape and torch.equal(a, b), what


def _check_batch_equals_separate(fits, bnfloop, capture, epochs):
    from dual_dmp_b200.step import MultiDualStep
    twins = [dict(f, posnet=copy.deepcopy(f["posnet"]), normnet=copy.deepcopy(f["normnet"])) for f in fits]
    multi = MultiDualStep(fits, bnfloop=bnfloop, capture=capture)
    got = []
    for ep in epochs:
        tot = multi.step(ep)
        got.append((tot.clone(), multi.parts.clone(), [p.clone() for p in multi.pos], [n.clone() for n in multi.norm]))
    torch.cuda.synchronize()
    if capture:
        assert len(multi._graphs) == 2
    for i, f in enumerate(twins):                     # one fit at a time, all epochs (graph_for's cache holds 64)
        single = _single(f, bnfloop, capture)
        for ep, (tot, parts, pos, nrm) in zip(epochs, got):
            t = single.step(ep)
            _eq(tot[i], t, f"total fit {i} epoch {ep}")
            _eq(parts[i], single.parts, f"parts fit {i} epoch {ep}")
            _eq(pos[i], single.pos, f"pos fit {i} epoch {ep}")
            _eq(nrm[i], single.norm, f"norm fit {i} epoch {ep}")
        torch.cuda.synchronize()
        for j, (net, twin, opt) in enumerate(((fits[i]["posnet"], f["posnet"], single.opt_pos),
                                              (fits[i]["normnet"], f["normnet"], single.opt_norm))):
            for (name, a), (_, b) in zip(net.state_dict().items(), twin.state_dict().items()):
                _eq(a, b, f"fit {i} net {j} {name}")              # parameters and BatchNorm running statistics
            seg = multi.opt.segment(2 * i + j)
            _eq(multi.opt.exp_avg[seg], opt.exp_avg, f"fit {i} net {j} exp_avg")
            _eq(multi.opt.exp_avg_sq[seg], opt.exp_avg_sq, f"fit {i} net {j} exp_avg_sq")
            _eq(multi.opt.step_count, opt.step_count, f"fit {i} net {j} step count")


@pytest.mark.parametrize("capture", [True, False])
def test_batch_equals_separate_fits(capture):
    _check_batch_equals_separate(_three_fits(), 2, capture, [97, 98, 99, 100, 101, 102])


def test_batch_of_one_equals_dual_step():
    _check_batch_equals_separate(_three_fits()[:1], 1, True, [97, 98, 99, 100, 101, 102])


def test_more_than_32_fits_captured():
    """40 fits = 80 network graphs, more than graph_for's cache keeps: the batch keeps its own reachable"""
    fits = []
    for s in range(40):
        n_mesh, s_mesh, _ = small_case("ico", 2 + s % 3, seed=100 + s)
        fits.append(_fit(n_mesh, s_mesh, 10 + s))
    _check_batch_equals_separate(fits, 1, True, [97, 98, 99, 100, 101, 102])


def _random_inputs(n_mesh, seed):
    g = torch.Generator().manual_seed(seed)
    V, F = len(n_mesh.vs), len(n_mesh.faces)
    pos = (torch.from_numpy(n_mesh.vs).float() + 0.05 * torch.randn(V, 3, generator=g)).to(DEV)
    nrm = torch.nn.functional.normalize(torch.from_numpy(n_mesh.fn).float() + 0.2 * torch.randn(F, 3, generator=g),
                                        dim=1).to(DEV)
    return pos, nrm


@pytest.mark.parametrize("sizes", [(10, 3, 25), (100, 100, 100)])
@pytest.mark.parametrize("loop", [0, 1, 5])
def test_dual_loss_multi_equals_per_mesh(sizes, loop):
    """every mesh equals its own ddmp_dual_loss; three 200K-face meshes need one cooperative launch each"""
    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200._lib import lib
    from dual_dmp_b200.graph import topology_for
    from dual_dmp_b200.multi import DeviceTables, DualLossMulti, loss_blocks, pack_launches
    meshes = [small_case("ico", n, seed=7 + i)[0] for i, n in enumerate(sizes)]
    if sizes == (10, 3, 25):
        meshes.append(small_case("open", 9)[0])
        meshes.append(_hub_case()[0])
    ks = [(3.0, 4.0, 4.0, 4.0, 1.0) if i % 2 == 0 else CAD_K for i in range(len(meshes))]
    topos = [topology_for(m, DEV) for m in meshes]
    tv = [torch.from_numpy(m.vs).to(DEV) for m in meshes]
    tf = [torch.from_numpy(m.fn).to(DEV) for m in meshes]
    ins = [_random_inputs(m, i) for i, m in enumerate(meshes)]
    poss = [p.requires_grad_() for p, _ in ins]
    nrms = [n.requires_grad_() for _, n in ins]
    plan = pack_launches([loss_blocks(t.V, t.F, lib.query("ddmp_dual_loss_grid", 0)) for t in topos],
                         lib.query("ddmp_dual_loss_grid", 1))
    if sizes == (100, 100, 100):
        assert len(plan) == 3, plan
    tot, parts = DualLossMulti.apply(DeviceTables(DEV), topos, tv, tf, ks, loop, 1.0, *poss, *nrms)
    tot.sum().backward()
    for i in range(len(meshes)):
        p1 = poss[i].detach().clone().requires_grad_()
        n1 = nrms[i].detach().clone().requires_grad_()
        t1, parts1 = F_.DualLoss.apply(p1, n1, tv[i], tf[i], topos[i], ks[i], loop, 1.0)
        t1.backward()
        _eq(tot[i], t1, f"total {i}")
        _eq(parts[i], parts1, f"parts {i}")
        _eq(poss[i].grad, p1.grad, f"gpos {i}")
        _eq(nrms[i].grad, n1.grad, f"gnrm {i}")


class _Params(torch.nn.Module):
    def __init__(self, sizes, seed):
        super().__init__()
        g = torch.Generator().manual_seed(seed)
        self.ps = torch.nn.ParameterList([torch.nn.Parameter(torch.randn(n, generator=g).to(DEV)) for n in sizes])


def test_group_adam_equals_fused_adam():
    """segments of 7 to 400,000 elements (more than the 4*148*256-element grid cap), with and without clipping"""
    from dual_dmp_b200.multi import DeviceTables
    from dual_dmp_b200.step import FusedAdam, GroupFusedAdam
    layouts = [[7, 300], [400_000, 5, 1000], [151_553], [3, 3, 3], [70_000, 90_000]]
    lrs = [0.01, 0.02, 0.005, 0.1, 0.01]
    clips = [None, 0.8, 0.5, None, 1e-3]
    mods = [_Params(sz, i) for i, sz in enumerate(layouts)]
    twins = [copy.deepcopy(m) for m in mods]
    group = GroupFusedAdam(mods, lrs, clips)
    singles = [FusedAdam(m, lr=lr, max_norm=c) for m, lr, c in zip(twins, lrs, clips)]
    tables = DeviceTables(DEV)
    g = torch.Generator().manual_seed(0)
    for step in range(4):
        for m, t in zip(mods, twins):
            for p, q in zip(m.parameters(), t.parameters()):
                grad = (torch.randn(p.shape, generator=g) * 10.0 ** (step - 1)).to(DEV)
                p.grad, q.grad = grad.clone(), grad.clone()
        group.step(tables)
        for s in singles:
            s.step()
    torch.cuda.synchronize()
    for i, s in enumerate(singles):
        seg = group.segment(i)
        _eq(group.flat[seg], s.flat, f"params {i}")
        _eq(group.exp_avg[seg], s.exp_avg, f"exp_avg {i}")
        _eq(group.exp_avg_sq[seg], s.exp_avg_sq, f"exp_avg_sq {i}")
        _eq(group.step_count, s.step_count, f"step count {i}")
        if clips[i] is not None:
            _eq(group.norms[i], s.norm, f"norm {i}")
    for m, t in zip(mods, twins):
        for p, q in zip(m.parameters(), t.parameters()):
            _eq(p, q, "parameter views")


def test_rejects_cpu_tensors_in_the_loss():
    from dual_dmp_b200.graph import topology_for
    from dual_dmp_b200.multi import DeviceTables, DualLossMulti
    m = small_case("ico", 3)[0]
    topo = topology_for(m, DEV)
    pos, nrm = _random_inputs(m, 0)
    with pytest.raises(RuntimeError, match="CUDA"):
        DualLossMulti.apply(DeviceTables(DEV), [topo], [torch.from_numpy(m.vs)], [torch.from_numpy(m.fn).to(DEV)],
                            [CAD_K], 1, 1.0, pos, nrm)
