"""Kernel-level parity (through the C ABI) against the CPU oracle / plain torch fp32-fp64 evaluations."""
import numpy as np
import pytest
import torch

from tests.helpers import rel_err, report, small_case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def graphs():
    from dual_dmp_b200.graph import GcnGraph
    from oracle.step_ref import make_dataset
    out = {}
    for kind, n in (("ico", 10), ("open", 9)):
        n_mesh, s_mesh, _ = small_case(kind, n)
        ds = make_dataset(n_mesh, s_mesh)
        V, F = len(n_mesh.vs), len(n_mesh.faces)
        out[kind] = dict(
            mesh=n_mesh, ds=ds,
            vg=GcnGraph(ds.edge_index, V, DEV, coords=ds.x_pos, reorder=True),
            vg_id=GcnGraph(ds.edge_index, V, DEV, reorder=False),
            fg=GcnGraph(ds.face_index, F, DEV, coords=ds.z2.detach()[:, :3], reorder=True),
            fg_id=GcnGraph(ds.face_index, F, DEV, reorder=False))
    return out


def lib_rows_per_block(C):
    from dual_dmp_b200._lib import lib
    return int(lib.query("ddmp_rows_per_block", C))


def _ref_aggregate(edge_index, n, H):
    from oracle.gcn_ref import gcn_norm_ref
    idx, w = gcn_norm_ref(edge_index, n, torch.float64)
    out = torch.zeros(n, H.shape[1], dtype=torch.float64)
    return out.index_add_(0, idx[1], w.view(-1, 1) * H.double().index_select(0, idx[0]))


@pytest.mark.parametrize("kind", ["ico", "open"])
def test_graph_is_bit_exact_and_weights_match(graphs, kind):
    from oracle.gcn_ref import gcn_norm_ref
    g = graphs[kind]
    for graph, ei in ((g["vg"], g["ds"].edge_index), (g["fg"], g["ds"].face_index), (g["vg_id"], g["ds"].edge_index)):
        idx, w = gcn_norm_ref(ei, graph.n)
        ref = idx.numpy()
        ref = ref[:, np.lexsort((ref[1], ref[0]))]
        assert np.array_equal(graph.to_edge_list(), ref)          # integer part: bit-exact
        assert graph.symmetric
        # weights: compare per (src, dst) pair
        rowptr = graph.rowptr.cpu().numpy().astype(np.int64)
        dst = np.repeat(np.arange(graph.n), np.diff(rowptr))
        p = graph.perm_host
        key = p[graph.col.cpu().numpy()] * graph.n + p[dst]
        wmap = dict(zip(key.tolist(), graph.w.cpu().numpy().tolist()))
        kref = (idx[0] * graph.n + idx[1]).numpy()
        got = np.array([wmap[k] for k in kref.tolist()], dtype=np.float32)
        assert np.abs(got - w.numpy()).max() <= 2.4e-7 * np.abs(w.numpy()).max()
        perm = np.sort(p)
        assert np.array_equal(perm, np.arange(graph.n))


@pytest.mark.parametrize("C", [32, 64, 128, 256, 512, 384, 12, 3])
@pytest.mark.parametrize("which", ["vg_id", "fg_id"])
def test_spmm_matches_oracle(graphs, C, which):
    from dual_dmp_b200 import functional as F_
    g = graphs["open"]
    graph = g[which]
    ei = g["ds"].edge_index if which.startswith("v") else g["ds"].face_index
    torch.manual_seed(C)
    H = torch.randn(graph.n, C)
    bias = torch.randn(C)
    ref = _ref_aggregate(ei, graph.n, H) + bias.double()
    Hd, bd = H.to(DEV), bias.to(DEV)
    if C in (32, 64, 128, 256, 512):
        Y, partials = F_.spmm_gcn(graph, Hd, bias=bd, stats=True)
        # partials: per row block (sum, M2 about the block mean); sum of squares = sum_b (M2_b + sum_b^2 / n_b)
        pb = partials.double().cpu()
        rpb = lib_rows_per_block(C)
        n_b = torch.full((pb.shape[0], 1), float(rpb), dtype=torch.float64)
        n_b[-1] = graph.n - (pb.shape[0] - 1) * rpb
        assert rel_err(pb[:, 0].sum(dim=0), ref.sum(dim=0)) < 1e-5
        assert rel_err((pb[:, 1] + pb[:, 0] ** 2 / n_b).sum(dim=0), (ref * ref).sum(dim=0)) < 1e-5
        Y2, partials2 = F_.spmm_gcn(graph, Hd, bias=bd, stats=True)
        assert torch.equal(Y, Y2) and torch.equal(partials, partials2)          # deterministic
        Y3 = F_.spmm_gcn(graph, Hd)
        assert rel_err(Y3, ref - bias.double()) < 2e-6
    else:
        Y = F_.spmm_gcn(graph, Hd, bias=bd)
    e = rel_err(Y, ref)
    report(f"spmm C={C} {which}", e)
    assert e < 2e-6


def test_spmm_reordered_graph_equals_permuted_reference(graphs):
    from dual_dmp_b200 import functional as F_
    g = graphs["ico"]
    graph, ei = g["fg"], g["ds"].face_index
    H = torch.randn(graph.n, 64)
    ref = _ref_aggregate(ei, graph.n, H)
    p = torch.from_numpy(graph.perm_host)
    Y = F_.spmm_gcn(graph, H[p].contiguous().to(DEV))          # rows in Morton order
    assert rel_err(Y.cpu(), ref[p]) < 2e-6


SHAPES = [(7, 32), (16, 32), (32, 64), (64, 128), (128, 256), (256, 512), (512, 256), (64, 32), (32, 16), (20, 12), (16, 4)]


@pytest.mark.parametrize("cin,cout", SHAPES)
@pytest.mark.parametrize("n", [1000, 4099])
def test_gemm_ffma(cin, cout, n):
    from dual_dmp_b200 import functional as F_
    torch.manual_seed(cin * 1000 + cout)
    X = torch.randn(n + 5, cin)
    W = torch.randn(cout, cin) / cin ** 0.5
    scale, shift = torch.rand(cin) + 0.5, torch.randn(cin)
    rmap = torch.randperm(n + 5)[:n].to(torch.int32)
    dH = torch.randn(n, cout)
    Xd, Wd, dHd = X.to(DEV), W.to(DEV), dH.to(DEV)
    sc, sh, rm = scale.to(DEV), shift.to(DEV), rmap.to(DEV)
    act = torch.nn.functional.leaky_relu(X.double() * scale.double() + shift.double(), 0.01)
    # xw: plain, with BN+LeakyReLU prologue, with row gather
    e1 = rel_err(F_.gemm_xw(Xd[:n].contiguous(), Wd, backend=1), X[:n].double() @ W.double().t())
    e2 = rel_err(F_.gemm_xw(Xd[:n].contiguous(), Wd, scale=sc, shift=sh, backend=1), act[:n] @ W.double().t())
    e3 = rel_err(F_.gemm_xw(Xd, Wd, row_map=rm, n=n, backend=1), X[rmap.long()].double() @ W.double().t())
    # dx
    e4 = rel_err(F_.gemm_dx(dHd, Wd, backend=1), dH.double() @ W.double())
    # dw: plain, prologue, gather
    e5 = rel_err(F_.gemm_dw(dHd, Xd[:n].contiguous(), cin, backend=1), dH.double().t() @ X[:n].double())
    e6 = rel_err(F_.gemm_dw(dHd, Xd[:n].contiguous(), cin, scale=sc, shift=sh, backend=1), dH.double().t() @ act[:n])
    e7 = rel_err(F_.gemm_dw(dHd, Xd, cin, row_map=rm, backend=1), dH.double().t() @ X[rmap.long()].double())
    report(f"gemm_ffma cin={cin} cout={cout} n={n}", (e1, e2, e3, e4, e5, e6, e7))
    assert max(e1, e2, e3, e4) < 5e-6, (e1, e2, e3, e4)
    assert max(e5, e6, e7) < 2e-5, (e5, e6, e7)
    a = F_.gemm_dw(dHd, Xd[:n].contiguous(), cin, backend=1)
    b = F_.gemm_dw(dHd, Xd[:n].contiguous(), cin, backend=1)
    assert torch.equal(a, b)                                                    # split-K is deterministic


@pytest.mark.parametrize("cin,cout", [(16, 32), (32, 64), (64, 32), (32, 16), (16, 4)])
def test_gemm_dw_narrow_kernel_many_splits(cin, cout):
    """dw_narrow_kernel (both widths < 64: 256-thread CTAs, split-K inside the CTA) with one partial per CTA for ~600
    CTAs and a ragged last chunk, against float64; deterministic"""
    from dual_dmp_b200 import functional as F_
    n = 200003
    torch.manual_seed(cin + cout)
    X = torch.randn(n, cin); dH = torch.randn(n, cout)
    scale, shift = torch.rand(cin) + 0.5, torch.randn(cin)
    act = torch.nn.functional.leaky_relu(X.double() * scale.double() + shift.double(), 0.01)
    Xd, dHd, sc, sh = X.to(DEV), dH.to(DEV), scale.to(DEV), shift.to(DEV)
    a = F_.gemm_dw(dHd, Xd, cin, scale=sc, shift=sh)
    e1 = rel_err(a, dH.double().t() @ act)
    e2 = rel_err(F_.gemm_dw(dHd, Xd, cin), dH.double().t() @ X.double())
    report(f"gemm_dw narrow cin={cin} cout={cout} n={n}", (e1, e2))
    assert a.shape == (cout, cin) and max(e1, e2) < 2e-5, (e1, e2)
    assert torch.equal(a, F_.gemm_dw(dHd, Xd, cin, scale=sc, shift=sh))


@pytest.mark.parametrize("C", [32, 64, 256, 512])
@pytest.mark.parametrize("n", [777, 5000])
def test_batchnorm_lrelu_forward_backward(C, n):
    """statistics finalize + lazy apply + backward against torch BatchNorm1d(train) -> LeakyReLU in float64"""
    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200.graph import GcnGraph
    torch.manual_seed(n + C)
    # statistics come from the SpMM epilogue: aggregate over a graph of isolated nodes (A_hat = I)
    graph = GcnGraph(torch.zeros(2, 0, dtype=torch.long), n, DEV, reorder=False)
    Y0 = (torch.randn(n, C) * (torch.rand(C) * 3 + 0.5) + torch.randn(C) * 2)
    gamma, beta = torch.rand(C) + 0.5, torch.randn(C)
    # keep every pre-activation away from the LeakyReLU kink: an element whose sign differs between float32 and
    # float64 would flip its slope (1 vs 0.01) and say nothing about the kernel
    for _ in range(3):
        z = (Y0.double() - Y0.double().mean(0)) / (Y0.double().var(0, unbiased=False) + 1e-5).sqrt() * gamma + beta
        Y0 = torch.where(z.abs() < 1e-3, Y0 + 0.05 * Y0.std(0), Y0)
    rm0, rv0 = torch.randn(C), torch.rand(C) + 0.5
    bn = torch.nn.BatchNorm1d(C).double()
    with torch.no_grad():
        bn.weight.copy_(gamma); bn.bias.copy_(beta); bn.running_mean.copy_(rm0); bn.running_var.copy_(rv0)
    yr = Y0.double().requires_grad_(True)
    xr = torch.nn.functional.leaky_relu(bn(yr), 0.01)
    gX = torch.randn(n, C)
    xr.backward(gX.double())

    Yd = Y0.to(DEV)
    Y, partials = F_.spmm_gcn(graph, Yd, stats=True)
    assert torch.equal(Y, Yd)
    rm, rv = rm0.to(DEV), rv0.to(DEV)
    st = F_.bn_stats_finalize(partials, n, gamma.to(DEV), beta.to(DEV), rm, rv)
    assert rel_err(rm, bn.running_mean) < 1e-5 and rel_err(rv, bn.running_var) < 1e-5
    x = torch.nn.functional.leaky_relu(Y * st[2] + st[3], 0.01)
    e_f = rel_err(x, xr)
    dY, dgamma, dbeta, dbias = F_.bn_lrelu_backward(gX.to(DEV), Y, st)
    e_b = (rel_err(dY, yr.grad), rel_err(dgamma, bn.weight.grad), rel_err(dbeta, bn.bias.grad))
    report(f"bn C={C} n={n}", (e_f,) + e_b)
    assert e_f < 2e-5 and max(e_b) < 5e-5, (e_f, e_b)
    assert dbias.abs().max() < 1e-3 * dY.abs().sum(dim=0).max()          # true gradient of a pre-BN bias is 0
    assert rel_err(F_.colsum(Y), Y0.double().sum(dim=0)) < 1e-5


@pytest.mark.parametrize("ratio", [0.0, 100.0, 1000.0, 1.0e4])
@pytest.mark.parametrize("C,n", [(32, 70001), (256, 33333), (512, 1001)])
def test_batchnorm_statistics_with_large_mean_over_sigma_default_and_reference(C, n, ratio):
    """the variance must not be formed as E[y^2] - E[y]^2 in float32 (SURVEY.md §7 hard part 3): the aggregation epilogue
    emits per-block (sum, M2 about the block mean) (Welford per thread, Chan merge per block) and the finalize combines
    them in float64, so the relative error of var / rstd grows like |mean|/sigma * 1e-7, not (mean/sigma)^2 * 1e-7.
    Also the partitioned-mode route (rank sums in float64 -> finalize_sums), on the default kernels and the reference
    kernel (gather kernel, shared-memory statistics)"""
    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200._lib import lib
    from dual_dmp_b200.graph import GcnGraph
    torch.manual_seed(C)
    sigma = torch.rand(C) * 2 + 0.5
    Y0 = torch.randn(n, C) * sigma + ratio * sigma * torch.where(torch.rand(C) < 0.5, -1.0, 1.0)
    graph = GcnGraph(torch.zeros(2, 0, dtype=torch.long), n, DEV, reorder=False)           # A_hat = I
    Yd = Y0.to(DEV)
    ref_mean = Yd.double().mean(0)
    ref_var = Yd.double().var(0, unbiased=False)
    gamma, beta = torch.ones(C, device=DEV), torch.zeros(C, device=DEV)
    tol = 2e-6 + 4e-7 * ratio
    prev = lib.query("ddmp_spmm_reference_kernel", 0)
    try:
        for ref in (0, 1):
            lib.query("ddmp_spmm_reference_kernel", ref)
            _, partials = F_.spmm_gcn(graph, Yd, stats=True)
            st = F_.bn_stats_finalize(partials, n, gamma, beta)
            e_mean = float((st[0].double() - ref_mean).abs().max() / ref_mean.abs().max().clamp_min(1.0))
            e_rstd = rel_err(st[1], torch.rsqrt(ref_var + 1e-5))
            st2 = F_.bn_stats_finalize_sums(F_.bn_rank_sums(partials, n), n, gamma, beta)
            report(f"bn stats |mean|/sigma={ratio:g} C={C} n={n} reference kernel {ref}", (e_mean, e_rstd))
            assert e_mean < 2e-7 and e_rstd < tol, (ref, e_mean, e_rstd, tol)
            assert torch.equal(st, st2)
    finally:
        lib.query("ddmp_spmm_reference_kernel", prev)


@pytest.mark.parametrize("cin,cout", [(64, 128), (128, 256), (256, 256), (512, 512), (512, 256), (256, 64), (128, 64)])
@pytest.mark.parametrize("n", [37, 640, 4099, 77777])
def test_gemm_f16_split_tma_epilogue_equals_staged_epilogue(cin, cout, n):
    """The fp16-split NT kernels write their result with TMA tensor stores (32 x 32 boxes out of a 128-byte-swizzled
    staging buffer, rows past n clipped by the unit); the staged ld.shared + st.global epilogue stays behind
    ddmp_gemm_tc_flags(16).  Same accumulators, same power-of-two unscale: the two must be IDENTICAL -- row counts below
    one box, not a multiple of 32, and many tiles per CTA; no write may land past row n."""
    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200._lib import lib
    torch.manual_seed(cin + cout + n)
    X = (torch.randn(n, cin) * (torch.rand(1, cin) * 3 + 0.1)).to(DEV)
    W = (torch.randn(cout, cin) / cin ** 0.5).to(DEV)
    W[1] *= 1e-5
    sc, sh = (torch.rand(cin) + 0.5).to(DEV), torch.randn(cin).to(DEV)
    dH = (torch.randn(n, cout) * 1e-3).to(DEV)
    b_act = (torch.nn.functional.leaky_relu(X * sc + sh, 0.01).abs().amax(0) * 1.5).contiguous()
    b_dh = dH.abs().amax(0).contiguous()
    prev = lib.query("ddmp_gemm_tc_flags", -1)
    try:
        res = {}
        for fl in (16, 0):
            lib.query("ddmp_gemm_tc_flags", fl)
            # outputs are views of larger poisoned buffers: a store past row n would be seen
            Hbuf = torch.full((n + 64, cout), 7.0, device=DEV)
            Gbuf = torch.full((n + 64, cin), 7.0, device=DEV)
            F_.gemm_xw(X, W, scale=sc, shift=sh, backend=2, amax=b_act, out=Hbuf[:n])
            F_.gemm_dx(dH, W, backend=2, amax=b_dh, out=Gbuf[:n])
            assert (Hbuf[n:] == 7.0).all() and (Gbuf[n:] == 7.0).all()
            res[fl] = (Hbuf[:n].clone(), Gbuf[:n].clone())
        assert torch.equal(res[0][0], res[16][0])
        assert torch.equal(res[0][1], res[16][1])
        act = torch.nn.functional.leaky_relu(X.double() * sc.double() + sh.double(), 0.01)
        assert rel_err(res[0][0], act @ W.double().t()) < 5e-6
        assert rel_err(res[0][1], dH.double() @ W.double()) < 5e-6
        assert rel_err(res[0][0][:, 1], act @ W[1].double()) < 5e-6       # a weight row 1e-5 of its tile's maximum
    finally:
        lib.query("ddmp_gemm_tc_flags", prev)


@pytest.mark.parametrize("kind", [0, 1])
def test_heads(kind):
    from dual_dmp_b200._lib import lib, ptr, stream_ptr
    torch.manual_seed(kind)
    n = 3001
    Y12 = torch.randn(n, 32)
    scale, shift = torch.rand(32) + 0.5, torch.randn(32) * 0.3
    lin1, lin2 = torch.nn.Linear(32, 16).double(), torch.nn.Linear(16, 3).double()
    x_pos = torch.randn(n, 3)
    perm = torch.randperm(n)
    g_out = torch.randn(n, 3)
    # float64 torch reference in the caller's numbering: row i of the reordered tensors is node perm[i]
    yr = Y12.double().requires_grad_(True)
    x = torch.nn.functional.leaky_relu(yr * scale.double() + shift.double(), 0.01)
    x.retain_grad()
    h = torch.nn.functional.leaky_relu(lin1(x), 0.01)
    o = lin2(h)
    if kind == 0:
        res = x_pos.double()[perm] + o
    else:
        t = torch.tanh(o)
        res = t * torch.reciprocal(torch.norm(t, dim=1, keepdim=True).expand(-1, 3) + 1e-12)
    res.backward(g_out.double()[perm])

    d = lambda t: t.float().contiguous().to(DEV)
    out = torch.empty(n, 3, device=DEV)
    h_save = torch.empty(n, 16, device=DEV)
    t_save = torch.empty(n, 4, device=DEV)
    W1, b1, W2, b2 = d(lin1.weight.detach()), d(lin1.bias.detach()), d(lin2.weight.detach()), d(lin2.bias.detach())
    permd = perm.to(torch.int32).to(DEV)
    st = stream_ptr(torch.device(DEV))
    # keep every device tensor in a variable: a temporary freed inside the argument list would be re-used by the next
    Yd, scd, shd, xpd, god = d(Y12), d(scale), d(shift), d(x_pos), d(g_out)
    lib.call("ddmp_head_fwd", kind, ptr(Yd), ptr(scd), ptr(shd), 0.01, ptr(W1), ptr(b1), ptr(W2), ptr(b2),
             ptr(permd), ptr(xpd), ptr(out), ptr(h_save), ptr(t_save), n, st)
    ref_out = torch.empty(n, 3, dtype=torch.float64)
    ref_out[perm] = res.detach()
    e_f = rel_err(out, ref_out)
    go, gh, gX = torch.empty(n, 4, device=DEV), torch.empty(n, 16, device=DEV), torch.empty(n, 32, device=DEV)
    lib.call("ddmp_head_bwd", kind, ptr(god), ptr(permd), ptr(W1), ptr(W2), ptr(h_save), ptr(t_save), 0.01,
             ptr(go), ptr(gh), ptr(gX), n, st)
    from dual_dmp_b200 import functional as F_
    e_x = rel_err(gX, x.grad)
    gW1 = F_.gemm_dw(gh, Yd, 32, scale=scd, shift=shd)
    gW2 = F_.gemm_dw(go, h_save, 16)[:3]
    e_w = (rel_err(gW1, lin1.weight.grad), rel_err(gW2, lin2.weight.grad), rel_err(F_.colsum(gh), lin1.bias.grad),
           rel_err(F_.colsum(go)[:3], lin2.bias.grad))
    report(f"head kind={kind}", (e_f, e_x) + e_w)
    assert e_f < 5e-6 and e_x < 2e-5 and max(e_w) < 5e-5, (e_f, e_x, e_w)


def test_gcnconv_operator_level(graphs):
    """conv(x, edge_index) drop-in for torch_geometric.nn.GCNConv: forward + all three gradients vs the oracle"""
    from dual_dmp_b200.util.networks import GCNConv
    from oracle.gcn_ref import GCNConvRef
    g = graphs["open"]
    for ei, n in ((g["ds"].edge_index, g["vg"].n), (g["ds"].face_index, g["fg"].n)):
        for cin, cout in ((7, 32), (64, 128), (20, 12)):
            torch.manual_seed(cin)
            ref = GCNConvRef(cin, cout)
            with torch.no_grad():
                ref.bias.normal_()
            conv = GCNConv(cin, cout).to(DEV)
            conv.load_state_dict(ref.state_dict())
            x = torch.randn(n, cin)
            xr = x.clone().requires_grad_(True)
            xd = x.to(DEV).requires_grad_(True)
            gy = torch.randn(n, cout)
            ref(xr, ei).backward(gy)
            y = conv(xd, ei)
            y.backward(gy.to(DEV))
            errs = (rel_err(y, ref(xr, ei)), rel_err(xd.grad, xr.grad), rel_err(conv.lin.weight.grad, ref.lin.weight.grad),
                    rel_err(conv.bias.grad, ref.bias.grad))
            report(f"gcnconv {cin}->{cout} n={n}", errs)
            assert max(errs) < 1e-4, errs


def test_directed_graph_backward_uses_transpose():
    from dual_dmp_b200.util.networks import GCNConv
    from oracle.gcn_ref import GCNConvRef
    torch.manual_seed(3)
    n = 50
    ei = torch.randint(0, n, (2, 300))
    ref = GCNConvRef(8, 32)
    conv = GCNConv(8, 32).to(DEV)
    conv.load_state_dict(ref.state_dict())
    x = torch.randn(n, 8)
    xr, xd = x.clone().requires_grad_(True), x.to(DEV).requires_grad_(True)
    gy = torch.randn(n, 32)
    ref(xr, ei).backward(gy)
    conv(xd, ei).backward(gy.to(DEV))
    assert rel_err(xd.grad, xr.grad) < 1e-4 and rel_err(conv.lin.weight.grad, ref.lin.weight.grad) < 1e-4


TC_SHAPES = [(64, 64), (64, 128), (128, 256), (256, 512), (512, 512), (512, 256), (256, 64), (128, 64)]


@pytest.mark.parametrize("cin,cout", TC_SHAPES)
@pytest.mark.parametrize("n", [640, 1000, 4099, 20011])
def test_gemm_tcgen05_3xtf32(cin, cout, n):
    """tcgen05 kind::tf32 path with the hi/lo split: fp32-level accuracy against a float64 evaluation"""
    from dual_dmp_b200 import functional as F_
    torch.manual_seed(cin * 1000 + cout + n)
    X = torch.randn(n + 5, cin)
    W = torch.randn(cout, cin) / cin ** 0.5
    scale, shift = torch.rand(cin) + 0.5, torch.randn(cin)
    rmap = torch.randperm(n + 5)[:n].to(torch.int32)
    dH = torch.randn(n, cout)
    Xd, Wd, dHd = X.to(DEV), W.to(DEV), dH.to(DEV)
    sc, sh, rm = scale.to(DEV), shift.to(DEV), rmap.to(DEV)
    Xn = Xd[:n].contiguous()
    act = torch.nn.functional.leaky_relu(X.double() * scale.double() + shift.double(), 0.01)
    e1 = rel_err(F_.gemm_xw(Xn, Wd, backend=2), X[:n].double() @ W.double().t())
    e2 = rel_err(F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=2), act[:n] @ W.double().t())
    e3 = rel_err(F_.gemm_xw(Xd, Wd, row_map=rm, n=n, backend=2), X[rmap.long()].double() @ W.double().t())
    e4 = rel_err(F_.gemm_dx(dHd, Wd, backend=2), dH.double() @ W.double())
    e5 = rel_err(F_.gemm_dw(dHd, Xn, cin, backend=2), dH.double().t() @ X[:n].double())
    e6 = rel_err(F_.gemm_dw(dHd, Xn, cin, scale=sc, shift=sh, backend=2), dH.double().t() @ act[:n])
    report(f"gemm_tc cin={cin} cout={cout} n={n}", (e1, e2, e3, e4, e5, e6))
    assert max(e1, e2, e3, e4) < 1e-5, (e1, e2, e3, e4)
    assert max(e5, e6) < 2e-5, (e5, e6)
    assert torch.equal(F_.gemm_dw(dHd, Xn, cin, scale=sc, shift=sh, backend=2),
                       F_.gemm_dw(dHd, Xn, cin, scale=sc, shift=sh, backend=2))
    a = F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=2)
    b = F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=2)
    assert torch.equal(a, b)
    # and it agrees with the FFMA kernel to fp32 rounding
    assert rel_err(a, F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=1)) < 1e-5


@pytest.mark.parametrize("n", [640, 1000, 4099, 20011])
def test_gemm_tcgen05_narrow_reduction_width(n):
    """32-wide reductions on the tensor-core kernels: X.W^T of the 32 -> 64 layer and dH.W of the 64 -> 32 layer (K = 32:
    one k-block of the 3xTF32 kernel) against float64, the FFMA kernel, and through the default dispatch"""
    from dual_dmp_b200 import functional as F_
    torch.manual_seed(n)
    X = torch.randn(n, 32); W = torch.randn(64, 32) / 32 ** 0.5
    scale, shift = torch.rand(32) + 0.5, torch.randn(32)
    act = torch.nn.functional.leaky_relu(X.double() * scale.double() + shift.double(), 0.01)
    Xd, Wd, sc, sh = X.to(DEV), W.to(DEV), scale.to(DEV), shift.to(DEV)
    e1 = rel_err(F_.gemm_xw(Xd, Wd, backend=2), X.double() @ W.double().t())
    a = F_.gemm_xw(Xd, Wd, scale=sc, shift=sh, backend=2)
    e2 = rel_err(a, act @ W.double().t())
    assert torch.equal(a, F_.gemm_xw(Xd, Wd, scale=sc, shift=sh)), "default dispatch must take the tensor-core kernel"
    assert rel_err(a, F_.gemm_xw(Xd, Wd, scale=sc, shift=sh, backend=1)) < 1e-5
    # 64 -> 32 layer
    X2 = torch.randn(n, 64); W2 = torch.randn(32, 64) / 8; dH = torch.randn(n, 32)
    sc2, sh2 = torch.rand(64) + 0.5, torch.randn(64)
    act2 = torch.nn.functional.leaky_relu(X2.double() * sc2.double() + sh2.double(), 0.01)
    X2d, W2d, dHd, sc2d, sh2d = X2.to(DEV), W2.to(DEV), dH.to(DEV), sc2.to(DEV), sh2.to(DEV)
    g = F_.gemm_dx(dHd, W2d, backend=2)
    e3 = rel_err(g, dH.double() @ W2.double())
    assert torch.equal(g, F_.gemm_dx(dHd, W2d))
    d = F_.gemm_dw(dHd, X2d, 64, scale=sc2d, shift=sh2d)          # stays on the FFMA kernel (measured faster)
    e4 = rel_err(d, dH.double().t() @ act2)
    # 32-wide OUTPUTS (a 32-column UMMA tile): X.W^T of the 64 -> 32 layer (with an operand bound, as the network calls
    # it: must not take the fp16-split kernel, whose tiles are >= 64 wide) and dH.W of the 32 -> 64 layer
    bound = (act2.abs().amax(0) * 1.5).float().to(DEV)
    h = F_.gemm_xw(X2d, W2d, scale=sc2d, shift=sh2d, backend=2, amax=bound)
    e5 = rel_err(h, act2 @ W2.double().t())
    assert h.shape == (n, 32) and torch.equal(h, F_.gemm_xw(X2d, W2d, scale=sc2d, shift=sh2d, amax=bound))
    dH3 = torch.randn(n, 64); dH3d = dH3.to(DEV)
    g3 = F_.gemm_dx(dH3d, Wd, backend=2, amax=dH3d.abs().amax().reshape(1))
    e6 = rel_err(g3, dH3.double() @ W.double())
    assert g3.shape == (n, 32) and torch.equal(g3, F_.gemm_dx(dH3d, Wd))
    report(f"gemm_tc narrow n={n}", (e1, e2, e3, e4, e5, e6))
    assert max(e1, e2, e3, e5, e6) < 1e-5 and e4 < 2e-5, (e1, e2, e3, e4, e5, e6)


@pytest.mark.parametrize("cin,cout", TC_SHAPES)
@pytest.mark.parametrize("n", [640, 4099, 20011])
def test_gemm_tcgen05_f16_split(cin, cout, n):
    """tcgen05 kind::f16 path (x*s = hi + lo in fp16, three MMAs, fp32 accumulate) given an operand bound: accuracy of
    an fp32 product sum against a float64 evaluation, for O(1) activations, for tiny gradients, and with a bound that
    is 1000x pessimistic (the BatchNorm bound at 1M rows)"""
    from dual_dmp_b200 import functional as F_
    torch.manual_seed(cin * 1000 + cout + n)
    X = torch.randn(n + 5, cin) * (torch.rand(1, cin) * 3 + 0.1)
    W = torch.randn(cout, cin) / cin ** 0.5
    W[3] = 0.0                                        # an all-zero weight row
    W[5] *= 1e-6
    scale, shift = torch.rand(cin) + 0.5, torch.randn(cin)
    rmap = torch.randperm(n + 5)[:n].to(torch.int32)
    dH = torch.randn(n, cout) * 1e-7 * torch.exp(torch.randn(n, 1))
    Xd, Wd, dHd = X.to(DEV), W.to(DEV), dH.to(DEV)
    sc, sh, rm = scale.to(DEV), shift.to(DEV), rmap.to(DEV)
    Xn = Xd[:n].contiguous()
    act = torch.nn.functional.leaky_relu(X.double() * scale.double() + shift.double(), 0.01)
    b_raw = X.abs().amax(0).to(DEV)                   # per-channel bounds (any array whose max bounds the operand)
    b_act = act.abs().amax(0).float().to(DEV)
    b_dh = dH.abs().amax(1)[::7].contiguous().to(DEV) if n > 700 else dH.abs().amax().reshape(1).to(DEV)
    b_dh = torch.cat([b_dh, dH.abs().amax().reshape(1).to(DEV)])
    e1 = rel_err(F_.gemm_xw(Xn, Wd, backend=2, amax=b_raw), X[:n].double() @ W.double().t())
    e2 = rel_err(F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=2, amax=b_act), act[:n] @ W.double().t())
    e2p = rel_err(F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=2, amax=b_act * 1000.0), act[:n] @ W.double().t())
    e3 = rel_err(F_.gemm_xw(Xd, Wd, row_map=rm, n=n, backend=2, amax=b_raw), X[rmap.long()].double() @ W.double().t())
    e4 = rel_err(F_.gemm_dx(dHd, Wd, backend=2, amax=b_dh), dH.double() @ W.double())
    t2 = rel_err(F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=2), act[:n] @ W.double().t())     # 3xTF32, same job
    t4 = rel_err(F_.gemm_dx(dHd, Wd, backend=2), dH.double() @ W.double())
    e5 = rel_err(F_.gemm_dw(dHd, Xn, cin, backend=2, amax_dh=b_dh, amax_x=b_raw), dH.double().t() @ X[:n].double())
    e6 = rel_err(F_.gemm_dw(dHd, Xn, cin, scale=sc, shift=sh, backend=2, amax_dh=b_dh, amax_x=b_act * 1000.0),
                 dH.double().t() @ act[:n])
    t6 = rel_err(F_.gemm_dw(dHd, Xn, cin, scale=sc, shift=sh, backend=2), dH.double().t() @ act[:n])
    assert max(e5, e6) < 2e-5 and e6 < 1.5 * t6 + 1e-7, (e5, e6, t6)
    assert torch.equal(F_.gemm_dw(dHd, Xn, cin, scale=sc, shift=sh, backend=2, amax_dh=b_dh, amax_x=b_act),
                       F_.gemm_dw(dHd, Xn, cin, scale=sc, shift=sh, backend=2, amax_dh=b_dh, amax_x=b_act))
    report(f"gemm_tc f16 cin={cin} cout={cout} n={n}", (e1, e2, e2p, e3, e4, e5, e6, "tf32:", t2, t4, t6))
    # the error is dominated by the tensor core's truncating fp32 accumulation (grows with K, same for 3xTF32)
    assert max(e1, e2, e2p, e3, e4) < 5e-6, (e1, e2, e2p, e3, e4)
    assert e2 < 1.5 * t2 + 1e-7 and e4 < 1.5 * t4 + 1e-7, (e2, t2, e4, t4)
    a = F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=2, amax=b_act)
    assert torch.equal(a, F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=2, amax=b_act))
    assert (a[:, 3] == 0).all()
    ref5 = act[:n] @ W[5].double()
    assert rel_err(a[:, 5], ref5) < 5e-6              # a weight row 1e-6 of the others keeps full accuracy
    assert rel_err(a, F_.gemm_xw(Xn, Wd, scale=sc, shift=sh, backend=2)) < 5e-6       # vs the 3xTF32 kernel


def test_fused_clip_adam_matches_torch():
    """ddmp_grad_norm + ddmp_adam_step_dev over flat buffers == clip_grad_norm_ + torch.optim.Adam (main.py:108-110)"""
    from dual_dmp_b200.step import FusedAdam
    torch.manual_seed(0)
    shapes = [(32, 7), (32,), (512, 256), (512,), (3, 16), (3,)]
    ref = torch.nn.ParameterList([torch.nn.Parameter(torch.randn(*s, device=DEV)) for s in shapes])
    mine = torch.nn.ParameterList([torch.nn.Parameter(p.detach().clone()) for p in ref])
    opt_ref = torch.optim.Adam(ref.parameters(), lr=0.01)
    opt = FusedAdam(mine, lr=0.01, max_norm=0.8)
    for it in range(5):
        grads = [torch.randn(*s, device=DEV) * (10.0 if it % 2 == 0 else 0.01) for s in shapes]   # clipped / not
        for p, q, g in zip(ref, mine, grads):
            p.grad, q.grad = g.clone(), g.clone()
        torch.nn.utils.clip_grad_norm_(ref.parameters(), 0.8)
        opt_ref.step()
        opt.step()
        for p, q in zip(ref, mine):
            assert rel_err(q, p) < 2e-6, (it, rel_err(q, p))
    assert int(opt.step_count) == 5
    assert all(q.data_ptr() >= opt.flat.data_ptr() for q in mine)         # parameters are views of the flat buffer


@pytest.mark.parametrize("C", [32, 64, 128, 256, 512])
@pytest.mark.parametrize("kind,n", [("ico", 3), ("ico", 10), ("open", 9), ("ico", 40)])
def test_spmm_default_kernels_equal_reference_kernel_bitwise(kind, n, C):
    """the default kernels (csrc/spmm_tile.cu, TMA-staged row block + shared-memory index stream, at C <= 128) against
    the reference kernel (csrc/spmm.cu, gathers only, ddmp_spmm_reference_kernel): both accumulate every row in the same
    CSR order, so Y, the BatchNorm partial sums and max|Y| must be IDENTICAL --
    closed and open meshes, Morton-ordered and caller-ordered graphs, row counts below / not a multiple of the row
    block, and the partitioned layout (H = [owned | halo] rows, only the owned rows computed)."""
    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200._lib import lib
    from dual_dmp_b200.graph import GcnGraph
    from oracle.step_ref import make_dataset
    n_mesh, s_mesh, _ = small_case(kind, n)
    ds = make_dataset(n_mesh, s_mesh)
    V, F = len(n_mesh.vs), len(n_mesh.faces)
    graphs_ = [GcnGraph(ds.edge_index, V, DEV, coords=ds.x_pos, reorder=True),
               GcnGraph(ds.face_index, F, DEV, coords=ds.z2.detach()[:, :3], reorder=True),
               GcnGraph(ds.face_index, F, DEV, reorder=False)]
    torch.manual_seed(C + n)
    prev = lib.query("ddmp_spmm_reference_kernel", 0)
    try:
        for graph in graphs_:
            H = torch.randn(graph.n, C, device=DEV)
            b = torch.randn(C, device=DEV)
            res = {}
            for ref in (0, 1):
                lib.query("ddmp_spmm_reference_kernel", ref)
                Y, partials, ab = F_.spmm_gcn(graph, H, bias=b, stats=True, amax=True)
                Yp = F_.spmm_gcn(graph, H)
                res[ref] = (Y, partials, ab.max(), Yp)
            assert torch.equal(res[0][0], res[1][0]) and torch.equal(res[0][3], res[1][3])
            assert torch.equal(res[0][1], res[1][1])
            assert float(res[0][2]) == float(res[1][2]) == float(res[1][0].abs().max())
            # partitioned layout: the last rows of H are "halo" rows that are only read
            n_own = graph.n - max(1, graph.n // 7)
            rp = graph.rowptr[: n_own + 1].contiguous()
            sub = type("G", (), dict(rowptr=rp, col=graph.col, w=graph.w, rowptr_t=rp, col_t=graph.col, w_t=graph.w))
            outs = []
            for ref in (0, 1):
                lib.query("ddmp_spmm_reference_kernel", ref)
                outs.append(F_.spmm_gcn(sub, H, bias=b, n_rows=n_own))
            assert outs[0].shape == (n_own, C) and torch.equal(outs[0], outs[1])
            assert torch.equal(outs[0], res[1][0][:n_own])
    finally:
        lib.query("ddmp_spmm_reference_kernel", prev)


@pytest.mark.parametrize("C", [256, 512])
@pytest.mark.parametrize("kind,n", [("ico", 3), ("open", 9), ("ico", 40)])
def test_spmm_tensor_memory_statistics_kernel_equals_reference_kernel_bitwise(kind, n, C):
    """spmm_gcn_stats_tmem_kernel (forward flavour of the wide layers: per-warp Welford state in TMEM through
    tcgen05.ld / tcgen05.st instead of 32 KB of shared memory; the default) keeps the warp -> row assignment, the
    per-element accumulation order and the Chan merge of spmm_gcn_kernel (ddmp_spmm_reference_kernel): Y and the
    (sum, M2) block partials must be IDENTICAL -- with and without bias, ragged last block, partitioned layout, repeated
    launches (TMEM allocation / release)."""
    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200._lib import lib
    from dual_dmp_b200.graph import GcnGraph
    from oracle.step_ref import make_dataset
    n_mesh, s_mesh, _ = small_case(kind, n)
    ds = make_dataset(n_mesh, s_mesh)
    V, F = len(n_mesh.vs), len(n_mesh.faces)
    graphs_ = [GcnGraph(ds.edge_index, V, DEV, coords=ds.x_pos, reorder=True),
               GcnGraph(ds.face_index, F, DEV, coords=ds.z2.detach()[:, :3], reorder=True)]
    torch.manual_seed(C + n)
    prev = lib.query("ddmp_spmm_reference_kernel", 0)
    try:
        for graph in graphs_:
            H = torch.randn(graph.n, C, device=DEV)
            b = torch.randn(C, device=DEV) * 3
            n_own = graph.n - max(1, graph.n // 7)
            rp = graph.rowptr[: n_own + 1].contiguous()
            sub = type("G", (), dict(rowptr=rp, col=graph.col, w=graph.w, rowptr_t=rp, col_t=graph.col, w_t=graph.w))
            res = {}
            for ref in (1, 0):
                lib.query("ddmp_spmm_reference_kernel", ref)
                out = []
                for _ in range(3):
                    out += [*F_.spmm_gcn(graph, H, bias=b, stats=True), *F_.spmm_gcn(graph, H, stats=True),
                            *F_.spmm_gcn(sub, H, bias=b, stats=True, n_rows=n_own)]
                res[ref] = out
            for i, (x, x0) in enumerate(zip(res[0], res[1])):
                assert torch.equal(x, x0), (i, graph.n, C)
    finally:
        lib.query("ddmp_spmm_reference_kernel", prev)
