"""Every CSR-walking kernel on long rows: hub vertices, fan caps and dense graph rows (tests/long_rows.py).

The meshes of the rest of the suite have a maximum valence of 6, so no aggregation row there is longer than one chunk
of (col, w) entries and no loss kernel runs a second batch of 8 neighbours.  Here:
  * aggregation over a non-mesh graph with rows of 1 ... 4097 entries, on every kernel setting, against float64:
    exactly (power-of-two weights and integer features make every fp32 partial sum exact, so Y must EQUAL the reference)
    and with real GCN weights under a rigorous per-row bound  |Y_i - ref_i| <= 2 (L_i + 1) 2^-24 sum_k |w_k H_ck| (+|b|);
  * the fused BatchNorm-backward aggregations against the unfused pair under the same kind of bound;
  * the losses, the geometry and the preprocessing on UV spheres, fan discs and fan-capped cylinders against the CPU
    oracle: the product's distance from the float64 oracle must stay within 3x the fp32 oracle's own distance + a floor;
  * a 1M-face UV sphere (poles of valence 2048), where the grid-stride loops of the fused loss kernel iterate.
"""
import numpy as np
import pytest
import torch

from tests import long_rows as LR
from tests.helpers import rel_err, report

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
U32 = 2.0 ** -24
U64 = 2.0 ** -53
WIDTHS = [32, 64, 128, 256, 512]
# ddmp_spmm_use_tile_kernel settings: mode (0 gather, 1 tile-staged for C <= 128, 2 tile-staged everywhere) | flags << 4
# (2: streaming stores, 4|8: Welford state in tensor memory at C = 512 / 256)
SETTINGS = [mode | (flags << 4) for mode in (0, 1, 2) for flags in (2, 4 | 8)]


# ---------------------------------------------------------------------------------------------------------------------
# aggregation
# ---------------------------------------------------------------------------------------------------------------------
def _sub(rowptr, col, w, n_rows):
    rp = rowptr[: n_rows + 1].contiguous()
    return type("G", (), dict(rowptr=rp, col=col, w=w, rowptr_t=rp, col_t=col, w_t=w))


@pytest.fixture(scope="module")
def agg():
    from dual_dmp_b200.graph import GcnGraph
    ei, n, coords = LR.aggregation_graph()
    eit = torch.from_numpy(ei)
    graphs = {"morton": GcnGraph(eit, n, DEV, coords=torch.from_numpy(coords), reorder=True),
              "caller": GcnGraph(eit, n, DEV, reorder=False)}
    assert graphs["morton"].symmetric and not graphs["morton"].identity and graphs["caller"].identity
    n_own = n - n // 7
    variants = {}
    for name, g in graphs.items():
        # power-of-two weights 2^0 ... 2^-3, a function of the entry's position
        k = torch.arange(g.nnz, device=DEV)
        w_exact = torch.ldexp(torch.ones(g.nnz, device=DEV), -((k * 7 + g.col.long() * 3) % 4)).float()
        variants[name] = (g.rowptr, g.col, g.w, w_exact, n)
        variants[name + "-partitioned"] = (g.rowptr, g.col, g.w, w_exact, n_own)   # H = [owned | halo] rows
    return dict(n=n, ei=ei, graphs=graphs, variants=variants)


def _csr64(rowptr, col, w, X, n_rows):
    """float64 sum_k w_k X[col_k] per row on the device (index_add_), a slice of channels at a time"""
    rp = rowptr[: n_rows + 1].long()
    nnz = int(rp[-1])
    dst = torch.repeat_interleave(torch.arange(n_rows, device=X.device), rp.diff())
    c, ww = col[:nnz].long(), w[:nnz].double().view(-1, 1)
    C = X.shape[1]
    out = torch.zeros(n_rows, C, dtype=torch.float64, device=X.device)
    step = max(1, (1 << 26) // max(nnz, 1))
    for c0 in range(0, C, step):
        out[:, c0:c0 + step].index_add_(0, dst, ww * X[:, c0:c0 + step].double().index_select(0, c))
    return out


def _row_len(rowptr, n_rows):
    return rowptr[: n_rows + 1].long().diff().double()


def _check_partials(partials, ref, C):
    """BatchNorm partials (sum, M2 about the block mean) per row block against the float64 column sums / sums of squares"""
    from dual_dmp_b200._lib import lib
    pb = partials.double()
    rpb = int(lib.query("ddmp_rows_per_block", C))
    n = ref.shape[0]
    assert pb.shape[0] == (n + rpb - 1) // rpb
    n_b = torch.full((pb.shape[0], 1), float(rpb), dtype=torch.float64, device=pb.device)
    n_b[-1] = n - (pb.shape[0] - 1) * rpb
    s = pb[:, 0].sum(0)
    q = (pb[:, 1] + pb[:, 0] ** 2 / n_b).sum(0)
    e_s = float(((s - ref.sum(0)).abs() / ref.abs().sum(0)).max())
    sq = (ref * ref).sum(0)
    e_q = float(((q - sq).abs() / sq).max())
    assert e_s < 1e-5 and e_q < 1e-5, (e_s, e_q)
    return max(e_s, e_q)


def _set(setting):
    from dual_dmp_b200._lib import lib
    lib.query("ddmp_spmm_use_tile_kernel", setting)


@pytest.fixture
def restore_setting():
    from dual_dmp_b200._lib import lib
    prev = lib.query("ddmp_spmm_use_tile_kernel", -1)
    lib.query("ddmp_spmm_use_tile_kernel", prev)
    try:
        yield
    finally:
        lib.query("ddmp_spmm_use_tile_kernel", prev)


def test_long_row_graph_csr_and_weights(agg):
    """the graph builder and ddmp_gcn_edge_weights (one thread walks a whole row) on rows of up to 4097 entries"""
    from oracle.gcn_ref import gcn_norm_ref
    idx, _ = gcn_norm_ref(torch.from_numpy(agg["ei"]), agg["n"])
    ref = idx.numpy()
    ref = ref[:, np.lexsort((ref[1], ref[0]))]
    for g in agg["graphs"].values():
        assert np.array_equal(g.to_edge_list(), ref)
        deg = g.rowptr.long().diff().double()
        dst = torch.repeat_interleave(torch.arange(g.n, device=DEV), g.rowptr.long().diff())
        w64 = deg[dst].rsqrt() * deg[g.col.long()].rsqrt()
        e = float(((g.w.double() - w64).abs() / w64).max())
        assert e <= 6 * U32, e                     # 1/sqrtf(deg): two roundings per factor, one for the product


@pytest.mark.parametrize("C", WIDTHS + [12])
def test_aggregation_is_exact_on_long_rows(agg, C, restore_setting):
    """power-of-two weights, integer H in [-64, 64], power-of-two bias: every product and partial sum is exact in fp32,
    so Y and max|Y| must EQUAL the float64 reference on every kernel setting -- a dropped, doubled or misplaced (col, w)
    entry of any chunk fails here with no tolerance involved"""
    from dual_dmp_b200 import functional as F_
    n = agg["n"]
    torch.manual_seed(C)
    H = torch.randint(-64, 65, (n, C), device=DEV).float()
    bias = (torch.ldexp(torch.ones(C), torch.randint(-3, 4, (C,))) * torch.where(torch.rand(C) < 0.5, -1.0, 1.0)).to(DEV)
    worst = 0.0
    for name, (rowptr, col, _, w_exact, n_rows) in agg["variants"].items():
        g = _sub(rowptr, col, w_exact, n_rows)
        ref0 = _csr64(rowptr, col, w_exact, H, n_rows)
        for setting in (SETTINGS if C != 12 else SETTINGS[:1]):
            _set(setting)
            for b in (None, bias):
                ref = ref0 if b is None else ref0 + b.double()
                Y = F_.spmm_gcn(g, H, bias=b, n_rows=n_rows)
                assert torch.equal(Y.double(), ref), (name, setting, float((Y.double() - ref).abs().max()))
                if C == 12:
                    continue
                Ys, partials = F_.spmm_gcn(g, H, bias=b, stats=True, n_rows=n_rows)
                assert torch.equal(Ys.double(), ref), (name, setting, "stats")
                worst = max(worst, _check_partials(partials, ref, C))
                Ya, ab = F_.spmm_gcn(g, H, bias=b, n_rows=n_rows, amax=True)
                assert torch.equal(Ya.double(), ref) and float(ab.max()) == float(ref.abs().max()), (name, setting)
    report(f"long rows: exact aggregation C={C}: Y bitwise = float64 on {len(SETTINGS)} settings; partials err", worst)


@pytest.mark.parametrize("C", WIDTHS + [12])
def test_aggregation_with_gcn_weights_within_a_priori_bound(agg, C, restore_setting):
    """real GCN weights (the graph's own fp32 w), random H and bias, against float64 index_add_ on the device, per row:
    |Y_i - ref_i| <= 2 (L_i + 1) 2^-24 (sum_k |w_k H_ck| + |b|)   (recursive fp32 summation of L_i products + bias)"""
    from dual_dmp_b200 import functional as F_
    n = agg["n"]
    torch.manual_seed(100 + C)
    H = torch.randn(n, C, device=DEV)
    bias = torch.randn(C, device=DEV)
    worst = 0.0
    for name, (rowptr, col, w, _, n_rows) in agg["variants"].items():
        g = _sub(rowptr, col, w, n_rows)
        ref = _csr64(rowptr, col, w, H, n_rows) + bias.double()
        bound = 2.0 * (_row_len(rowptr, n_rows) + 1.0).view(-1, 1) * U32 * \
            (_csr64(rowptr, col, w.abs(), H.abs(), n_rows) + bias.double().abs()) + 1e-30
        for setting in (SETTINGS if C != 12 else SETTINGS[:1]):
            _set(setting)
            outs = [F_.spmm_gcn(g, H, bias=bias, n_rows=n_rows)]
            if C != 12:
                outs.append(F_.spmm_gcn(g, H, bias=bias, stats=True, n_rows=n_rows)[0])
            for Y in outs:
                r = (Y.double() - ref).abs() / bound
                worst = max(worst, float(r.max()))
                assert (r <= 1.0).all(), (name, setting, float(r.max()))
    report(f"long rows: GCN-weight aggregation C={C}: max |Y - ref| / a-priori bound", worst)


@pytest.mark.parametrize("C", WIDTHS)
def test_aggregation_kernels_bitwise_equal_on_long_rows(agg, C, restore_setting):
    """tile-staged (shared-memory and global (col, w) streams), gather, gather with streaming stores, and the TMEM
    statistics flavour all accumulate every row in CSR order: Y, the block partials and max|Y| are IDENTICAL"""
    from dual_dmp_b200 import functional as F_
    n = agg["n"]
    torch.manual_seed(200 + C)
    H = torch.randn(n, C, device=DEV)
    b = torch.randn(C, device=DEV) * 3
    for name, (rowptr, col, w, _, n_rows) in agg["variants"].items():
        g = _sub(rowptr, col, w, n_rows)
        res = {}
        for setting in [0] + SETTINGS:
            _set(setting)
            y1, p1 = F_.spmm_gcn(g, H, bias=b, stats=True, n_rows=n_rows)
            y2, p2 = F_.spmm_gcn(g, H, stats=True, n_rows=n_rows)
            y3, ab = F_.spmm_gcn(g, H, bias=b, amax=True, n_rows=n_rows)
            y4 = F_.spmm_gcn(g, H, n_rows=n_rows)
            assert float(ab.max()) == float(y3.abs().max())
            res[setting] = (y1, p1, y2, p2, y3, y4, ab.max())
        for setting, out in res.items():
            for i, (x, x0) in enumerate(zip(out, res[0])):
                assert torch.equal(x, x0), (name, setting, i)
    report(f"long rows: aggregation kernels bitwise equal C={C}", len(res))


def _ident(n):
    from dual_dmp_b200.graph import GcnGraph
    return GcnGraph(torch.zeros(2, 0, dtype=torch.long), n, DEV, reorder=False)


@pytest.mark.parametrize("C", WIDTHS)
def test_fused_bn_backward_aggregation_on_long_rows(agg, C):
    """ddmp_spmm_bn_bwd (dY recomputed in the gather) and ddmp_spmm_bn_bwd_tile (dY formed in shared memory; global (col, w)
    stream in the heavy row blocks) against ddmp_bn_bwd_apply + the backward aggregation, per row within
    sum_k |w_k| (4 (L_i + 1) 2^-24 |dY_ck| + 16 2^-24 T_ck), T = |scale| (|gZ| + |c1| + |c2| rstd (|Y| + |mean|)) the
    magnitude of the terms dY is formed from; dgamma / dbeta equal, conv-bias gradient and max|dH| checked, reruns equal"""
    from dual_dmp_b200 import functional as F_
    worst = 0.0
    for name, g in agg["graphs"].items():
        n = g.n
        torch.manual_seed(300 + C)
        Y = (torch.randn(n, C) * 1.5 + 0.3).to(DEV)
        gX = torch.randn(n, C, device=DEV)
        st = F_.bn_stats_finalize(F_.spmm_gcn(_ident(n), Y, stats=True)[1], n, (torch.rand(C) + 0.5).to(DEV),
                                  torch.randn(C).to(DEV))
        sc, sh, mu, rs = (st[i].double() for i in (2, 3, 0, 1))
        for _ in range(3):        # away from the LeakyReLU kink: the slope must not depend on rounding
            z = Y.double() * sc + sh
            Y = torch.where(z.abs() < 1e-3, Y + 0.05, Y)
        dY, dgamma, dbeta, dbias = F_.bn_lrelu_backward(gX, Y, st)
        dH_ref = F_.spmm_gcn(g, dY, transposed=True)
        z = Y.double() * sc + sh
        gZ = torch.where(z > 0, gX.double(), gX.double() * F_.SLOPE)
        c1, c2 = dbeta.double() / n, dgamma.double() / n
        T = sc.abs() * (gZ.abs() + c1.abs() + c2.abs() * rs * (Y.double().abs() + mu.abs()))
        aw = g.w.abs()
        bound = 4.0 * (_row_len(g.rowptr, n) + 1.0).view(-1, 1) * U32 * _csr64(g.rowptr, g.col, aw, dY.abs(), n) + \
            16.0 * U32 * _csr64(g.rowptr, g.col, aw, T, n) + 1e-30
        dH1, dgamma1, dbeta1, dbias1 = F_.bn_bwd_spmm_fused(g, gX, Y, st)
        dH2, dgamma2, dbeta2, dbias2, ab = F_.bn_bwd_spmm_tile(g, gX, Y, st, amax=True)
        for which, dH, dg, db, dbb in (("gather", dH1, dgamma1, dbeta1, dbias1), ("tile", dH2, dgamma2, dbeta2, dbias2)):
            r = float(((dH.double() - dH_ref.double()).abs() / bound).max())
            worst = max(worst, r)
            assert r <= 1.0, (name, which, r)
            assert torch.equal(dg, dgamma) and torch.equal(db, dbeta), (name, which)
            assert (dbb - dbias).abs().max() <= 1e-5 * dY.abs().sum(dim=0).max(), (name, which)
        assert float(ab.max()) == float(dH2.abs().max())
        assert torch.equal(F_.bn_bwd_spmm_fused(g, gX, Y, st)[0], dH1)
        assert torch.equal(F_.bn_bwd_spmm_tile(g, gX, Y, st)[0], dH2)
    report(f"long rows: fused BN backward aggregation C={C}: max |dH - unfused| / bound", worst)


# ---------------------------------------------------------------------------------------------------------------------
# losses, geometry, preprocessing
# ---------------------------------------------------------------------------------------------------------------------
LOSS_MESHES = LR.LOSS_MESHES
_mesh_cache = {}


def _mesh(kind, m, rings):
    from dual_dmp_b200.util.mesh import Mesh
    key = (kind, m, rings)
    if key not in _mesh_cache:
        vs, faces = LR.make_mesh(kind, m, rings)
        _mesh_cache[key] = Mesh(vs=vs, faces=faces)
    return _mesh_cache[key]


def _kinks(pos, nrm, mesh):
    """faces within reach of rounding of a sign() of the losses: |(p_k - c) . n| of pos_norm, |n - fn| of norm_rec"""
    faces = torch.from_numpy(mesh.faces).to(pos.device)
    tri = pos.double()[faces]
    pc = tri - tri.mean(dim=1, keepdim=True)
    dot = (pc * nrm.double().unsqueeze(1)).sum(dim=2).abs()
    scale = pc.norm(dim=2).amax(dim=1, keepdim=True) + 1e-5 * tri.abs().amax(dim=(1, 2)).view(-1, 1)
    bad = (dot < 1e-3 * scale).any(dim=1)
    fn = torch.from_numpy(mesh.fn).to(pos.device)
    return bad | ((nrm.double() - fn).abs() < 1e-4).any(dim=1)


def _loss_inputs(mesh, seed, new_fn=None):
    """noisy positions and predicted normals away from every sign() kink; ``new_fn(pos, nrm)`` gives the filtered
    normals of the bilateral filter, whose L1 term has a kink too"""
    g = torch.Generator().manual_seed(seed)
    V, F = len(mesh.vs), len(mesh.faces)
    pos = torch.from_numpy(mesh.vs).float() + 0.05 * torch.randn(V, 3, generator=g)
    fn = torch.from_numpy(mesh.fn).float()
    nrm = torch.nn.functional.normalize(fn + 0.3 * torch.randn(F, 3, generator=g), dim=1)
    for _ in range(20):
        bad = _kinks(pos, nrm, mesh)
        if new_fn is not None:
            bad = bad | ((new_fn(pos, nrm).double() - nrm.double()).abs() < 1e-4).any(dim=1)
        if not bad.any():
            return pos, nrm
        k = int(bad.sum())
        nrm[bad] = torch.nn.functional.normalize(fn[bad] + 0.3 * torch.randn(k, 3, generator=g), dim=1)
    raise AssertionError("could not move the inputs away from the kinks")


def _eval_losses(mod, pos, nrm, mesh, loop, dev):
    """the five losses one at a time: values, gradients w.r.t. pos and nrm (zeros where a loss does not depend on one),
    and the filtered normals"""
    vals, grads, new_fn = [], [], None
    for i in range(5):
        p = pos.clone().to(dev).requires_grad_(True)
        q = nrm.clone().to(dev).requires_grad_(True)
        if i == 0:
            l = mod.pos_rec_loss(p, mesh.vs)
        elif i == 1:
            l = mod.mesh_laplacian_loss(p, mesh)
        elif i == 2:
            l = mod.norm_rec_loss(q, mesh.fn)
        elif i == 3:
            l, new_fn = mod.fn_bnf_loss(p, q, mesh, loop=loop)
        else:
            l = mod.pos_norm_loss(p, q, mesh)
        gp, gq = torch.autograd.grad(l, [p, q], allow_unused=True)
        vals.append(float(l.detach()))
        grads += [torch.zeros_like(p) if gp is None else gp.detach(), torch.zeros_like(q) if gq is None else gq.detach()]
    return vals, grads, new_fn.detach()


def _within_fp32_oracle(name, got, o32, o64, floor):
    """the product's distance from the float64 oracle <= 3x the fp32 oracle's own distance + floor"""
    if isinstance(got, float):
        e_p, e_o = abs(got - o64) / (abs(o64) + 1e-30), abs(o32 - o64) / (abs(o64) + 1e-30)
    else:
        e_p, e_o = rel_err(got, o64), rel_err(o32, o64)
    assert e_p <= 3.0 * e_o + floor, (name, e_p, e_o)
    return e_p, e_o


@pytest.mark.parametrize("loop", [0, 1, 5])
@pytest.mark.parametrize("kind,m,rings", LOSS_MESHES)
def test_losses_on_hub_meshes_against_oracle(kind, m, rings, loop):
    from dual_dmp_b200.util import loss as L
    from oracle import loss_ref as R
    mesh = _mesh(kind, m, rings)

    def oracle_new_fn(p, q):
        return R.fn_bnf_loss(p.double(), q.double(), mesh, loop=loop)[1]

    pos, nrm = _loss_inputs(mesh, seed=m + rings, new_fn=oracle_new_fn if loop > 0 else None)
    vp, gp, nfp = _eval_losses(L, pos, nrm, mesh, loop, DEV)
    v32, g32, nf32 = _eval_losses(R, pos, nrm, mesh, loop, "cpu")
    v64, g64, nf64 = _eval_losses(R, pos.double(), nrm.double(), mesh, loop, "cpu")
    errs = []
    names = ["pos_rec", "laplacian", "norm_rec", "bnf", "pos_norm"]
    for i in range(5):
        errs.append(_within_fp32_oracle(names[i], vp[i], v32[i], v64[i], 1e-6))
        for j, wrt in enumerate(("pos", "nrm")):
            errs.append(_within_fp32_oracle(f"d {names[i]} / d {wrt}", gp[2 * i + j], g32[2 * i + j], g64[2 * i + j], 2e-6))
    errs.append(_within_fp32_oracle("filtered normals", nfp, nf32, nf64, 2e-6))
    report(f"long rows: losses {kind}{m}x{rings} F={len(mesh.faces)} loop={loop}: (product, fp32 oracle) vs float64",
           [tuple(f"{x:.2e}" for x in e) for e in errs])


@pytest.mark.parametrize("kind,m,rings", LOSS_MESHES[:3])
@pytest.mark.parametrize("loop,scale,k", [(0, 1.0, (3.0, 4.0, 4.0, 4.0, 1.0)), (1, 1.0, (3.0, 4.0, 4.0, 4.0, 1.0)),
                                          (1, 0.0, (3.0, 4.0, 4.0, 4.0, 1.0)), (5, 1.0, (3.0, 0.0, 3.0, 4.0, 2.0))])
def test_fused_dual_loss_equals_separate_losses_on_hub_meshes(kind, m, rings, loop, scale, k):
    from dual_dmp_b200.util import loss as L
    mesh = _mesh(kind, m, rings)

    def product_new_fn(p, q):
        return L.fn_bnf_loss(p.to(DEV), q.to(DEV), mesh, loop=max(loop, 1))[1].cpu()

    pos0, nrm0 = _loss_inputs(mesh, seed=7 * m + loop, new_fn=product_new_fn)
    res = _dual_vs_separate(pos0.to(DEV), nrm0.to(DEV), mesh, k, loop, scale)
    report(f"long rows: fused vs separate losses {kind}{m}x{rings} loop={loop} scale={scale}", res)


def _dual_vs_separate(pos0, nrm0, mesh, k, loop, scale):
    from dual_dmp_b200.util import loss as L
    res = []
    for fused in (True, False):
        p = pos0.clone().requires_grad_(True)
        q = nrm0.clone().requires_grad_(True)
        if fused:
            total, parts = L.dual_loss(p, q, mesh, mesh.vs, mesh.fn, k, loop, scale)
        else:
            l4, _ = L.fn_bnf_loss(p, q, mesh, loop=loop)
            ls = [L.pos_rec_loss(p, mesh.vs), L.mesh_laplacian_loss(p, mesh), L.norm_rec_loss(q, mesh.fn), l4 * scale,
                  L.pos_norm_loss(p, q, mesh)]
            total = k[0] * ls[0] + k[1] * ls[1] + k[2] * ls[2] + k[3] * ls[3] + k[4] * ls[4]
            parts = torch.stack([x.double() for x in ls])
        (total * 1.7).backward()
        res.append((total.detach(), parts.detach(), p.grad, q.grad))
    (ta, pa, gpa, gqa), (tb, pb, gpb, gqb) = res
    assert ta.dtype == tb.dtype == torch.float64
    assert abs(float(ta) - float(tb)) <= 1e-6 * abs(float(tb))
    assert torch.allclose(pa, pb, rtol=1e-6, atol=1e-9), (pa, pb)
    # d/dpos sums a hub's whole Laplacian and corner rows; the two paths scale the summands in a different order, so
    # they may differ by the rounding of a sum of L terms: per vertex, not relative to the largest gradient
    e_p = float(((gpa - gpb).abs() / _gpos_bound(pos0, nrm0, mesh, k, 1.7, pb)).max())
    e_q = rel_err(gqa, gqb)
    assert e_p <= 1.0 and e_q < 2e-6, (e_p, e_q)
    p = pos0.clone().requires_grad_(True)
    q = nrm0.clone().requires_grad_(True)
    t2, parts2 = L.dual_loss(p, q, mesh, mesh.vs, mesh.fn, k, loop, scale)
    (t2 * 1.7).backward()
    assert torch.equal(t2, ta) and torch.equal(parts2, pa) and torch.equal(p.grad, gpa) and torch.equal(q.grad, gqa)
    return e_p, e_q, pa


def _gpos_bound(pos, nrm, mesh, k, gout, parts):
    """per-vertex bound on the difference of two fp32 evaluations of d(gout * total)/d pos: 8 (L_i + 4) 2^-24 times the
    sum of the magnitudes of the summands (pos_rec; the Laplacian residuals of i and of its neighbours / their degree;
    the pos_norm corner messages, |coef| <= 4/3 k5 / V), L_i the longer of vertex i's Laplacian and corner rows"""
    dev = pos.device
    V = len(mesh.vs)
    p, t = pos.double(), torch.from_numpy(mesh.vs).to(dev)
    e = torch.from_numpy(mesh.edges.astype(np.int64)).to(dev)
    src, dst = torch.cat([e[:, 0], e[:, 1]]), torch.cat([e[:, 1], e[:, 0]])
    deg = torch.bincount(src, minlength=V).double().view(-1, 1)
    d = (p - torch.zeros_like(p).index_add_(0, src, p[dst]) / deg).abs()
    lap = d + torch.zeros_like(p).index_add_(0, src, (d / deg)[dst])
    corners = torch.from_numpy(mesh.faces.reshape(-1)).to(dev)
    ncorner = torch.bincount(corners, minlength=V).double().view(-1, 1)
    cor = torch.zeros(V, dtype=torch.float64, device=dev).index_add_(
        0, corners, nrm.double().abs().amax(dim=1).repeat_interleave(3)).view(-1, 1)
    S = gout * (abs(k[0]) / (V * float(parts[0])) * (p - t).abs() + abs(k[1]) / (V * float(parts[1])) * lap +
                4.0 / 3.0 * abs(k[4]) / V * cor)
    return 8.0 * (torch.maximum(deg, ncorner) + 4.0) * U32 * S + 1e-30


@pytest.mark.parametrize("kind,m,rings", LR.GEOM_MESHES)
def test_geometry_on_hub_meshes_against_oracle(kind, m, rings):
    """compute_fn (+ its corner-gather backward), compute_vn, vertex_updating (per-vertex loops over the incident faces)"""
    from dual_dmp_b200.util import models as M
    from oracle import models_ref as MR
    mesh = _mesh(kind, m, rings)
    V, F = len(mesh.vs), len(mesh.faces)
    g = torch.Generator().manual_seed(m)
    pos = torch.from_numpy(mesh.vs).float() + 0.05 * torch.randn(V, 3, generator=g)
    gfn = torch.randn(F, 3, generator=g)
    errs = []
    outs = {}
    for tag, dev, dt in (("p", DEV, torch.float32), ("32", "cpu", torch.float32), ("64", "cpu", torch.float64)):
        x = pos.to(dev, dt).clone().requires_grad_(True)
        fn = (M if tag == "p" else MR).compute_fn(x, mesh.faces)
        fn.backward(gfn.to(dev, dt))
        vn_in = torch.from_numpy(mesh.fn).float()
        if tag == "p":
            vn = M.compute_vn(x.detach(), vn_in.to(DEV), mesh.faces)
        else:
            vn = MR.compute_vn(x.detach(), vn_in.to(dt), mesh.faces)
        outs[tag] = [fn.detach(), x.grad, vn]
        if V <= 4000:
            nrm = torch.from_numpy(mesh.fn).float()
            if tag == "p":
                outs[tag].append(M.vertex_updating(pos.to(DEV), nrm.to(DEV), mesh, loop=3))
            else:
                outs[tag].append(MR.vertex_updating(pos.to(dt), nrm.to(dt), mesh, loop=3))
    for i, name in enumerate(["compute_fn", "d compute_fn / d vs", "compute_vn", "vertex_updating"][: len(outs["p"])]):
        errs.append(_within_fp32_oracle(name, outs["p"][i], outs["32"][i], outs["64"][i], 2e-6))
    report(f"long rows: geometry {kind}{m}x{rings}: (product, fp32 oracle) vs float64",
           [tuple(f"{x:.2e}" for x in e) for e in errs])


@pytest.mark.parametrize("kind,m,rings", LR.PREP_MESHES)
def test_preprocess_on_hub_meshes(kind, m, rings):
    """DeviceMesh smoothing sweeps and vertex normals (float64, one thread walks a vertex's whole row) against
    synth.laplacian_smooth / synth.vertex_normals within a-priori float64 bounds"""
    from dual_dmp_b200 import preprocess, synth
    vs, faces = LR.make_mesh(kind, m, rings)
    vs = vs + 0.05 * np.random.default_rng(m).standard_normal(vs.shape)
    dm = preprocess.DeviceMesh(vs, faces, DEV)
    e = synth.unique_edges(faces, len(vs))
    maxdeg = int(LR.valences(faces, len(vs)).max())
    steps = 5
    sm = preprocess.smooth(dm, steps=steps).cpu().numpy()
    ref = synth.laplacian_smooth(vs, e, steps)
    # each sweep: a sum of deg + 1 rows then a division, twice (device, numpy); the sweep itself is non-expansive
    tol = 4.0 * steps * (maxdeg + 2) * U64 * np.abs(vs).max()
    e_s = np.abs(sm - ref).max()
    assert e_s <= tol, (e_s, tol)
    vn = dm.vertex_normals().cpu().numpy()
    fn, _ = synth.face_normals_areas(vs, faces)
    vref = synth.vertex_normals(vs, faces, fn)
    raw = np.zeros_like(vs)
    for c in range(3):
        raw[:, c] = np.bincount(faces.reshape(-1), weights=np.repeat(fn[:, c], 3), minlength=len(vs))
    # a face normal is as well conditioned as its cross product: kappa = |a| |b| / |a x b| (large for the slivers next to
    # the poles); the two evaluations may round the cross product differently, then sum L unit normals and normalise
    a, b = vs[faces[:, 1]] - vs[faces[:, 0]], vs[faces[:, 2]] - vs[faces[:, 0]]
    kappa = np.linalg.norm(a, axis=1) * np.linalg.norm(b, axis=1) / np.linalg.norm(np.cross(a, b), axis=1)
    d_fn = np.bincount(faces.reshape(-1), weights=np.repeat(6.0 * U64 * (kappa + 1.0), 3), minlength=len(vs))
    L = np.bincount(faces.reshape(-1), minlength=len(vs)).astype(np.float64)
    bound = 4.0 * (d_fn + 2.0 * (L + 2.0) * U64 * L) / np.linalg.norm(raw, axis=1) + 16.0 * U64
    r = (np.abs(vn - vref).max(axis=1) / bound).max()
    assert r <= 1.0, r
    report(f"long rows: preprocess {kind}{m}x{rings}: smooth err / bound, vertex normals err / bound", (e_s / tol, r))


# ---------------------------------------------------------------------------------------------------------------------
# one size where the grid-stride loops iterate
# ---------------------------------------------------------------------------------------------------------------------
def test_one_million_face_uv_sphere():
    """999,424 faces / 499,714 vertices, poles of valence 2048: the fused loss kernel (#SMs x occupancy blocks) walks
    several vertices and faces per thread.  dual_loss = separate kernels (and reruns equal); pos_rec, norm_rec and the
    Laplacian term against a float64 evaluation on the device; the aggregation at C = 64 and 512 within the per-row bound"""
    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200.graph import GcnGraph
    from dual_dmp_b200.util import loss as L
    from dual_dmp_b200.util.mesh import Mesh
    vs, faces = LR.uv_sphere(2048, 244)
    mesh = Mesh(vs=vs, faces=faces)
    V, F = len(vs), len(faces)
    assert F == 999_424 and LR.valences(faces, V).max() == 2048
    g = torch.Generator(device=DEV).manual_seed(0)
    pos = (torch.from_numpy(vs).to(DEV) + 0.05 * torch.randn(V, 3, device=DEV, generator=g, dtype=torch.float64)).float()
    fn = torch.from_numpy(mesh.fn).to(DEV)
    nrm = torch.nn.functional.normalize(fn + 0.3 * torch.randn(F, 3, device=DEV, generator=g, dtype=torch.float64),
                                        dim=1).float()
    for _ in range(20):
        bad = _kinks(pos, nrm, mesh)
        bad = bad | ((L.fn_bnf_loss(pos, nrm, mesh, loop=1)[1] - nrm).abs() < 1e-4).any(dim=1)
        if not bad.any():
            break
        k = int(bad.sum())
        nrm[bad] = torch.nn.functional.normalize(fn[bad] + 0.3 * torch.randn(k, 3, device=DEV, generator=g,
                                                                             dtype=torch.float64), dim=1).float()
    assert not bad.any()
    e_p, e_q, parts = _dual_vs_separate(pos, nrm, mesh, (3.0, 4.0, 4.0, 4.0, 1.0), 1, 1.0)

    # float64 evaluation on the device
    p64, t64 = pos.double(), torch.from_numpy(mesh.vs).to(DEV)
    pos_rec = torch.sqrt(((t64 - p64) ** 2).sum() / V + 1e-6)
    norm_rec = (nrm.double() - fn).abs().sum() / F
    e = torch.from_numpy(mesh.edges.astype(np.int64)).to(DEV)
    src, dst = torch.cat([e[:, 0], e[:, 1]]), torch.cat([e[:, 1], e[:, 0]])
    deg = torch.zeros(V, dtype=torch.float64, device=DEV).index_add_(0, src, torch.ones_like(src, dtype=torch.float64))
    d = p64 - torch.zeros_like(p64).index_add_(0, src, p64[dst]) / deg.view(-1, 1)
    lap = torch.sqrt((d ** 2).sum() / V + 1e-12)
    # fp32 residual of vertex i: deg_i - 1 additions, a division, a subtraction, per component
    amax = torch.zeros(V, dtype=torch.float64, device=DEV).scatter_reduce_(0, src, p64.abs().amax(1)[dst], "amax")
    delta = 2.0 * (deg + 2.0) * U32 * (p64.abs().amax(1) + amax) * 3 ** 0.5
    lap_tol = float(torch.sqrt((delta ** 2).sum() / V)) + 8 * U32 * float(lap)
    sep = [float(L.pos_rec_loss(pos, mesh.vs)), float(L.mesh_laplacian_loss(pos, mesh)),
           float(L.norm_rec_loss(nrm, mesh.fn))]
    errs = []
    for got_pr, got_lap, got_nr in ((float(parts[0]), float(parts[1]), float(parts[2])), tuple(sep)):
        errs += [abs(got_pr - float(pos_rec)) / float(pos_rec), abs(got_nr - float(norm_rec)) / float(norm_rec),
                 abs(got_lap - float(lap)) / lap_tol]
        assert errs[-3] < 1e-11 and errs[-2] < 1e-11 and errs[-1] <= 1.0, errs

    # aggregation over the vertex graph (Morton order), default kernel setting
    ei = torch.cat([e.t(), e.t().flip(0)], dim=1)
    graph = GcnGraph(ei.cpu(), V, DEV, coords=pos.cpu(), reorder=True)
    worst = 0.0
    for C in (64, 512):
        torch.manual_seed(C)
        H = torch.randn(V, C, device=DEV)
        b = torch.randn(C, device=DEV)
        ref = _csr64(graph.rowptr, graph.col, graph.w, H, V) + b.double()
        bound = 2.0 * (_row_len(graph.rowptr, V) + 1.0).view(-1, 1) * U32 * \
            (_csr64(graph.rowptr, graph.col, graph.w.abs(), H.abs(), V) + b.double().abs()) + 1e-30
        for Y in (F_.spmm_gcn(graph, H, bias=b), F_.spmm_gcn(graph, H, bias=b, stats=True)[0]):
            r = float(((Y.double() - ref).abs() / bound).max())
            worst = max(worst, r)
            assert r <= 1.0, (C, r)
        del H, ref, bound
    report("long rows: 1M-face UV sphere: fused vs separate grads, pos_rec / norm_rec rel, laplacian err / bound, "
           "aggregation err / bound", (e_p, e_q, errs, worst))
