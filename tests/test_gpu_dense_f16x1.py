"""The single-product mode of the dense transforms (DDMP_GEMM_F16X1, dense_precision="f16x1") on the GPU:
  * accuracy of gemm_xw (with and without the fused BatchNorm + LeakyReLU prologue, with row_map), gemm_dx and gemm_dw
    on every tcgen05 shape of the networks, at 1,000 rows, 1M rows and a ragged row count, against float64 with the
    rigorous elementwise bound restated in tests/test_f16x1_cpu.py; the error must also be clearly larger than the
    3-term kernels' (which proves the 1-term kernel ran);
  * bitwise-equal reruns; no leak of the mode into the default path (calls, and fits of one MultiDualStep);
  * coverage: a 1-term DualStep launches the 1-term instantiation for every fp16-split GEMM of its step;
  * the end-to-end MAD bar of tests/test_gpu_e2e_mad.py, with both weight sets, in "f16x1" mode."""
import copy
import json
import os
import re
import sys
from collections import Counter

import numpy as np
import pytest
import torch

from tests.helpers import report, small_case
from tests.test_f16x1_cpu import gemm_bound, scale_from_bits

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
# (Cin, Cout) of every trunk layer whose three transforms run on the fp16-split kernels (util/networks.py widths)
SHAPES = [(64, 128), (128, 256), (256, 256), (256, 512), (512, 512), (512, 256), (256, 128), (128, 64)]
ROWS = [1000, 1003520, 200003]
SLOPE = 0.01


def _operands(n, cin, cout, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    X = (torch.randn(n, cin, generator=g) * (torch.rand(1, cin, generator=g) * 3 + 0.2)).to(DEV)
    W = (torch.randn(cout, cin, generator=g) / cin ** 0.5).to(DEV)
    dH = (torch.randn(n, cout, generator=g) * 1e-3).to(DEV)
    sc = (torch.rand(cin, generator=g) + 0.5).to(DEV)
    sh = torch.randn(cin, generator=g).to(DEV)
    return X, W, dH, sc, sh


def _act64(X, sc, sh):
    z = X.double() * sc.double() + sh.double()
    return torch.where(z > 0, z, z * SLOPE)


def _scale(bound_tensor):
    return float(scale_from_bits([float(bound_tensor.abs().max())])[0][0])


def _check(C, A64, B64, s_a, s_b, what):
    """elementwise bound; returns the largest error relative to |A||B| (the measure the 3-term path is compared on)"""
    ref = A64 @ B64
    err = (C.double() - ref).abs()
    bnd = gemm_bound(A64, B64, s_a, s_b)
    ratio = float((err / bnd).max())
    assert ratio <= 1.0, (what, ratio)
    return float((err / (A64.abs() @ B64.abs()).clamp_min(1e-300)).max())


@pytest.mark.parametrize("n", ROWS)
@pytest.mark.parametrize("cin,cout", SHAPES)
def test_accuracy_against_float64(cin, cout, n):
    from dual_dmp_b200 import functional as F_
    X, W, dH, sc, sh = _operands(n, cin, cout, 1000 * cin + cout + n % 997)
    act = _act64(X, sc, sh)
    b_act = (act.abs().amax(0) * 1.25).float().contiguous()              # per-channel bounds, like the BatchNorm bound
    b_x = (X.abs().amax(0) * 2.0).contiguous()
    b_dh = dH.abs().amax(1).reshape(-1)[:4096].contiguous()              # row-block style maxima (a prefix is a
    b_dh = torch.cat([b_dh, dH.abs().max().reshape(1)])                  # smaller array with the same maximum)
    s_act, s_x, s_dh = _scale(b_act), _scale(b_x), _scale(b_dh)
    s_w_rows = torch.from_numpy(scale_from_bits(W.abs().amax(1).cpu().numpy())[0]).to(DEV)    # xw: per output column
    s_w_cols = torch.from_numpy(scale_from_bits(W.abs().amax(0).cpu().numpy())[0]).to(DEV)    # dx: per output column
    perm = torch.randperm(n, generator=torch.Generator(device="cpu").manual_seed(n)).to(DEV)
    row_map = perm.to(torch.int32)
    Wt64, W64 = W.double().t(), W.double()
    worst = {}
    for mode in ("f16x1", "fp32"):
        kw = dict(backend=2, dense_precision=mode)
        res = {
            "xw_act": (F_.gemm_xw(X, W, scale=sc, shift=sh, amax=b_act, **kw), act, Wt64, s_act, s_w_rows),
            "xw": (F_.gemm_xw(X, W, amax=b_x, **kw), X.double(), Wt64, s_x, s_w_rows),
            "xw_rowmap": (F_.gemm_xw(X, W, row_map=row_map, scale=sc, shift=sh, amax=b_act, **kw), act[perm], Wt64,
                          s_act, s_w_rows),
            "dx": (F_.gemm_dx(dH, W, amax=b_dh, **kw), dH.double(), W64, s_dh, s_w_cols),
            "dw": (F_.gemm_dw(dH, X, cin, scale=sc, shift=sh, amax_dh=b_dh, amax_x=b_act, **kw), dH.double().t(), act,
                   s_dh, s_act),
        }
        for name, (C, A64, B64, s_a, s_b) in res.items():
            if mode == "f16x1":
                worst[name] = [_check(C, A64, B64, s_a, s_b, (name, cin, cout, n)), None]
            else:
                ref = A64 @ B64
                worst[name][1] = float(((C.double() - ref).abs() / (A64.abs() @ B64.abs()).clamp_min(1e-300)).max())
        del res
    report(f"f16x1 {cin}->{cout} n={n}: max |C-C64|/(|A||B|) 1-term vs 3-term", worst)
    # the 1-term kernel ran: its worst error is >= 32x the 3-term one's on every case measured on a B200 (dW at 1M
    # rows, where the rounding errors of 2048-row chains average out, is the closest); 10x leaves room for other data
    for name, (e1, e3) in worst.items():
        assert e1 > 10 * e3, (name, e1, e3)


def test_deterministic_and_no_leak_into_the_default_path():
    from dual_dmp_b200 import functional as F_
    X, W, dH, sc, sh = _operands(300007, 256, 512, 7)
    b = (_act64(X, sc, sh).abs().amax(0) * 1.25).float().contiguous()
    b_dh = dH.abs().max().reshape(1)
    calls = [lambda m: F_.gemm_xw(X, W, scale=sc, shift=sh, amax=b, dense_precision=m),
             lambda m: F_.gemm_dx(dH, W, amax=b_dh, dense_precision=m),
             lambda m: F_.gemm_dw(dH, X, 256, scale=sc, shift=sh, amax_dh=b_dh, amax_x=b, dense_precision=m)]
    for call in calls:
        before = call("fp32")
        one = call("f16x1")
        again = [call("f16x1") for _ in range(2)]
        after = call("fp32")
        assert torch.equal(before, after)                                    # the 3-term result does not move
        assert all(torch.equal(one, a) for a in again)                       # bitwise-equal reruns
        assert not torch.equal(one, before)


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


F16 = re.compile(r"(tc_gemm_nt16x2_kernel|tc_gemm_nt16_kernel|tc_gemm_tn16x2_kernel|tc_gemm_tn16_kernel|"
                 r"tc_prep_b16_kernel)<([^>]*)>")


def _split(names):
    """fp16-split launches as (family, term count) and every other launch by name"""
    f16, other = Counter(), Counter()
    for nm in names:
        m = F16.search(nm)
        if m:
            f16[(m.group(1), int(m.group(2).split(",")[-1]))] += 1
        elif "Memcpy" not in nm and "Memset" not in nm:
            other[nm] += 1
    return f16, other


@pytest.mark.parametrize("n_ico", [9, 40])
def test_coverage_of_a_dual_step(n_ico):
    """every fp16-split GEMM of a step (9 trunk layers x xw, dx, dw x 2 networks = 54, and 36 weight images) runs the
    1-term instantiation in "f16x1" mode, and nothing else changes: the same other kernels, the same count"""
    from dual_dmp_b200.step import DualStep
    from dual_dmp_b200.util.datamaker import dataset_from_meshes
    from dual_dmp_b200.util.networks import NormalNet, PosNet
    n_mesh, s_mesh, _ = small_case("ico", n_ico)
    ds = dataset_from_meshes(n_mesh, s_mesh)
    runs = {}
    for mode in ("fp32", "f16x1"):
        torch.manual_seed(0)
        posnet, normnet = PosNet(DEV).to(DEV), NormalNet(DEV).to(DEV)
        st = DualStep(posnet, normnet, ds, n_mesh, capture=False, dense_precision=mode)
        st.step(1)
        runs[mode] = _split(_kernels(lambda: st.step(2)))
    (f3, o3), (f1, o1) = runs["fp32"], runs["f16x1"]
    report(f"f16x1 coverage ico {n_ico}", {"fp32": dict(f3), "f16x1": dict(f1)})
    assert all(t == 3 for _, t in f3) and all(t == 1 for _, t in f1)
    gemms = lambda c: sum(v for (fam, _), v in c.items() if fam != "tc_prep_b16_kernel")   # noqa: E731
    assert gemms(f3) == gemms(f1) == 54
    assert sum(f3.values()) == sum(f1.values()) == 54 + 36
    assert Counter(f for f, _ in f3.elements()) == Counter(f for f, _ in f1.elements())
    assert o3 == o1


def test_multi_fit_mode_does_not_leak_into_other_fits():
    from dual_dmp_b200.step import DualStep, MultiDualStep
    from dual_dmp_b200.util.datamaker import dataset_from_meshes
    from dual_dmp_b200.util.networks import NormalNet, PosNet
    cases = [small_case("ico", 10), small_case("open", 12), small_case("ico", 8)]
    modes = ["fp32", "f16x1", "fp32"]
    fits = []
    for i, ((n_mesh, s_mesh, _), mode) in enumerate(zip(cases, modes)):
        torch.manual_seed(i + 1)
        fits.append(dict(posnet=PosNet(DEV).to(DEV), normnet=NormalNet(DEV).to(DEV),
                         dataset=dataset_from_meshes(n_mesh, s_mesh), n_mesh=n_mesh, dense_precision=mode))
    twins = [dict(f, posnet=copy.deepcopy(f["posnet"]), normnet=copy.deepcopy(f["normnet"])) for f in fits]
    multi = MultiDualStep(fits)
    epochs = list(range(98, 104))
    got = []
    for ep in epochs:
        multi.step(ep)
        got.append(([p.clone() for p in multi.pos], [q.clone() for q in multi.norm]))
    for i, f in enumerate(twins):
        single = DualStep(f["posnet"], f["normnet"], f["dataset"], f["n_mesh"], dense_precision=f["dense_precision"])
        for j, ep in enumerate(epochs):
            single.step(ep)
            same = torch.equal(single.pos, got[j][0][i]) and torch.equal(single.norm, got[j][1][i])
            if modes[i] == "fp32":
                assert same, (i, ep)
    # the f16x1 fit really ran in its own mode: its trajectory differs from the same fit in fp32
    f = fits[1]
    torch.manual_seed(2)
    p32, n32 = PosNet(DEV).to(DEV), NormalNet(DEV).to(DEV)
    ref = DualStep(p32, n32, f["dataset"], f["n_mesh"])
    for ep in epochs:
        ref.step(ep)
    assert not torch.equal(ref.pos, got[-1][0][1])


def _stats(mad):
    mad = np.asarray(mad)
    return {"final": float(mad[-1]), "tail10": float(mad[-10:].mean()), "half2": float(mad[50:].mean())}


@pytest.mark.parametrize("config", ["default", "cad"])
def test_f16x1_meets_the_end_to_end_mad_bar(golden_dir, config):
    """the statements of tests/test_gpu_e2e_mad.py, for the product in "f16x1" mode (five DualStep trajectories and the
    drop-in loop, all with dense_precision="f16x1")"""
    sys.path.insert(0, os.path.join(ROOT, "scripts"))
    import e2e_mad
    gold = json.load(open(os.path.join(golden_dir, f"e2e_mad_{config}.json")))
    case = small_case("ico", gold["n"])
    assert len(case[0].faces) == gold["faces"]
    k, bnfloop = e2e_mad.CONFIGS[config]
    ref = [_stats(r["mad"]) for r in gold["oracle_runs"]]
    ref_curves = np.array([r["mad"] for r in gold["oracle_runs"]])
    half_ref = np.array([r["half2"] for r in ref])
    fin_ref = np.array([r["final"] for r in ref])
    early_ref = ref_curves[:, :10].min(axis=1)
    prods = {}
    for path, perturb in [("dualstep", i) for i in range(5)] + [("dropin", 0)]:
        run = e2e_mad.run_product(case, k, bnfloop, gold["iters"], gold["seed"], path, lambda s: None, perturb=perturb,
                                  dense_precision="f16x1")
        mad = np.array(run["mad"])
        assert mad.shape == ref_curves.shape[1:] and np.isfinite(mad).all()
        st = _stats(mad)
        st["early_min"] = float(mad[:10].min())
        prods[f"{path}/{perturb}"] = st
    report(f"e2e MAD {config} f16x1: product runs {prods}", "oracle runs %s" % ref)
    for name, st in prods.items():
        assert abs(st["half2"] - half_ref.mean()) <= 3.0 * half_ref.std(ddof=1) + 0.02 * half_ref.mean(), (name, st, half_ref)
        assert abs(st["final"] - fin_ref.mean()) <= 3.0 * fin_ref.std(ddof=1) + 0.02 * fin_ref.mean(), (name, st, fin_ref)
        assert st["early_min"] < 0.2 * gold["initial_mad"]
        assert early_ref.min() * 0.9 <= st["early_min"] <= early_ref.max() * 1.1, (name, st["early_min"], early_ref)
    level_ref = float(np.mean(half_ref))
    level = float(np.mean([p["half2"] for p in prods.values()]))
    rel = abs(level - level_ref) / level_ref
    report(f"e2e MAD {config} f16x1: product ensemble level / oracle ensemble level / rel diff", (level, level_ref, rel))
    assert rel <= 0.02, (level, level_ref)
