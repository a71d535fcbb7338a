"""The numerical contract of the single-product mode of the fp16-split tensor-core GEMMs (DDMP_GEMM_F16X1,
csrc/gemm_tc.cu "single-product mode", DESIGN.md 4.2), restated on the CPU the way tests/test_f16_split_cpu.py restates
the three-term split: the power-of-two scale from a bound, the error of one fp16 product, and the elementwise bound of
a whole 1-term GEMM that tests/test_gpu_dense_f16x1.py checks the CUDA kernels against.

The bound.  With hi = fl16(s x) (round to nearest, u = 2^-11) each normal-range rounding has |delta| <= u / (1 + u), so
one product hi_a * hi_b (exact in fp32: 11 + 11 significant bits) differs from (s_a a)(s_b b) by at most
(2u + u^2)|s_a a||s_b b| (in fact (2u - u^2 + O(u^3))).  Summing K such products in fp32 -- any order, each addition
truncated or rounded, error <= 2^-23 of the partial sum -- adds at most (K - 1) 2^-23 (1 + 2u) sum|a||b| to first
order.  Unscaling by powers of two is exact.  So

    |C - C64| <= (2^-10 + K 2^-23) (|A| |B|) + subnormal term,

where the second-order terms fit in the slack between 2u - u^2 and 2^-10 for K <= 4096.  An operand element whose
scaled magnitude is below 2^-14 rounds to an fp16 subnormal with an absolute error of at most 2^-25 (half of the
subnormal spacing 2^-24); divided by its scale, that is the subnormal term (``gemm_bound``).
"""
import numpy as np
import torch

U16 = 2.0 ** -11


def scale_from_bits(bound):
    """mirror of tc::scale_from_bits: E = biased exponent of the bound, clamped to [16, 252]; s = 2^(141-E)"""
    bits = np.abs(np.asarray(bound, dtype=np.float32)).view(np.uint32)
    E = np.clip((bits >> 23) & 0xFF, 16, 252).astype(np.int64)
    return np.ldexp(1.0, 141 - E), np.ldexp(1.0, E - 141)


def gemm_bound(A, B, s_a, s_b):
    """elementwise bound of |C - A B| for the 1-term kernel, all float64 tensors: A [M, K], B [K, N]; s_a the scale of A
    (a number or one per row of A), s_b the scale of B (a number or one per column of B)"""
    K = A.shape[1]
    absA, absB = A.abs(), B.abs()
    s_a = torch.as_tensor(s_a, dtype=torch.float64, device=A.device).reshape(-1, 1)
    s_b = torch.as_tensor(s_b, dtype=torch.float64, device=A.device).reshape(1, -1)
    rel = (2.0 ** -10 + K * 2.0 ** -23) * (absA @ absB)
    sub = 2.0 ** -25 * (1 + 2 * U16) * (absB.sum(0, keepdim=True) / s_a + absA.sum(1, keepdim=True) / s_b)
    return rel + sub + K * 2.0 ** -50 / (s_a * s_b)


def fl16(x):
    return torch.as_tensor(x).to(torch.float16).to(torch.float64)


def truncating_fp32_matmul(a, b):
    """sum_k a[:, k] b[k, :] accumulated in fp32 with every addition truncated toward zero (the worst case of the
    tensor core's accumulator); a, b float64 holding fp16 values, so each product is exact"""
    acc = np.zeros((a.shape[0], b.shape[1]), dtype=np.float64)
    for k in range(a.shape[1]):
        s = acc + np.outer(a[:, k], b[k, :])
        t = s.astype(np.float32)                                       # round to nearest ...
        over = np.abs(t.astype(np.float64)) > np.abs(s)                # ... then one step toward zero where it rounded up
        t[over] = np.nextafter(t[over], np.float32(0))
        acc = t.astype(np.float64)
    return acc


def test_scale_selection_from_a_bound():
    rng = np.random.RandomState(0)
    bound = np.exp(rng.uniform(np.log(1e-20), np.log(1e20), 5000)).astype(np.float32)
    s, inv = scale_from_bits(bound)
    assert np.all(s * inv == 1.0) and np.all(np.log2(s) == np.round(np.log2(s)))
    scaled = bound.astype(np.float64) * s
    assert np.all(scaled < 2.0 ** 15) and np.all(scaled >= 2.0 ** 14)   # hi = fl16(s x) never overflows
    # every element below the bound, scaled, is representable without overflow and keeps 11 bits down to 2^-14
    x = bound * rng.uniform(-1, 1, bound.shape).astype(np.float32)
    hi = fl16(torch.from_numpy(x.astype(np.float64) * s)).numpy()
    assert np.all(np.isfinite(hi))


def test_per_product_bound():
    """|fl16(s_a a) fl16(s_b b) / (s_a s_b) - a b| <= (2u + u^2)|a||b| inside the normal fp16 range"""
    torch.manual_seed(3)
    a = torch.randn(400000, dtype=torch.float64) * torch.exp(torch.randn(400000, dtype=torch.float64) * 2)
    b = torch.randn(400000, dtype=torch.float64) * torch.exp(torch.randn(400000, dtype=torch.float64) * 2)
    s_a, _ = scale_from_bits([float(a.abs().max())])
    s_b, _ = scale_from_bits([float(b.abs().max())])
    sa, sb = a.float().double() * s_a[0], b.float().double() * s_b[0]     # fp32 operands, scaled exactly
    normal = (sa.abs() >= 2.0 ** -14) & (sb.abs() >= 2.0 ** -14)
    err = (fl16(sa) * fl16(sb) - sa * sb).abs()
    lim = (2 * U16 + U16 ** 2) * (sa * sb).abs()
    assert bool((err[normal] <= lim[normal]).all())
    worst = float((err[normal] / (sa * sb).abs()[normal]).max())
    assert worst > 1.5 * U16                                             # the bound is nearly attained: one product
    # outside the normal range the rounding error is absolute: at most 2^-25 per scaled element
    e_a = (fl16(sa) - sa).abs()
    assert float(e_a[sa.abs() < 2.0 ** -14].max()) <= 2.0 ** -25


def test_elementwise_gemm_bound_holds_and_is_not_loose():
    torch.manual_seed(4)
    M, K, N = 96, 512, 48
    A = (torch.randn(M, K) * (torch.rand(1, K) * 3 + 0.1)).double()
    A[::7, ::5] *= 1e-7                                                  # elements that become fp16 subnormals
    W = (torch.randn(N, K) / K ** 0.5).double()
    bound_a = float(A.abs().max()) * 3.0                                # a pessimistic bound, as the callers supply
    s_a, _ = scale_from_bits([bound_a])
    s_w, _ = scale_from_bits(W.abs().amax(1).float().numpy())           # per weight row = per output column
    ha = fl16(A.float().double() * s_a[0])
    hw = fl16(W.float().double() * torch.from_numpy(s_w)[:, None])
    C = truncating_fp32_matmul(ha.numpy(), hw.t().numpy()) / s_a[0] / s_w[None, :]
    ref = A @ W.t()
    bnd = gemm_bound(A, W.t(), s_a[0], s_w)
    err = (torch.from_numpy(C) - ref).abs()
    assert bool((err <= bnd).all()), float((err / bnd).max())
    # the 1-term result is clearly less accurate than the 3-term one (test_f16_split_cpu.py: < 2e-7 relative)
    rel = float((torch.from_numpy(C) - ref).norm() / ref.norm())
    assert 1e-5 < rel < 2.0 ** -10, rel
    # and the bound is within a small factor of the worst error actually seen (it is an error bound, not a guess)
    assert float((err / bnd).max()) > 1e-3


def test_bit_value_matches_the_header():
    import os
    import re
    from dual_dmp_b200 import functional as F_
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "include", "ddmp_b200.h")).read()
    m = re.search(r"#define DDMP_GEMM_F16X1 (0x[0-9a-fA-F]+|\d+)", text)
    assert m and int(m.group(1), 0) == F_.GEMM_F16X1
    for b in (0, 1, 2):                                                  # a modifier: clear of every backend value
        assert b & F_.GEMM_F16X1 == 0
    assert F_._with_precision(2, "f16x1") == 2 | F_.GEMM_F16X1 and F_._with_precision(2, "fp32") == 2


def test_precision_names_are_checked():
    import pytest
    from dual_dmp_b200 import functional as F_
    from dual_dmp_b200.step import set_dense_precision
    with pytest.raises(ValueError):
        F_.check_dense_precision("fp16")

    class Net:
        dense_precision = "fp32"
    a, b = Net(), Net()
    set_dense_precision((a, b), None)
    assert a.dense_precision == b.dense_precision == "fp32"
    set_dense_precision((a, b), "f16x1")
    assert a.dense_precision == b.dense_precision == "f16x1"
    with pytest.raises(ValueError):
        set_dense_precision((a,), "tf32")


def test_cli_flags():
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("fit_many", os.path.join(root, "scripts", "fit_many.py"))
    fm = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fm)
    assert fm.parse_args(["d"]).dense_precision == "fp32"
    assert fm.parse_args(["d", "--dense-precision", "f16x1"]).dense_precision == "f16x1"
