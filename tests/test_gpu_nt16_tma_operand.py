"""The fp16-split NT kernels (X.W^T, dH.W) feed their A operand by TMA at K <= 256, and at K = 512 when the BatchNorm +
LeakyReLU prologue is fused: raw fp32 tiles stream into a shared-memory ring and the producer warps transform shared ->
shared.  ddmp_gemm_tc_flags(32) keeps the register-fed producers everywhere.  Same arithmetic, same layout, same MMA
order: the two must give IDENTICAL results."""
import os
import subprocess
import sys

import pytest
import torch

from tests.helpers import rel_err

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _inputs(n, K, N, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    X = torch.randn(n, K, device=DEV, generator=g) * (torch.rand(1, K, device=DEV, generator=g) * 3 + 0.1)
    W = torch.randn(N, K, device=DEV, generator=g) / K ** 0.5
    W[1] *= 1e-5
    sc = torch.rand(K, device=DEV, generator=g) + 0.5
    sh = torch.randn(K, device=DEV, generator=g)
    return X, W, sc, sh


def _run_both(fn, n, width):
    """fn(out) under flags 32 and 0, each into a view of a poisoned, over-long buffer"""
    from dual_dmp_b200._lib import lib
    prev = lib.query("ddmp_gemm_tc_flags", -1)
    res = {}
    try:
        for fl in (32, 0):
            lib.query("ddmp_gemm_tc_flags", fl)
            buf = torch.full((n + 300, width), 7.0, device=DEV)
            fn(buf[:n])
            torch.cuda.synchronize()
            assert (buf[n:] == 7.0).all(), f"flags={fl}: a store landed past row {n}"
            res[fl] = buf[:n].clone()
            del buf
    finally:
        lib.query("ddmp_gemm_tc_flags", prev)
    return res


@pytest.mark.parametrize("K", [64, 128, 256, 512])
@pytest.mark.parametrize("N", [64, 128, 256, 512])
@pytest.mark.parametrize("n", [37, 640, 4099, 77777, 1003520])
def test_tma_operand_equals_register_operand(K, N, n):
    """xw with and without the BatchNorm + LeakyReLU prologue (reduction over K = Cin) and dx (reduction over
    K = Cout) on every K x N: row counts below one tile, not a multiple of 32, and many tiles per CTA."""
    from dual_dmp_b200 import functional as F_
    X, W, sc, sh = _inputs(n, K, N, seed=K * 7 + N * 13 + n)
    b_act = (torch.nn.functional.leaky_relu(X * sc + sh, 0.01).abs().amax(0) * 1.5).contiguous()
    b_x = X.abs().amax(0).contiguous()
    # dx: dH [n, K] . Wd [K, N], Wd = W^T
    dH = X * 1e-3
    Wd = W.t().contiguous()
    b_dh = dH.abs().amax(0).contiguous()
    cases = {
        "xw_act": (lambda out: F_.gemm_xw(X, W, scale=sc, shift=sh, backend=2, amax=b_act, out=out), N),
        "xw": (lambda out: F_.gemm_xw(X, W, backend=2, amax=b_x, out=out), N),
        "dx": (lambda out: F_.gemm_dx(dH, Wd, backend=2, amax=b_dh, out=out), N),
    }
    for name, (fn, width) in cases.items():
        res = _run_both(fn, n, width)
        assert torch.equal(res[0], res[32]), f"{name}: TMA-fed and register-fed results differ"
        if n <= 4099:
            if name == "xw_act":
                ref = torch.nn.functional.leaky_relu(X.double() * sc.double() + sh.double(), 0.01) @ W.double().t()
            elif name == "xw":
                ref = X.double() @ W.double().t()
            else:
                ref = dH.double() @ Wd.double()
            assert rel_err(res[0], ref) < 5e-6, name
        del res


_PROBE = r"""
import sys, torch
sys.path.insert(0, sys.argv[1])
from dual_dmp_b200 import functional as F_
from dual_dmp_b200._lib import lib
dev = "cuda:0"
n = 1000
def call(K, N, row_map=None, flags=0, act=False):
    lib.query("ddmp_gemm_tc_flags", flags)
    X = torch.randn(n, K, device=dev); W = torch.randn(N, K, device=dev)
    sc, sh = (torch.rand(K, device=dev) + 0.5, torch.randn(K, device=dev)) if act else (None, None)
    F_.gemm_xw(X, W, row_map=row_map, scale=sc, shift=sh, backend=2, amax=(X.abs().amax(0) * 2 + 3).contiguous())
    torch.cuda.synchronize()
    print(f"probe K={K} N={N} map={row_map is not None} flags={flags} act={act}", file=sys.stderr, flush=True)
call(64, 128); call(256, 256); call(256, 64)
call(512, 256, act=True); call(512, 128, act=True)
call(512, 256); call(512, 128)
call(128, 256, row_map=torch.randperm(n, device=dev).int())
call(512, 256, row_map=torch.randperm(n, device=dev).int(), act=True)
call(128, 128, flags=32); call(512, 256, flags=32, act=True)
"""


def test_register_operand_where_tma_does_not_pay():
    """The TMA-fed configuration serves K <= 256, and K = 512 with the BatchNorm + LeakyReLU prologue, without a row
    gather; K = 512 without the prologue, the fused row gather (a_map) and flags bit 5 keep the register-fed
    producers.  Read from the kernels' cycle-trace lines (DDMP_TC_TRACE=1)."""
    env = dict(os.environ, DDMP_TC_TRACE="1")
    env.pop("DDMP_TC_F16_FLAGS", None)
    p = subprocess.run([sys.executable, "-c", _PROBE, ROOT], env=env, capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr
    lines = p.stderr.splitlines()
    kinds = []
    for i, ln in enumerate(lines):
        if ln.startswith("probe"):
            tr = [l for l in lines[:i] if l.startswith("[ddmp trace]")]
            assert tr, ln
            kinds.append(tr[-1].split(" A=")[1].split()[0])
    assert kinds == ["tma", "tma", "tma", "tma", "tma", "registers", "registers", "registers", "registers", "registers",
                     "registers"], (kinds, p.stderr)
