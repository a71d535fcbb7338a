"""A/B of the fp16-split NT kernels (X.W^T and dH.W) at the 1M-face shapes: ddmp_gemm_tc_flags settings given on the command
line (0 = the default configuration, 16 = staged epilogue instead of TMA stores, 32 = register-fed A operand everywhere;
default: 0 16), interleaved per shape in ONE process."""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dual_dmp_b200 import functional as F_
from dual_dmp_b200._lib import lib

dev = "cuda:0"
n = 1003520
settings = [int(a) for a in sys.argv[1:]] or [0, 16]
shapes = [(64, 128), (128, 256), (256, 256), (256, 512), (512, 512), (512, 256), (256, 128), (128, 64)]
weight = {(256, 256): 2}
tot = {s: 0.0 for s in settings}
flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)
for cin, cout in shapes:
    X = torch.randn(n, cin, device=dev); W = torch.randn(cout, cin, device=dev) / cin ** 0.5
    dH = torch.randn(n, cout, device=dev)
    sc = torch.rand(cin, device=dev) + 0.5; sh = torch.randn(cin, device=dev)
    bx = (torch.nn.functional.leaky_relu(X[:65536] * sc + sh, 0.01).abs().amax(0) * 1.5).contiguous()
    bd = dH[:65536].abs().amax(0).mul(1.5).contiguous()
    H = torch.empty(n, cout, device=dev); G = torch.empty(n, cin, device=dev)
    for name, fn in (("xw", lambda: F_.gemm_xw(X, W, scale=sc, shift=sh, backend=2, amax=bx, out=H)),
                     ("dx", lambda: F_.gemm_dx(dH, W, backend=2, amax=bd, out=G))):
        line = f"{name} {cin:4d}->{cout:4d}"
        for s in settings:
            lib.query("ddmp_gemm_tc_flags", s)
            fn(); torch.cuda.synchronize()
            ms = 0.0
            for _ in range(5):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(); e1.record(); torch.cuda.synchronize()
                ms += e0.elapsed_time(e1) / 5
            tot[s] += ms * weight.get((cin, cout), 1)
            line += f" | flags={s:2d} {ms:7.3f} ms {2.0 * n * cin * cout / ms / 1e9:6.1f} TF"
        print(line, flush=True)
    del X, dH, H, G
for s in settings:
    print(f"flags {s}: {tot[s]:.3f} ms for the 18 NT launches of one 1M-row net pass (x1.5 per step)")
lib.query("ddmp_gemm_tc_flags", 0)
