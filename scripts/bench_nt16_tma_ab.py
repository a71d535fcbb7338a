"""A/B of the two pipeline configurations of the fp16-split NT kernels (X.W^T and dH.W) at the 1M-face shapes.

  ab     [--flags F ...] [--reps R]   ddmp_gemm_tc_flags settings interleaved per shape and per repetition in ONE process
                                     (0 = the selection of run_nt16, 16 = staged epilogue instead of TMA stores, 32 =
                                     register-fed A operand everywhere; default: 32 0); the L2 is overwritten before
                                     every timed call; median ms, and the share of the shape's floor
  trace  [--flags F]                 DDMP_TC_TRACE=1 cycle counters of CTA 0, one line per shape (stderr of the library)

The floor of a call is the larger of its HBM bytes (A read + C written) / 6.55 TB/s (measured copy peak of the B200)
and its fp32-equivalent FLOPs / 459 TFLOP/s (a third of the sustained bf16 rate: three fp16 MMAs per product)."""
import argparse, os, statistics, sys

ap = argparse.ArgumentParser()
ap.add_argument("mode", choices=("ab", "trace"))
ap.add_argument("--flags", type=int, nargs="+", default=None)
ap.add_argument("--reps", type=int, default=9)
ap.add_argument("--rows", type=int, default=1003520)
args = ap.parse_args()
if args.mode == "trace":
    os.environ["DDMP_TC_TRACE"] = "1"              # read once by the library, before its first GEMM
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dual_dmp_b200 import functional as F_
from dual_dmp_b200._lib import lib

assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
dev = "cuda:0"
n = args.rows
settings = args.flags or ([32, 0] if args.mode == "ab" else [0])
# (Cin, Cout) of the transforms of one net pass: xw reduces over Cin, dx over Cout
shapes = [(64, 128), (128, 256), (256, 256), (256, 512), (512, 512), (512, 256), (256, 128), (128, 64)]
HBM, MMA = 6.55e12, 459e12


def floor_ms(K, N):
    return max(n * (K + N) * 4 / HBM, 2.0 * n * K * N / MMA) * 1e3


flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)
print(f"{torch.cuda.get_device_name(0)}, rows={n}, settings={settings}, reps={args.reps}", flush=True)
for cin, cout in shapes:
    X = torch.randn(n, cin, device=dev); W = torch.randn(cout, cin, device=dev) / cin ** 0.5
    dH = torch.randn(n, cout, device=dev)
    sc = torch.rand(cin, device=dev) + 0.5; sh = torch.randn(cin, device=dev)
    bx = (torch.nn.functional.leaky_relu(X[:65536] * sc + sh, 0.01).abs().amax(0) * 1.5).contiguous()
    bd = dH[:65536].abs().amax(0).mul(1.5).contiguous()
    H = torch.empty(n, cout, device=dev); G = torch.empty(n, cin, device=dev)
    calls = (("xw", cin, cout, lambda: F_.gemm_xw(X, W, scale=sc, shift=sh, backend=2, amax=bx, out=H)),
             ("dx", cout, cin, lambda: F_.gemm_dx(dH, W, backend=2, amax=bd, out=G)))
    for name, K, N, fn in calls:
        line = f"{name} {cin:4d}->{cout:4d} K={K:3d} N={N:3d} floor {floor_ms(K, N):.3f} ms"
        if args.mode == "trace":
            for s in settings:
                lib.query("ddmp_gemm_tc_flags", s)
                fn(); torch.cuda.synchronize()           # warm-up (also dumps a trace line)
                print(f"{line} flags={s}", flush=True)
                sys.stdout.flush()
                fn(); torch.cuda.synchronize()
            continue
        times = {s: [] for s in settings}
        for s in settings:
            lib.query("ddmp_gemm_tc_flags", s)
            fn()
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for s in settings:
                lib.query("ddmp_gemm_tc_flags", s)
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); fn(); e1.record(); torch.cuda.synchronize()
                times[s].append(e0.elapsed_time(e1))
        for s in settings:
            med = statistics.median(times[s])
            line += (f" | flags={s:2d} {med:7.3f} ms (min {min(times[s]):.3f} max {max(times[s]):.3f})"
                     f" {100 * floor_ms(K, N) / med:5.1f}% of floor")
        if len(settings) == 2:
            a, b = (statistics.median(times[s]) for s in settings)
            line += f" | flags={settings[1]} vs {settings[0]}: {100 * (a - b) / a:+.1f}% faster"
        print(line, flush=True)
    del X, dH, H, G
lib.query("ddmp_gemm_tc_flags", 0)
