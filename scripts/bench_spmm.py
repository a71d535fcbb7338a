"""Micro-benchmark of the GCN aggregation kernels on the 1M-face graphs (both flavours, every width).
usage: bench_spmm.py [setting ...]   setting = 0: the default kernels, 1: the reference gather kernel
(ddmp_spmm_reference_kernel, include/ddmp_b200.h); default: both.  All settings are measured in ONE process on the same
graphs, interleaved per shape."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from dual_dmp_b200 import functional as F_, synth
from dual_dmp_b200._lib import lib
from dual_dmp_b200.graph import GcnGraph
from dual_dmp_b200.util.mesh import Mesh
dev = "cuda:0"
settings = [int(a) for a in sys.argv[1:]] or [0, 1]
vs, faces = synth.icosphere(224)
m = Mesh(vs=vs * 100, faces=faces)
F, V = len(faces), len(vs)
fg = GcnGraph(torch.from_numpy(m.f_edges), F, dev, coords=torch.from_numpy(m.fc))
e = torch.from_numpy(m.edges.T.astype("int64")); vg = GcnGraph(torch.cat([e, e[[1, 0]]], dim=1), V, dev, coords=torch.from_numpy(m.vs))
flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)          # 256 MB > L2
tot_b = {s: 0.0 for s in settings}; tot_t = {s: 0.0 for s in settings}
for name, g in (("vertex", vg), ("face", fg)):
    for C in (32, 64, 128, 256, 512):
        H = torch.randn(g.n, C, device=dev); b = torch.randn(C, device=dev)
        byt = 4 * ((g.n + 1) + 2 * g.nnz + 2 * g.n * C)
        for flav, fn in (("fwd(stats+bias)", lambda: F_.spmm_gcn(g, H, bias=b, stats=True)), ("bwd(plain)", lambda: F_.spmm_gcn(g, H, amax=True))):
            line = f"{name:6s} C={C:3d} {flav:16s}"
            for s in settings:
                lib.query("ddmp_spmm_reference_kernel", s)
                fn(); torch.cuda.synchronize()
                ms = 0.0
                for _ in range(5):
                    flush.zero_()
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
                    ms += e0.elapsed_time(e1) / 5
                w = 2 if C == 256 else 1          # a step has twice as many 256-wide launches
                tot_b[s] += byt * w; tot_t[s] += ms * w
                line += f" | s={s:2d} {ms:7.3f} ms {byt / ms / 1e6:6.0f} GB/s"
            print(line, flush=True)
        del H
for s in settings:
    print(f"setting {s}: step-weighted {tot_b[s] / tot_t[s] / 1e6:.0f} GB/s, {2 * tot_t[s]:.2f} ms per step (48 launches)")
lib.query("ddmp_spmm_reference_kernel", 0)
