"""torch.autograd.Function layer over the C ABI (libddmp_b200).  Host glue only: every FLOP runs in the library's
hand-written sm_100a kernels; PyTorch provides device memory, streams and the autograd graph.

``GcnNetFunction`` runs a whole network (12 x [X.W^T -> A_hat aggregate + bias -> BatchNorm -> LeakyReLU] + head)
as ONE autograd node with a hand-written backward, so only the pre-BatchNorm tensor of each layer is saved; the
activated tensors are recomputed on load by the consumers (SURVEY.md §7 hard part 2).
"""
from __future__ import annotations

import torch

from ._lib import lib, ptr, require_cuda, set_device, stream_ptr
from .graph import GcnGraph

SLOPE = 0.01        # nn.LeakyReLU() default (reference util/networks.py:44,105)
BN_EPS = 1e-5
BN_MOMENTUM = 0.1
GEMM_BACKEND = 0    # DDMP_GEMM_AUTO; tests may set 1 (FFMA) / 2 (tcgen05)
# accuracy contract of the dense transforms, chosen per call / per network (include/ddmp_b200.h DDMP_GEMM_F16X1):
# "fp32" = the fp16-split tensor-core kernels emulate fp32 with three products (default); "f16x1" = one fp16 product
GEMM_F16X1 = 0x10   # DDMP_GEMM_F16X1, OR-ed into the backend argument
DENSE_PRECISIONS = ("fp32", "f16x1")

HEAD_POS, HEAD_NORM = 0, 1


def _f32(t, what):
    return require_cuda(t, torch.float32, what)


# ---------------------------------------------------------------------------------------------------------------------
# thin op wrappers (used by the autograd functions and, one by one, by the parity tests)
# ---------------------------------------------------------------------------------------------------------------------
def num_row_blocks(n: int, C: int) -> int:
    return int(lib.query("ddmp_num_row_blocks", n, C))


AMAX_WIDTHS = (64, 128, 256, 512)      # widths whose aggregation kernel has the amax epilogue and feed tensor-core GEMMs


def num_elem_blocks(n: int, C: int) -> int:
    """row blocks of the element-wise kernels (BatchNorm backward reduce / apply, column sums)"""
    return int(lib.query("ddmp_num_elem_blocks", n, C))


def spmm_gcn(graph: GcnGraph, H, bias=None, stats=False, transposed=False, out=None, n_rows=None, amax=False):
    """n_rows < H.shape[0] in the partitioned mode: H = [owned | halo] rows, only the owned rows are computed.
    ``amax``: also return the per-row-block maxima of |Y| (operand bound of the fp16-split GEMMs)"""
    n, C = H.shape
    if n_rows is not None:
        n = n_rows
    rowptr, col, w = (graph.rowptr_t, graph.col_t, graph.w_t) if transposed else (graph.rowptr, graph.col, graph.w)
    Y = out if out is not None else torch.empty(n, C, dtype=torch.float32, device=H.device)
    partials = torch.empty(num_row_blocks(n, C), 2, C, dtype=torch.float32, device=H.device) if stats else None
    ab = torch.empty(int(lib.query("ddmp_spmm_amax_len", n, C)), dtype=torch.float32, device=H.device) if amax else None
    lib.call("ddmp_spmm_gcn", ptr(rowptr), ptr(col), ptr(w), ptr(H), ptr(bias), ptr(Y), ptr(partials), ptr(ab), n, C,
             stream_ptr(H.device))
    if amax:
        return (Y, partials, ab) if stats else (Y, ab)
    return (Y, partials) if stats else Y


def check_dense_precision(dense_precision: str) -> str:
    if dense_precision not in DENSE_PRECISIONS:
        raise ValueError(f"dense_precision must be one of {DENSE_PRECISIONS}, got {dense_precision!r}")
    return dense_precision


def _with_precision(backend: int, dense_precision: str) -> int:
    return backend | GEMM_F16X1 if check_dense_precision(dense_precision) == "f16x1" else backend


def _gemm_ws(n, Cin, Cout, device, backend):
    if backend == 1:
        return None, 0
    nbytes = int(lib.query("ddmp_gemm_workspace_bytes", n, Cin, Cout))
    if nbytes == 0:
        return None, 0
    return torch.empty(nbytes // 4, dtype=torch.float32, device=device), nbytes


def gemm_xw(X, W, row_map=None, scale=None, shift=None, out=None, n=None, backend=None, amax=None,
            dense_precision="fp32"):
    """``amax``: optional device tensor whose largest magnitude bounds |act(X)| -> fp16-split tensor-core kernel.
    ``dense_precision="f16x1"``: that kernel runs with one fp16 product instead of three (no effect elsewhere)"""
    n = X.shape[0] if n is None else n
    Cout, Cin = W.shape
    H = out if out is not None else torch.empty(n, Cout, dtype=torch.float32, device=X.device)
    backend = GEMM_BACKEND if backend is None else backend
    ws, ws_bytes = _gemm_ws(n, Cin, Cout, X.device, backend)
    lib.call("ddmp_gemm_xw", ptr(X), ptr(row_map), ptr(scale), ptr(shift), SLOPE, ptr(W), ptr(H), ptr(ws), ws_bytes,
             n, Cin, Cout, ptr(amax), 0 if amax is None else amax.numel(), _with_precision(backend, dense_precision),
             stream_ptr(X.device))
    return H


def gemm_dx(dH, W, out=None, backend=None, amax=None, dense_precision="fp32"):
    n = dH.shape[0]
    Cout, Cin = W.shape
    gX = out if out is not None else torch.empty(n, Cin, dtype=torch.float32, device=dH.device)
    backend = GEMM_BACKEND if backend is None else backend
    ws, ws_bytes = _gemm_ws(n, Cin, Cout, dH.device, backend)
    lib.call("ddmp_gemm_dx", ptr(dH), ptr(W), ptr(gX), ptr(ws), ws_bytes, n, Cin, Cout, ptr(amax),
             0 if amax is None else amax.numel(), _with_precision(backend, dense_precision), stream_ptr(dH.device))
    return gX


def gemm_dw(dH, X, Cin, row_map=None, scale=None, shift=None, backend=None, amax_dh=None, amax_x=None,
            dense_precision="fp32"):
    n, Cout = dH.shape
    dW = torch.empty(Cout, Cin, dtype=torch.float32, device=dH.device)
    ws_bytes = int(lib.query("ddmp_gemm_dw_workspace_bytes", n, Cin, Cout))
    ws = torch.empty(max(ws_bytes, 16) // 4, dtype=torch.float32, device=dH.device)
    lib.call("ddmp_gemm_dw", ptr(dH), ptr(X), ptr(row_map), ptr(scale), ptr(shift), SLOPE, ptr(dW), ptr(ws),
             ws_bytes, n, Cin, Cout, ptr(amax_dh), 0 if amax_dh is None else amax_dh.numel(), ptr(amax_x),
             0 if amax_x is None else amax_x.numel(),
             _with_precision(GEMM_BACKEND if backend is None else backend, dense_precision), stream_ptr(dH.device))
    return dW


def partials_to_sums(partials):
    """[nblk, sets, C] row-block partials -> [sets, C] (fixed order, float64 accumulate)"""
    nblk, sets, C = partials.shape
    out = torch.empty(sets, C, dtype=torch.float32, device=partials.device)
    lib.call("ddmp_colsum_finalize", ptr(partials), nblk, sets, C, ptr(out), stream_ptr(partials.device))
    return out


def colsum(X):
    n, C = X.shape
    nblk = num_elem_blocks(n, C)
    partials = torch.empty(nblk, 1, C, dtype=torch.float32, device=X.device)
    out = torch.empty(C, dtype=torch.float32, device=X.device)
    st = stream_ptr(X.device)
    lib.call("ddmp_colsum_partials", ptr(X), ptr(partials), n, C, st)
    lib.call("ddmp_colsum_finalize", ptr(partials), nblk, 1, C, ptr(out), st)
    return out


def bn_stats_finalize(partials, n, gamma, beta, running_mean=None, running_var=None):
    nblk, _, C = partials.shape
    stats = torch.empty(5, C, dtype=torch.float32, device=partials.device)   # mean, rstd, scale, shift, bound
    lib.call("ddmp_bn_stats_finalize", ptr(partials), nblk, n, C, ptr(gamma), ptr(beta), BN_EPS, BN_MOMENTUM,
             ptr(running_mean), ptr(running_var), ptr(stats[0]), ptr(stats[1]), ptr(stats[2]), ptr(stats[3]),
             ptr(stats[4]), stream_ptr(partials.device))
    return stats


def bn_rank_sums(partials, n):
    """partitioned mode: this rank's per-channel (sum y, sum y^2) in float64 [2, C] from the aggregation partials"""
    nblk, _, C = partials.shape
    sums = torch.empty(2, C, dtype=torch.float64, device=partials.device)
    lib.call("ddmp_bn_stats_rank_sums", ptr(partials), nblk, n, C, ptr(sums), stream_ptr(partials.device))
    return sums


def bn_stats_finalize_sums(sums, n, gamma, beta, running_mean=None, running_var=None):
    """batch statistics from (all-reduced) float64 sums [2, C] and the global row count"""
    C = sums.shape[1]
    stats = torch.empty(5, C, dtype=torch.float32, device=sums.device)
    lib.call("ddmp_bn_stats_finalize_sums", ptr(sums), n, C, ptr(gamma), ptr(beta), BN_EPS, BN_MOMENTUM,
             ptr(running_mean), ptr(running_var), ptr(stats[0]), ptr(stats[1]), ptr(stats[2]), ptr(stats[3]),
             ptr(stats[4]), stream_ptr(sums.device))
    return stats


def bn_stats_finalize_peer(partials, n_local, comm, gamma, beta, running_mean=None, running_var=None):
    """partitioned mode: rank reduction + one-shot all-reduce over NVLink peer memory + BatchNorm table, one kernel"""
    nblk, _, C = partials.shape
    stats = torch.empty(5, C, dtype=torch.float32, device=partials.device)
    peer = comm.peer
    lib.call("ddmp_bn_stats_finalize_peer", ptr(partials), nblk, n_local, C, peer.ptrs, peer.rank, peer.world,
             peer.next_seq(), comm.n_global, ptr(gamma), ptr(beta), BN_EPS, BN_MOMENTUM, ptr(running_mean),
             ptr(running_var), ptr(stats[0]), ptr(stats[1]), ptr(stats[2]), ptr(stats[3]), ptr(stats[4]),
             stream_ptr(partials.device))
    return stats


def act_bound(stats):
    """per-channel upper bound of |lrelu(scale*Y+shift)| (training-mode batch statistics only), else None"""
    return stats[4] if stats.shape[0] > 4 else None


def bn_lrelu_backward(gX, Y, stats, dY_out=None, comm=None):
    """gX = dL/d lrelu(bn(Y))  ->  (dY, dgamma, dbeta, dbias).  ``comm`` (partitioned mode): the two column sums
    are all-reduced over the ranks before they are used; dbias stays a per-rank partial (all-reduced with the
    weight gradients)."""
    n, C = Y.shape
    dev = Y.device
    st = stream_ptr(dev)
    nblk = num_elem_blocks(n, C)
    partials = torch.empty(nblk, 2, C, dtype=torch.float32, device=dev)
    small = torch.empty(5, C, dtype=torch.float32, device=dev)             # dgamma, dbeta, c1, c2, dbias
    mean, rstd, scale, shift = stats[0], stats[1], stats[2], stats[3]
    lib.call("ddmp_bn_bwd_reduce", ptr(gX), ptr(Y), ptr(mean), ptr(rstd), ptr(scale), ptr(shift), SLOPE,
             ptr(partials), n, C, st)
    if comm is None:
        lib.call("ddmp_bn_bwd_finalize", ptr(partials), nblk, n, C, ptr(small[0]), ptr(small[1]), ptr(small[2]),
                 ptr(small[3]), st)
    elif getattr(comm, "peer", None) is not None:
        peer = comm.peer
        lib.call("ddmp_bn_bwd_finalize_peer", ptr(partials), nblk, C, peer.ptrs, peer.rank, peer.world, peer.next_seq(),
                 comm.n_global, ptr(small[0]), ptr(small[1]), ptr(small[2]), ptr(small[3]), st)
    else:
        sums = comm.allreduce_(partials_to_sums(partials))
        lib.call("ddmp_bn_bwd_finalize", ptr(sums), 1, comm.n_global, C, ptr(small[0]), ptr(small[1]), ptr(small[2]),
                 ptr(small[3]), st)
    dY = dY_out if dY_out is not None else torch.empty_like(Y)
    lib.call("ddmp_bn_bwd_apply", ptr(gX), ptr(Y), ptr(mean), ptr(rstd), ptr(scale), ptr(shift), SLOPE,
             ptr(small[2]), ptr(small[3]), ptr(dY), ptr(partials), n, C, st)
    lib.call("ddmp_colsum_finalize", ptr(partials), nblk, 1, C, ptr(small[4]), st)
    return dY, small[0], small[1], small[4]


bn_bwd_spmm_tile = None     # never called: bench.py's per-phase timer patches this name; goes with that line of bench.py


# ---------------------------------------------------------------------------------------------------------------------
# operator-level GCNConv  (drop-in for torch_geometric.nn.GCNConv.forward, reference util/networks.py:15-26)
# ---------------------------------------------------------------------------------------------------------------------
class GCNConvFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, graph: GcnGraph):
        set_device(x.device)
        x, weight = _f32(x, "GCNConv x"), _f32(weight, "GCNConv weight")
        if graph.perm is not None:
            raise RuntimeError("operator-level GCNConv expects a graph built with reorder=False")
        H = gemm_xw(x, weight)
        Y = spmm_gcn(graph, H, bias=None if bias is None else _f32(bias, "GCNConv bias"))
        ctx.save_for_backward(x, weight)
        ctx.graph, ctx.has_bias = graph, bias is not None
        return Y

    @staticmethod
    def backward(ctx, gY):
        x, weight = ctx.saved_tensors
        set_device(gY.device)
        gY = _f32(gY, "GCNConv grad")
        dH = spmm_gcn(ctx.graph, gY, transposed=True)
        gx = gemm_dx(dH, weight) if ctx.needs_input_grad[0] else None
        gW = gemm_dw(dH, x, weight.shape[1]) if ctx.needs_input_grad[1] else None
        gb = colsum(gY) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return gx, gW, gb, None


# ---------------------------------------------------------------------------------------------------------------------
# whole network: 12 GCN layers + head
# ---------------------------------------------------------------------------------------------------------------------
class GcnNetFunction(torch.autograd.Function):
    """forward(graph, kind, training, bn_buffers, taps, x_in, x_pos, *params[, dense_precision])

    params = [W_1, b_1, gamma_1, beta_1, ..., W_12, b_12, gamma_12, beta_12, W_lin1, b_lin1, W_lin2, b_lin2]
    dense_precision: optional trailing string, "fp32" (default) or "f16x1"; passed to every trunk GEMM of the forward
    and the backward (the layers whose fp16-split tensor-core kernels it affects: DDMP_GEMM_F16X1).
    bn_buffers = [(running_mean_l, running_var_l)] updated in place (training) or read (eval).
    taps: optional list that receives (Y_l, stats_l) per layer, then (h_head, None), for the per-layer parity tests.
    """

    @staticmethod
    def forward(ctx, graph: GcnGraph, kind: int, training: bool, bn_buffers, taps, x_in, x_pos, *params):
        dev = x_in.device
        set_device(dev)
        ctx.has_precision = bool(params) and isinstance(params[-1], str)
        dense = check_dense_precision(params[-1]) if ctx.has_precision else "fp32"
        if ctx.has_precision:
            params = params[:-1]
        n = graph.n
        x_in = _f32(x_in, "net input")
        L = (len(params) - 4) // 4
        Ws = [_f32(params[4 * i], "conv weight") for i in range(L)]
        bs = [_f32(params[4 * i + 1], "conv bias") for i in range(L)]
        gammas = [_f32(params[4 * i + 2], "bn weight") for i in range(L)]
        betas = [_f32(params[4 * i + 3], "bn bias") for i in range(L)]
        W1, b1, W2, b2 = (_f32(p, "head parameter") for p in params[4 * L:])
        if x_in.shape != (n, Ws[0].shape[1]):
            raise RuntimeError(f"net input has shape {tuple(x_in.shape)}, expected {(n, Ws[0].shape[1])}")
        cmax = max(w.shape[0] for w in Ws)
        comm = graph if hasattr(graph, "exchange") else None        # partitioned mode (dual_dmp_b200.partition)
        n_ext = graph.n_ext if comm is not None else n
        Hbuf = torch.empty(n_ext * cmax, dtype=torch.float32, device=dev)
        Ys, stats = [], []
        for l in range(L):
            cout = Ws[l].shape[0]
            H = Hbuf[: n_ext * cout].view(n_ext, cout)               # [owned | halo] rows
            if l == 0:
                gemm_xw(x_in, Ws[0], row_map=graph.perm, out=H, n=n, dense_precision=dense)
            else:
                gemm_xw(Ys[l - 1], Ws[l], scale=stats[l - 1][2], shift=stats[l - 1][3], out=H,
                        amax=act_bound(stats[l - 1]), dense_precision=dense)
            if comm is not None:
                comm.exchange(H)
            if training:
                Y, partials = spmm_gcn(graph, H, bias=bs[l], stats=True, n_rows=n)
                rm, rv = bn_buffers[l]
                if comm is None:
                    st = bn_stats_finalize(partials, n, gammas[l], betas[l], rm, rv)
                elif getattr(comm, "peer", None) is not None:
                    st = bn_stats_finalize_peer(partials, n, comm, gammas[l], betas[l], rm, rv)
                else:
                    sums = comm.allreduce_(bn_rank_sums(partials, n))          # float64 (sum y, sum y^2)
                    st = bn_stats_finalize_sums(sums, comm.n_global, gammas[l], betas[l], rm, rv)
            else:
                Y = spmm_gcn(graph, H, bias=bs[l], n_rows=n)
                rm, rv = bn_buffers[l]
                st = torch.empty(4, cout, dtype=torch.float32, device=dev)      # mean, rstd, scale, shift (no bound)
                lib.call("ddmp_bn_eval_stats", ptr(rm), ptr(rv), ptr(gammas[l]), ptr(betas[l]), BN_EPS, cout, ptr(st[0]),
                         ptr(st[1]), ptr(st[2]), ptr(st[3]), stream_ptr(dev))
            Ys.append(Y)
            stats.append(st)
            if taps is not None:
                taps.append((Y, st))
        out = torch.empty(n, 3, dtype=torch.float32, device=dev)
        h_save = torch.empty(n, 16, dtype=torch.float32, device=dev)
        t_save = torch.empty(n, 4, dtype=torch.float32, device=dev) if kind == HEAD_NORM else None
        xp = _f32(x_pos, "x_pos") if kind == HEAD_POS else None
        lib.call("ddmp_head_fwd", kind, ptr(Ys[-1]), ptr(stats[-1][2]), ptr(stats[-1][3]), SLOPE, ptr(W1), ptr(b1),
                 ptr(W2), ptr(b2), ptr(graph.perm), ptr(xp), ptr(out), ptr(h_save), ptr(t_save), n, stream_ptr(dev))
        if taps is not None:
            taps.append((h_save, None))           # head: post-LeakyReLU hidden layer (its sign = active set)
        ctx.save_for_backward(x_in, *Ws, W1, W2)
        ctx.graph, ctx.kind, ctx.L = graph, kind, L
        ctx.Ys, ctx.stats, ctx.h_save, ctx.t_save = Ys, stats, h_save, t_save
        ctx.training = training
        ctx.dense_precision = dense
        return out

    @staticmethod
    def backward(ctx, g_out):
        if not ctx.training:
            raise RuntimeError("backward through eval-mode BatchNorm is not part of the Dual-DMP hot path")
        saved = ctx.saved_tensors
        x_in, Ws, W1, W2 = saved[0], saved[1:1 + ctx.L], saved[-2], saved[-1]
        graph, L, kind, dense = ctx.graph, ctx.L, ctx.kind, ctx.dense_precision
        Ys, stats = ctx.Ys, ctx.stats
        dev = g_out.device
        set_device(dev)
        st = stream_ptr(dev)
        n = graph.n
        g_out = _f32(g_out, "net output gradient")
        cmax = max(w.shape[0] for w in Ws)
        # ---- head ----
        go = torch.empty(n, 4, dtype=torch.float32, device=dev)
        gh = torch.empty(n, 16, dtype=torch.float32, device=dev)
        comm = graph if hasattr(graph, "exchange") else None
        n_ext = graph.n_ext if comm is not None else n
        bufA = torch.empty(n * cmax, dtype=torch.float32, device=dev)      # gX (grad wrt activated layer output)
        bufB = torch.empty(n_ext * cmax, dtype=torch.float32, device=dev)  # dY ([owned | halo])
        bufC = torch.empty(n * cmax, dtype=torch.float32, device=dev)      # dH
        gX = bufA[: n * 32].view(n, 32)
        lib.call("ddmp_head_bwd", kind, ptr(g_out), ptr(graph.perm), ptr(W1), ptr(W2), ptr(ctx.h_save),
                 ptr(ctx.t_save), SLOPE, ptr(go), ptr(gh), ptr(gX), n, st)
        sL = stats[L - 1]
        gW_lin1 = gemm_dw(gh, Ys[L - 1], 32, scale=sL[2], shift=sL[3])
        gb_lin1 = colsum(gh)
        gW_lin2 = gemm_dw(go, ctx.h_save, 16)[:3].contiguous()
        gb_lin2 = colsum(go)[:3].contiguous()
        # ---- trunk, last layer first ----
        grads = [None] * (4 * L)
        for l in range(L - 1, -1, -1):
            cout, cin = Ws[l].shape
            dH = bufC[: n * cout].view(n, cout)
            dY = bufB[: n_ext * cout].view(n_ext, cout)
            _, dgamma, dbeta, dbias = bn_lrelu_backward(gX, Ys[l], stats[l], dY_out=dY, comm=comm)
            if comm is not None:
                comm.exchange(dY)                   # A_hat symmetric: the backward needs dY of the halo rows
            dh_max = None                           # row-block maxima of |dH| when the aggregation kernel provides them
            if cout in AMAX_WIDTHS and l > 0:
                _, dh_max = spmm_gcn(graph, dY, transposed=True, out=dH, n_rows=n, amax=True)
            else:
                spmm_gcn(graph, dY, transposed=True, out=dH, n_rows=n)
            if l == 0:
                gW = gemm_dw(dH, x_in, cin, row_map=graph.perm, dense_precision=dense)
            else:
                gW = gemm_dw(dH, Ys[l - 1], cin, scale=stats[l - 1][2], shift=stats[l - 1][3], amax_dh=dh_max,
                             amax_x=act_bound(stats[l - 1]) if dh_max is not None else None, dense_precision=dense)
                gX = bufA[: n * cin].view(n, cin)
                gemm_dx(dH, Ws[l], out=gX, amax=dh_max, dense_precision=dense)
            grads[4 * l: 4 * l + 4] = [gW, dbias, dgamma, dbeta]
        g_xpos = g_out if (kind == HEAD_POS and ctx.needs_input_grad[6]) else None
        ctx.Ys = ctx.stats = ctx.h_save = ctx.t_save = None
        all_grads = [*grads, gW_lin1, gb_lin1, gW_lin2, gb_lin2]
        if comm is not None:
            # weight / bias gradients are sums over rows: one all-reduce of the flattened per-rank partials
            # (dgamma / dbeta were already reduced inside the layer loop and are identical on every rank)
            idx = [i for i in range(len(all_grads)) if not (i < 4 * L and i % 4 in (2, 3))]
            flat = comm.allreduce_(torch.cat([all_grads[i].reshape(-1) for i in idx]))
            off = 0
            for i in idx:
                k = all_grads[i].numel()
                all_grads[i] = flat[off: off + k].view_as(all_grads[i])
                off += k
        return (None, None, None, None, None, None, g_xpos, *all_grads) + ((None,) if ctx.has_precision else ())


# ---------------------------------------------------------------------------------------------------------------------
# losses (reference util/loss.py) and geometry (reference util/models.py)
# ---------------------------------------------------------------------------------------------------------------------
class PosRecLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, target64, topo):
        set_device(pos.device)
        pos = _f32(pos, "pos_rec_loss pos")
        loss = torch.empty((), dtype=torch.float64, device=pos.device)
        lib.call("ddmp_loss_pos_rec_fwd", ptr(pos), ptr(target64), ptr(loss), ptr(topo.scratch), pos.shape[0],
                 stream_ptr(pos.device))
        ctx.save_for_backward(pos, target64, loss)
        return loss

    @staticmethod
    def backward(ctx, gout):
        pos, target64, loss = ctx.saved_tensors
        set_device(pos.device)
        gpos = torch.empty_like(pos)
        gout = gout.to(torch.float64).contiguous()
        lib.call("ddmp_loss_pos_rec_bwd", ptr(pos), ptr(target64), ptr(loss), ptr(gout), ptr(gpos), pos.shape[0],
                 stream_ptr(pos.device))
        return gpos, None, None


class LaplacianLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, topo):
        set_device(pos.device)
        pos = _f32(pos, "mesh_laplacian_loss pos")
        d = torch.empty_like(pos)
        loss = torch.empty((), dtype=torch.float32, device=pos.device)
        lib.call("ddmp_loss_lap_fwd", ptr(pos), ptr(topo.lap_rowptr), ptr(topo.lap_col), ptr(d), ptr(loss),
                 ptr(topo.scratch), pos.shape[0], stream_ptr(pos.device))
        ctx.save_for_backward(d, loss)
        ctx.topo = topo
        return loss

    @staticmethod
    def backward(ctx, gout):
        d, loss = ctx.saved_tensors
        topo = ctx.topo
        set_device(d.device)
        gpos = torch.empty_like(d)
        gout = gout.to(torch.float32).contiguous()
        lib.call("ddmp_loss_lap_bwd", ptr(d), ptr(topo.lap_rowptr), ptr(topo.lap_col), ptr(loss), ptr(gout),
                 ptr(gpos), d.shape[0], stream_ptr(d.device))
        return gpos, None


class NormRecLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, nrm, target64, topo):
        set_device(nrm.device)
        nrm = _f32(nrm, "norm_rec_loss norm")
        loss = torch.empty((), dtype=torch.float64, device=nrm.device)
        lib.call("ddmp_loss_norm_rec_fwd", ptr(nrm), ptr(target64), ptr(loss), ptr(topo.scratch), nrm.shape[0],
                 stream_ptr(nrm.device))
        ctx.save_for_backward(nrm, target64)
        return loss

    @staticmethod
    def backward(ctx, gout):
        nrm, target64 = ctx.saved_tensors
        set_device(nrm.device)
        g = torch.empty_like(nrm)
        gout = gout.to(torch.float64).contiguous()
        lib.call("ddmp_loss_norm_rec_bwd", ptr(nrm), ptr(target64), ptr(gout), ptr(g), nrm.shape[0],
                 stream_ptr(nrm.device))
        return g, None, None


class PosNormLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, nrm, topo):
        set_device(pos.device)
        pos, nrm = _f32(pos, "pos_norm_loss pos"), _f32(nrm, "pos_norm_loss norm")
        loss = torch.empty((), dtype=torch.float32, device=pos.device)
        lib.call("ddmp_loss_pos_norm_fwd", ptr(pos), ptr(nrm), ptr(topo.faces), ptr(loss), ptr(topo.scratch),
                 topo.V, topo.F, stream_ptr(pos.device))
        ctx.save_for_backward(pos, nrm)
        ctx.topo = topo
        return loss

    @staticmethod
    def backward(ctx, gout):
        pos, nrm = ctx.saved_tensors
        topo = ctx.topo
        set_device(pos.device)
        gpos, gnrm = torch.empty_like(pos), torch.empty_like(nrm)
        tmp = torch.empty(topo.F, 9, dtype=torch.float32, device=pos.device)
        gout = gout.to(torch.float32).contiguous()
        lib.call("ddmp_loss_pos_norm_bwd", ptr(pos), ptr(nrm), ptr(topo.faces), ptr(topo.corner_ptr),
                 ptr(topo.corner_slot), ptr(gout), ptr(tmp), ptr(gpos), ptr(gnrm), topo.V, topo.F,
                 stream_ptr(pos.device))
        return gpos, gnrm, None


class BnfLoss(torch.autograd.Function):
    """fn_bnf_loss: returns (loss, new_fn); ``pos`` is detached by the reference (util/loss.py:91)."""

    @staticmethod
    def forward(ctx, pos, fn, topo, loop):
        dev = fn.device
        set_device(dev)
        st = stream_ptr(dev)
        pos, fn = _f32(pos, "fn_bnf_loss pos"), _f32(fn, "fn_bnf_loss fn")
        F = topo.F
        fc = torch.empty(F, 3, dtype=torch.float32, device=dev)
        fa = torch.empty(F, dtype=torch.float32, device=dev)
        wca = torch.empty(F, 3, dtype=torch.float32, device=dev)
        sigma_c = torch.empty((), dtype=torch.float32, device=dev)
        lib.call("ddmp_bnf_setup", ptr(pos), ptr(topo.faces), ptr(topo.f2f), ptr(fc), ptr(fa), ptr(wca),
                 ptr(sigma_c), ptr(topo.scratch), F, st)
        normals = [fn]
        for _ in range(loop):
            nxt = torch.empty_like(fn)
            lib.call("ddmp_bnf_iter_fwd", ptr(normals[-1]), ptr(topo.f2f), ptr(wca), ptr(nxt), F, st)
            normals.append(nxt)
        loss = torch.empty((), dtype=torch.float32, device=dev)
        lib.call("ddmp_bnf_loss_fwd", ptr(normals[-1]), ptr(fn), ptr(loss), ptr(topo.scratch), F, st)
        ctx.topo, ctx.normals, ctx.wca, ctx.loop = topo, normals, wca, loop
        new_fn = normals[-1] if loop > 0 else fn.clone()
        ctx.mark_non_differentiable(new_fn)
        return loss, new_fn

    @staticmethod
    def backward(ctx, gout, _g_new_fn):
        topo, normals, wca, loop = ctx.topo, ctx.normals, ctx.wca, ctx.loop
        fn = normals[0]
        dev = fn.device
        set_device(dev)
        st = stream_ptr(dev)
        F = topo.F
        if loop == 0:
            return None, torch.zeros_like(fn), None, None
        gout = gout.to(torch.float32).contiguous()
        g_last = torch.empty_like(fn)
        lib.call("ddmp_bnf_loss_bwd", ptr(normals[-1]), ptr(fn), ptr(gout), ptr(g_last), F, st)
        g = g_last
        msg = torch.empty(F, 9, dtype=torch.float32, device=dev)
        for t in range(loop - 1, -1, -1):
            g_in = torch.empty_like(fn)
            lib.call("ddmp_bnf_iter_bwd", ptr(normals[t]), ptr(g), ptr(topo.f2f), ptr(topo.rslot), ptr(wca),
                     ptr(g_last) if t == 0 else None, ptr(msg), ptr(g_in), F, st)
            g = g_in
        ctx.normals = None
        return None, g, None, None


class DualLoss(torch.autograd.Function):
    """The loss phase of one iteration (reference main.py:94-106) as one cooperative kernel: returns the weighted total
    (float64) and the five terms; the gradients w.r.t. ``pos`` / ``norm`` are produced by the same launch and only
    scaled by the upstream gradient in ``backward``."""

    @staticmethod
    def forward(ctx, pos, nrm, tgt_vs, tgt_fn, topo, k, loop, bnf_scale):
        dev = pos.device
        set_device(dev)
        pos, nrm = _f32(pos, "dual_loss pos"), _f32(nrm, "dual_loss norm")
        tgt_vs = require_cuda(tgt_vs, torch.float64, "dual_loss target positions")
        tgt_fn = require_cuda(tgt_fn, torch.float64, "dual_loss target normals")
        V, F = topo.V, topo.F
        if pos.shape != (V, 3) or nrm.shape != (F, 3) or tgt_vs.shape != (V, 3) or tgt_fn.shape != (F, 3):
            raise RuntimeError("dual_loss: shapes do not match the mesh")
        nbytes = int(lib.query("ddmp_dual_loss_workspace_bytes", V, F, int(loop)))
        ws = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
        gpos, gnrm = torch.empty_like(pos), torch.empty_like(nrm)
        losses = torch.empty(6, dtype=torch.float64, device=dev)
        lib.call("ddmp_dual_loss", ptr(pos), ptr(nrm), ptr(tgt_vs), ptr(tgt_fn), ptr(topo.faces), ptr(topo.f2f),
                 ptr(topo.rslot), ptr(topo.lap_rowptr), ptr(topo.lap_col), ptr(topo.corner_ptr), ptr(topo.corner_slot),
                 float(k[0]), float(k[1]), float(k[2]), float(k[3]), float(k[4]), float(bnf_scale), int(loop), ptr(ws),
                 nbytes, ptr(gpos), ptr(gnrm), ptr(losses), V, F, stream_ptr(dev))
        ctx.save_for_backward(gpos, gnrm)
        parts = losses[:5]
        ctx.mark_non_differentiable(parts)
        return losses[5], parts

    @staticmethod
    def backward(ctx, gout, _gparts):
        gpos, gnrm = ctx.saved_tensors
        g = gout.to(torch.float32)
        return gpos * g, gnrm * g, None, None, None, None, None, None


class FaceNormals(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pos, topo):
        set_device(pos.device)
        pos = _f32(pos, "compute_fn vs")
        fn = torch.empty(topo.F, 3, dtype=torch.float32, device=pos.device)
        lib.call("ddmp_face_normals_fwd", ptr(pos), ptr(topo.faces), ptr(fn), topo.F, stream_ptr(pos.device))
        ctx.save_for_backward(pos)
        ctx.topo = topo
        return fn

    @staticmethod
    def backward(ctx, gfn):
        (pos,) = ctx.saved_tensors
        topo = ctx.topo
        set_device(pos.device)
        gfn = _f32(gfn, "compute_fn grad")
        tmp = torch.empty(topo.F, 9, dtype=torch.float32, device=pos.device)
        gpos = torch.empty_like(pos)
        lib.call("ddmp_face_normals_bwd", ptr(pos), ptr(topo.faces), ptr(topo.corner_ptr), ptr(topo.corner_slot),
                 ptr(gfn), ptr(tmp), ptr(gpos), topo.V, topo.F, stream_ptr(pos.device))
        return gpos, None


def mad_device(n1, n2, topo) -> torch.Tensor:
    set_device(n1.device)
    n1, n2 = _f32(n1, "mad norm1"), _f32(n2, "mad norm2")
    out = torch.empty((), dtype=torch.float64, device=n1.device)
    lib.call("ddmp_mad", ptr(n1), ptr(n2), ptr(out), ptr(topo.scratch), n1.shape[0], stream_ptr(n1.device))
    return out
