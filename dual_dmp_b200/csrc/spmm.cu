// GCN aggregation: symmetric-normalised SpMM over CSR, row-segmented, deterministic (no atomics).
//   Y[i,:] = sum_k w[k] * H[col[k],:] (+ bias), optional BatchNorm partial statistics in the epilogue.
// Replaces torch_geometric GCNConv.propagate (index_select -> mul -> torch_scatter.scatter_add) called from
// reference util/networks.py:51-62,112-123, and its backward (A_hat is symmetric, so backward = same kernel).
//
// Mapping: a "row group" of G = min(32, C/4) lanes owns one output row at a time and keeps it in NV = C/(4G)
// float4 accumulators per lane; 128-bit gathers of H rows; the (col, w) stream of a row is fetched with ONE
// coalesced load per G entries (lane j takes entry j) and broadcast with group-scoped shuffles.  A CTA of 256
// threads walks `rows_per_block` consecutive rows (consecutive groups take consecutive rows, so neighbour rows
// gathered by one CTA overlap in L1).  Roofline: HBM; algorithmic bytes 4*[(n+1) + 2*nnz + 2*n*C].
#include <stdlib.h>

#include "common.cuh"

namespace ddmp {

template <int C, bool STATS, bool BIAS>
__global__ void __launch_bounds__(256, (STATS || C >= 512) ? 3 : 4)
spmm_gcn_kernel(const int* __restrict__ rowptr, const int* __restrict__ col, const float* __restrict__ w,
                const float* __restrict__ H, const float* __restrict__ bias, float* __restrict__ Y,
                float* __restrict__ partials, float* __restrict__ amax_blocks, int64_t n, int rows_per_block,
                int blocks_per_cta) {
    constexpr int G = (C / 4 < 32) ? (C / 4) : 32;
    constexpr int NV = C / (4 * G);
    constexpr int GROUPS = 256 / G;
    constexpr int U = (NV >= 4) ? 2 : 4;

    const int lane = threadIdx.x & 31;
    const int lg = lane % G;
    const int gid = threadIdx.x / G;
    const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << ((lane / G) * G));

    float4 bsum[NV];
#pragma unroll
    for (int v = 0; v < NV; ++v) {
        bsum[v] = BIAS ? ldg4(bias + (v * G + lg) * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // BatchNorm partial sums live in shared memory, one private [2][C] slice per row group (keeping them in
    // registers costs 8*NV registers and halves the occupancy of the widest instantiation: ncu, profiles/)
    // What this buffer costs is L1, not instructions: forcing a shared-memory carve-out on the PLAIN flavour slows it
    // from 0.474 to 0.635 ms (vertex graph, C = 512), past the statistics flavour (0.591); with the moments in registers
    // (256-channel slices) the time does not change (profiles/spmm_slice_ab_r2.txt).
    __shared__ __align__(16) float red[STATS ? GROUPS * 2 * C : 4];
    __shared__ float wmax[8];
    float* myred = red + gid * 2 * C;
    // A CTA walks `blocks_per_cta` consecutive row blocks (1 by default, see launch_spmm).
    const int64_t nblk = (n + rows_per_block - 1) / rows_per_block;
    const int64_t blk_begin = (int64_t)blockIdx.x * blocks_per_cta;
    const int64_t blk_end = (blk_begin + blocks_per_cta < nblk) ? (blk_begin + blocks_per_cta) : nblk;
    for (int64_t blk = blk_begin; blk < blk_end; ++blk) {
    const int64_t row0 = blk * rows_per_block;
    const int64_t row_end = (row0 + rows_per_block < n) ? (row0 + rows_per_block) : n;
    float amx = 0.f;                                 // max |Y| over this thread's outputs of the row block
    float wcnt = 0.f;                                // rows this group has folded into its running statistics
    if (STATS) {
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            st4(myred + (v * G + lg) * 4, make_float4(0.f, 0.f, 0.f, 0.f));
            st4(myred + C + (v * G + lg) * 4, make_float4(0.f, 0.f, 0.f, 0.f));
        }
    }

    // Software pipeline over the rows of a group: (rowptr, first col/w chunk) of the NEXT row are fetched while the
    // gathers of the current row are in flight, so the rowptr -> col -> H dependent-load chain is paid once per
    // group instead of once per row (narrow widths are latency-, not bandwidth-bound).
    int64_t r = row0 + gid;
    int start = 0, end = 0, myc = 0;
    float myw = 0.f;
    if (r < row_end) {
        start = __ldg(rowptr + r);
        end = __ldg(rowptr + r + 1);
        const int kk = start + lg;
        if (kk < end) { myc = __ldg(col + kk); myw = __ldg(w + kk); }
    }
    for (; r < row_end; r += GROUPS) {
        const int64_t rn = r + GROUPS;
        int nstart = 0, nend = 0, nmyc = 0;
        float nmyw = 0.f;
        if (rn < row_end) {
            nstart = __ldg(rowptr + rn);
            nend = __ldg(rowptr + rn + 1);
        }
        float4 acc[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);

        for (int k0 = start; k0 < end; k0 += G) {
            if (k0 != start) {                       // rows longer than G entries: further chunks are loaded here
                const int kk = k0 + lg;
                myc = (kk < end) ? __ldg(col + kk) : 0;
                myw = (kk < end) ? __ldg(w + kk) : 0.f;
            }
            const int cnt = (end - k0 < G) ? (end - k0) : G;
            int j = 0;
            for (; j + U <= cnt; j += U) {
                int cj[U];
                float wj[U];
                float4 x[U][NV];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    cj[u] = __shfl_sync(gmask, myc, j + u, G);
                    wj[u] = __shfl_sync(gmask, myw, j + u, G);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const float* hp = H + (int64_t)cj[u] * C;
#pragma unroll
                    for (int v = 0; v < NV; ++v) x[u][v] = ldg4(hp + (v * G + lg) * 4);
                }
                if (k0 == start && j == 0 && rn < row_end) {   // next row's first chunk, behind the gathers in flight
                    const int kk = nstart + lg;
                    if (kk < nend) { nmyc = __ldg(col + kk); nmyw = __ldg(w + kk); }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
#pragma unroll
                    for (int v = 0; v < NV; ++v) {
                        acc[v].x = fmaf(wj[u], x[u][v].x, acc[v].x);
                        acc[v].y = fmaf(wj[u], x[u][v].y, acc[v].y);
                        acc[v].z = fmaf(wj[u], x[u][v].z, acc[v].z);
                        acc[v].w = fmaf(wj[u], x[u][v].w, acc[v].w);
                    }
                }
            }
            for (; j < cnt; ++j) {
                const int c1 = __shfl_sync(gmask, myc, j, G);
                const float w1 = __shfl_sync(gmask, myw, j, G);
                const float* hp = H + (int64_t)c1 * C;
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    const float4 x = ldg4(hp + (v * G + lg) * 4);
                    acc[v].x = fmaf(w1, x.x, acc[v].x);
                    acc[v].y = fmaf(w1, x.y, acc[v].y);
                    acc[v].z = fmaf(w1, x.z, acc[v].z);
                    acc[v].w = fmaf(w1, x.w, acc[v].w);
                }
            }
        }
        if (rn < row_end && (end - start) < U) {     // short row: the prefetch slot inside the unrolled loop was skipped
            const int kk = nstart + lg;
            if (kk < nend) { nmyc = __ldg(col + kk); nmyw = __ldg(w + kk); }
        }
        float* yp = Y + r * C;
        wcnt += 1.f;
        const float winv = 1.f / wcnt;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            float4 o = acc[v];
            if (BIAS) {
                o.x += bsum[v].x; o.y += bsum[v].y; o.z += bsum[v].z; o.w += bsum[v].w;
            }
            // streaming (evict-first) store: this kernel never re-reads Y, and keeping it out of L2 leaves the cache to the
            // gathered rows (+1 % on the wide layers)
            __stcs(reinterpret_cast<float4*>(yp + (v * G + lg) * 4), o);
            // only when requested: without this condition ptxas spills the row loop's state in the plain flavour
            if (amax_blocks) amx = fmaxf(fmaxf(amx, fmaxf(fabsf(o.x), fabsf(o.y))), fmaxf(fabsf(o.z), fabsf(o.w)));
            if (STATS) {                            // Welford: running mean and M2 of this group's rows (see bn.cu)
                float4 s = *reinterpret_cast<float4*>(myred + (v * G + lg) * 4);
                float4 q = *reinterpret_cast<float4*>(myred + C + (v * G + lg) * 4);
                float d;
                d = o.x - s.x; s.x = fmaf(d, winv, s.x); q.x = fmaf(d, o.x - s.x, q.x);
                d = o.y - s.y; s.y = fmaf(d, winv, s.y); q.y = fmaf(d, o.y - s.y, q.y);
                d = o.z - s.z; s.z = fmaf(d, winv, s.z); q.z = fmaf(d, o.z - s.z, q.z);
                d = o.w - s.w; s.w = fmaf(d, winv, s.w); q.w = fmaf(d, o.w - s.w, q.w);
                st4(myred + (v * G + lg) * 4, s);
                st4(myred + C + (v * G + lg) * 4, q);
            }
        }
        start = nstart; end = nend; myc = nmyc; myw = nmyw;
    }

    if (STATS) {
        // merge the GROUPS row groups of this CTA channel-wise in group order (Chan et al.): block (sum, M2 about its mean)
        __syncthreads();
        float* outp = partials + blk * 2 * C;
        const int rows_blk = (int)(row_end - row0);
        for (int ch = threadIdx.x; ch < C; ch += 256) {
            float n_a = 0.f, mean = 0.f, m2 = 0.f;
#pragma unroll 4
            for (int g = 0; g < GROUPS; ++g) {
                if (g < rows_blk) {
                    const float n_b = (float)((rows_blk - g + GROUPS - 1) / GROUPS);
                    const float mb = red[g * 2 * C + ch], qb = red[g * 2 * C + C + ch];
                    const float n = n_a + n_b;
                    const float d = mb - mean;
                    mean = fmaf(d, n_b / n, mean);
                    m2 += qb + d * d * (n_a * n_b / n);
                    n_a = n;
                }
            }
            outp[ch] = mean * n_a;
            outp[C + ch] = m2;
        }
        __syncthreads();
    }
    if (amax_blocks) {                               // operand bound for the fp16-split GEMMs that consume Y
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) amx = fmaxf(amx, __shfl_xor_sync(0xffffffffu, amx, o));
        if (lane == 0) wmax[threadIdx.x >> 5] = amx;
        __syncthreads();
        if (threadIdx.x == 0) {
            float m = wmax[0];
#pragma unroll
            for (int i = 1; i < 8; ++i) m = fmaxf(m, wmax[i]);
            amax_blocks[blk] = m;
        }
        __syncthreads();
    }
    }   // row blocks of this CTA
}

// ---- forward flavour of the wide layers (C = 256 / 512) with the Welford state in TENSOR MEMORY ------------------------
// The kernel above keeps a private (mean, M2) pair per warp and channel in shared memory: 32 KB per CTA at C = 512,
// 96 KB per SM -- taken from the L1 that serves the gathers, which is what makes the forward flavour 20-27 % slower than
// the plain one (profiles/spmm_slice_ab_r2.txt: a shared-memory carve-out alone slows the PLAIN flavour past it).
// Registers are no alternative (32 more per thread halve the occupancy).  But the SM has 256 KB of tensor memory that an
// aggregation kernel never touches: a warp reads and writes its own 32 lanes x 8*NV columns with tcgen05.ld / tcgen05.st
// (.32x32b: thread i <-> TMEM lane 32*(warp%4)+i), which is exactly "one private slot per thread".  State layout: warp w,
// lane i, float4 index v: columns (w/4)*8*NV + 8*v + {0..3} = running mean, + {4..7} = M2.  64 columns per CTA at C = 512,
// 32 at C = 256; 3 (4 at C = 256) CTAs per SM allocate 192 (128) of the 512 columns.  (The tcgen05 GEMM kernels of the other network's stream
// fill the register file on their own, so an SM never hosts both kinds of CTA and tcgen05.alloc cannot wait on them.)
// Same arithmetic and merge order as the kernel above: Y and the block moments are bitwise identical.
__device__ __forceinline__ void tmem_ld8(uint32_t taddr, float4& a, float4& b) {
    uint32_t r0, r1, r2, r3, r4, r5, r6, r7;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3), "=r"(r4), "=r"(r5), "=r"(r6), "=r"(r7)
                 : "r"(taddr)
                 : "memory");
    a = make_float4(__uint_as_float(r0), __uint_as_float(r1), __uint_as_float(r2), __uint_as_float(r3));
    b = make_float4(__uint_as_float(r4), __uint_as_float(r5), __uint_as_float(r6), __uint_as_float(r7));
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const float4& a, const float4& b) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"r"(taddr),
                 "r"(__float_as_uint(a.x)), "r"(__float_as_uint(a.y)), "r"(__float_as_uint(a.z)), "r"(__float_as_uint(a.w)),
                 "r"(__float_as_uint(b.x)), "r"(__float_as_uint(b.y)), "r"(__float_as_uint(b.z)), "r"(__float_as_uint(b.w))
                 : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

template <int C, bool BIAS>
__global__ void __launch_bounds__(256, C >= 512 ? 3 : 4)
spmm_gcn_stats_tmem_kernel(const int* __restrict__ rowptr, const int* __restrict__ col, const float* __restrict__ w,
                           const float* __restrict__ H, const float* __restrict__ bias, float* __restrict__ Y,
                           float* __restrict__ partials, int64_t n, int rows_per_block) {
    constexpr int NV = C / 128;             // float4 per lane
    constexpr int GROUPS = 8;
    constexpr int U = (NV >= 4) ? 2 : 4;
    constexpr uint32_t WCOLS = 8 * NV;      // TMEM columns of one warp's state
    constexpr uint32_t TCOLS = 2 * WCOLS < 32 ? 32 : 2 * WCOLS;
    const int lane = threadIdx.x & 31;
    const int gid = threadIdx.x >> 5;
    __shared__ __align__(16) float red[GROUPS * 2 * 128];       // 8 KB merge buffer (128 channels per round)
    __shared__ uint32_t tmem_slot;

    if (gid == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(
                         (uint32_t)__cvta_generic_to_shared(&tmem_slot)),
                     "r"(TCOLS)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tbase = tmem_slot;
    const uint32_t taddr = tbase + ((uint32_t)((gid & 3) * 32) << 16) + (uint32_t)(gid >> 2) * WCOLS;

    const int64_t row0 = (int64_t)blockIdx.x * rows_per_block;
    const int64_t row_end = (row0 + rows_per_block < n) ? (row0 + rows_per_block) : n;
    {
        const float4 z = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int v = 0; v < NV; ++v) tmem_st8(taddr + 8 * v, z, z);
        tmem_wait_st();
    }
    float wcnt = 0.f;

    int64_t r = row0 + gid;
    int start = 0, end = 0, myc = 0;
    float myw = 0.f;
    if (r < row_end) {
        start = __ldg(rowptr + r);
        end = __ldg(rowptr + r + 1);
        const int kk = start + lane;
        if (kk < end) { myc = __ldg(col + kk); myw = __ldg(w + kk); }
    }
    for (; r < row_end; r += GROUPS) {
        const int64_t rn = r + GROUPS;
        int nstart = 0, nend = 0, nmyc = 0;
        float nmyw = 0.f;
        if (rn < row_end) {
            nstart = __ldg(rowptr + rn);
            nend = __ldg(rowptr + rn + 1);
        }
        float4 acc[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) acc[v] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int k0 = start; k0 < end; k0 += 32) {
            if (k0 != start) {
                const int kk = k0 + lane;
                myc = (kk < end) ? __ldg(col + kk) : 0;
                myw = (kk < end) ? __ldg(w + kk) : 0.f;
            }
            const int cnt = (end - k0 < 32) ? (end - k0) : 32;
            int j = 0;
            for (; j + U <= cnt; j += U) {
                int cj[U];
                float wj[U];
                float4 x[U][NV];
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    cj[u] = __shfl_sync(0xffffffffu, myc, j + u);
                    wj[u] = __shfl_sync(0xffffffffu, myw, j + u);
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
                    const float* hp = H + (int64_t)cj[u] * C;
#pragma unroll
                    for (int v = 0; v < NV; ++v) x[u][v] = ldg4(hp + (v * 32 + lane) * 4);
                }
                if (k0 == start && j == 0 && rn < row_end) {   // next row's first chunk, behind the gathers in flight
                    const int kk = nstart + lane;
                    if (kk < nend) { nmyc = __ldg(col + kk); nmyw = __ldg(w + kk); }
                }
#pragma unroll
                for (int u = 0; u < U; ++u) {
#pragma unroll
                    for (int v = 0; v < NV; ++v) {
                        acc[v].x = fmaf(wj[u], x[u][v].x, acc[v].x);
                        acc[v].y = fmaf(wj[u], x[u][v].y, acc[v].y);
                        acc[v].z = fmaf(wj[u], x[u][v].z, acc[v].z);
                        acc[v].w = fmaf(wj[u], x[u][v].w, acc[v].w);
                    }
                }
            }
            for (; j < cnt; ++j) {
                const int c1 = __shfl_sync(0xffffffffu, myc, j);
                const float w1 = __shfl_sync(0xffffffffu, myw, j);
                const float* hp = H + (int64_t)c1 * C;
#pragma unroll
                for (int v = 0; v < NV; ++v) {
                    const float4 x = ldg4(hp + (v * 32 + lane) * 4);
                    acc[v].x = fmaf(w1, x.x, acc[v].x);
                    acc[v].y = fmaf(w1, x.y, acc[v].y);
                    acc[v].z = fmaf(w1, x.z, acc[v].z);
                    acc[v].w = fmaf(w1, x.w, acc[v].w);
                }
            }
        }
        if (rn < row_end && (end - start) < U) {     // short row: the prefetch slot inside the unrolled loop was skipped
            const int kk = nstart + lane;
            if (kk < nend) { nmyc = __ldg(col + kk); nmyw = __ldg(w + kk); }
        }
        // ---- epilogue: bias, store, Welford update of this warp's state in tensor memory ----
        float4 s4[NV], q4[NV];
#pragma unroll
        for (int v = 0; v < NV; ++v) tmem_ld8(taddr + 8 * v, s4[v], q4[v]);
        float* yp = Y + r * C;
        wcnt += 1.f;
        const float winv = 1.f / wcnt;
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            if (BIAS) {
                const float4 b = ldg4(bias + (v * 32 + lane) * 4);           // L1-resident; not worth 4*NV registers
                acc[v].x += b.x; acc[v].y += b.y; acc[v].z += b.z; acc[v].w += b.w;
            }
            __stcs(reinterpret_cast<float4*>(yp + (v * 32 + lane) * 4), acc[v]);
        }
        tmem_wait_ld();
#pragma unroll
        for (int v = 0; v < NV; ++v) {
            const float4 o = acc[v];
            float4 s = s4[v], q = q4[v];
            float d;
            d = o.x - s.x; s.x = fmaf(d, winv, s.x); q.x = fmaf(d, o.x - s.x, q.x);
            d = o.y - s.y; s.y = fmaf(d, winv, s.y); q.y = fmaf(d, o.y - s.y, q.y);
            d = o.z - s.z; s.z = fmaf(d, winv, s.z); q.z = fmaf(d, o.z - s.z, q.z);
            d = o.w - s.w; s.w = fmaf(d, winv, s.w); q.w = fmaf(d, o.w - s.w, q.w);
            tmem_st8(taddr + 8 * v, s, q);
        }
        tmem_wait_st();
        start = nstart; end = nend; myc = nmyc; myw = nmyw;
    }

    // merge the 8 warps channel-wise in warp order (Chan et al.), 128 channels per round through the 8 KB buffer
    float* outp = partials + (int64_t)blockIdx.x * 2 * C;
    const int rows_blk = (int)(row_end - row0);
    float* myred = red + gid * 2 * 128;
#pragma unroll
    for (int v = 0; v < NV; ++v) {
        float4 s, q;
        tmem_ld8(taddr + 8 * v, s, q);
        tmem_wait_ld();
        st4(myred + lane * 4, s);
        st4(myred + 128 + lane * 4, q);
        __syncthreads();
        if (threadIdx.x < 128) {
            const int ch = threadIdx.x;
            float n_a = 0.f, mu = 0.f, m2 = 0.f;
#pragma unroll 4
            for (int g = 0; g < GROUPS; ++g) {
                if (g < rows_blk) {
                    const float n_b = (float)((rows_blk - g + GROUPS - 1) / GROUPS);
                    const float mb = red[g * 256 + ch], qb = red[g * 256 + 128 + ch];
                    const float nn = n_a + n_b;
                    const float d = mb - mu;
                    mu = fmaf(d, n_b / nn, mu);
                    m2 += qb + d * d * (n_a * n_b / nn);
                    n_a = nn;
                }
            }
            outp[v * 128 + ch] = mu * n_a;
            outp[C + v * 128 + ch] = m2;
        }
        __syncthreads();
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (gid == 0) {
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tbase), "r"(TCOLS) : "memory");
    }
}

// Any width: one warp per row, lanes stride over channels (operator-level GCNConv with unusual widths).
__global__ void __launch_bounds__(256)
spmm_gcn_generic_kernel(const int* __restrict__ rowptr, const int* __restrict__ col, const float* __restrict__ w,
                        const float* __restrict__ H, const float* __restrict__ bias, float* __restrict__ Y,
                        int64_t n, int C) {
    const int lane = threadIdx.x & 31;
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (r >= n) return;
    const int start = rowptr[r], end = rowptr[r + 1];
    for (int c = lane; c < C; c += 32) {
        float acc = 0.f;
        for (int k = start; k < end; ++k) acc = fmaf(__ldg(w + k), __ldg(H + (int64_t)__ldg(col + k) * C + c), acc);
        Y[r * C + c] = acc + (bias ? bias[c] : 0.f);
    }
}

__global__ void gcn_edge_weights_kernel(const int* __restrict__ rowptr, const int* __restrict__ col,
                                        float* __restrict__ w, int64_t n) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n) return;
    const int start = rowptr[r], end = rowptr[r + 1];
    // deg^-1/2 as an IEEE 1/sqrt, like torch.pow(deg, -0.5) on the reference path
    const float di = 1.0f / sqrtf((float)(end - start));
    for (int k = start; k < end; ++k) {
        const int j = col[k];
        const float dj = 1.0f / sqrtf((float)(rowptr[j + 1] - rowptr[j]));
        w[k] = di * dj;
    }
}

template <int C>
static int launch_spmm(const int* rowptr, const int* col, const float* w, const float* H, const float* bias,
                       float* Y, float* partials, float* amax_blocks, int64_t n, bool reference, cudaStream_t st) {
    const int rpb = ddmp_rows_per_block(C);
    const int64_t nblk = ceil_div(n, rpb);
    // consecutive row blocks per CTA (DDMP_SPMM_CHUNK).  Default 1: walking 4 or 8 neighbouring blocks per CTA to
    // keep gathered rows in L1 measured 9 % SLOWER step-weighted on B200 (3,565 vs 3,927 GB/s, scripts/bench_spmm.py)
    // -- fewer, longer CTAs lose more to the tail than the extra L1 hits win back.
    static const int chunk_env = [] { const char* e = getenv("DDMP_SPMM_CHUNK"); return e ? atoi(e) : 1; }();
    int bpc = chunk_env < 1 ? 1 : chunk_env;
    while (bpc > 1 && ceil_div(nblk, bpc) < 8 * kNumSMs) --bpc;
    const unsigned grid = (unsigned)ceil_div(nblk, bpc);
    if (!reference && partials && !amax_blocks && (C == 256 || C == 512) && bpc == 1) {
        // wide forward flavour: Welford state in tensor memory (spmm_gcn_stats_tmem_kernel).  1M-row graphs, vertex /
        // face: C = 512 0.592 -> 0.525 / 0.938 -> 0.862 ms; C = 256 0.331 -> 0.296 / 0.483 -> 0.449 ms once the kernel
        // runs 4 CTAs per SM (at 3 it measured the same as the 16 KB shared-memory state): profiles/spmm_tmem_ab_r2.txt
        constexpr int CT = (C == 256 || C == 512) ? C : 256;
        if (bias) spmm_gcn_stats_tmem_kernel<CT, true><<<(unsigned)nblk, 256, 0, st>>>(rowptr, col, w, H, bias, Y, partials, n, rpb);
        else spmm_gcn_stats_tmem_kernel<CT, false><<<(unsigned)nblk, 256, 0, st>>>(rowptr, col, w, H, bias, Y, partials, n, rpb);
        return check_launch("spmm_gcn_stats_tmem");
    }
    if (partials) {
        if (bias) spmm_gcn_kernel<C, true, true><<<grid, 256, 0, st>>>(rowptr, col, w, H, bias, Y, partials, amax_blocks, n, rpb, bpc);
        else spmm_gcn_kernel<C, true, false><<<grid, 256, 0, st>>>(rowptr, col, w, H, bias, Y, partials, amax_blocks, n, rpb, bpc);
    } else {
        if (bias) spmm_gcn_kernel<C, false, true><<<grid, 256, 0, st>>>(rowptr, col, w, H, bias, Y, partials, amax_blocks, n, rpb, bpc);
        else spmm_gcn_kernel<C, false, false><<<grid, 256, 0, st>>>(rowptr, col, w, H, bias, Y, partials, amax_blocks, n, rpb, bpc);
    }
    return check_launch("spmm_gcn");
}

// ddmp_spmm_reference_kernel: the gather kernel with shared-memory statistics at every width
static std::atomic<int> g_reference_kernel{0};

}  // namespace ddmp

extern "C" {

int ddmp_gcn_edge_weights(const int32_t* rowptr, const int32_t* col, float* w, int64_t n, void* stream) {
    DDMP_REQUIRE(rowptr && col && w && n >= 0, "gcn_edge_weights: null pointer or negative n");
    if (n == 0) return DDMP_OK;
    ddmp::gcn_edge_weights_kernel<<<(unsigned)ddmp::ceil_div(n, 256), 256, 0, ddmp::as_stream(stream)>>>(rowptr, col, w, n);
    return ddmp::check_launch("gcn_edge_weights");
}

int ddmp_spmm_gcn(const int32_t* rowptr, const int32_t* col, const float* w, const float* H, const float* bias,
                  float* Y, float* stats_partials, float* amax_blocks, int64_t n, int32_t C, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(n >= 0 && C > 0, "spmm_gcn: bad shape n=%lld C=%d", (long long)n, C);
    if (n == 0) return DDMP_OK;
    DDMP_REQUIRE(rowptr && col && w && H && Y, "spmm_gcn: null pointer");
    cudaStream_t st = as_stream(stream);
    const bool ref = g_reference_kernel.load(std::memory_order_relaxed) != 0;
    if (!ref && spmm_tile_supported(n, C))
        return spmm_tile_launch(rowptr, col, w, H, bias, Y, stats_partials, amax_blocks, n, C, st);
    switch (C) {
        case 32: return launch_spmm<32>(rowptr, col, w, H, bias, Y, stats_partials, amax_blocks, n, ref, st);
        case 64: return launch_spmm<64>(rowptr, col, w, H, bias, Y, stats_partials, amax_blocks, n, ref, st);
        case 128: return launch_spmm<128>(rowptr, col, w, H, bias, Y, stats_partials, amax_blocks, n, ref, st);
        case 256: return launch_spmm<256>(rowptr, col, w, H, bias, Y, stats_partials, amax_blocks, n, ref, st);
        case 512: return launch_spmm<512>(rowptr, col, w, H, bias, Y, stats_partials, amax_blocks, n, ref, st);
        default: break;
    }
    if (stats_partials || amax_blocks) {
        set_error("spmm_gcn: the statistics / amax epilogues support C in {32,64,128,256,512}, got %d", C);
        return DDMP_ERR_UNSUPPORTED;
    }
    spmm_gcn_generic_kernel<<<(unsigned)ceil_div(n, 8), 256, 0, st>>>(rowptr, col, w, H, bias, Y, n, C);
    return check_launch("spmm_gcn_generic");
}

int ddmp_spmm_reference_kernel(int on) { return ddmp::g_reference_kernel.exchange(on != 0, std::memory_order_relaxed); }

int64_t ddmp_spmm_amax_len(int64_t n, int32_t C) { return ddmp_num_row_blocks(n, C); }

}  // extern "C"
