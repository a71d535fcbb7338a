// GCN aggregation, tile-staged variant: the row block's OWN rows of H arrive in shared memory through ONE TMA tensor
// copy (cp.async.bulk.tensor.2d, SASS UTMALDG) and its (rowptr, col, w) stream through coalesced loads into shared
// memory, so the gathers of a Morton-ordered mesh graph -- 85-92 % of whose neighbour references fall inside the
// block (measured on the 1M-face icosphere, DESIGN.md §4.1) -- are shared-memory reads; only the references that
// leave the block go to L1/L2.  Replaces torch_geometric GCNConv.propagate (index_select -> mul -> scatter_add,
// reference util/networks.py:51-62,112-123) like spmm.cu; same epilogues (bias, BatchNorm partial sums, max|Y|).
//
// Mapping: CTA = row block of R rows, all C <= 128 channels, 256 threads.  A group of G = C/4 lanes owns one output
// row at a time (one float4 per lane); the 256/G groups walk the block's rows.  No global dependent-load chain is left
// in the loop: rowptr / col / w come from shared memory, in-block rows from the tile.
//   C = 32      : R = 256  (tile 32 KB)
//   C = 64, 128 : R = 128  (tile 32 / 64 KB)
// The wider layers run the gather kernel (spmm.cu): there a TMA tile of whole rows does not fit, and a 128-channel
// slice per CTA measured slower (DESIGN.md §4.1).
// Deterministic: no atomics; per-CTA BatchNorm partials are combined in group order.
// Roofline: HBM; algorithmic bytes 4*[(n+1) + 2*nnz + 2*n*C] (SURVEY.md §8d).
#include <cuda.h>

#include "common.cuh"

namespace ddmp {

namespace tile {

constexpr int kThreads = 256;
constexpr int kMetaPerRow = 9;          // (col, w) entries per row kept in shared memory (mesh graphs: <= 8 incl. loop)

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}" ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}
// 2-D tile of a row-major [rows, C] fp32 tensor: coordinates (c0 = first channel, c1 = first row)
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];"
        ::"r"(smem_u32(dst)), "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar)) : "memory");
}

struct Args {
    const int* rowptr;
    const int* col;
    const float* w;
    const float* H;
    const float* bias;
    float* Y;
    float* partials;      // [nblk][2][C] or null
    float* amax;          // [nblk] or null
    int64_t n;
};

template <int C, int R, bool STATS, bool BIAS>
__global__ void __launch_bounds__(kThreads)
spmm_tile_kernel(const __grid_constant__ CUtensorMap hmap, const Args a) {
    constexpr int G = C / 4;
    constexpr int GROUPS = kThreads / G;
    constexpr int kMetaCap = R * kMetaPerRow;
    static_assert(GROUPS * 2 * C * 4 <= R * C * 4, "the statistics scratch aliases the tile");
    extern __shared__ unsigned char smem_raw[];
    unsigned char* base = smem_raw + ((128u - (smem_u32(smem_raw) & 127u)) & 127u);    // TMA destination: 128 B aligned
    float* tile = reinterpret_cast<float*>(base);                                       // [R][C]
    float* red = tile;                                                                  // [GROUPS][2*C], after the loop
    int* scol = reinterpret_cast<int*>(base + (size_t)R * C * 4);                       // [kMetaCap]
    float* sw = reinterpret_cast<float*>(scol + kMetaCap);                              // [kMetaCap]
    int* srow = reinterpret_cast<int*>(sw + kMetaCap);                                  // [R + 1]
    uint64_t* barp = reinterpret_cast<uint64_t*>(srow + R + 2 + ((R & 1) ? 1 : 0));     // 8 B aligned
    float* wmax = reinterpret_cast<float*>(barp + 1);                                   // [kThreads / 32]
    uint64_t& bar = *barp;

    const int64_t blk = blockIdx.x;
    const int64_t row0 = blk * R;
    const int rows = (int)((row0 + R <= a.n) ? R : (a.n - row0));
    const int lane = threadIdx.x & 31;
    const int lg = threadIdx.x % G;
    const int gid = threadIdx.x / G;

    if (threadIdx.x == 0) {
        mbar_init(&bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        mbar_expect_tx(&bar, (uint32_t)(R * C * 4));             // rows past n are zero-filled and still counted
        tma_load_2d(tile, &hmap, 0, (int)row0, &bar);
    }
    // (rowptr, col, w) of the block -> shared memory, while the tile is in flight
    for (int i = threadIdx.x; i <= rows; i += kThreads) srow[i] = __ldg(a.rowptr + row0 + i);
    __syncthreads();
    const int kb = srow[0];
    const int nk = srow[rows] - kb;
    const bool meta_in_smem = nk <= kMetaCap;
    if (meta_in_smem) {
        for (int i = threadIdx.x; i < nk; i += kThreads) {
            scol[i] = __ldg(a.col + kb + i);
            sw[i] = __ldg(a.w + kb + i);
        }
    }
    float4 bsum = make_float4(0.f, 0.f, 0.f, 0.f);
    if (BIAS) bsum = ldg4(a.bias + lg * 4);
    float4 ssum = make_float4(0.f, 0.f, 0.f, 0.f), qsum = make_float4(0.f, 0.f, 0.f, 0.f);     // running mean, M2
    float cnt = 0.f;
    float amx = 0.f;
    __syncthreads();
    mbar_wait(&bar, 0);

    const float* Hs = a.H + lg * 4;
    for (int r = gid; r < rows; r += GROUPS) {
        const int s = srow[r] - kb, e = srow[r + 1] - kb;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        int k = s;
        // four references at a time: the (rare) out-of-block gathers of a batch are in flight together
        for (; k + 4 <= e; k += 4) {
            int c[4];
            float wv[4];
            float4 x[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                c[u] = meta_in_smem ? scol[k + u] : __ldg(a.col + kb + k + u);
                wv[u] = meta_in_smem ? sw[k + u] : __ldg(a.w + kb + k + u);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                const int64_t lc = (int64_t)c[u] - row0;
                if ((uint64_t)lc < (uint64_t)rows) x[u] = *reinterpret_cast<const float4*>(tile + (int)lc * C + lg * 4);
                else x[u] = ldg4(Hs + (int64_t)c[u] * C);
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
                acc.x = fmaf(wv[u], x[u].x, acc.x); acc.y = fmaf(wv[u], x[u].y, acc.y);
                acc.z = fmaf(wv[u], x[u].z, acc.z); acc.w = fmaf(wv[u], x[u].w, acc.w);
            }
        }
        for (; k < e; ++k) {
            const int c1 = meta_in_smem ? scol[k] : __ldg(a.col + kb + k);
            const float w1 = meta_in_smem ? sw[k] : __ldg(a.w + kb + k);
            const int64_t lc = (int64_t)c1 - row0;
            float4 x;
            if ((uint64_t)lc < (uint64_t)rows) x = *reinterpret_cast<const float4*>(tile + (int)lc * C + lg * 4);
            else x = ldg4(Hs + (int64_t)c1 * C);
            acc.x = fmaf(w1, x.x, acc.x); acc.y = fmaf(w1, x.y, acc.y);
            acc.z = fmaf(w1, x.z, acc.z); acc.w = fmaf(w1, x.w, acc.w);
        }
        if (BIAS) { acc.x += bsum.x; acc.y += bsum.y; acc.z += bsum.z; acc.w += bsum.w; }
        st4(a.Y + (row0 + r) * C + lg * 4, acc);
        amx = fmaxf(fmaxf(amx, fmaxf(fabsf(acc.x), fabsf(acc.y))), fmaxf(fabsf(acc.z), fabsf(acc.w)));
        if (STATS) {                                // Welford: running mean and M2 of this thread's rows (see bn.cu)
            cnt += 1.f;
            const float inv = 1.f / cnt;
            float d;
            d = acc.x - ssum.x; ssum.x = fmaf(d, inv, ssum.x); qsum.x = fmaf(d, acc.x - ssum.x, qsum.x);
            d = acc.y - ssum.y; ssum.y = fmaf(d, inv, ssum.y); qsum.y = fmaf(d, acc.y - ssum.y, qsum.y);
            d = acc.z - ssum.z; ssum.z = fmaf(d, inv, ssum.z); qsum.z = fmaf(d, acc.z - ssum.z, qsum.z);
            d = acc.w - ssum.w; ssum.w = fmaf(d, inv, ssum.w); qsum.w = fmaf(d, acc.w - ssum.w, qsum.w);
        }
    }

    if (STATS) {
        // per-group (mean, M2) -> shared memory (over the tile, which is dead now); then one thread per channel merges the
        // groups in group order (Chan et al.) and writes the block's (sum, M2 about the block mean)
        __syncthreads();
        st4(red + gid * 2 * C + lg * 4, ssum);
        st4(red + gid * 2 * C + C + lg * 4, qsum);
        __syncthreads();
        float* outp = a.partials + blk * 2 * C;
        for (int ch = threadIdx.x; ch < C; ch += kThreads) {
            float n_a = 0.f, mean = 0.f, m2 = 0.f;
#pragma unroll 4
            for (int g = 0; g < GROUPS; ++g) {
                const float n_b = (float)((rows - g + GROUPS - 1) / GROUPS);      // rows g, g+GROUPS, ... of this block
                if (g < rows) {
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
    }
    if (a.amax) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) amx = fmaxf(amx, __shfl_xor_sync(0xffffffffu, amx, o));
        if (lane == 0) wmax[threadIdx.x >> 5] = amx;
        __syncthreads();
        if (threadIdx.x == 0) {
            float m = wmax[0];
#pragma unroll
            for (int i = 1; i < kThreads / 32; ++i) m = fmaxf(m, wmax[i]);
            a.amax[blk] = m;
        }
    }
}

template <int C, int R>
constexpr size_t smem_bytes() {
    return 128 + (size_t)R * C * 4 + (size_t)R * kMetaPerRow * 8 + (size_t)(R + 4) * 4 + 8 + (kThreads / 32) * 4 + 16;
}

template <int C, int R>
static int launch(const Args& a, cudaStream_t st) {
    CUtensorMap map;
    int rc = make_tensor_map_2d(&map, a.H, a.n, C, R, C, false, "spmm_tile");
    if (rc != DDMP_OK) return rc;
    const int64_t nblk = ceil_div(a.n, R);
    const bool stats = a.partials != nullptr, bias = a.bias != nullptr;
    const size_t smem = smem_bytes<C, R>();
    static PerDeviceOnce configured;
    if (configured.need()) {
        const int mx = (int)smem;
        DDMP_CUDA(cudaFuncSetAttribute(spmm_tile_kernel<C, R, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
        DDMP_CUDA(cudaFuncSetAttribute(spmm_tile_kernel<C, R, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
        DDMP_CUDA(cudaFuncSetAttribute(spmm_tile_kernel<C, R, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
        DDMP_CUDA(cudaFuncSetAttribute(spmm_tile_kernel<C, R, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, mx));
        configured.mark();
    }
    if (stats) {
        if (bias) spmm_tile_kernel<C, R, true, true><<<(unsigned)nblk, kThreads, smem, st>>>(map, a);
        else spmm_tile_kernel<C, R, true, false><<<(unsigned)nblk, kThreads, smem, st>>>(map, a);
    } else {
        if (bias) spmm_tile_kernel<C, R, false, true><<<(unsigned)nblk, kThreads, smem, st>>>(map, a);
        else spmm_tile_kernel<C, R, false, false><<<(unsigned)nblk, kThreads, smem, st>>>(map, a);
    }
    return check_launch("spmm_tile");
}

}  // namespace tile

// the widths where this kernel beats the gather kernel on B200 (1M-face graphs, profiles/spmm_tile_ab_r2.txt); the TMA
// row coordinate is a 32-bit int
bool spmm_tile_supported(int64_t n, int C) {
    return n < (1ll << 31) && (C == 32 || C == 64 || C == 128);
}

int spmm_tile_launch(const int* rowptr, const int* col, const float* w, const float* H, const float* bias, float* Y,
                     float* partials, float* amax, int64_t n, int C, cudaStream_t st) {
    tile::Args a{rowptr, col, w, H, bias, Y, partials, amax, n};
    const int rpb = ddmp_rows_per_block(C);               // the BatchNorm partials are laid out per row block
    if (C == 32 && rpb == 256) return tile::launch<32, 256>(a, st);
    if (C == 64 && rpb == 128) return tile::launch<64, 128>(a, st);
    if (C == 128 && rpb == 128) return tile::launch<128, 128>(a, st);
    set_error("spmm_tile: no instantiation for C=%d rows_per_block=%d", C, rpb);
    return DDMP_ERR_UNSUPPORTED;
}

}  // namespace ddmp
