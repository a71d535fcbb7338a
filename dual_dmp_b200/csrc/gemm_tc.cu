// Dense feature transform on the 5th-generation tensor cores (DDMP_GEMM_TC): fp32 products emulated with three MMAs
// on error-compensated operand splits, fp32 accumulation in TMEM (the 1e-4 parity contract rules out plain TF32 /
// fp16, SURVEY.md §7 hard part 1).  Two splits:
//   * fp16 (kind::f16, default when the caller supplies operand bounds): s*x = hi + lo in fp16, operands scaled by
//     powers of two from device-side bounds -- section "fp32 emulation with three fp16 MMAs" below;
//   * TF32 (kind::tf32): x = hi + lo in TF32, no range restriction, half the MMA rate.
//
//   NT kernels (xw, dx):  C[M=rows, N] = act(A)[rows, K] * B[N, K]^T        A, B K-major
//   TN kernels (dw)    :  C[M, N] = sum_rows A[rows, M]^T * act(B)[rows, N]  A, B MN-major, split-K over rows
//
// The activation operand cannot go to the tensor core as loaded: the previous layer's BatchNorm + LeakyReLU, the scale
// and the hi/lo split are applied while the tile is staged, so producer warps do  ld.global -> transform -> st.shared
// into the 128-byte-swizzled UMMA canonical layout (fp16 kernels at K <= 256: raw fp32 tiles by TMA, then
// ld.shared -> transform -> st.shared); the (pre-split, pre-swizzled) weights arrive by cp.async.bulk.
// One elected thread issues the MMAs; `full`/`empty` mbarriers per smem stage; tcgen05.commit releases a stage /
// publishes the accumulator; dedicated warps drain the double-buffered TMEM accumulator.  CTA pairs (cta_group::2)
// where the shapes allow.  Kernel inventory and measured behaviour: DESIGN.md §4.2, profiles/README.md.
#include <cuda.h>
#include <cuda_fp16.h>
#include <stdlib.h>

#include <atomic>
#include <type_traits>

#include "common.cuh"

namespace ddmp {
namespace tc {

constexpr int kProducerWarps = 8;
constexpr int kProducerThreads = kProducerWarps * 32;
constexpr int BM = 128;                              // UMMA M
constexpr int BK = 32;                               // 32 fp32 = 128 bytes = one swizzle atom row
constexpr int UMMA_K = 8;                            // kind::tf32

// ---- PTX wrappers ---------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra.uni WAIT_DONE;\n"
        "bra.uni WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// tf32 split x = hi + lo: hi = x rounded to 10 mantissa bits (round-half-up in magnitude with an integer add, 2
// ops instead of the ~5 that cvt.rna.tf32 expands to), lo = exact remainder x - hi with its low 13 bits cleared
// (|lo| <= 2^-11 |x|, so the dropped part is <= 2^-22 |x|).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
    hi = (__float_as_uint(x) + 0x1000u) & 0xFFFFE000u;
    lo = __float_as_uint(x - __uint_as_float(hi)) & 0xFFFFE000u;
}
__device__ __forceinline__ void sts128(uint32_t saddr, const uint4& v) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
                 : "memory");
}
__device__ __forceinline__ float lrelu_max(float z, float slope) { return fmaxf(z, z * slope); }   // 0 < slope < 1

// ---- descriptors ----------------------------------------------------------------------------------------------------
// shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start>>4 [0,14) | LBO>>4 [16,30) | SBO>>4 [32,46) |
// version=1 [46,48) | layout_type [61,64) (2 = SWIZZLE_128B, 1 = SWIZZLE_128B_BASE32B)
__device__ __forceinline__ uint64_t make_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes,
                                              uint32_t layout_type = 2) {
    uint64_t d = 0;
    d |= (uint64_t)((saddr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)layout_type << 61;
    return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor) for kind::tf32, fp32 accumulate
__host__ __device__ constexpr uint32_t make_idesc(int M, int N, bool a_mn_major, bool b_mn_major) {
    return (1u << 4)                       // c_format = F32
           | (2u << 7) | (2u << 10)        // a_format = b_format = TF32
           | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}

// byte offset of (row r, 16-byte chunk c) inside a K-major SWIZZLE_128B tile whose rows are 128 bytes
__device__ __forceinline__ uint32_t sw128(uint32_t r, uint32_t c) { return r * 128u + ((c ^ (r & 7u)) << 4); }


// ---- NT kernel, version 2: persistent, B streamed by TMA bulk copies, epilogue overlapped ---------------------------
// The weights (B operand) are split into hi/lo and laid out ONCE per call in the exact swizzled shared-memory image
// (tc_prep_b_kernel: [n_tile][k_block][hi|lo][BN rows x 128 B]), so a stage's B part is one contiguous blob that a
// single thread streams with cp.async.bulk (SASS UBLKCP) onto the stage's `full` mbarrier.  Only the activation
// operand still goes through the producer warps (BatchNorm + LeakyReLU + split need registers).  CTAs are persistent
// (tile = blockIdx.x + i*gridDim.x, n-tile fastest so the CTAs that share an A row block run together), the
// accumulator is double-buffered in TMEM (2 x BN columns) and four dedicated warps drain tile i while tile i+1 is
// being multiplied.
constexpr int kV2Threads = 16 * 32;   // warps 0-7 producers | 8 MMA | 9 B loader | 10,11 idle | 12-15 epilogue

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

struct Nt2Args {
    const float* A;
    const uint8_t* Bimg;  // pre-split, pre-swizzled weights
    float* C;
    const int* a_map;
    const float* scale;
    const float* shift;
    float slope;
    int64_t M;
    int N, K;
    int tiles_n;
    int64_t num_tiles;
};

// W [N,K] (or, transposed, W^T given as [K,N]) -> image; one thread per (n, 16-byte chunk of K)
// byte offset of (row r, 16-byte chunk c) in a K-major tile with rows of KB*4 bytes: SWIZZLE_128B (KB=32) / _64B (KB=16)
template <int KB>
__device__ __forceinline__ uint32_t swz(uint32_t r, uint32_t c) {
    if constexpr (KB == 32) return r * 128u + ((c ^ (r & 7u)) << 4);
    else return r * 64u + ((c ^ ((r >> 1) & 3u)) << 4);
}

template <int KB>
__global__ void tc_prep_b_kernel(const float* __restrict__ W, int transposed, uint8_t* __restrict__ img, int N, int K,
                                 int BN) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int kc = K / 4;
    if (i >= (int64_t)N * kc) return;
    const int n = (int)(i / kc), k = (int)(i % kc) * 4;
    float4 v;
    if (!transposed) {
        v = ldg4(W + (int64_t)n * K + k);
    } else {
        v.x = __ldg(W + (int64_t)(k + 0) * N + n); v.y = __ldg(W + (int64_t)(k + 1) * N + n);
        v.z = __ldg(W + (int64_t)(k + 2) * N + n); v.w = __ldg(W + (int64_t)(k + 3) * N + n);
    }
    uint4 hi, lo;
    split_tf32(v.x, hi.x, lo.x); split_tf32(v.y, hi.y, lo.y); split_tf32(v.z, hi.z, lo.z); split_tf32(v.w, hi.w, lo.w);
    const int n_tile = n / BN, r = n % BN, kb = k / KB, c = (k % KB) / 4;
    const int num_kb = K / KB;
    const int64_t base = ((int64_t)n_tile * num_kb + kb) * 2 * ((int64_t)BN * KB * 4);
    const uint32_t off = swz<KB>((uint32_t)r, (uint32_t)c);
    *reinterpret_cast<uint4*>(img + base + off) = hi;
    *reinterpret_cast<uint4*>(img + base + (int64_t)BN * KB * 4 + off) = lo;
}

template <int BN, int STAGES, bool DEEP, int KB>
__global__ void __launch_bounds__(kV2Threads, 1) tc_gemm_nt2_kernel(const Nt2Args g) {
    constexpr int BK = KB;                           // shadows the file-level BK inside this kernel
    constexpr uint32_t ROW_BYTES = KB * 4;           // 128 (SWIZZLE_128B) or 64 (SWIZZLE_64B)
    constexpr uint32_t CPR = KB / 4;                 // 16-byte chunks per row
    constexpr uint32_t SBO = 8 * ROW_BYTES;          // 8-row swizzle atom
    constexpr uint32_t LTYPE = (KB == 32) ? 2u : 4u; // descriptor layout type
    constexpr uint32_t A_BYTES = BM * ROW_BYTES;
    constexpr uint32_t B_BYTES = BN * ROW_BYTES;
    constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    constexpr uint32_t TMEM_COLS = 2 * BN;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* acc_full = empty_bar + STAGES;     // [2]
    uint64_t* acc_empty = acc_full + 2;          // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
    uint8_t* staging = smem + STAGES * STAGE_BYTES + 256;   // 4 epilogue warps x 32 rows x 128 B

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_kb = g.K / BK;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar + s, kProducerWarps + 1);
            mbar_init(empty_bar + s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(acc_full + b, 1);
            mbar_init(acc_empty + b, 4);
        }
        fence_barrier_init();
    }
    if (warp == 8) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t smem_base = smem_u32(smem);

    if (warp < kProducerWarps) {
        // ===== A producers: flattened (tile, k-block) iteration space, global loads issued two iterations ahead =====
        const int t = threadIdx.x;
        const uint32_t c = t % CPR;
        const bool has_act = g.scale != nullptr;
        constexpr int NJ = BM * CPR / kProducerThreads;      // float4 per thread per k-block
        constexpr int RPP = kProducerThreads / CPR;          // rows covered by one pass of the producer threads
        if constexpr (!DEEP) {
            // loads of a k-block are issued at the top of its own iteration (one iteration of prefetch over the wait)
            uint32_t it = 0;
            for (int64_t tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x) {
                const int64_t m0 = (tile / g.tiles_n) * BM;
                int64_t src_row[NJ];
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int64_t m = m0 + (t / CPR) + j * RPP;
                    src_row[j] = (m < g.M) ? (g.a_map ? (int64_t)__ldg(g.a_map + m) : m) : -1;
                }
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    const int k0 = kb * BK + c * 4;
                    float4 av[NJ];
#pragma unroll
                    for (int j = 0; j < NJ; ++j)
                        av[j] = (src_row[j] >= 0) ? ldg4(g.A + src_row[j] * g.K + k0)
                                                                       : make_float4(0.f, 0.f, 0.f, 0.f);
                    float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (has_act) { sc = ldg4(g.scale + k0); sh = ldg4(g.shift + k0); }
                    mbar_wait(empty_bar + s, ph ^ 1u);
                    const uint32_t st = smem_base + s * STAGE_BYTES;
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        const uint32_t row = (t / CPR) + j * RPP;
                        float4 a = av[j];
                        if (has_act && src_row[j] >= 0) {
                            a.x = lrelu_max(fmaf(a.x, sc.x, sh.x), g.slope); a.y = lrelu_max(fmaf(a.y, sc.y, sh.y), g.slope);
                            a.z = lrelu_max(fmaf(a.z, sc.z, sh.z), g.slope); a.w = lrelu_max(fmaf(a.w, sc.w, sh.w), g.slope);
                        }
                        uint4 hi, lo;
                        split_tf32(a.x, hi.x, lo.x); split_tf32(a.y, hi.y, lo.y);
                        split_tf32(a.z, hi.z, lo.z); split_tf32(a.w, hi.w, lo.w);
                        const uint32_t off = swz<KB>(row, c);
                        sts128(st + off, hi);
                        sts128(st + A_BYTES + off, lo);
                    }
                    fence_proxy_async();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(full_bar + s);
                }
            }
        } else {
            const int64_t my_tiles = (g.num_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x;
            const int64_t total = my_tiles * num_kb;
            float4 av[2][NJ];
            bool ok[2][NJ];
            // prefetch cursor (advanced incrementally: no divisions in the loop)
            int64_t pf_tile = blockIdx.x;
            int pf_kb = 0;
            int64_t pf_left = total;
            auto issue = [&](auto slot_c) {
                constexpr int slot = decltype(slot_c)::value;      // compile-time slot keeps av[][] in registers
                if (pf_left <= 0) return;
                const int64_t m0 = (int64_t)((uint32_t)pf_tile / (uint32_t)g.tiles_n) * BM;   // num_tiles < 2^31
                const int k0 = pf_kb * BK + c * 4;
    #pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const int64_t m = m0 + (t / CPR) + j * RPP;
                    ok[slot][j] = m < g.M;
                    if (ok[slot][j]) {
                        const int64_t src = g.a_map ? (int64_t)__ldg(g.a_map + m) : m;
                        av[slot][j] = ldg4(g.A + src * g.K + k0);
                    } else {
                        av[slot][j] = make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                }
                --pf_left;
                if (++pf_kb == num_kb) { pf_kb = 0; pf_tile += gridDim.x; }
            };
            using S0 = std::integral_constant<int, 0>;
            using S1 = std::integral_constant<int, 1>;
            issue(S0{});
            issue(S1{});
            int s = 0, kb_cur = 0;
            uint32_t ph = 0;
            auto step = [&](auto slot_c) {
                constexpr int slot = decltype(slot_c)::value;
                const int k0 = kb_cur * BK + c * 4;
                float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
                if (has_act) { sc = ldg4(g.scale + k0); sh = ldg4(g.shift + k0); }
                mbar_wait(empty_bar + s, ph ^ 1u);
                const uint32_t st = smem_base + s * STAGE_BYTES;
    #pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    const uint32_t row = (t / CPR) + j * RPP;
                    float4 a = av[slot][j];
                    if (has_act && ok[slot][j]) {
                        a.x = lrelu_max(fmaf(a.x, sc.x, sh.x), g.slope); a.y = lrelu_max(fmaf(a.y, sc.y, sh.y), g.slope);
                        a.z = lrelu_max(fmaf(a.z, sc.z, sh.z), g.slope); a.w = lrelu_max(fmaf(a.w, sc.w, sh.w), g.slope);
                    }
                    uint4 hi, lo;
                    split_tf32(a.x, hi.x, lo.x); split_tf32(a.y, hi.y, lo.y);
                    split_tf32(a.z, hi.z, lo.z); split_tf32(a.w, hi.w, lo.w);
                    const uint32_t off = swz<KB>(row, c);
                    sts128(st + off, hi);
                    sts128(st + A_BYTES + off, lo);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(full_bar + s);
                if (++s == STAGES) { s = 0; ph ^= 1u; }
                if (++kb_cur == num_kb) kb_cur = 0;
                issue(slot_c);                                    // refill the slot just consumed
            };
            for (int64_t it = 0; it < total; it += 2) {
                step(S0{});
                if (it + 1 < total) step(S1{});
            }
        }
    } else if (warp == 8) {
        // ===== MMA issuer =====
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc(BM, BN, false, false);
            uint32_t it = 0, tile_no = 0;
            for (int64_t tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++tile_no) {
                const uint32_t buf = tile_no & 1u;
                mbar_wait(acc_empty + buf, ((tile_no >> 1) & 1u) ^ 1u);
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * BN;
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(full_bar + s, ph);
                    tc_fence_after();
                    const uint32_t sa = smem_base + s * STAGE_BYTES;
#pragma unroll
                    for (int ks = 0; ks < BK / UMMA_K; ++ks) {
                        const uint32_t koff = ks * UMMA_K * 4;
                        const uint64_t a_hi = make_desc(sa + koff, 16, SBO, LTYPE);
                        const uint64_t a_lo = make_desc(sa + A_BYTES + koff, 16, SBO, LTYPE);
                        const uint64_t b_hi = make_desc(sa + 2 * A_BYTES + koff, 16, SBO, LTYPE);
                        const uint64_t b_lo = make_desc(sa + 2 * A_BYTES + B_BYTES + koff, 16, SBO, LTYPE);
                        umma_tf32(d_tmem, a_lo, b_hi, idesc, (kb | ks) != 0);
                        umma_tf32(d_tmem, a_hi, b_lo, idesc, 1);
                        umma_tf32(d_tmem, a_hi, b_hi, idesc, 1);
                    }
                    umma_commit(empty_bar + s);
                }
                umma_commit(acc_full + buf);
            }
        }
        __syncwarp();
    } else if (warp == 9) {
        // ===== B loader: one bulk copy per stage =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int64_t tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x) {
                const int tn = (int)(tile % g.tiles_n);
                const uint8_t* src = g.Bimg + (int64_t)tn * num_kb * (2 * (int64_t)B_BYTES);
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(empty_bar + s, ph ^ 1u);
                    mbar_arrive_expect_tx(full_bar + s, 2 * B_BYTES);
                    bulk_g2s(smem_base + s * STAGE_BYTES + 2 * A_BYTES, src + (int64_t)kb * (2 * (int64_t)B_BYTES),
                             2 * B_BYTES, full_bar + s);
                }
            }
        }
        __syncwarp();
    } else if (warp >= 12) {
        // ===== epilogue: TMEM -> registers -> (smem transpose) -> global, overlapped with the next tile's main loop =====
        // tcgen05.ld hands every thread one ROW (32 columns); writing that straight out makes each warp store touch 32
        // rows x 16 B.  A 16-KB swizzled staging tile per warp turns it into 4 rows x 128 B per store instruction.
        const int q = warp & 3;
        const uint32_t stg = smem_u32(staging) + (uint32_t)q * (32u * 128u);
        uint32_t tile_no = 0;
        for (int64_t tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++tile_no) {
            const uint32_t buf = tile_no & 1u;
            const int64_t mrow0 = (tile / g.tiles_n) * BM + q * 32;
            const int n0 = (int)(tile % g.tiles_n) * BN;
            mbar_wait(acc_full + buf, (tile_no >> 1) & 1u);
            tc_fence_after();
#pragma unroll 1
            for (int cb = 0; cb < BN; cb += 32) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN + (uint32_t)cb, v);
#pragma unroll
                for (int i = 0; i < 8; ++i)          // row = lane, 16-byte chunk i -> swizzled chunk i ^ (lane & 7)
                    sts128(stg + (uint32_t)lane * 128u + (uint32_t)((i ^ (lane & 7)) << 4),
                           make_uint4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int r = j * 4 + (lane >> 3), cc = lane & 7;
                    uint4 o;
                    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                                 : "=r"(o.x), "=r"(o.y), "=r"(o.z), "=r"(o.w)
                                 : "r"(stg + (uint32_t)r * 128u + (uint32_t)((cc ^ (r & 7)) << 4)));
                    const int64_t m = mrow0 + r;
                    if (m < g.M)
                        *reinterpret_cast<uint4*>(g.C + m * g.N + n0 + cb + cc * 4) = o;
                }
                __syncwarp();
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(acc_empty + buf);
        }
    }
    __syncthreads();
    if (warp == 8) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

template <int BN, int STAGES, bool DEEP, int KB>
static int launch_nt2_impl(const Nt2Args& g, cudaStream_t st) {
    constexpr size_t smem = (size_t)STAGES * (2 * BM * KB * 4 + 2 * BN * KB * 4) + 1024 + 256 + 4 * 32 * 128;
    static PerDeviceOnce configured;
    if (configured.need()) {
        DDMP_CUDA(cudaFuncSetAttribute(tc_gemm_nt2_kernel<BN, STAGES, DEEP, KB>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured.mark();
    }
    const int64_t grid = g.num_tiles < kNumSMs ? g.num_tiles : kNumSMs;
    tc_gemm_nt2_kernel<BN, STAGES, DEEP, KB><<<(unsigned)grid, kV2Threads, smem, st>>>(g);
    return check_launch("tc_gemm_nt2");
}
// K-block: 32 fp32 = one 128-byte swizzle row.  Measured on B200 (profiles/gemm_ab_r1.txt): a 16-wide k-block
// (SWIZZLE_64B, twice the stages) is 10-15 % slower, and a 2-deep register prefetch 8 % slower than issuing the loads at the
// top of the iteration -- the kernel is throughput-, not latency-bound; both variants were dropped.
template <int BN, int STAGES32>
static int launch_nt2(const Nt2Args& g, cudaStream_t st) {
    return launch_nt2_impl<BN, STAGES32, false, 32>(g, st);
}

// B = W [N,K] row-major (transposed == 0) or B = W^T where W is [K,N] row-major (transposed == 1)
static int run_nt2(const float* A, const int* a_map, const float* scale, const float* shift, float slope,
                   const float* W, int transposed, void* workspace, float* C, int64_t M, int N, int K,
                   cudaStream_t st) {
    const int BN = (N % 256 == 0) ? 256 : ((N % 128 == 0) ? 128 : ((N % 64 == 0) ? 64 : 32));
    uint8_t* img = reinterpret_cast<uint8_t*>(workspace);
    const int64_t chunks = (int64_t)N * (K / 4);
    tc_prep_b_kernel<32><<<(unsigned)ceil_div(chunks, 256), 256, 0, st>>>(W, transposed, img, N, K, BN);
    int rc = check_launch("tc_prep_b");
    if (rc) return rc;
    Nt2Args g{};
    g.A = A; g.Bimg = img; g.C = C; g.a_map = a_map; g.scale = scale; g.shift = shift; g.slope = slope;
    g.M = M; g.N = N; g.K = K; g.tiles_n = N / BN;
    g.num_tiles = ceil_div(M, BM) * g.tiles_n;
    DDMP_REQUIRE(g.num_tiles < (1ll << 31), "tc gemm: too many tiles");
    if (BN == 256) return launch_nt2<256, 2>(g, st);
    if (BN == 128) return launch_nt2<128, 3>(g, st);
    if (BN == 64) return launch_nt2<64, 4>(g, st);
    return launch_nt2<32, 4>(g, st);              // 32-wide outputs of the narrow layers (xw 64 -> 32, dx of 32 -> 64)
}

// ---- CTA pairs (cta_group::2): helpers of the fp16-split pair kernels below ---------------------------------------------
// Two CTAs of one cluster (same TPC) compute a 256-row tile with M=256 MMAs issued by the leader CTA: each CTA stages its
// own 128 rows of A and only HALF of the B tile, the tensor core reads both halves, and each CTA's TMEM receives its 128
// output rows.  Synchronisation across the pair: the peer's producers / B-loader arrive on the peer's own `full` barrier; a
// relay thread there forwards it to the leader's `peer_ready` barrier (remote mbarrier arrive); tcgen05.commit with the
// multicast mask 0b11 releases a stage / publishes the accumulator in both CTAs; the peer's epilogue warps arrive remotely
// on the leader's `acc_empty`.  (The 3xTF32 pair kernel this scheme was first built for, round 1, gained 0-4 % over the
// single-CTA kernel and was removed when the fp16 split became the default.)
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t cta) {
    asm volatile(
        "{\n"
        ".reg .b32 remaddr;\n"
        "mapa.shared::cluster.u32 remaddr, %0, %1;\n"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [remaddr];\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(cta)
        : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "WAITC_LOOP:\n"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra.uni WAITC_DONE;\n"
        "bra.uni WAITC_LOOP;\n"
        "WAITC_DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_2cta(uint32_t* dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2cta(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_commit_2cta(uint64_t* bar) {
    asm volatile(
        "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
            smem_u32(bar)),
        "h"((uint16_t)3)
        : "memory");
}
// ---- fp32 emulation with three fp16 MMAs (kind::f16) ----------------------------------------------------------------
// x*s = hi + lo with hi = fp16(x*s), lo = fp16(x*s - hi): two round-to-nearest 11-bit pieces carry 22+ bits of x, so
// hi*hi + hi*lo + lo*hi (fp32 accumulation in TMEM) has the accuracy of an fp32 product sum (measured: closer to the
// float64 result than the 3xTF32 split, whose pieces are truncated).  kind::f16 issues at twice the kind::tf32 rate
// and every operand byte count halves (shared-memory reads/writes, the weight image streamed from L2).
// fp16 has 5 exponent bits, so each operand is multiplied by a power of two `s` (exact) chosen from an upper bound of
// its magnitude: s*|x| < 2^15.  Elements more than 2^17 below the bound lose low bits of `lo` (absolute error
// <= 2^-40 of the bound).  The caller supplies the bound as a device array whose maximum is taken in-kernel
// (`amax`): the BatchNorm bound |gamma|*sqrt(n-1)+|beta| for activated inputs (no sample is more than sqrt(n-1)
// biased standard deviations from the batch mean), per-row-block maxima written by the aggregation kernel for
// gradients.  Weights are scaled per output row by the prep kernel.  Without a bound the 3xTF32 kernels run.
constexpr int BK16 = 64;                             // 64 fp16 = 128 bytes = one swizzle atom row
constexpr int UMMA_K16 = 16;                         // kind::f16

__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                         uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// instruction descriptor for kind::f16 with fp16 inputs (a_format = b_format = 0), fp32 accumulate
__host__ __device__ constexpr uint32_t make_idesc16(int M, int N, bool a_mn_major, bool b_mn_major) {
    return (1u << 4) | ((a_mn_major ? 1u : 0u) << 15) | ((b_mn_major ? 1u : 0u) << 16) | ((uint32_t)(N >> 3) << 17) |
           ((uint32_t)(M >> 4) << 24);
}
// bits of a non-negative float bound -> s = 2^(141-E) (s*bound < 2^15) and 1/s; E = biased exponent, clamped so that
// both stay normal floats (an all-zero operand gets a huge but finite scale; inf/NaN propagate through s*x)
__device__ __forceinline__ void scale_from_bits(uint32_t bits, float& s, float& inv_s) {
    uint32_t E = (bits >> 23) & 0xFFu;
    E = E < 16u ? 16u : (E > 252u ? 252u : E);
    s = __uint_as_float((268u - E) << 23);
    inv_s = __uint_as_float((E - 14u) << 23);
}
__device__ __forceinline__ void split_f16x2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
    const __half2 h = __floats2half2_rn(x0, x1);                     // x0 -> low half (lower address)
    const float2 hf = __half22float2(h);
    const __half2 l = __floats2half2_rn(x0 - hf.x, x1 - hf.y);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}
// 8 consecutive k values (already scaled) -> one 16-byte chunk of hi and one of lo
__device__ __forceinline__ void split_f16x8(const float4& a, const float4& b, uint4& hi, uint4& lo) {
    split_f16x2(a.x, a.y, hi.x, lo.x); split_f16x2(a.z, a.w, hi.y, lo.y);
    split_f16x2(b.x, b.y, hi.z, lo.z); split_f16x2(b.z, b.w, hi.w, lo.w);
}
// max |arr[i]| over the whole CTA -> bits, via `slot` (shared, zeroed before the preceding __syncthreads)
__device__ __forceinline__ void block_amax_bits(const float* __restrict__ arr, int64_t len, uint32_t* slot) {
    uint32_t m = 0;
    for (int64_t i = threadIdx.x; i < len; i += blockDim.x) {
        const uint32_t b = __float_as_uint(fabsf(__ldg(arr + i)));
        m = b > m ? b : m;
    }
    m = __reduce_max_sync(0xffffffffu, m);
    if ((threadIdx.x & 31) == 0) atomicMax(slot, m);                 // integer max: order-independent
}

struct Nt16Args {
    const float* A;
    const uint8_t* Bimg;     // fp16 hi/lo image of the scaled weights: [n_tile][k_block][hi|lo][BN rows x 128 B]
    const float* inv_sw;     // [N] 1 / (scale of weight row n)
    float* C;
    const int* a_map;
    const float* scale;
    const float* shift;
    float slope;
    const float* amax;       // bound of |act(A)|: max over this array
    int64_t amax_len;
    unsigned long long* trace;   // profiling only (DDMP_TC_TRACE=1): per-role cycle counters of CTA 0
    int flags;               // DDMP_TC_F16_FLAGS. bit 0: prefetch the next tile's A rows into L2; bit 3: unstaged epilogue
    int64_t M;
    int N, K;
    int tiles_n;
    int64_t num_tiles;
};

// A-operand producer of the fp16-split NT kernels.  16 consecutive lanes read the 256 bytes (64 fp32) a row
// contributes to the k-block, so one warp-wide 16-byte load covers 2 rows x 256 B = four full 128-byte lines (an
// earlier mapping gave every thread 8 consecutive k as two 16-byte loads: each warp load then touched eight
// half-used lines and the LSU data pipe, at 77 % busy, bounded the kernel: ncu, profiles/).  A thread's 4 k values
// become 8 bytes of hi and 8 bytes of lo; the pair of lanes that shares a 16-byte swizzle chunk writes its halves.
constexpr int kProdNJ = BM * 16 / kProducerThreads;      // rows per thread per k-block (8)
constexpr int kProdRPP = kProducerThreads / 16;          // rows covered by one pass of the producer threads (16)
__device__ __forceinline__ void sts64(uint32_t saddr, uint32_t x, uint32_t y) {
    asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(saddr), "r"(x), "r"(y) : "memory");
}
// A k-block touches 256 bytes of each of the tile's 128 rows (stride K*4), and the next 256 bytes of the same rows a
// microsecond later: DRAM sees short scattered bursts (measured: every shape of the fp16-split kernel ran at
// ~3.6 TB/s of operand + result traffic).  Pulling the NEXT tile's rows into L2 as whole rows while the current tile
// is multiplied makes the DRAM reads long and sequential and turns the producers' loads into L2 hits.
template <class Args>
__device__ __forceinline__ void prefetch_tile_l2(const Args& g, int64_t m0) {
    const int t = threadIdx.x;
    if (t >= BM) return;
    const int64_t m = m0 + t;
    if (m >= g.M) return;
    const int64_t r = g.a_map ? (int64_t)__ldg(g.a_map + m) : m;
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(g.A + r * g.K), "r"((uint32_t)g.K * 4u) : "memory");
}
// 16-byte read-only load the compiler may not move: the prefetch below depends on the loads of the NEXT k-block being
// issued before the current one is transformed (plain __ldg loads get sunk below the transform to save registers).
__device__ __forceinline__ float4 ldg4_pinned(const float* p) {
    float4 v;
    asm volatile("ld.global.nc.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}
// The producer loop of a CTA: (tile, k-block) pairs flattened, the loads of pair i+1 in flight while pair i is
// transformed (two register buffers, ping-pong by unrolling).  Cycle counters (DDMP_TC_TRACE) showed the producers,
// not the tensor pipe, set the pace of the fp16-split kernel: per k-block 420 cycles issuing loads, ~100 waiting for
// a free stage and 1600 between the wait and the arrive, most of it load latency, while the MMA thread waited
// 1100 cycles per k-block for `full`.
template <int STAGES, class Args, class WaitEmpty>
__device__ __forceinline__ void produce_loop(const Args& g, int64_t first_tile, int64_t tile_step, int64_t row_mul,
                                                    int64_t row_add, int num_kb, float s_a, uint32_t smem_base,
                                                    uint32_t stage_bytes, uint32_t a_bytes, uint64_t* full_bar,
                                                    uint64_t* empty_bar, WaitEmpty wait_empty) {
    constexpr int NJ = kProdNJ, RPP = kProdRPP;
    const int t = threadIdx.x, lane = threadIdx.x & 31;
    const int c8 = (t & 15) * 4;
    const uint32_t c4 = t & 15;
    const bool has_act = g.scale != nullptr;
    const int64_t my_tiles = first_tile < g.num_tiles ? (g.num_tiles - first_tile + tile_step - 1) / tile_step : 0;
    const uint32_t total = (uint32_t)(my_tiles * num_kb);
    // load cursor
    int64_t lc_tile = first_tile;
    int lc_kb = 0;
    const float* rp[NJ];                                  // row pointers of the cursor's tile (nullptr: past the end)
    auto set_rows = [&](int64_t tile) {
        const int64_t m0 = (tile / g.tiles_n) * row_mul + row_add;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const int64_t m = m0 + (t >> 4) + j * RPP;
            const int64_t r = (m < g.M) ? (g.a_map ? (int64_t)__ldg(g.a_map + m) : m) : -1;
            rp[j] = r >= 0 ? g.A + r * g.K + c8 : nullptr;
        }
        if ((g.flags & 1) && tile + tile_step < g.num_tiles)
            prefetch_tile_l2(g, ((tile + tile_step) / g.tiles_n) * row_mul + row_add);
    };
    auto load = [&](float4 (&buf)[NJ], uint32_t& vmask, int& k0) {
        k0 = lc_kb * BK16;
        vmask = 0;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            if (rp[j]) {
                buf[j] = ldg4_pinned(rp[j] + k0);
                vmask |= 1u << j;
            } else {
                buf[j] = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        if (++lc_kb == num_kb) {
            lc_kb = 0;
            lc_tile += tile_step;
            if (lc_tile < g.num_tiles) set_rows(lc_tile);
        }
    };
    auto process = [&](float4 (&buf)[NJ], uint32_t vmask, int k0, uint32_t it) {
        const int s = it % STAGES;
        const uint32_t ph = (it / STAGES) & 1;
        const bool tr = g.trace && blockIdx.x == 0 && t == 0;
        long long c1 = 0, c2 = 0, c3 = 0;
        // the power-of-two operand scale is folded into the affine part (LeakyReLU is positively homogeneous)
        float4 sc = make_float4(s_a, s_a, s_a, s_a), sh = make_float4(0.f, 0.f, 0.f, 0.f);
        if (has_act) {
            sc = ldg4(g.scale + k0 + c8);
            sh = ldg4(g.shift + k0 + c8);
            sc.x *= s_a; sc.y *= s_a; sc.z *= s_a; sc.w *= s_a;
            sh.x *= s_a; sh.y *= s_a; sh.z *= s_a; sh.w *= s_a;
        }
        if (tr) c1 = clock64();
        wait_empty(empty_bar + s, ph ^ 1u);
        if (tr) c2 = clock64();
        const uint32_t st = smem_base + s * stage_bytes;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const uint32_t row = (t >> 4) + j * RPP;
            float4 a = buf[j];
            if (has_act) {
                if (vmask & (1u << j)) {
                    a.x = lrelu_max(fmaf(a.x, sc.x, sh.x), g.slope); a.y = lrelu_max(fmaf(a.y, sc.y, sh.y), g.slope);
                    a.z = lrelu_max(fmaf(a.z, sc.z, sh.z), g.slope); a.w = lrelu_max(fmaf(a.w, sc.w, sh.w), g.slope);
                }
            } else {
                a.x *= s_a; a.y *= s_a; a.z *= s_a; a.w *= s_a;
            }
            uint32_t h0, l0, h1, l1;
            split_f16x2(a.x, a.y, h0, l0);
            split_f16x2(a.z, a.w, h1, l1);
            const uint32_t off = sw128(row, c4 >> 1) + ((c4 & 1u) << 3);
            sts64(st + off, h0, h1);
            sts64(st + a_bytes + off, l0, l1);
        }
        long long cA = 0, cB = 0;
        if (tr) cA = clock64();
        fence_proxy_async();
        if (tr) cB = clock64();
        __syncwarp();
        if (tr) c3 = clock64();
        if (lane == 0) mbar_arrive(full_bar + s);
        if (tr) {
            g.trace[1] += (unsigned long long)(c2 - c1);     // wait for a free stage
            g.trace[2] += (unsigned long long)(c3 - c2);     // wait for data + transform + stores + fence
            g.trace[3] += 1ull;
            g.trace[14] += (unsigned long long)(cA - c2);    // ... of which: data wait + transform + store issue
            g.trace[15] += (unsigned long long)(cB - cA);    // ... fence.proxy.async
        }
    };
    float4 buf0[NJ], buf1[NJ];
    uint32_t vm0 = 0, vm1 = 0;
    int k0 = 0, k1 = 0;
    if (total > 0) {
        set_rows(lc_tile);
        load(buf0, vm0, k0);
    }
    for (uint32_t it = 0; it < total; it += 2) {
        if (it + 1 < total) load(buf1, vm1, k1);
        process(buf0, vm0, k0, it);
        if (it + 1 >= total) break;
        if (it + 2 < total) load(buf0, vm0, k0);
        process(buf1, vm1, k1, it + 1);
    }
}

// ---- A operand by TMA (no row gather; where run_nt16 selects it) -----------------------------------------------------
// The register-fed producers above keep at most two k-blocks of A in flight per warp (~64 KB per SM) and pay the load
// latency plus the transform once per k-block, which set the pace at K <= 256 (2-4 k-blocks of ~1.5 k MMA cycles per
// tile) and wherever the BatchNorm + LeakyReLU prologue is applied.  Here one thread streams the raw fp32 A tile into a ring of `RAW` slots with TMA tensor loads
// (two 128-row x 32-column boxes per k-block, 128-byte swizzle: the inner box dimension is limited to 128 bytes), and
// the producer warps become shared -> shared transform warps: ld.shared -> BatchNorm + LeakyReLU + scale -> hi/lo split
// -> st.shared, the same arithmetic and the same output layout as produce_loop, so the products are bitwise equal.
// Rows past M arrive zero-filled; their transformed values only reach accumulator rows that are never stored.
constexpr uint32_t kRawBoxBytes = BM * 128;                    // 128 rows x 32 fp32
constexpr uint32_t kRawSlotBytes = 2 * kRawBoxBytes;           // one k-block of A: 128 rows x 64 fp32

__device__ __forceinline__ void tma_load_2d(uint32_t dst_smem, const CUtensorMap* map, int c0, int c1, uint64_t* bar) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(
            dst_smem),
        "l"(map), "r"(c0), "r"(c1), "r"(smem_u32(bar))
        : "memory");
}
__device__ __forceinline__ float4 lds128f(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr)
                 : "memory");
    return v;
}

// one elected thread: the (tile, k-block) sequence of produce/transform_loop, A rows row_mul*(tile/tiles_n)+row_add
template <int RAW, class Args>
__device__ __forceinline__ void tma_a_loop(const Args& g, const CUtensorMap* amap, int64_t first_tile, int64_t tile_step,
                                           int64_t row_mul, int64_t row_add, int num_kb, uint32_t raw_base,
                                           uint64_t* raw_full, uint64_t* raw_empty) {
    const bool tr = g.trace && blockIdx.x == 0;
    uint32_t it = 0;
    for (int64_t tile = first_tile; tile < g.num_tiles; tile += tile_step) {
        const int row0 = (int)((tile / g.tiles_n) * row_mul + row_add);
        for (int kb = 0; kb < num_kb; ++kb, ++it) {
            const int r = it % RAW;
            const uint32_t rph = (it / RAW) & 1;
            long long c0 = 0;
            if (tr) c0 = clock64();
            mbar_wait(raw_empty + r, rph ^ 1u);
            if (tr) g.trace[12] += (unsigned long long)(clock64() - c0);   // A loader: wait for a free raw slot
            mbar_arrive_expect_tx(raw_full + r, kRawSlotBytes);
            const uint32_t dst = raw_base + (uint32_t)r * kRawSlotBytes;
            tma_load_2d(dst, amap, kb * BK16, row0, raw_full + r);
            tma_load_2d(dst + kRawBoxBytes, amap, kb * BK16 + 32, row0, raw_full + r);
        }
    }
}

template <int STAGES, int RAW, class Args, class WaitEmpty>
__device__ __forceinline__ void transform_loop(const Args& g, int64_t first_tile, int64_t tile_step, int num_kb, float s_a,
                                               uint32_t smem_base, uint32_t raw_base, uint32_t stage_bytes,
                                               uint32_t a_bytes, uint64_t* full_bar, uint64_t* empty_bar,
                                               uint64_t* raw_full, uint64_t* raw_empty, WaitEmpty wait_empty) {
    constexpr int NJ = kProdNJ, RPP = kProdRPP;
    const int t = threadIdx.x, lane = threadIdx.x & 31;
    const uint32_t c4 = t & 15;                           // 4 consecutive k of the k-block: 16-byte chunk c4 & 7 of box c4 >> 3
    const int c8 = (int)c4 * 4;
    const bool has_act = g.scale != nullptr;
    const bool tr = g.trace && blockIdx.x == 0 && t == 0;
    const int64_t my_tiles = first_tile < g.num_tiles ? (g.num_tiles - first_tile + tile_step - 1) / tile_step : 0;
    const uint32_t total = (uint32_t)(my_tiles * num_kb);
    const uint32_t rd = raw_base + (c4 >> 3) * kRawBoxBytes;
    int kb = 0;
    for (uint32_t it = 0; it < total; ++it) {
        const int s = it % STAGES, r = it % RAW;
        const uint32_t ph = (it / STAGES) & 1, rph = (it / RAW) & 1;
        const int k0 = kb * BK16;
        if (++kb == num_kb) kb = 0;
        long long c1 = 0, c2 = 0, c3 = 0, cA = 0, cB = 0, c4t = 0;
        float4 sc = make_float4(s_a, s_a, s_a, s_a), sh = make_float4(0.f, 0.f, 0.f, 0.f);
        if (has_act) {
            sc = ldg4(g.scale + k0 + c8);
            sh = ldg4(g.shift + k0 + c8);
            sc.x *= s_a; sc.y *= s_a; sc.z *= s_a; sc.w *= s_a;
            sh.x *= s_a; sh.y *= s_a; sh.z *= s_a; sh.w *= s_a;
        }
        if (tr) c1 = clock64();
        mbar_wait(raw_full + r, rph);
        if (tr) c2 = clock64();
        const uint32_t raw = rd + (uint32_t)r * kRawSlotBytes;
        float4 av[NJ];
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const uint32_t row = (t >> 4) + j * RPP;
            av[j] = lds128f(raw + row * 128u + (((c4 & 7u) ^ (row & 7u)) << 4));
        }
        wait_empty(empty_bar + s, ph ^ 1u);
        if (tr) c3 = clock64();
        const uint32_t st = smem_base + s * stage_bytes;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const uint32_t row = (t >> 4) + j * RPP;
            float4 a = av[j];
            if (has_act) {
                a.x = lrelu_max(fmaf(a.x, sc.x, sh.x), g.slope); a.y = lrelu_max(fmaf(a.y, sc.y, sh.y), g.slope);
                a.z = lrelu_max(fmaf(a.z, sc.z, sh.z), g.slope); a.w = lrelu_max(fmaf(a.w, sc.w, sh.w), g.slope);
            } else {
                a.x *= s_a; a.y *= s_a; a.z *= s_a; a.w *= s_a;
            }
            uint32_t h0, l0, h1, l1;
            split_f16x2(a.x, a.y, h0, l0);
            split_f16x2(a.z, a.w, h1, l1);
            const uint32_t off = sw128(row, c4 >> 1) + ((c4 & 1u) << 3);
            sts64(st + off, h0, h1);
            sts64(st + a_bytes + off, l0, l1);
        }
        if (tr) cA = clock64();
        fence_proxy_async();
        if (tr) cB = clock64();
        __syncwarp();
        if (tr) c4t = clock64();
        if (lane == 0) {
            mbar_arrive(raw_empty + r);
            mbar_arrive(full_bar + s);
        }
        if (tr) {
            g.trace[11] += (unsigned long long)(c2 - c1);    // wait for the raw A slot (TMA)
            g.trace[1] += (unsigned long long)(c3 - c2);     // shared loads + wait for a free stage
            g.trace[2] += (unsigned long long)(c4t - c3);    // transform + stores + fence
            g.trace[3] += 1ull;
            g.trace[14] += (unsigned long long)(cA - c3);    // ... of which: transform + store issue
            g.trace[15] += (unsigned long long)(cB - cA);    // ... fence.proxy.async
        }
    }
}
// Epilogue of the fp16-split NT kernels: one warp drains its 32 rows x BN columns of the accumulator.
// tcgen05.ld hands every thread one ROW; the 32 x 32 block goes through a swizzled staging tile so that a store
// instruction writes 4 rows x 128 B, and the column scales are applied on the way out (there a lane owns 4 fixed
// columns, so one 16-byte load of the scales serves the whole block).  The TMEM load of the next block is in flight
// while the current one is written: the drain of a 128 x 256 tile took 13.5 k cycles when everything was serial,
// which is what bounded the K <= 256 shapes (4 k-blocks of ~2.9 k cycles per tile).
__device__ __forceinline__ void tmem_ld32_async(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]),
          "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),
          "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),
          "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

template <class Args>
__device__ __forceinline__ void epilogue_block32(const Args& g, uint32_t (&v)[32], float inv_sa, uint32_t stg, int lane,
                                                 int64_t mrow0, int ncol0) {
    const int cc = lane & 7;
    float4 w = ldg4(g.inv_sw + ncol0 + cc * 4);          // scales of the 4 columns this lane stores
    if (g.flags & 8) {                                   // A/B switch: no staging, thread-per-row 16-byte stores (slower)
        const int64_t m = mrow0 + lane;
        if (m < g.M) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float4 ws = ldg4(g.inv_sw + ncol0 + 4 * i);
                st4(g.C + m * g.N + ncol0 + 4 * i,
                    make_float4(__uint_as_float(v[4 * i]) * inv_sa * ws.x, __uint_as_float(v[4 * i + 1]) * inv_sa * ws.y,
                                __uint_as_float(v[4 * i + 2]) * inv_sa * ws.z, __uint_as_float(v[4 * i + 3]) * inv_sa * ws.w));
            }
        }
        return;
    }
#pragma unroll
    for (int i = 0; i < 8; ++i)              // row = lane, 16-byte chunk i -> swizzled chunk i ^ (lane & 7)
        sts128(stg + (uint32_t)lane * 128u + (uint32_t)((i ^ (lane & 7)) << 4),
               make_uint4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]));
    w.x *= inv_sa; w.y *= inv_sa; w.z *= inv_sa; w.w *= inv_sa;
    __syncwarp();
    uint4 o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int r = j * 4 + (lane >> 3);
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(o[j].x), "=r"(o[j].y), "=r"(o[j].z), "=r"(o[j].w)
                     : "r"(stg + (uint32_t)r * 128u + (uint32_t)((cc ^ (r & 7)) << 4)));
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
        const int64_t m = mrow0 + j * 4 + (lane >> 3);
        if (m < g.M)
            st4(g.C + m * g.N + ncol0 + cc * 4,
                make_float4(__uint_as_float(o[j].x) * w.x, __uint_as_float(o[j].y) * w.y,
                            __uint_as_float(o[j].z) * w.z, __uint_as_float(o[j].w) * w.w));
    }
    __syncwarp();
}
// taddr = TMEM address of (this warp's lane quarter, first column of the accumulator buffer)
template <int BN, class Args>
__device__ __forceinline__ void epilogue_tile(const Args& g, uint32_t taddr, float inv_sa, uint32_t stg, int lane,
                                              int64_t mrow0, int n0) {
    static_assert(BN % 64 == 0, "two 32-column blocks per iteration");
    uint32_t va[32], vb[32];
    tmem_ld32_async(taddr, va);
#pragma unroll 1
    for (int cb = 0; cb < BN; cb += 64) {
        const bool tr = g.trace && blockIdx.x == 0 && threadIdx.x == 12 * 32;
        long long q0 = 0;
        if (tr) q0 = clock64();
        tmem_wait_ld();                                  // va has landed
        if (tr) g.trace[13] += (unsigned long long)(clock64() - q0);   // exposed TMEM load latency
        tmem_ld32_async(taddr + (uint32_t)cb + 32u, vb);
        epilogue_block32(g, va, inv_sa, stg, lane, mrow0, n0 + cb);
        tmem_wait_ld();                                  // vb has landed
        if (cb + 64 < BN) tmem_ld32_async(taddr + (uint32_t)cb + 64u, va);
        epilogue_block32(g, vb, inv_sa, stg, lane, mrow0, n0 + cb + 32);
    }
}

// ---- epilogue through TMA tensor stores (default) -------------------------------------------------------------------
// The staged epilogue above spends 70 % of its 11-13 k cycles per 128 x 256 tile moving the staging tile to global memory
// with ld.shared + st.global from 4 warps that share the LSU with the 8 producer warps -- which is what bounds every
// K <= 256 shape (4 k-blocks of ~1.5 k cycles per tile).  Here a warp writes its 32 x 32 block (already unscaled) into a
// 128-byte-swizzled 4 KB staging buffer and ONE lane hands it to the TMA unit (cp.async.bulk.tensor.2d.global.shared::cta,
// SASS UTMASTG; tensor map of C with box 32 x 32 fp32, SWIZZLE_128B; rows past M are clipped by the unit).  Two staging
// buffers per warp: the next block is written while the previous one is being read out.  A lane owns a ROW here, so it
// needs the unscale factors of all 32 columns of the block: eight warp-uniform 16-byte loads of inv_sw (one transaction
// each, L1-resident) issued before the TMEM load is awaited; powers of two, so the products equal the staged path's.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src_smem, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.tile.bulk_group [%0, {%1, %2}], [%3];" ::"l"(map), "r"(c0),
                 "r"(c1), "r"(src_smem)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read1() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }

constexpr uint32_t kStageWarpBytes = 2u * 32u * 128u;          // two 32 x 128 B staging buffers per epilogue warp
constexpr uint32_t kStagingBytes = 4u * kStageWarpBytes;       // 32 KB

__device__ __forceinline__ void store_block32_tma(const CUtensorMap* cmap, const uint32_t (&v)[32],
                                                  const float4 (&cs)[8], float inv_sa, uint32_t stg, int lane, int mrow0,
                                                  int ncol0) {
    if (lane == 0) bulk_wait_read1();                // the store that read this buffer two blocks ago has drained it
    __syncwarp();
#pragma unroll
    for (int i = 0; i < 8; ++i)                      // row = lane, 16-byte chunk i -> swizzled chunk i ^ (lane & 7)
        sts128(stg + (uint32_t)lane * 128u + (uint32_t)((i ^ (lane & 7)) << 4),
               make_uint4(__float_as_uint(__uint_as_float(v[4 * i]) * (cs[i].x * inv_sa)),
                          __float_as_uint(__uint_as_float(v[4 * i + 1]) * (cs[i].y * inv_sa)),
                          __float_as_uint(__uint_as_float(v[4 * i + 2]) * (cs[i].z * inv_sa)),
                          __float_as_uint(__uint_as_float(v[4 * i + 3]) * (cs[i].w * inv_sa))));
    fence_proxy_async();
    __syncwarp();
    if (lane == 0) {
        tma_store_2d(cmap, stg, ncol0, mrow0);
        bulk_commit();
    }
}
// stg: this warp's two staging buffers (1024-byte aligned); inv_sw: 1 / (scale of weight row n), 16-byte aligned
template <int BN>
__device__ __forceinline__ void epilogue_tile_tma(const CUtensorMap* cmap, const float* __restrict__ inv_sw, uint32_t taddr,
                                                  float inv_sa, uint32_t stg, int lane, int64_t mrow0, int n0) {
    static_assert(BN % 64 == 0, "two 32-column blocks per iteration");
    uint32_t va[32], vb[32];
    float4 cs[8];
    tmem_ld32_async(taddr, va);
#pragma unroll 1
    for (int cb = 0; cb < BN; cb += 64) {
#pragma unroll
        for (int i = 0; i < 8; ++i) cs[i] = ldg4(inv_sw + n0 + cb + 4 * i);
        tmem_wait_ld();                                  // va has landed
        tmem_ld32_async(taddr + (uint32_t)cb + 32u, vb);
        store_block32_tma(cmap, va, cs, inv_sa, stg, lane, (int)mrow0, n0 + cb);
#pragma unroll
        for (int i = 0; i < 8; ++i) cs[i] = ldg4(inv_sw + n0 + cb + 32 + 4 * i);
        tmem_wait_ld();                                  // vb has landed
        if (cb + 64 < BN) tmem_ld32_async(taddr + (uint32_t)cb + 64u, va);
        store_block32_tma(cmap, vb, cs, inv_sa, stg + 32u * 128u, lane, (int)mrow0, n0 + cb + 32);
    }
}

// W [N,K] (or, transposed, W^T given as [K,N]) -> per-row scaled fp16 hi/lo image; one warp per weight row n
__global__ void tc_prep_b16_kernel(const float* __restrict__ W, int transposed, uint8_t* __restrict__ img,
                                   float* __restrict__ inv_sw, int N, int K, int BN) {
    const int n = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (n >= N) return;
    const int chunks = K / 8;
    auto load8 = [&](int c, float4& a, float4& b) {
        const int k = c * 8;
        if (!transposed) {
            a = ldg4(W + (int64_t)n * K + k);
            b = ldg4(W + (int64_t)n * K + k + 4);
        } else {
            a.x = __ldg(W + (int64_t)(k + 0) * N + n); a.y = __ldg(W + (int64_t)(k + 1) * N + n);
            a.z = __ldg(W + (int64_t)(k + 2) * N + n); a.w = __ldg(W + (int64_t)(k + 3) * N + n);
            b.x = __ldg(W + (int64_t)(k + 4) * N + n); b.y = __ldg(W + (int64_t)(k + 5) * N + n);
            b.z = __ldg(W + (int64_t)(k + 6) * N + n); b.w = __ldg(W + (int64_t)(k + 7) * N + n);
        }
    };
    uint32_t m = 0;
    for (int c = lane; c < chunks; c += 32) {
        float4 a, b;
        load8(c, a, b);
        const float mx = fmaxf(fmaxf(fmaxf(fabsf(a.x), fabsf(a.y)), fmaxf(fabsf(a.z), fabsf(a.w))),
                               fmaxf(fmaxf(fabsf(b.x), fabsf(b.y)), fmaxf(fabsf(b.z), fabsf(b.w))));
        const uint32_t bits = __float_as_uint(mx);
        m = bits > m ? bits : m;
    }
    m = __reduce_max_sync(0xffffffffu, m);
    float s, inv_s;
    scale_from_bits(m, s, inv_s);
    if (lane == 0) inv_sw[n] = inv_s;
    const int n_tile = n / BN, r = n % BN, num_kb = K / BK16;
    const int64_t half_bytes = (int64_t)BN * 128;
    for (int c = lane; c < chunks; c += 32) {
        float4 a, b;
        load8(c, a, b);
        a.x *= s; a.y *= s; a.z *= s; a.w *= s; b.x *= s; b.y *= s; b.z *= s; b.w *= s;
        uint4 hi, lo;
        split_f16x8(a, b, hi, lo);
        const int kb = c / 8, cc = c % 8;
        const int64_t base = ((int64_t)n_tile * num_kb + kb) * 2 * half_bytes;
        const uint32_t off = sw128((uint32_t)r, (uint32_t)cc);
        *reinterpret_cast<uint4*>(img + base + off) = hi;
        *reinterpret_cast<uint4*>(img + base + half_bytes + off) = lo;
    }
}

// RAW = 0: A by the register-fed producers (produce_loop); RAW > 0: A by TMA into RAW raw slots (tma_a_loop +
// transform_loop).  ACC: depth of the TMEM accumulator ring (ACC x BN columns).
template <int BN, int STAGES, int RAW, int ACC>
__global__ void __launch_bounds__(kV2Threads, 1) tc_gemm_nt16_kernel(const __grid_constant__ CUtensorMap cmap,
                                                                     const __grid_constant__ CUtensorMap amap,
                                                                     const Nt16Args g) {
    constexpr uint32_t A_BYTES = BM * 128;           // 128 rows x 64 fp16, one of hi / lo
    constexpr uint32_t B_BYTES = BN * 128;
    constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    constexpr uint32_t TMEM_COLS = ACC * BN;
    static_assert(TMEM_COLS <= 512 && (TMEM_COLS & (TMEM_COLS - 1)) == 0, "TMEM allocation: power of two <= 512");
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* raw = smem + STAGES * STAGE_BYTES;              // RAW x 32 KB of fp32 A (1 KB aligned)
    uint8_t* staging = raw + RAW * kRawSlotBytes;            // 4 epilogue warps x 2 buffers x 32 rows x 128 B (1 KB aligned)
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(staging + kStagingBytes);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* acc_full = empty_bar + STAGES;     // [ACC]
    uint64_t* acc_empty = acc_full + ACC;        // [ACC]
    uint64_t* raw_full = acc_empty + ACC;        // [RAW]
    uint64_t* raw_empty = raw_full + RAW;        // [RAW]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(raw_empty + RAW);
    uint32_t* amax_slot = tmem_slot + 1;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int num_kb = g.K / BK16;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar + s, kProducerWarps + 1);
            mbar_init(empty_bar + s, 1);
        }
        for (int b = 0; b < ACC; ++b) {
            mbar_init(acc_full + b, 1);
            mbar_init(acc_empty + b, 4);
        }
        for (int r = 0; r < RAW; ++r) {
            mbar_init(raw_full + r, 1);
            mbar_init(raw_empty + r, kProducerWarps);
        }
        *amax_slot = 0u;
        fence_barrier_init();
    }
    if (warp == 8) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    block_amax_bits(g.amax, g.amax_len, amax_slot);
    __syncthreads();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t smem_base = smem_u32(smem);
    float s_a, inv_sa;
    scale_from_bits(*amax_slot, s_a, inv_sa);

    if (warp < kProducerWarps) {
        // ===== A producers (see produce_loop / transform_loop) =====
        auto wait_empty = [](uint64_t* bar, uint32_t parity) { mbar_wait(bar, parity); };
        if constexpr (RAW > 0)
            transform_loop<STAGES, RAW>(g, (int64_t)blockIdx.x, (int64_t)gridDim.x, num_kb, s_a, smem_base,
                                        smem_u32(raw), STAGE_BYTES, A_BYTES, full_bar, empty_bar, raw_full, raw_empty,
                                        wait_empty);
        else
            produce_loop<STAGES>(g, (int64_t)blockIdx.x, (int64_t)gridDim.x, (int64_t)BM, 0, num_kb, s_a,
                                 smem_base, STAGE_BYTES, A_BYTES, full_bar, empty_bar, wait_empty);
    } else if (warp == 8) {
        // ===== MMA issuer =====
        if (lane == 0) {
            constexpr uint32_t idesc = make_idesc16(BM, BN, false, false);
            const bool tr = g.trace && blockIdx.x == 0;
            uint32_t it = 0, tile_no = 0;
            for (int64_t tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++tile_no) {
                const uint32_t buf = tile_no % ACC;
                long long a0 = 0;
                if (tr) a0 = clock64();
                mbar_wait(acc_empty + buf, ((tile_no / ACC) & 1u) ^ 1u);
                if (tr) g.trace[7] += (unsigned long long)(clock64() - a0);   // wait for a free accumulator
                tc_fence_after();
                const uint32_t d_tmem = tmem_base + buf * BN;
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    long long c0 = 0;
                    if (tr) c0 = clock64();
                    mbar_wait(full_bar + s, ph);
                    if (tr) {
                        g.trace[4] += (unsigned long long)(clock64() - c0);     // MMA thread: wait stage full
                        g.trace[6] += 1ull;
                    }
                    tc_fence_after();
                    const uint32_t sa = smem_base + s * STAGE_BYTES;
#pragma unroll
                    for (int ks = 0; ks < BK16 / UMMA_K16; ++ks) {
                        const uint32_t koff = ks * UMMA_K16 * 2;
                        const uint64_t a_hi = make_desc(sa + koff, 16, 1024);
                        const uint64_t a_lo = make_desc(sa + A_BYTES + koff, 16, 1024);
                        const uint64_t b_hi = make_desc(sa + 2 * A_BYTES + koff, 16, 1024);
                        const uint64_t b_lo = make_desc(sa + 2 * A_BYTES + B_BYTES + koff, 16, 1024);
                        umma_f16(d_tmem, a_lo, b_hi, idesc, (kb | ks) != 0);
                        umma_f16(d_tmem, a_hi, b_lo, idesc, 1);
                        umma_f16(d_tmem, a_hi, b_hi, idesc, 1);
                    }
                    umma_commit(empty_bar + s);
                }
                umma_commit(acc_full + buf);
            }
        }
        __syncwarp();
    } else if (warp == 9) {
        // ===== B loader: one bulk copy per stage =====
        if (lane == 0) {
            uint32_t it = 0;
            for (int64_t tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x) {
                const int tn = (int)(tile % g.tiles_n);
                const uint8_t* src = g.Bimg + (int64_t)tn * num_kb * (2 * (int64_t)B_BYTES);
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(empty_bar + s, ph ^ 1u);
                    mbar_arrive_expect_tx(full_bar + s, 2 * B_BYTES);
                    bulk_g2s(smem_base + s * STAGE_BYTES + 2 * A_BYTES, src + (int64_t)kb * (2 * (int64_t)B_BYTES),
                             2 * B_BYTES, full_bar + s);
                }
            }
        }
        __syncwarp();
    } else if (warp == 10) {
        // ===== A loader (RAW > 0): TMA tensor loads into the raw ring =====
        if constexpr (RAW > 0) {
            if (lane == 0)
                tma_a_loop<RAW>(g, &amap, (int64_t)blockIdx.x, (int64_t)gridDim.x, (int64_t)BM, 0, num_kb, smem_u32(raw),
                                raw_full, raw_empty);
        }
        __syncwarp();
    } else if (warp >= 12) {
        // ===== epilogue: TMEM -> registers (unscale) -> swizzled staging tile -> global =====
        const int q = warp & 3;
        const uint32_t stg = smem_u32(staging) + (uint32_t)q * kStageWarpBytes;
        const bool staged = (g.flags & 16) != 0;         // A/B switch: the ld.shared + st.global epilogue
        uint32_t tile_no = 0;
        for (int64_t tile = blockIdx.x; tile < g.num_tiles; tile += gridDim.x, ++tile_no) {
            const uint32_t buf = tile_no % ACC;
            const int64_t mrow0 = (tile / g.tiles_n) * BM + q * 32;
            const int n0 = (int)(tile % g.tiles_n) * BN;
            const bool tr = g.trace && blockIdx.x == 0 && warp == 12 && lane == 0;
            long long e0 = 0;
            if (tr) e0 = clock64();
            mbar_wait(acc_full + buf, (tile_no / ACC) & 1u);
            if (tr) {
                const long long e1 = clock64();
                g.trace[8] += (unsigned long long)(e1 - e0);                 // epilogue: wait accumulator
                g.trace[9] -= (unsigned long long)e1;                        // epilogue: drain (completed below)
            }
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN;
            if (staged) epilogue_tile<BN>(g, taddr, inv_sa, stg, lane, mrow0, n0);
            else epilogue_tile_tma<BN>(&cmap, g.inv_sw, taddr, inv_sa, stg, lane, mrow0, n0);
            tc_fence_before();
            __syncwarp();
            if (tr) {
                g.trace[9] += (unsigned long long)clock64();
                g.trace[10] += 1ull;
            }
            if (lane == 0) mbar_arrive(acc_empty + buf);
        }
        if (lane == 0) bulk_wait_all();                  // the staging buffers must outlive the last tensor stores
    }
    __syncthreads();
    if (warp == 8) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// dynamic shared memory of the fp16-split NT kernels: split stages, raw A slots, epilogue staging, barriers
constexpr size_t nt16_smem(int stages, uint32_t b_bytes, int raw) {
    return (size_t)stages * (2 * BM * 128 + 2 * b_bytes) + (size_t)raw * kRawSlotBytes + kStagingBytes + 1024 + 256;
}

// tensor map of A [M, K] for the raw ring: 128-row x 32-column boxes, 128-byte swizzle, rows past M zero-filled
static int make_a_map(CUtensorMap* amap, const Nt16Args& g, const char* who) {
    return make_tensor_map_2d(amap, g.A, g.M, g.K, BM, 32, true, who);
}

template <int BN, int STAGES, int RAW, int ACC>
static int launch_nt16(const Nt16Args& g, cudaStream_t st) {
    constexpr size_t smem = nt16_smem(STAGES, BN * 128, RAW);
    static_assert(smem <= 232448, "shared memory of the fp16-split NT kernel");
    static PerDeviceOnce configured;
    if (configured.need()) {
        DDMP_CUDA(cudaFuncSetAttribute(tc_gemm_nt16_kernel<BN, STAGES, RAW, ACC>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured.mark();
    }
    CUtensorMap cmap;                                    // result tensor [M, N], 32 x 32 boxes, 128-byte swizzle
    int rc = make_tensor_map_2d(&cmap, g.C, g.M, g.N, 32, 32, true, "tc_gemm_nt16");
    if (rc != DDMP_OK) return rc;
    CUtensorMap amap = cmap;                             // unused by the register-fed configuration
    if (RAW > 0 && (rc = make_a_map(&amap, g, "tc_gemm_nt16 A")) != DDMP_OK) return rc;
    const int64_t grid = g.num_tiles < kNumSMs ? g.num_tiles : kNumSMs;
    tc_gemm_nt16_kernel<BN, STAGES, RAW, ACC><<<(unsigned)grid, kV2Threads, smem, st>>>(cmap, amap, g);
    return check_launch("tc_gemm_nt16");
}

// fp16-split NT kernel on CTA pairs (cta_group::2, synchronisation scheme above): each CTA
// stages its 128 rows of A and HALF of the weight tile, so the bytes a CTA pulls from L2 per k-block drop from 96 KB to
// 64 KB (with the MMA time halved by kind::f16, the weight stream re-read for every row tile is what saturates the
// SM's L2 port) and a third pipeline stage fits.
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                              uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// RAW = 0: A by the register-fed producers; RAW > 0: A by TMA into RAW raw slots (as in tc_gemm_nt16_kernel)
template <int STAGES, int RAW>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kV2Threads, 1)
tc_gemm_nt16x2_kernel(const __grid_constant__ CUtensorMap cmap, const __grid_constant__ CUtensorMap amap,
                      const Nt16Args g) {
    constexpr int BN = 256;
    constexpr uint32_t A_BYTES = BM * 128;
    constexpr uint32_t B_HALF = (BN / 2) * 128;          // this CTA's half of the weight tile, one of hi / lo
    constexpr uint32_t B_FULL = BN * 128;
    constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_HALF;
    constexpr uint32_t TMEM_COLS = 2 * BN;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* raw = smem + STAGES * STAGE_BYTES;              // RAW x 32 KB of fp32 A (1 KB aligned)
    uint8_t* staging = raw + RAW * kRawSlotBytes;            // 1 KB aligned (128-byte swizzle of the tensor stores)
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(staging + kStagingBytes);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* peer_ready = empty_bar + STAGES;
    uint64_t* acc_full = peer_ready + STAGES;
    uint64_t* acc_empty = acc_full + 2;
    uint64_t* raw_full = acc_empty + 2;          // [RAW]
    uint64_t* raw_empty = raw_full + RAW;        // [RAW]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(raw_empty + RAW);
    uint32_t* amax_slot = tmem_slot + 1;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int num_kb = g.K / BK16;
    const int64_t num_pairs = gridDim.x / 2, pair = blockIdx.x / 2;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar + s, kProducerWarps + 1);
            mbar_init(empty_bar + s, 1);
            mbar_init(peer_ready + s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(acc_full + b, 1);
            mbar_init(acc_empty + b, 8);
        }
        for (int r = 0; r < RAW; ++r) {
            mbar_init(raw_full + r, 1);
            mbar_init(raw_empty + r, kProducerWarps);
        }
        *amax_slot = 0u;
        fence_barrier_init();
    }
    cluster_sync_all();
    if (warp == 8) tmem_alloc_2cta(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    block_amax_bits(g.amax, g.amax_len, amax_slot);
    __syncthreads();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t smem_base = smem_u32(smem);
    float s_a, inv_sa;
    scale_from_bits(*amax_slot, s_a, inv_sa);

    if (warp < kProducerWarps) {
        auto wait_empty = [](uint64_t* bar, uint32_t parity) { mbar_wait_cluster(bar, parity); };
        if constexpr (RAW > 0)
            transform_loop<STAGES, RAW>(g, pair, num_pairs, num_kb, s_a, smem_base, smem_u32(raw), STAGE_BYTES, A_BYTES,
                                        full_bar, empty_bar, raw_full, raw_empty, wait_empty);
        else
            produce_loop<STAGES>(g, pair, num_pairs, (int64_t)(2 * BM), (int64_t)rank * BM, num_kb, s_a,
                                 smem_base, STAGE_BYTES, A_BYTES, full_bar, empty_bar, wait_empty);
    } else if (warp == 8) {
        if (lane == 0) {
            uint32_t it = 0, tile_no = 0;
            if (rank == 0) {
                constexpr uint32_t idesc = make_idesc16(2 * BM, BN, false, false);
                for (int64_t tile = pair; tile < g.num_tiles; tile += num_pairs, ++tile_no) {
                    const uint32_t buf = tile_no & 1u;
                    long long a0 = 0;
                    if (g.trace && blockIdx.x == 0) a0 = clock64();
                    mbar_wait_cluster(acc_empty + buf, ((tile_no >> 1) & 1u) ^ 1u);
                    if (g.trace && blockIdx.x == 0) g.trace[7] += (unsigned long long)(clock64() - a0);   // wait acc free
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + buf * BN;
                    for (int kb = 0; kb < num_kb; ++kb, ++it) {
                        const int s = it % STAGES;
                        const uint32_t ph = (it / STAGES) & 1;
                        const bool tr = g.trace && blockIdx.x == 0;
                        long long c0 = 0, c1 = 0, c2 = 0;
                        if (tr) c0 = clock64();
                        mbar_wait(full_bar + s, ph);
                        if (tr) c1 = clock64();
                        mbar_wait_cluster(peer_ready + s, ph);
                        if (tr) {
                            c2 = clock64();
                            g.trace[4] += (unsigned long long)(c1 - c0);     // MMA thread: wait own stage full
                            g.trace[5] += (unsigned long long)(c2 - c1);     // wait peer stage full
                            g.trace[6] += 1ull;
                        }
                        tc_fence_after();
                        const uint32_t sa = smem_base + s * STAGE_BYTES;
#pragma unroll
                        for (int ks = 0; ks < BK16 / UMMA_K16; ++ks) {
                            const uint32_t koff = ks * UMMA_K16 * 2;
                            const uint64_t a_hi = make_desc(sa + koff, 16, 1024);
                            const uint64_t a_lo = make_desc(sa + A_BYTES + koff, 16, 1024);
                            const uint64_t b_hi = make_desc(sa + 2 * A_BYTES + koff, 16, 1024);
                            const uint64_t b_lo = make_desc(sa + 2 * A_BYTES + B_HALF + koff, 16, 1024);
                            umma_f16_2cta(d_tmem, a_lo, b_hi, idesc, (kb | ks) != 0);
                            umma_f16_2cta(d_tmem, a_hi, b_lo, idesc, 1);
                            umma_f16_2cta(d_tmem, a_hi, b_hi, idesc, 1);
                        }
                        umma_commit_2cta(empty_bar + s);
                    }
                    umma_commit_2cta(acc_full + buf);
                }
            } else {
                for (int64_t tile = pair; tile < g.num_tiles; tile += num_pairs) {
                    for (int kb = 0; kb < num_kb; ++kb, ++it) {
                        const int s = it % STAGES;
                        const uint32_t ph = (it / STAGES) & 1;
                        mbar_wait(full_bar + s, ph);
                        mbar_arrive_remote(peer_ready + s, 0);
                    }
                }
            }
        }
        __syncwarp();
    } else if (warp == 9) {
        if (lane == 0) {
            uint32_t it = 0;
            for (int64_t tile = pair; tile < g.num_tiles; tile += num_pairs) {
                const int tn = (int)(tile % g.tiles_n);
                const uint8_t* src = g.Bimg + (int64_t)tn * num_kb * (2 * (int64_t)B_FULL) + (int64_t)rank * B_HALF;
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait_cluster(empty_bar + s, ph ^ 1u);
                    mbar_arrive_expect_tx(full_bar + s, 2 * B_HALF);
                    const uint8_t* sk = src + (int64_t)kb * (2 * (int64_t)B_FULL);
                    const uint32_t dst = smem_base + s * STAGE_BYTES + 2 * A_BYTES;
                    bulk_g2s(dst, sk, B_HALF, full_bar + s);
                    bulk_g2s(dst + B_HALF, sk + B_FULL, B_HALF, full_bar + s);
                }
            }
        }
        __syncwarp();
    } else if (warp == 10) {
        // ===== A loader (RAW > 0): TMA tensor loads of this CTA's 128 rows into the raw ring =====
        if constexpr (RAW > 0) {
            if (lane == 0)
                tma_a_loop<RAW>(g, &amap, pair, num_pairs, (int64_t)(2 * BM), (int64_t)rank * BM, num_kb, smem_u32(raw),
                                raw_full, raw_empty);
        }
        __syncwarp();
    } else if (warp >= 12) {
        const int q = warp & 3;
        const uint32_t stg = smem_u32(staging) + (uint32_t)q * kStageWarpBytes;
        const bool staged = (g.flags & 16) != 0;         // A/B switch: the ld.shared + st.global epilogue
        uint32_t tile_no = 0;
        for (int64_t tile = pair; tile < g.num_tiles; tile += num_pairs, ++tile_no) {
            const uint32_t buf = tile_no & 1u;
            const int64_t mrow0 = (tile / g.tiles_n) * (2 * BM) + rank * BM + q * 32;
            const int n0 = (int)(tile % g.tiles_n) * BN;
            const bool tr = g.trace && blockIdx.x == 0 && warp == 12 && lane == 0;
            long long e0 = 0;
            if (tr) e0 = clock64();
            mbar_wait_cluster(acc_full + buf, (tile_no >> 1) & 1u);
            if (tr) {
                const long long e1 = clock64();
                g.trace[8] += (unsigned long long)(e1 - e0);                 // epilogue: wait accumulator
                g.trace[9] -= (unsigned long long)e1;                        // epilogue: drain (completed below)
            }
            tc_fence_after();
            const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + buf * BN;
            if (staged) epilogue_tile<BN>(g, taddr, inv_sa, stg, lane, mrow0, n0);
            else epilogue_tile_tma<BN>(&cmap, g.inv_sw, taddr, inv_sa, stg, lane, mrow0, n0);
            tc_fence_before();
            __syncwarp();
            if (tr) {
                g.trace[9] += (unsigned long long)clock64();
                g.trace[10] += 1ull;
            }
            if (lane == 0) {
                if (rank == 0) mbar_arrive(acc_empty + buf);
                else mbar_arrive_remote(acc_empty + buf, 0);
            }
        }
        if (lane == 0) bulk_wait_all();                  // the staging buffers must outlive the last tensor stores
    }
    tc_fence_before();
    cluster_sync_all();
    if (warp == 8) {
        tc_fence_after();
        tmem_dealloc_2cta(tmem_base, TMEM_COLS);
    }
}

template <int STAGES, int RAW>
static int launch_nt16x2(const Nt16Args& g0, cudaStream_t st) {
    constexpr size_t smem = nt16_smem(STAGES, 128 * 128, RAW);
    static_assert(smem <= 232448, "shared memory of the CTA-pair fp16-split NT kernel");
    static PerDeviceOnce configured;
    if (configured.need()) {
        DDMP_CUDA(cudaFuncSetAttribute(tc_gemm_nt16x2_kernel<STAGES, RAW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
        configured.mark();
    }
    Nt16Args g = g0;
    g.num_tiles = ceil_div(g.M, 2 * BM) * g.tiles_n;
    CUtensorMap cmap;                                    // result tensor [M, N], 32 x 32 boxes, 128-byte swizzle
    int rc = make_tensor_map_2d(&cmap, g.C, g.M, g.N, 32, 32, true, "tc_gemm_nt16x2");
    if (rc != DDMP_OK) return rc;
    CUtensorMap amap = cmap;                             // unused by the register-fed configuration
    if (RAW > 0 && (rc = make_a_map(&amap, g, "tc_gemm_nt16x2 A")) != DDMP_OK) return rc;
    const int64_t pairs = g.num_tiles < kNumSMs / 2 ? g.num_tiles : kNumSMs / 2;
    tc_gemm_nt16x2_kernel<STAGES, RAW><<<(unsigned)(2 * pairs), kV2Threads, smem, st>>>(cmap, amap, g);
    return check_launch("tc_gemm_nt16x2");
}

// switches of the fp16-split NT kernels (environment DDMP_TC_F16_FLAGS, ddmp_gemm_tc_flags): bit 0 = prefetch the next
// tile's A rows into L2, bit 1 = the same for K <= 256 only, bit 3 = unstaged epilogue, bit 4 = staged ld.shared + st.global
// epilogue instead of TMA stores, bit 5 = the previous configuration (register-fed A operand everywhere, CTA pairs for
// every N % 256 == 0)
int f16_flags(int set) {
    static std::atomic<int> v{-1};
    int cur = v.load(std::memory_order_relaxed);
    if (cur < 0) {
        const char* e = getenv("DDMP_TC_F16_FLAGS");
        cur = e ? (atoi(e) & 0xffff) : 0;
        v.store(cur, std::memory_order_relaxed);
    }
    if (set >= 0) v.store(set & 0xffff, std::memory_order_relaxed);
    return cur;
}

static bool f16_split_enabled() {
    static const bool v = [] { const char* e = getenv("DDMP_TC_SPLIT"); return !(e && e[0] == 't'); }();   // "tf32"
    return v;
}

static int run_nt16(const float* A, const int* a_map, const float* scale, const float* shift, float slope,
                    const float* W, int transposed, void* workspace, float* C, int64_t M, int N, int K,
                    const float* amax, int64_t amax_len, cudaStream_t st) {
    int flags = f16_flags(-1);
    if ((flags & 2) && K <= 256) flags |= 1;         // bit 1: the L2 prefetch only where it measured faster (K <= 256)
    // (TMA tensor coordinates are 32-bit: row counts near 2^31 keep the register-fed producers)
    // TMA-fed A (DESIGN.md §4.2): at K <= 256, and at K = 512 when the BatchNorm + LeakyReLU prologue is fused (there
    // the transform makes the register-fed producers the bound); without the prologue the producers keep pace at
    // K = 512 and the raw ring's extra shared-memory traffic measured ~3 % slower.  The fused row gather (a_map) has
    // no TMA tile form.
    const bool tma_a = (K <= 256 || scale != nullptr) && a_map == nullptr && !(flags & 32) && M < (1ll << 31) - 2 * BM;
    // N % 256 == 0 at K <= 128: a CTA pair's 128 x 256 tile has ~3 k cycles of MMA against 8-9 k cycles of drain, so
    // 128-wide single-CTA tiles with the 4-deep accumulator ring are faster there (12-16 %); at K >= 256 the pair is faster
    const int BN = (N % 256 == 0 && !(tma_a && K <= 128)) ? 256 : ((N % 128 == 0) ? 128 : 64);
    uint8_t* img = reinterpret_cast<uint8_t*>(workspace);
    float* inv_sw = reinterpret_cast<float*>(img + (int64_t)N * K * 4);          // after the hi + lo images
    tc_prep_b16_kernel<<<(unsigned)ceil_div((int64_t)N * 32, 256), 256, 0, st>>>(W, transposed, img, inv_sw, N, K, BN);
    int rc = check_launch("tc_prep_b16");
    if (rc) return rc;
    Nt16Args g{};
    g.A = A; g.Bimg = img; g.inv_sw = inv_sw; g.C = C; g.a_map = a_map; g.scale = scale; g.shift = shift;
    g.slope = slope; g.amax = amax; g.amax_len = amax_len;
    g.flags = flags;
    static const bool trace = [] { const char* e = getenv("DDMP_TC_TRACE"); return e && e[0] == '1'; }();
    static unsigned long long* trace_buf = nullptr;
    if (trace) {
        if (!trace_buf) cudaMalloc(&trace_buf, 16 * sizeof(unsigned long long));
        cudaMemsetAsync(trace_buf, 0, 16 * sizeof(unsigned long long), st);
        g.trace = trace_buf;
    }
    auto dump_trace = [&](int rc) {
        if (trace && rc == 0) {
            unsigned long long h[16];
            cudaStreamSynchronize(st);
            cudaMemcpy(h, trace_buf, sizeof(h), cudaMemcpyDeviceToHost);
            // cycles of CTA 0 per k-block (producer thread 0, MMA thread, A loader) or per tile (epilogue warp 12)
            auto per = [](unsigned long long x, unsigned long long n) { return n ? x / n : 0ull; };
            fprintf(stderr, "[ddmp trace] M=%lld N=%d K=%d A=%s | producer/kb: wait_raw %llu wait_free %llu data+store %llu "
                    "(n=%llu) [transform+stores %llu fence %llu] | tma_a/kb: wait_slot %llu | mma/kb: wait_full %llu "
                    "wait_peer %llu (n=%llu) | mma/tile: wait_acc %llu | epilogue/tile: wait %llu drain %llu (n=%llu) "
                    "[staged tmem wait %llu]\n",
                    (long long)M, N, K, tma_a ? "tma" : "registers", per(h[11], h[3]), per(h[1], h[3]), per(h[2], h[3]),
                    h[3], per(h[14], h[3]), per(h[15], h[3]), per(h[12], h[3]), per(h[4], h[6]), per(h[5], h[6]), h[6],
                    per(h[7], h[10]), per(h[8], h[10]), per(h[9], h[10]), h[10], per(h[13], h[10]));
        }
        return rc;
    };
    g.M = M; g.N = N; g.K = K; g.tiles_n = N / BN;
    g.num_tiles = ceil_div(M, BM) * g.tiles_n;
    DDMP_REQUIRE(g.num_tiles < (1ll << 31), "tc gemm: too many tiles");
    static const bool one_cta = [] { const char* e = getenv("DDMP_TC_2CTA"); return e && e[0] == '0'; }();
    if (BN == 256 && one_cta) return dump_trace(launch_nt16<256, 2, 0, 2>(g, st));
    if (tma_a) {                                     // one split stage traded for the raw fp32 slots
        if (BN == 256) return dump_trace(launch_nt16x2<2, 2>(g, st));
        if (BN == 128) return dump_trace(launch_nt16<128, 2, 2, 4>(g, st));
        return dump_trace(launch_nt16<64, 2, 3, 4>(g, st));
    }
    if (BN == 256) return dump_trace(launch_nt16x2<3, 0>(g, st));
    if (BN == 128) return dump_trace(launch_nt16<128, 3, 0, 2>(g, st));
    return dump_trace(launch_nt16<64, 4, 0, 2>(g, st));
}

// ---- TN kernel (dW) -------------------------------------------------------------------------------------------------
// dW[M=Cout, N=Cin] = sum over rows r of A[r, m] * act(B)[r, n].  Both operands are MN-major: a K index is a graph
// row, and a row of dH / X is contiguous along the channel.  SWIZZLE_128B MN-major canonical layout (CUTLASS
// mma_traits_sm100.hpp "make_umma_desc<Major::MN>"): element (mn, k) of a stage lives at
//     (mn/32)*LBO + (k/8)*1024 + (k%8)*128 + ((((mn%32)/4) ^ (k%8)) * 16) + (mn%4)*4
// Work item = (row segment of kSegRows rows, output tile); items are dealt round-robin to persistent CTAs with the
// tile index fastest, so CTAs running together read the same rows (L2 reuse).  Every item writes its own partial
// tile; a fixed-order float64 reduction sums the segments (deterministic, and it bounds the fp32 accumulation
// length inside TMEM to kSegRows: the tensor core truncates when it accumulates, so the error grows linearly
// with the chain length, measured ~7e-9 per row).
#ifndef DDMP_SEG_ROWS
#define DDMP_SEG_ROWS 2048
#endif
constexpr int kSegRows = DDMP_SEG_ROWS;

struct TnArgs {
    const float* A;       // dH [rows, M] row-major
    const float* B;       // X  [rows, N] row-major (pre-BatchNorm), act over n when scale != null
    float* P;             // partials [num_seg][M][N]
    const float* scale;
    const float* shift;
    float slope;
    int64_t rows;
    int M, N;
    int tiles_m, tiles_n;
    int64_t num_items;
};

template <int BN, int STAGES, int PW>
__global__ void __launch_bounds__(PW * 32 + 32, 1) tc_gemm_tn_kernel(const TnArgs g) {
    constexpr int kPT = PW * 32;                     // producer threads (PW warps) + one MMA warp
    constexpr uint32_t A_BYTES = BM * 128;           // 32 k-rows x 128 m x 4 B
    constexpr uint32_t B_BYTES = BN * 128;
    constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;
    constexpr uint32_t LBO = (BK / 4) * 512;         // next 32-wide MN block (layout [mn_blk][k4_grp][4][128B])
    constexpr uint32_t SBO = 512;                    // next group of 4 k-rows
    constexpr int A_CH = BM / 4, B_CH = BN / 4;      // 16-byte chunks per k-row
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* accum_bar = empty_bar + STAGES;        // MMA -> epilogue: accumulator of this item complete
    uint64_t* drained_bar = accum_bar + 1;           // epilogue -> MMA: TMEM may be overwritten
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(drained_bar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar + s, PW);
            mbar_init(empty_bar + s, 1);
        }
        mbar_init(accum_bar, 1);
        mbar_init(drained_bar, PW);
        fence_barrier_init();
    }
    if (warp == PW) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t smem_base = smem_u32(smem);
    const int tiles = g.tiles_m * g.tiles_n;

    uint32_t it = 0;                                 // pipeline iteration counter, runs across items
    uint32_t item_no = 0;
    for (int64_t item = blockIdx.x; item < g.num_items; item += gridDim.x, ++item_no) {
        const int tile = (int)(item % tiles);
        const int64_t seg = item / tiles;
        const int m0 = (tile / g.tiles_n) * BM, n0 = (tile % g.tiles_n) * BN;
        const int64_t r0 = seg * kSegRows;
        const int64_t r1 = (r0 + kSegRows < g.rows) ? (r0 + kSegRows) : g.rows;
        const int num_kb = (int)((r1 - r0 + BK - 1) / BK);

        if (warp < PW) {
            const int t = threadIdx.x;
            // A: 32 chunks per k-row (BM=128) -> 8 k-rows per pass of 256 threads; B: B_CH chunks per k-row
            const uint32_t a_cm = t % A_CH, a_r = t / A_CH;                    // a_r in [0, 256/A_CH)
            const uint32_t b_cm = t % B_CH, b_r = t / B_CH;
            constexpr int A_PASS = kPT / A_CH, B_PASS = kPT / B_CH;
            const bool a_ok = (m0 + (int)a_cm * 4) < g.M;
            const bool has_act = g.scale != nullptr;
            float4 sc = make_float4(1.f, 1.f, 1.f, 1.f), sh = make_float4(0.f, 0.f, 0.f, 0.f);
            if (has_act) { sc = ldg4(g.scale + n0 + b_cm * 4); sh = ldg4(g.shift + n0 + b_cm * 4); }
            const uint32_t a_off0 = (a_cm / 8) * LBO, b_off0 = (b_cm / 8) * LBO;
            float4 av[BK / A_PASS], bv[BK / B_PASS];
            // global loads of k-block kb+1 are issued right after the stores of kb, so their latency overlaps the
            // wait for the next free stage (the MMA of an earlier block) instead of being exposed every iteration
            auto issue = [&](int kb) {
                if (kb >= num_kb) return;
                const int64_t rb = r0 + (int64_t)kb * BK;
#pragma unroll
                for (int j = 0; j < BK / A_PASS; ++j) {
                    const int64_t r = rb + a_r + j * A_PASS;
                    av[j] = (r < r1 && a_ok) ? ldg4(g.A + r * g.M + m0 + a_cm * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int j = 0; j < BK / B_PASS; ++j) {
                    const int64_t r = rb + b_r + j * B_PASS;
                    bv[j] = (r < r1) ? ldg4(g.B + r * g.N + n0 + b_cm * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            issue(0);
            for (int kb = 0; kb < num_kb; ++kb, ++it) {
                const int s = it % STAGES;
                const uint32_t ph = (it / STAGES) & 1;
                const int64_t rb = r0 + (int64_t)kb * BK;
                mbar_wait(empty_bar + s, ph ^ 1u);
                const uint32_t st = smem_base + s * STAGE_BYTES;
#pragma unroll
                for (int j = 0; j < BK / A_PASS; ++j) {
                    const uint32_t k = a_r + j * A_PASS;                        // k-row inside the stage
                    uint4 hi, lo;
                    split_tf32(av[j].x, hi.x, lo.x); split_tf32(av[j].y, hi.y, lo.y);
                    split_tf32(av[j].z, hi.z, lo.z); split_tf32(av[j].w, hi.w, lo.w);
                    const uint32_t off = a_off0 + (k >> 2) * SBO + (k & 3u) * 128u + ((((a_cm & 7u) >> 1) ^ (k & 3u)) << 5) +
                                         ((a_cm & 1u) << 4);
                    sts128(st + off, hi);
                    sts128(st + A_BYTES + off, lo);
                }
#pragma unroll
                for (int j = 0; j < BK / B_PASS; ++j) {
                    const uint32_t k = b_r + j * B_PASS;
                    float4 b = bv[j];
                    if (has_act && (rb + k) < r1) {
                        b.x = lrelu_max(fmaf(b.x, sc.x, sh.x), g.slope); b.y = lrelu_max(fmaf(b.y, sc.y, sh.y), g.slope);
                        b.z = lrelu_max(fmaf(b.z, sc.z, sh.z), g.slope); b.w = lrelu_max(fmaf(b.w, sc.w, sh.w), g.slope);
                    }
                    uint4 hi, lo;
                    split_tf32(b.x, hi.x, lo.x); split_tf32(b.y, hi.y, lo.y);
                    split_tf32(b.z, hi.z, lo.z); split_tf32(b.w, hi.w, lo.w);
                    const uint32_t off = b_off0 + (k >> 2) * SBO + (k & 3u) * 128u + ((((b_cm & 7u) >> 1) ^ (k & 3u)) << 5) +
                                         ((b_cm & 1u) << 4);
                    sts128(st + 2 * A_BYTES + off, hi);
                    sts128(st + 2 * A_BYTES + B_BYTES + off, lo);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(full_bar + s);
                issue(kb + 1);
            }
            // ---- epilogue of this item ----
            mbar_wait(accum_bar, item_no & 1u);
            tc_fence_after();
            constexpr int PARTS = PW / 4;                // warps sharing one TMEM lane quarter split the columns
            constexpr int CPART = (BN / PARTS) < 32 ? 32 : (BN / PARTS);
            const int q = warp & 3, part = warp >> 2;
            const int m = m0 + q * 32 + lane;
            float* prow = g.P + (seg * g.M + m) * (int64_t)g.N + n0;
#pragma unroll 1
            for (int cb = part * CPART; cb < (part + 1) * CPART && cb < BN; cb += 32) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)cb, v);
                if (m < g.M) {
#pragma unroll
                    for (int e = 0; e < 32; e += 4)
                        st4(prow + cb + e, make_float4(__uint_as_float(v[e]), __uint_as_float(v[e + 1]),
                                                       __uint_as_float(v[e + 2]), __uint_as_float(v[e + 3])));
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(drained_bar);
        } else {
            if (lane == 0) {
                constexpr uint32_t idesc = make_idesc(BM, BN, true, true);
                if (item_no > 0) {                    // wait until the previous item's accumulator has been read out
                    mbar_wait(drained_bar, (item_no - 1) & 1u);
                    tc_fence_after();
                }
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(full_bar + s, ph);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + s * STAGE_BYTES);
#pragma unroll
                    for (int ks = 0; ks < BK / UMMA_K; ++ks) {
                        const uint32_t koff = ks * 2u * SBO;                    // 8 k-rows = two 4-row groups
                        const uint64_t a_hi = make_desc(sa + koff, LBO, SBO, 1);
                        const uint64_t a_lo = make_desc(sa + A_BYTES + koff, LBO, SBO, 1);
                        const uint64_t b_hi = make_desc(sa + 2 * A_BYTES + koff, LBO, SBO, 1);
                        const uint64_t b_lo = make_desc(sa + 2 * A_BYTES + B_BYTES + koff, LBO, SBO, 1);
                        umma_tf32(tmem_base, a_lo, b_hi, idesc, (kb | ks) != 0);
                        umma_tf32(tmem_base, a_hi, b_lo, idesc, 1);
                        umma_tf32(tmem_base, a_hi, b_hi, idesc, 1);
                    }
                    umma_commit(empty_bar + s);
                }
                umma_commit(accum_bar);
            } else {
                it += num_kb;
            }
            __syncwarp();
        }
    }
    __syncthreads();
    if (warp == PW) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

// out[i] = sum_seg partials[seg][i], float64 accumulate, fixed order: a CTA owns 32 outputs, 8 z-lanes per output add
// every 8th segment in ascending order (independent, coalesced loads) and the lane sums are folded in lane order.
// (One thread per output walking all ~490 segments in a dependent chain took 74 us whatever the output size -- 18
// launches, 1.1 ms per step at 1M faces.)
__global__ void __launch_bounds__(256)
seg_reduce_kernel(const float* __restrict__ partials, float* __restrict__ out, int64_t count, int64_t segs) {
    __shared__ double red[8][33];
    const int o = threadIdx.x & 31, zl = threadIdx.x >> 5;
    const int64_t i = (int64_t)blockIdx.x * 32 + o;
    double s = 0.0;
    if (i < count) {
#pragma unroll 4
        for (int64_t z = zl; z < segs; z += 8) s += (double)__ldg(partials + z * count + i);
    }
    red[zl][o] = s;
    __syncthreads();
    if (zl == 0 && i < count) {
        double v = red[0][o];
#pragma unroll
        for (int z = 1; z < 8; ++z) v += red[z][o];
        out[i] = (float)v;
    }
}

template <int BN, int STAGES, int PW>
static int launch_tn_impl(const TnArgs& g, cudaStream_t st) {
    constexpr size_t smem = (size_t)STAGES * (2 * BM * 128 + 2 * BN * 128) + 1024 + 256;
    static PerDeviceOnce configured;
    if (configured.need()) {
        DDMP_CUDA(cudaFuncSetAttribute(tc_gemm_tn_kernel<BN, STAGES, PW>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
        configured.mark();
    }
    const int64_t grid = g.num_items < kNumSMs ? g.num_items : kNumSMs;
    tc_gemm_tn_kernel<BN, STAGES, PW><<<(unsigned)grid, PW * 32 + 32, smem, st>>>(g);
    return check_launch("tc_gemm_tn");
}
// producer warps: both operands are split in flight here, so the transform is issue-bound with 8 warps (ncu: 42 %
// issue utilisation, tensor pipe 45 %); DDMP_TC_TN_WARPS=8 restores the narrow version for A/B runs
template <int BN, int STAGES>
static int launch_tn(const TnArgs& g, cudaStream_t st) {
    static const int pw = [] { const char* e = getenv("DDMP_TC_TN_WARPS"); return (e && atoi(e) == 8) ? 8 : 16; }();
    if (pw == 16 && BN >= 128) return launch_tn_impl<BN, STAGES, 16>(g, st);
    return launch_tn_impl<BN, STAGES, 8>(g, st);
}

// ---- TN kernel (dW), fp16 split --------------------------------------------------------------------------------------
// Same work decomposition as tc_gemm_tn_kernel (row segments x output tiles, float64 segment reduction); operands are
// scaled by powers of two from their bounds (`amax_a`: row-block maxima of dH from the aggregation kernel, `amax_b`:
// the BatchNorm bound of act(X)), split into fp16 hi/lo and stored MN-major in the 16-bit SWIZZLE_128B canonical
// layout: element (mn, k) of a stage at
//     (mn/64)*LBO + (k/8)*1024 + (k%8)*128 + ((((mn%64)/8) ^ (k%8)) * 16) + (mn%8)*2,    LBO = (BK16/8)*1024
// i.e. a k-row (one graph row) of 64 channels is one 128-byte line, exactly how it lies in global memory.
struct Tn16Args {
    const float* A;       // dH [rows, M] row-major
    const float* B;       // X  [rows, N] row-major (pre-BatchNorm), act over n when scale != null
    float* P;             // partials [num_seg][M][N]
    const float* scale;
    const float* shift;
    float slope;
    const float* amax_a;
    int64_t amax_a_len;
    const float* amax_b;
    int64_t amax_b_len;
    int64_t rows;
    int M, N;
    int tiles_m, tiles_n;
    int64_t num_items;
};

template <int BN, int STAGES>
__global__ void __launch_bounds__(16 * 32 + 32, 1) tc_gemm_tn16_kernel(const Tn16Args g) {
    constexpr int PW = 16;
    constexpr int kPT = PW * 32;
    constexpr uint32_t A_BYTES = BM * BK16 * 2;      // 64 k-rows x 128 m x 2 B
    constexpr uint32_t B_BYTES = BN * BK16 * 2;
    constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + 2 * B_BYTES;
    constexpr uint32_t TMEM_COLS = BN < 32 ? 32 : BN;
    constexpr uint32_t LBO = (BK16 / 8) * 1024;      // next 64-wide MN block
    constexpr uint32_t SBO = 1024;                   // next group of 8 k-rows
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* accum_bar = empty_bar + STAGES;
    uint64_t* drained_bar = accum_bar + 1;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(drained_bar + 1);
    uint32_t* amax_slot = tmem_slot + 1;             // [2]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar + s, PW);
            mbar_init(empty_bar + s, 1);
        }
        mbar_init(accum_bar, 1);
        mbar_init(drained_bar, PW);
        amax_slot[0] = 0u;
        amax_slot[1] = 0u;
        fence_barrier_init();
    }
    if (warp == PW) tmem_alloc(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    block_amax_bits(g.amax_a, g.amax_a_len, amax_slot);
    block_amax_bits(g.amax_b, g.amax_b_len, amax_slot + 1);
    __syncthreads();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t smem_base = smem_u32(smem);
    float s_a, inv_sa, s_b, inv_sb;
    scale_from_bits(amax_slot[0], s_a, inv_sa);
    scale_from_bits(amax_slot[1], s_b, inv_sb);
    const int tiles = g.tiles_m * g.tiles_n;

    uint32_t it = 0;
    uint32_t item_no = 0;
    for (int64_t item = blockIdx.x; item < g.num_items; item += gridDim.x, ++item_no) {
        const int tile = (int)(item % tiles);
        const int64_t seg = item / tiles;
        const int m0 = (tile / g.tiles_n) * BM, n0 = (tile % g.tiles_n) * BN;
        const int64_t r0 = seg * kSegRows;
        const int64_t r1 = (r0 + kSegRows < g.rows) ? (r0 + kSegRows) : g.rows;
        const int num_kb = (int)((r1 - r0 + BK16 - 1) / BK16);

        if (warp < PW) {
            const int t = threadIdx.x;
            // one float4 (4 channels) per thread and k-row: consecutive lanes read consecutive 16 bytes of a graph
            // row, and write the 8-byte half of the 16-byte swizzle chunk they share with their neighbour
            constexpr int A_C4 = BM / 4, B_C4 = BN / 4;                        // float4 per k-row
            const uint32_t a_c4 = t % A_C4, a_r = t / A_C4;
            const uint32_t b_c4 = t % B_C4, b_r = t / B_C4;
            constexpr int A_PASS = kPT / A_C4, B_PASS = kPT / B_C4;            // k-rows per pass of the producers
            constexpr int A_N = BK16 / A_PASS, B_N = BK16 / B_PASS;
            const bool a_ok = (m0 + (int)a_c4 * 4) < g.M;
            const bool has_act = g.scale != nullptr;
            float4 sc = make_float4(s_b, s_b, s_b, s_b), sh = make_float4(0.f, 0.f, 0.f, 0.f);
            if (has_act) {
                sc = ldg4(g.scale + n0 + b_c4 * 4);
                sh = ldg4(g.shift + n0 + b_c4 * 4);
                sc.x *= s_b; sc.y *= s_b; sc.z *= s_b; sc.w *= s_b;
                sh.x *= s_b; sh.y *= s_b; sh.z *= s_b; sh.w *= s_b;
            }
            const uint32_t a_cm = a_c4 >> 1, b_cm = b_c4 >> 1;                 // 16-byte chunk (8 channels)
            const uint32_t a_off0 = (a_cm / 8) * LBO + ((a_c4 & 1u) << 3), b_off0 = (b_cm / 8) * LBO + ((b_c4 & 1u) << 3);
            const uint32_t a_cj = a_cm & 7u, b_cj = b_cm & 7u;
            float4 av[A_N], bv[B_N];
            auto issue = [&](int kb) {
                if (kb >= num_kb) return;
                const int64_t rb = r0 + (int64_t)kb * BK16;
#pragma unroll
                for (int j = 0; j < A_N; ++j) {
                    const int64_t r = rb + a_r + j * A_PASS;
                    av[j] = (r < r1 && a_ok) ? ldg4(g.A + r * g.M + m0 + a_c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int j = 0; j < B_N; ++j) {
                    const int64_t r = rb + b_r + j * B_PASS;
                    bv[j] = (r < r1) ? ldg4(g.B + r * g.N + n0 + b_c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            issue(0);
            for (int kb = 0; kb < num_kb; ++kb, ++it) {
                const int s = it % STAGES;
                const uint32_t ph = (it / STAGES) & 1;
                const int64_t rb = r0 + (int64_t)kb * BK16;
                mbar_wait(empty_bar + s, ph ^ 1u);
                const uint32_t st = smem_base + s * STAGE_BYTES;
#pragma unroll
                for (int j = 0; j < A_N; ++j) {
                    const uint32_t k = a_r + j * A_PASS;
                    float4 a = av[j];
                    a.x *= s_a; a.y *= s_a; a.z *= s_a; a.w *= s_a;
                    uint32_t h0, l0, h1, l1;
                    split_f16x2(a.x, a.y, h0, l0);
                    split_f16x2(a.z, a.w, h1, l1);
                    const uint32_t off = a_off0 + (k >> 3) * SBO + (k & 7u) * 128u + ((a_cj ^ (k & 7u)) << 4);
                    sts64(st + off, h0, h1);
                    sts64(st + A_BYTES + off, l0, l1);
                }
#pragma unroll
                for (int j = 0; j < B_N; ++j) {
                    const uint32_t k = b_r + j * B_PASS;
                    float4 a = bv[j];
                    if (has_act) {
                        if ((rb + k) < r1) {
                            a.x = lrelu_max(fmaf(a.x, sc.x, sh.x), g.slope); a.y = lrelu_max(fmaf(a.y, sc.y, sh.y), g.slope);
                            a.z = lrelu_max(fmaf(a.z, sc.z, sh.z), g.slope); a.w = lrelu_max(fmaf(a.w, sc.w, sh.w), g.slope);
                        }
                    } else {
                        a.x *= s_b; a.y *= s_b; a.z *= s_b; a.w *= s_b;
                    }
                    uint32_t h0, l0, h1, l1;
                    split_f16x2(a.x, a.y, h0, l0);
                    split_f16x2(a.z, a.w, h1, l1);
                    const uint32_t off = b_off0 + (k >> 3) * SBO + (k & 7u) * 128u + ((b_cj ^ (k & 7u)) << 4);
                    sts64(st + 2 * A_BYTES + off, h0, h1);
                    sts64(st + 2 * A_BYTES + B_BYTES + off, l0, l1);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(full_bar + s);
                issue(kb + 1);
            }
            // ---- epilogue of this item ----
            mbar_wait(accum_bar, item_no & 1u);
            tc_fence_after();
            constexpr int PARTS = PW / 4;
            constexpr int CPART = (BN / PARTS) < 32 ? 32 : (BN / PARTS);
            const int q = warp & 3, part = warp >> 2;
            const int m = m0 + q * 32 + lane;
            float* prow = g.P + (seg * g.M + m) * (int64_t)g.N + n0;
            const float inv = inv_sa * inv_sb;       // both are normal powers of two well inside the float range
#pragma unroll 1
            for (int cb = part * CPART; cb < (part + 1) * CPART && cb < BN; cb += 32) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)cb, v);
                if (m < g.M) {
#pragma unroll
                    for (int e = 0; e < 32; e += 4)
                        st4(prow + cb + e, make_float4(__uint_as_float(v[e]) * inv, __uint_as_float(v[e + 1]) * inv,
                                                       __uint_as_float(v[e + 2]) * inv, __uint_as_float(v[e + 3]) * inv));
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(drained_bar);
        } else {
            if (lane == 0) {
                constexpr uint32_t idesc = make_idesc16(BM, BN, true, true);
                if (item_no > 0) {
                    mbar_wait(drained_bar, (item_no - 1) & 1u);
                    tc_fence_after();
                }
                for (int kb = 0; kb < num_kb; ++kb, ++it) {
                    const int s = it % STAGES;
                    const uint32_t ph = (it / STAGES) & 1;
                    mbar_wait(full_bar + s, ph);
                    tc_fence_after();
                    const uint32_t sa = smem_u32(smem + s * STAGE_BYTES);
#pragma unroll
                    for (int ks = 0; ks < BK16 / UMMA_K16; ++ks) {
                        const uint32_t koff = ks * 2u * SBO;                    // 16 k-rows = two 8-row groups
                        const uint64_t a_hi = make_desc(sa + koff, LBO, SBO, 2);
                        const uint64_t a_lo = make_desc(sa + A_BYTES + koff, LBO, SBO, 2);
                        const uint64_t b_hi = make_desc(sa + 2 * A_BYTES + koff, LBO, SBO, 2);
                        const uint64_t b_lo = make_desc(sa + 2 * A_BYTES + B_BYTES + koff, LBO, SBO, 2);
                        umma_f16(tmem_base, a_lo, b_hi, idesc, (kb | ks) != 0);
                        umma_f16(tmem_base, a_hi, b_lo, idesc, 1);
                        umma_f16(tmem_base, a_hi, b_hi, idesc, 1);
                    }
                    umma_commit(empty_bar + s);
                }
                umma_commit(accum_bar);
            } else {
                it += num_kb;
            }
            __syncwarp();
        }
    }
    __syncthreads();
    if (warp == PW) {
        tc_fence_after();
        tmem_dealloc(tmem_base, TMEM_COLS);
    }
}

template <int BN, int STAGES>
static int launch_tn16(const Tn16Args& g, cudaStream_t st) {
    constexpr size_t smem = (size_t)STAGES * (2 * BM * BK16 * 2 + 2 * BN * BK16 * 2) + 1024 + 256;
    static PerDeviceOnce configured;
    if (configured.need()) {
        DDMP_CUDA(cudaFuncSetAttribute(tc_gemm_tn16_kernel<BN, STAGES>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
        configured.mark();
    }
    const int64_t grid = g.num_items < kNumSMs ? g.num_items : kNumSMs;
    tc_gemm_tn16_kernel<BN, STAGES><<<(unsigned)grid, 16 * 32 + 32, smem, st>>>(g);
    return check_launch("tc_gemm_tn16");
}

// TN kernel on CTA pairs (cta_group::2): the pair owns a 256 x (256*NACC) tile of dW.  Each CTA splits its 128
// channels of dH and 128*NACC channels of X per k-row, the MMAs (M = 256, N = 256 per accumulator) read both CTAs'
// halves, and each CTA's TMEM receives its 128 output rows x 256*NACC columns.  Against the single-CTA kernel
// (128 x 256 tiles) every element of dH is split once instead of Cin/256 times and every element of X Cout/256
// instead of Cout/128 times: the producer work per MMA -- which bounds this kernel -- halves for 512 x 512.
template <int NACC>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(16 * 32 + 32, 1) tc_gemm_tn16x2_kernel(const Tn16Args g) {
    constexpr int PW = 16;
    constexpr int kPT = PW * 32;
    constexpr int STAGES = (NACC == 2) ? 2 : 3;
    constexpr uint32_t A_BYTES = BM * BK16 * 2;          // this CTA's 128 dH channels x 64 k-rows, one of hi / lo
    constexpr uint32_t B_BLK = 128 * BK16 * 2;           // this CTA's 128 X channels of one accumulator
    constexpr uint32_t STAGE_BYTES = 2 * A_BYTES + NACC * 2 * B_BLK;
    constexpr uint32_t TMEM_COLS = NACC * 256;
    constexpr uint32_t LBO = (BK16 / 8) * 1024;
    constexpr uint32_t SBO = 1024;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
    uint64_t* empty_bar = full_bar + STAGES;
    uint64_t* peer_ready = empty_bar + STAGES;           // leader only
    uint64_t* accum_bar = peer_ready + STAGES;
    uint64_t* drained_bar = accum_bar + 1;               // leader only: both CTAs have read the accumulators out
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(drained_bar + 1);
    uint32_t* amax_slot = tmem_slot + 1;                 // [2]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const int64_t num_pairs = gridDim.x / 2, pair = blockIdx.x / 2;
    if (threadIdx.x == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(full_bar + s, PW);
            mbar_init(empty_bar + s, 1);
            mbar_init(peer_ready + s, 1);
        }
        mbar_init(accum_bar, 1);
        mbar_init(drained_bar, 2 * PW);
        amax_slot[0] = 0u;
        amax_slot[1] = 0u;
        fence_barrier_init();
    }
    cluster_sync_all();
    if (warp == PW) tmem_alloc_2cta(tmem_slot, TMEM_COLS);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    block_amax_bits(g.amax_a, g.amax_a_len, amax_slot);
    block_amax_bits(g.amax_b, g.amax_b_len, amax_slot + 1);
    __syncthreads();
    const uint32_t tmem_base = *tmem_slot;
    const uint32_t smem_base = smem_u32(smem);
    float s_a, inv_sa, s_b, inv_sb;
    scale_from_bits(amax_slot[0], s_a, inv_sa);
    scale_from_bits(amax_slot[1], s_b, inv_sb);
    const int tiles = g.tiles_m * g.tiles_n;             // pair tiles: 256 x (256*NACC)

    uint32_t it = 0;
    uint32_t item_no = 0;
    for (int64_t item = pair; item < g.num_items; item += num_pairs, ++item_no) {
        const int tile = (int)(item % tiles);
        const int64_t seg = item / tiles;
        const int m0 = (tile / g.tiles_n) * 256 + (int)rank * 128;     // this CTA's dH channels / output rows
        const int n0 = (tile % g.tiles_n) * 256 * NACC;                // first column of the pair tile
        const int64_t r0 = seg * kSegRows;
        const int64_t r1 = (r0 + kSegRows < g.rows) ? (r0 + kSegRows) : g.rows;
        const int num_kb = (int)((r1 - r0 + BK16 - 1) / BK16);

        if (warp < PW) {
            const int t = threadIdx.x;
            constexpr int A_C4 = 32, B_C4 = NACC * 32;                         // float4 per k-row (this CTA's part)
            const uint32_t a_c4 = t % A_C4, a_r = t / A_C4;
            const uint32_t b_c4 = t % B_C4, b_r = t / B_C4;
            constexpr int A_PASS = kPT / A_C4, B_PASS = kPT / B_C4;
            constexpr int A_N = BK16 / A_PASS, B_N = BK16 / B_PASS;
            const uint32_t b_acc = b_c4 / 32, b_in = b_c4 % 32;                // accumulator block, float4 inside it
            const int b_ch = n0 + (int)b_acc * 256 + (int)rank * 128 + (int)b_in * 4;   // global X channel
            const bool has_act = g.scale != nullptr;
            float4 sc = make_float4(s_b, s_b, s_b, s_b), sh = make_float4(0.f, 0.f, 0.f, 0.f);
            if (has_act) {
                sc = ldg4(g.scale + b_ch);
                sh = ldg4(g.shift + b_ch);
                sc.x *= s_b; sc.y *= s_b; sc.z *= s_b; sc.w *= s_b;
                sh.x *= s_b; sh.y *= s_b; sh.z *= s_b; sh.w *= s_b;
            }
            const uint32_t a_cm = a_c4 >> 1, b_cm = b_in >> 1;
            const uint32_t a_off0 = (a_cm / 8) * LBO + ((a_c4 & 1u) << 3);
            const uint32_t b_off0 = 2 * A_BYTES + b_acc * (2 * B_BLK) + (b_cm / 8) * LBO + ((b_in & 1u) << 3);
            const uint32_t a_cj = a_cm & 7u, b_cj = b_cm & 7u;
            float4 av[A_N], bv[B_N];
            auto issue = [&](int kb) {
                if (kb >= num_kb) return;
                const int64_t rb = r0 + (int64_t)kb * BK16;
#pragma unroll
                for (int j = 0; j < A_N; ++j) {
                    const int64_t r = rb + a_r + j * A_PASS;
                    av[j] = (r < r1) ? ldg4(g.A + r * g.M + m0 + a_c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
#pragma unroll
                for (int j = 0; j < B_N; ++j) {
                    const int64_t r = rb + b_r + j * B_PASS;
                    bv[j] = (r < r1) ? ldg4(g.B + r * g.N + b_ch) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            issue(0);
            for (int kb = 0; kb < num_kb; ++kb, ++it) {
                const int s = it % STAGES;
                const uint32_t ph = (it / STAGES) & 1;
                const int64_t rb = r0 + (int64_t)kb * BK16;
                mbar_wait_cluster(empty_bar + s, ph ^ 1u);
                const uint32_t st = smem_base + s * STAGE_BYTES;
#pragma unroll
                for (int j = 0; j < A_N; ++j) {
                    const uint32_t k = a_r + j * A_PASS;
                    float4 a = av[j];
                    a.x *= s_a; a.y *= s_a; a.z *= s_a; a.w *= s_a;
                    uint32_t h0, l0, h1, l1;
                    split_f16x2(a.x, a.y, h0, l0);
                    split_f16x2(a.z, a.w, h1, l1);
                    const uint32_t off = a_off0 + (k >> 3) * SBO + (k & 7u) * 128u + ((a_cj ^ (k & 7u)) << 4);
                    sts64(st + off, h0, h1);
                    sts64(st + A_BYTES + off, l0, l1);
                }
#pragma unroll
                for (int j = 0; j < B_N; ++j) {
                    const uint32_t k = b_r + j * B_PASS;
                    float4 a = bv[j];
                    if (has_act) {
                        if ((rb + k) < r1) {
                            a.x = lrelu_max(fmaf(a.x, sc.x, sh.x), g.slope); a.y = lrelu_max(fmaf(a.y, sc.y, sh.y), g.slope);
                            a.z = lrelu_max(fmaf(a.z, sc.z, sh.z), g.slope); a.w = lrelu_max(fmaf(a.w, sc.w, sh.w), g.slope);
                        }
                    } else {
                        a.x *= s_b; a.y *= s_b; a.z *= s_b; a.w *= s_b;
                    }
                    uint32_t h0, l0, h1, l1;
                    split_f16x2(a.x, a.y, h0, l0);
                    split_f16x2(a.z, a.w, h1, l1);
                    const uint32_t off = b_off0 + (k >> 3) * SBO + (k & 7u) * 128u + ((b_cj ^ (k & 7u)) << 4);
                    sts64(st + off, h0, h1);
                    sts64(st + B_BLK + off, l0, l1);
                }
                fence_proxy_async();
                __syncwarp();
                if (lane == 0) mbar_arrive(full_bar + s);
                issue(kb + 1);
            }
            // ---- epilogue of this item: this CTA's 128 rows x 256*NACC columns ----
            mbar_wait_cluster(accum_bar, item_no & 1u);
            tc_fence_after();
            constexpr int PARTS = PW / 4;
            constexpr int CPART = (256 * NACC) / PARTS;
            const int q = warp & 3, part = warp >> 2;
            const int m = m0 + q * 32 + lane;
            float* prow = g.P + (seg * g.M + m) * (int64_t)g.N + n0;
            const float inv = inv_sa * inv_sb;
#pragma unroll 1
            for (int cb = part * CPART; cb < (part + 1) * CPART; cb += 32) {
                uint32_t v[32];
                tmem_ld32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)cb, v);
                if (m < g.M) {
#pragma unroll
                    for (int e = 0; e < 32; e += 4)
                        st4(prow + cb + e, make_float4(__uint_as_float(v[e]) * inv, __uint_as_float(v[e + 1]) * inv,
                                                       __uint_as_float(v[e + 2]) * inv, __uint_as_float(v[e + 3]) * inv));
                }
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if (rank == 0) mbar_arrive(drained_bar);
                else mbar_arrive_remote(drained_bar, 0);
            }
        } else {
            if (lane == 0) {
                if (rank == 0) {
                    constexpr uint32_t idesc = make_idesc16(256, 256, true, true);
                    if (item_no > 0) {
                        mbar_wait_cluster(drained_bar, (item_no - 1) & 1u);
                        tc_fence_after();
                    }
                    for (int kb = 0; kb < num_kb; ++kb, ++it) {
                        const int s = it % STAGES;
                        const uint32_t ph = (it / STAGES) & 1;
                        mbar_wait(full_bar + s, ph);
                        mbar_wait_cluster(peer_ready + s, ph);
                        tc_fence_after();
                        const uint32_t sa = smem_base + s * STAGE_BYTES;
#pragma unroll
                        for (int ks = 0; ks < BK16 / UMMA_K16; ++ks) {
                            const uint32_t koff = ks * 2u * SBO;
                            const uint64_t a_hi = make_desc(sa + koff, LBO, SBO, 2);
                            const uint64_t a_lo = make_desc(sa + A_BYTES + koff, LBO, SBO, 2);
#pragma unroll
                            for (int j = 0; j < NACC; ++j) {
                                const uint32_t sb = sa + 2 * A_BYTES + j * (2 * B_BLK) + koff;
                                const uint64_t b_hi = make_desc(sb, LBO, SBO, 2);
                                const uint64_t b_lo = make_desc(sb + B_BLK, LBO, SBO, 2);
                                const uint32_t d = tmem_base + j * 256;
                                umma_f16_2cta(d, a_lo, b_hi, idesc, (kb | ks) != 0);
                                umma_f16_2cta(d, a_hi, b_lo, idesc, 1);
                                umma_f16_2cta(d, a_hi, b_hi, idesc, 1);
                            }
                        }
                        umma_commit_2cta(empty_bar + s);
                    }
                    umma_commit_2cta(accum_bar);
                } else {
                    for (int kb = 0; kb < num_kb; ++kb, ++it) {
                        const int s = it % STAGES;
                        const uint32_t ph = (it / STAGES) & 1;
                        mbar_wait(full_bar + s, ph);
                        mbar_arrive_remote(peer_ready + s, 0);
                    }
                }
            } else {
                it += num_kb;
            }
            __syncwarp();
        }
    }
    tc_fence_before();
    cluster_sync_all();
    if (warp == PW) {
        tc_fence_after();
        tmem_dealloc_2cta(tmem_base, TMEM_COLS);
    }
}

template <int NACC>
static int launch_tn16x2(const Tn16Args& g, cudaStream_t st) {
    constexpr int STAGES = (NACC == 2) ? 2 : 3;
    constexpr size_t smem = (size_t)STAGES * (2 * BM * BK16 * 2 + NACC * 2 * 128 * BK16 * 2) + 1024 + 256;
    static PerDeviceOnce configured;
    if (configured.need()) {
        DDMP_CUDA(cudaFuncSetAttribute(tc_gemm_tn16x2_kernel<NACC>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
        configured.mark();
    }
    const int64_t pairs = g.num_items < kNumSMs / 2 ? g.num_items : kNumSMs / 2;
    tc_gemm_tn16x2_kernel<NACC><<<(unsigned)(2 * pairs), 16 * 32 + 32, smem, st>>>(g);
    return check_launch("tc_gemm_tn16x2");
}

}  // namespace tc

static inline bool tc_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Both the reduction width and the output width of the NT kernels may be as small as 32 (one k-block / a 32-column UMMA
// tile of the 3xTF32 kernel): at 1M rows X.W^T 32 -> 64 takes 0.118 ms instead of 0.195 on the FFMA kernel, dH.W of the
// 64 -> 32 layer 0.105 instead of 0.153 (profiles/gemm_narrow_ab_r2.txt).  The TN kernel with a 32-row M tile (dH^T.X of
// the 64 -> 32 layer) measured SLOWER than FFMA (0.342 vs 0.297 ms: it pays for a whole 128-row tile); the narrow dW
// products have their own FFMA kernel (gemm_ffma.cu: dw_narrow_kernel).
bool tc_supported_xw(int64_t n, int32_t Cin, int32_t Cout) {
    return n > 0 && Cin >= 32 && Cout >= 32 && Cin % 32 == 0 && Cout % 32 == 0 && Cout <= 4096;
}
bool tc_supported_dx(int64_t n, int32_t Cin, int32_t Cout) {
    return n > 0 && Cin >= 32 && Cout >= 32 && Cout % 32 == 0 && Cin % 32 == 0 && Cin <= 4096;
}
bool tc_supported_dw(int64_t n, int32_t Cin, int32_t Cout) {
    return n > 0 && Cin >= 64 && Cout >= 64 && Cin % 64 == 0 && Cout % 4 == 0 && Cin <= 4096 && Cout <= 4096;
}

int64_t tc_gemm_nt_workspace_bytes(int32_t Cin, int32_t Cout) { return 2ll * Cin * Cout * (int64_t)sizeof(float); }

int tc_gemm_xw(const float* X, const int32_t* row_map, const float* scale, const float* shift, float slope,
               const float* W, float* H, void* workspace, int64_t workspace_bytes, int64_t n, int32_t Cin,
               int32_t Cout, const float* amax, int64_t amax_len, cudaStream_t st) {
    DDMP_REQUIRE(tc_aligned16(X) && tc_aligned16(W) && tc_aligned16(H), "tc_gemm_xw: pointers must be 16-byte aligned");
    DDMP_REQUIRE(workspace && tc_aligned16(workspace) && workspace_bytes >= tc_gemm_nt_workspace_bytes(Cin, Cout),
                 "tc_gemm_xw: workspace too small");
    if (amax && amax_len > 0 && Cin % tc::BK16 == 0 && Cout % 64 == 0 && tc::f16_split_enabled())
        return tc::run_nt16(X, row_map, scale, shift, slope, W, 0, workspace, H, n, Cout, Cin, amax, amax_len, st);
    return tc::run_nt2(X, row_map, scale, shift, slope, W, 0, workspace, H, n, Cout, Cin, st);
}

// gX[n,Cin] = dH[n,Cout] * W[Cout,Cin]: B operand (K-major) is W^T, built directly into the swizzled image.
int tc_gemm_dx(const float* dH, const float* W, float* gX, void* workspace, int64_t workspace_bytes, int64_t n,
               int32_t Cin, int32_t Cout, const float* amax, int64_t amax_len, cudaStream_t st) {
    DDMP_REQUIRE(tc_aligned16(dH) && tc_aligned16(W) && tc_aligned16(gX), "tc_gemm_dx: pointers must be 16-byte aligned");
    DDMP_REQUIRE(workspace && tc_aligned16(workspace) && workspace_bytes >= tc_gemm_nt_workspace_bytes(Cin, Cout),
                 "tc_gemm_dx: workspace too small");
    if (amax && amax_len > 0 && Cout % tc::BK16 == 0 && Cin % 64 == 0 && tc::f16_split_enabled())
        return tc::run_nt16(dH, nullptr, nullptr, nullptr, 0.f, W, 1, workspace, gX, n, Cin, Cout, amax, amax_len, st);
    return tc::run_nt2(dH, nullptr, nullptr, nullptr, 0.f, W, 1, workspace, gX, n, Cin, Cout, st);
}

int64_t tc_gemm_dw_workspace_bytes(int64_t n, int32_t Cin, int32_t Cout) {
    return ceil_div(n, tc::kSegRows) * (int64_t)Cin * Cout * (int64_t)sizeof(float);
}

int tc_gemm_dw(const float* dH, const float* X, const int32_t* row_map, const float* scale, const float* shift,
               float slope, float* dW, void* workspace, int64_t workspace_bytes, int64_t n, int32_t Cin, int32_t Cout,
               const float* amax_dh, int64_t amax_dh_len, const float* amax_x, int64_t amax_x_len, cudaStream_t st) {
    DDMP_REQUIRE(row_map == nullptr, "tc_gemm_dw: row_map is only supported by the FFMA path");
    DDMP_REQUIRE(workspace && workspace_bytes >= tc_gemm_dw_workspace_bytes(n, Cin, Cout),
                 "tc_gemm_dw: workspace too small (%lld bytes)", (long long)workspace_bytes);
    DDMP_REQUIRE(tc_aligned16(dH) && tc_aligned16(X) && tc_aligned16(workspace), "tc_gemm_dw: 16-byte alignment");
    const int64_t count = (int64_t)Cin * Cout;
    // fp16 split: 10-30 % faster than 3xTF32 on every shape (1M rows: 512->512 2.39 vs 2.71 ms, 64->128 0.27 vs 0.36);
    // both operands are split by the producer warps here, which bounds this kernel.  DDMP_TC_TN16=0 -> 3xTF32
    static const bool tn16_off = [] { const char* e = getenv("DDMP_TC_TN16"); return e && e[0] == '0'; }();
    if (amax_dh && amax_x && amax_dh_len > 0 && amax_x_len > 0 && Cout % 4 == 0 && tc::f16_split_enabled() &&
        !tn16_off) {
        tc::Tn16Args h{};
        h.A = dH; h.B = X; h.P = reinterpret_cast<float*>(workspace); h.scale = scale; h.shift = shift; h.slope = slope;
        h.amax_a = amax_dh; h.amax_a_len = amax_dh_len; h.amax_b = amax_x; h.amax_b_len = amax_x_len;
        h.rows = n; h.M = Cout; h.N = Cin;
        h.tiles_m = (int)ceil_div(Cout, tc::BM);
        const int64_t segs16 = ceil_div(n, tc::kSegRows);
        int rc16;
        static const bool tn_one_cta = [] { const char* e = getenv("DDMP_TC_2CTA"); return e && e[0] == '0'; }();
        if (!tn_one_cta && Cout % 256 == 0 && Cin % 256 == 0) {
            h.tiles_m = Cout / 256;
            if (Cin % 512 == 0) { h.tiles_n = Cin / 512; h.num_items = segs16 * h.tiles_m * h.tiles_n; rc16 = tc::launch_tn16x2<2>(h, st); }
            else { h.tiles_n = Cin / 256; h.num_items = segs16 * h.tiles_m * h.tiles_n; rc16 = tc::launch_tn16x2<1>(h, st); }
        }
        else if (Cin % 256 == 0) { h.tiles_n = Cin / 256; h.num_items = segs16 * h.tiles_m * h.tiles_n; rc16 = tc::launch_tn16<256, 2>(h, st); }
        else if (Cin % 128 == 0) { h.tiles_n = Cin / 128; h.num_items = segs16 * h.tiles_m * h.tiles_n; rc16 = tc::launch_tn16<128, 3>(h, st); }
        else { h.tiles_n = Cin / 64; h.num_items = segs16 * h.tiles_m * h.tiles_n; rc16 = tc::launch_tn16<64, 4>(h, st); }
        if (rc16) return rc16;
        tc::seg_reduce_kernel<<<(unsigned)ceil_div(count, 32), 256, 0, st>>>(h.P, dW, count, segs16);
        return check_launch("tc seg_reduce");
    }
    tc::TnArgs g{};
    g.A = dH; g.B = X; g.P = reinterpret_cast<float*>(workspace); g.scale = scale; g.shift = shift; g.slope = slope;
    g.rows = n; g.M = Cout; g.N = Cin;
    g.tiles_m = (int)ceil_div(Cout, tc::BM);
    const int64_t segs = ceil_div(n, tc::kSegRows);
    int rc;
    if (Cin % 256 == 0) { g.tiles_n = Cin / 256; g.num_items = segs * g.tiles_m * g.tiles_n; rc = tc::launch_tn<256, 2>(g, st); }
    else if (Cin % 128 == 0) { g.tiles_n = Cin / 128; g.num_items = segs * g.tiles_m * g.tiles_n; rc = tc::launch_tn<128, 3>(g, st); }
    else { g.tiles_n = Cin / 64; g.num_items = segs * g.tiles_m * g.tiles_n; rc = tc::launch_tn<64, 4>(g, st); }
    if (rc) return rc;
    tc::seg_reduce_kernel<<<(unsigned)ceil_div(count, 32), 256, 0, st>>>(g.P, dW, count, segs);
    return check_launch("tc seg_reduce");
}

}  // namespace ddmp
