// Shared device/host helpers for libddmp_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include <atomic>

#include "../../include/ddmp_b200.h"

namespace ddmp {

// ---- error convention: 0 = ok, negative = failure, message in a thread-local buffer (include/ddmp_b200.h) ----
void set_error(const char* fmt, ...);
int check_launch(const char* what);   // also counts the launch (ddmp_launch_count)
long long launch_count();

#define DDMP_REQUIRE(cond, ...)                                   \
    do {                                                          \
        if (!(cond)) {                                            \
            ::ddmp::set_error(__VA_ARGS__);                       \
            return DDMP_ERR_INVALID;                              \
        }                                                         \
    } while (0)

#define DDMP_CUDA(call)                                                                      \
    do {                                                                                     \
        cudaError_t e__ = (call);                                                            \
        if (e__ != cudaSuccess) {                                                            \
            ::ddmp::set_error("%s failed: %s", #call, cudaGetErrorString(e__));              \
            return DDMP_ERR_CUDA;                                                            \
        }                                                                                    \
    } while (0)

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

constexpr int kNumSMs = 148;          // B200
constexpr float kLeakySlope = 0.01f;  // nn.LeakyReLU() default, reference util/networks.py:44,105

// ---- device helpers ----------------------------------------------------------------------------------------
__device__ __forceinline__ float lrelu(float z, float slope) { return z > 0.f ? z : z * slope; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Block-wide sum of one double per thread, fixed combination order (deterministic). Result valid in thread 0.
template <int THREADS>
__device__ __forceinline__ double block_sum(double v, double* smem /* >= THREADS/32 */) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) smem[wid] = v;
    __syncthreads();
    double r = 0.0;
    if (threadIdx.x == 0) {
#pragma unroll
        for (int i = 0; i < THREADS / 32; ++i) r += smem[i];
    }
    __syncthreads();
    return r;
}

// "Last block finalises" pattern: every block publishes its partial, the block that arrives last (atomic ticket)
// sums ALL partials in index order, so the result does not depend on which block was last.  The ticket counter
// must be zero on entry and is reset to zero by the last block (self-cleaning workspace).
__device__ __forceinline__ bool publish_and_am_last(unsigned int* ticket, unsigned int nblocks) {
    __shared__ bool is_last;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = atomicAdd(ticket, 1u);
        is_last = (t == nblocks - 1);
        if (is_last) *ticket = 0u;
    }
    __syncthreads();
    if (is_last) __threadfence();
    return is_last;
}

// "Done once per device" flag for per-device function attributes (cudaFuncSetAttribute is per device/context, the
// library can be driven on several devices of one process through ddmp_set_device, and launchers are called from the
// main thread and from the autograd thread): one bit per device ordinal, set with an atomic OR.
struct PerDeviceOnce {
    std::atomic<unsigned long long> done{0ull};
    static unsigned long long bit() {
        int d = 0;
        cudaGetDevice(&d);
        return 1ull << (d & 63);
    }
    bool need() const { return (done.load(std::memory_order_acquire) & bit()) == 0ull; }
    void mark() { done.fetch_or(bit(), std::memory_order_release); }
};

// 2-D tensor map (TMA descriptor) of a row-major fp32 [outer, inner] tensor, box = [box_outer, box_inner]; swizzle128:
// CU_TENSOR_MAP_SWIZZLE_128B (box_inner * 4 must be 128 bytes) else no swizzle.  `map` points to a CUtensorMap (128 bytes,
// 64-byte aligned).  cuTensorMapEncodeTiled is resolved through the runtime, so the library has no link-time dependency
// on libcuda.so (it must load on boxes without a driver: tests/test_cabi.py).
int make_tensor_map_2d(void* map, const float* base, int64_t outer, int64_t inner, int box_outer, int box_inner,
                       bool swizzle128, const char* who);

// tile-staged aggregation kernel (spmm_tile.cu)
bool spmm_tile_supported(int64_t n, int C);
int spmm_tile_launch(const int* rowptr, const int* col, const float* w, const float* H, const float* bias, float* Y,
                     float* partials, float* amax, int64_t n, int C, cudaStream_t st);

__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }

}  // namespace ddmp
