// Library-level entry points and the error channel of libddmp_b200.
#include <stdarg.h>
#include <stdlib.h>
#include <atomic>
#include <string.h>

#include <cuda.h>

#include "common.cuh"

namespace ddmp {

typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                             const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                             CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeFn encode_fn() {
    static EncodeFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        return reinterpret_cast<EncodeFn>(p);
    }();
    return fn;
}

int make_tensor_map_2d(void* map, const float* base, int64_t outer, int64_t inner, int box_outer, int box_inner,
                       bool swizzle128, const char* who) {
    // the driver call needs a current context on THIS thread: the autograd engine's thread may reach its first kernel of
    // a backward pass before any runtime call has bound the primary context to it
    static thread_local const bool bound = (cudaFree(nullptr), true);
    (void)bound;
    EncodeFn enc = encode_fn();
    if (!enc) {
        set_error("%s: cuTensorMapEncodeTiled is not available from this driver", who);
        return DDMP_ERR_CUDA;
    }
    const cuuint64_t dims[2] = {(cuuint64_t)inner, (cuuint64_t)outer};
    const cuuint64_t strides[1] = {(cuuint64_t)inner * 4};
    const cuuint32_t box[2] = {(cuuint32_t)box_inner, (cuuint32_t)box_outer};
    const cuuint32_t estr[2] = {1, 1};
    CUresult rc = enc(reinterpret_cast<CUtensorMap*>(map), CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base),
                      dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                      swizzle128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_NONE,
                      CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) {
        set_error("%s: cuTensorMapEncodeTiled failed (CUresult %d) for base=%p [%lld x %lld] box=%dx%d", who, (int)rc,
                  (const void*)base, (long long)outer, (long long)inner, box_outer, box_inner);
        return DDMP_ERR_CUDA;
    }
    return DDMP_OK;
}

static thread_local char g_err[512] = "";
static std::atomic<long long> g_launches{0};

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

long long launch_count() { return g_launches.load(); }

int check_launch(const char* what) {
    g_launches.fetch_add(1);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: kernel launch failed: %s", what, cudaGetErrorString(e));
        return DDMP_ERR_CUDA;
    }
    return DDMP_OK;
}

}  // namespace ddmp

extern "C" {

int ddmp_version(void) { return 100; }

int64_t ddmp_launch_count(void) { return (int64_t)ddmp::launch_count(); }

const char* ddmp_last_error(void) { return ddmp::g_err; }

int ddmp_set_device(int device) {
    int cur = -1;
    DDMP_CUDA(cudaGetDevice(&cur));
    if (cur != device) DDMP_CUDA(cudaSetDevice(device));
    return DDMP_OK;
}

int ddmp_device_info(int* sm_count, int* cc_major, int* cc_minor) {
    int dev = 0;
    DDMP_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp p;
    DDMP_CUDA(cudaGetDeviceProperties(&p, dev));
    if (sm_count) *sm_count = p.multiProcessorCount;
    if (cc_major) *cc_major = p.major;
    if (cc_minor) *cc_minor = p.minor;
    return DDMP_OK;
}

int ddmp_rows_per_block(int32_t C) {
    if (C <= 0) return 0;
    // 128 rows per CTA for the wide layers, 256 for the narrow ones: >= 3,900 CTAs at 1M rows (a grid of 980 CTAs,
    // as with 1024 rows per block, leaves a mostly empty second wave: ncu, profiles/)
    // 128 rows per CTA from width 64 up (tile-staged kernel at C = 64: 32 KB tile, 5 CTAs per SM -- 2.6-2.9 / 4.2-4.8 TB/s
    // on the vertex / face graph against 1.9 / 3.2 with 256 rows)
    return C <= 32 ? 256 : 128;
}

// Row block of the element-wise BatchNorm-backward / column-sum kernels (bn.cu).  Independent of the aggregation kernel's
// block: 512 rows keep >= 1,900 CTAs at 1M rows while the [blocks][sets][C] partials -- which the finalize kernels
// re-read with only C/8 CTAs -- shrink 4x against 128-row blocks (finalize: 46 us -> ~12 us at C = 512, 48 per step).
int ddmp_elem_rows_per_block(int32_t C) { return C > 0 ? 512 : 0; }

int64_t ddmp_num_elem_blocks(int64_t n, int32_t C) {
    const int r = ddmp_elem_rows_per_block(C);
    if (r <= 0 || n <= 0) return 0;
    return (n + r - 1) / r;
}

int64_t ddmp_num_row_blocks(int64_t n, int32_t C) {
    int r = ddmp_rows_per_block(C);
    if (r <= 0 || n <= 0) return 0;
    return (n + r - 1) / r;
}

}  // extern "C"
