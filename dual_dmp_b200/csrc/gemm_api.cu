// Backend dispatch of the dense feature transform (include/ddmp_b200.h "dense feature transform").
// AUTO: tcgen05 3xTF32 where both channel widths are >= 64 (tensor-pipe bound), FFMA below (memory bound).
// DDMP_GEMM_F16X1 on top of any backend: the fp16-split kernels among these run with one product instead of three.
#include "common.cuh"

namespace ddmp {
int ffma_gemm_xw(const float*, const int32_t*, const float*, const float*, float, const float*, float*, int64_t,
                 int32_t, int32_t, cudaStream_t);
int ffma_gemm_dx(const float*, const float*, float*, int64_t, int32_t, int32_t, cudaStream_t);
int64_t ffma_gemm_dw_workspace_bytes(int64_t, int32_t, int32_t);
int ffma_gemm_dw(const float*, const float*, const int32_t*, const float*, const float*, float, float*, void*,
                 int64_t, int64_t, int32_t, int32_t, cudaStream_t);
#ifdef DDMP_WITH_TC
bool tc_supported_xw(int64_t n, int32_t Cin, int32_t Cout);
bool tc_supported_dx(int64_t n, int32_t Cin, int32_t Cout);
bool tc_supported_dw(int64_t n, int32_t Cin, int32_t Cout);
int64_t tc_gemm_nt_workspace_bytes(int32_t, int32_t);
int tc_gemm_xw(const float*, const int32_t*, const float*, const float*, float, const float*, float*, void*, int64_t,
               int64_t, int32_t, int32_t, const float*, int64_t, int, cudaStream_t);
int tc_gemm_dx(const float*, const float*, float*, void*, int64_t, int64_t, int32_t, int32_t, const float*, int64_t, int,
               cudaStream_t);
namespace tc { int f16_flags(int set); }
int64_t tc_gemm_dw_workspace_bytes(int64_t, int32_t, int32_t);
int tc_gemm_dw(const float*, const float*, const int32_t*, const float*, const float*, float, float*, void*,
               int64_t, int64_t, int32_t, int32_t, const float*, int64_t, const float*, int64_t, int, cudaStream_t);
#else
static bool tc_supported_xw(int64_t, int32_t, int32_t) { return false; }
static bool tc_supported_dx(int64_t, int32_t, int32_t) { return false; }
static bool tc_supported_dw(int64_t, int32_t, int32_t) { return false; }
static int64_t tc_gemm_nt_workspace_bytes(int32_t, int32_t) { return 0; }
static int tc_gemm_xw(const float*, const int32_t*, const float*, const float*, float, const float*, float*, void*,
                      int64_t, int64_t, int32_t, int32_t, const float*, int64_t, int, cudaStream_t) {
    return DDMP_ERR_UNSUPPORTED;
}
static int tc_gemm_dx(const float*, const float*, float*, void*, int64_t, int64_t, int32_t, int32_t, const float*,
                      int64_t, int, cudaStream_t) {
    return DDMP_ERR_UNSUPPORTED;
}
static int64_t tc_gemm_dw_workspace_bytes(int64_t, int32_t, int32_t) { return 0; }
static int tc_gemm_dw(const float*, const float*, const int32_t*, const float*, const float*, float, float*, void*,
                      int64_t, int64_t, int32_t, int32_t, const float*, int64_t, const float*, int64_t, int, cudaStream_t) {
    return DDMP_ERR_UNSUPPORTED;
}
#endif

// DDMP_GEMM_F16X1 is a modifier of the backend argument: split it off; it selects the term count of the fp16-split
// tcgen05 kernels (3, or 1 with the bit) and changes nothing else
static inline int gemm_terms(int& backend) {
    const int terms = (backend & DDMP_GEMM_F16X1) ? 1 : 3;
    backend &= ~DDMP_GEMM_F16X1;
    return terms;
}
}  // namespace ddmp

extern "C" {

int ddmp_gemm_tc_flags(int flags) {
#ifdef DDMP_WITH_TC
    return ddmp::tc::f16_flags(flags);
#else
    (void)flags;
    return 0;
#endif
}

int64_t ddmp_gemm_workspace_bytes(int64_t n, int32_t Cin, int32_t Cout) {
    using namespace ddmp;
    if (n <= 0 || Cin <= 0 || Cout <= 0) return 0;
    return (tc_supported_xw(n, Cin, Cout) || tc_supported_dx(n, Cin, Cout)) ? tc_gemm_nt_workspace_bytes(Cin, Cout) : 0;
}

int ddmp_gemm_xw(const float* X, const int32_t* row_map, const float* scale, const float* shift, float slope,
                 const float* W, float* H, void* workspace, int64_t workspace_bytes, int64_t n, int32_t Cin,
                 int32_t Cout, const float* amax, int64_t amax_len, int backend, void* stream) {
    using namespace ddmp;
    const int terms = gemm_terms(backend);
    DDMP_REQUIRE(n >= 0 && Cin > 0 && Cout > 0, "gemm_xw: bad shape");
    if (n == 0) return DDMP_OK;
    DDMP_REQUIRE(X && W && H, "gemm_xw: null pointer");
    DDMP_REQUIRE((scale == nullptr) == (shift == nullptr), "gemm_xw: scale and shift must come together");
    const bool tc_ok = tc_supported_xw(n, Cin, Cout) && workspace != nullptr;
    if (backend == DDMP_GEMM_TC && !tc_ok) {
        set_error("gemm_xw: tcgen05 path does not support n=%lld Cin=%d Cout=%d", (long long)n, Cin, Cout);
        return DDMP_ERR_UNSUPPORTED;
    }
    if (backend == DDMP_GEMM_TC || (backend == DDMP_GEMM_AUTO && tc_ok))
        return tc_gemm_xw(X, row_map, scale, shift, slope, W, H, workspace, workspace_bytes, n, Cin, Cout, amax,
                          amax_len, terms, as_stream(stream));
    return ffma_gemm_xw(X, row_map, scale, shift, slope, W, H, n, Cin, Cout, as_stream(stream));
}

int ddmp_gemm_dx(const float* dH, const float* W, float* gX, void* workspace, int64_t workspace_bytes, int64_t n,
                 int32_t Cin, int32_t Cout, const float* amax, int64_t amax_len, int backend, void* stream) {
    using namespace ddmp;
    const int terms = gemm_terms(backend);
    DDMP_REQUIRE(n >= 0 && Cin > 0 && Cout > 0, "gemm_dx: bad shape");
    if (n == 0) return DDMP_OK;
    DDMP_REQUIRE(dH && W && gX, "gemm_dx: null pointer");
    const bool tc_ok = tc_supported_dx(n, Cin, Cout) && workspace != nullptr;
    if (backend == DDMP_GEMM_TC && !tc_ok) {
        set_error("gemm_dx: tcgen05 path does not support n=%lld Cin=%d Cout=%d", (long long)n, Cin, Cout);
        return DDMP_ERR_UNSUPPORTED;
    }
    if (backend == DDMP_GEMM_TC || (backend == DDMP_GEMM_AUTO && tc_ok))
        return tc_gemm_dx(dH, W, gX, workspace, workspace_bytes, n, Cin, Cout, amax, amax_len, terms,
                          as_stream(stream));
    return ffma_gemm_dx(dH, W, gX, n, Cin, Cout, as_stream(stream));
}

int64_t ddmp_gemm_dw_workspace_bytes(int64_t n, int32_t Cin, int32_t Cout) {
    using namespace ddmp;
    if (n <= 0 || Cin <= 0 || Cout <= 0) return 0;
    int64_t a = ffma_gemm_dw_workspace_bytes(n, Cin, Cout);
    int64_t b = tc_supported_dw(n, Cin, Cout) ? tc_gemm_dw_workspace_bytes(n, Cin, Cout) : 0;
    return a > b ? a : b;
}

int ddmp_gemm_dw(const float* dH, const float* X, const int32_t* row_map, const float* scale, const float* shift,
                 float slope, float* dW, void* workspace, int64_t workspace_bytes, int64_t n, int32_t Cin,
                 int32_t Cout, const float* amax_dh, int64_t amax_dh_len, const float* amax_x, int64_t amax_x_len,
                 int backend, void* stream) {
    using namespace ddmp;
    const int terms = gemm_terms(backend);
    DDMP_REQUIRE(dH && X && dW, "gemm_dw: null pointer");
    DDMP_REQUIRE((scale == nullptr) == (shift == nullptr), "gemm_dw: scale and shift must come together");
    DDMP_REQUIRE(n > 0 && Cin > 0 && Cout > 0, "gemm_dw: bad shape");
    const bool tc_ok = tc_supported_dw(n, Cin, Cout);
    if (backend == DDMP_GEMM_TC && !tc_ok) {
        set_error("gemm_dw: tcgen05 path does not support n=%lld Cin=%d Cout=%d", (long long)n, Cin, Cout);
        return DDMP_ERR_UNSUPPORTED;
    }
    if (backend == DDMP_GEMM_TC || (backend == DDMP_GEMM_AUTO && tc_ok))
        return tc_gemm_dw(dH, X, row_map, scale, shift, slope, dW, workspace, workspace_bytes, n, Cin, Cout,
                          amax_dh, amax_dh_len, amax_x, amax_x_len, terms, as_stream(stream));
    return ffma_gemm_dw(dH, X, row_map, scale, shift, slope, dW, workspace, workspace_bytes, n, Cin, Cout,
                        as_stream(stream));
}

}  // extern "C"
