// Fused loss / geometry kernels of the Dual-DMP step (reference util/loss.py, util/models.py).
// Every scalar is produced by ONE launch: per-block float64 partials, then the last-arriving block sums them in
// block order (deterministic).  Gradients that the library computes with scatter-add (index_put_ accumulate)
// are gathers here: vertex <- incident face corners (corner CSR), face <- neighbour faces (reverse-slot map).
#include "common.cuh"

namespace ddmp {

constexpr int kLossThreads = 256;
constexpr int kLossMaxBlocks = 1024;
struct LossScratch {
    unsigned int ticket;
    unsigned int pad[63];
    double partials[kLossMaxBlocks];
};

static inline unsigned loss_grid(int64_t count) {
    int64_t g = ceil_div(count, kLossThreads);
    if (g > 4 * kNumSMs) g = 4 * kNumSMs;
    if (g < 1) g = 1;
    return (unsigned)g;
}

// finish a scalar reduction over blocks blk = 0..nblk-1: returns true in thread 0 of the last block with the total in
// `total`
__device__ __forceinline__ bool finish_sum_of(double local, LossScratch* sc, double& total, unsigned blk, unsigned nblk) {
    __shared__ double sm[kLossThreads / 32];
    const double b = block_sum<kLossThreads>(local, sm);
    if (threadIdx.x == 0) sc->partials[blk] = b;
    const bool last = publish_and_am_last(&sc->ticket, nblk);
    if (last && threadIdx.x == 0) {
        double t = 0.0;
        for (unsigned i = 0; i < nblk; ++i) t += __ldcg(&sc->partials[i]);
        total = t;
        return true;
    }
    return false;
}
__device__ __forceinline__ bool finish_sum(double local, LossScratch* sc, double& total) {
    return finish_sum_of(local, sc, total, blockIdx.x, gridDim.x);
}

#define GRID_STRIDE(i, count) \
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < (count); i += (int64_t)gridDim.x * blockDim.x)

// ---- pos_rec (reference util/loss.py:16-35 "rmse"; float64 through type promotion at :27) ---------------------
__global__ void __launch_bounds__(kLossThreads)
pos_rec_fwd_kernel(const float* __restrict__ pos, const double* __restrict__ tgt, double* loss, LossScratch* sc,
                   int64_t V) {
    double acc = 0.0;
    GRID_STRIDE(e, 3 * V) {
        const double d = tgt[e] - (double)pos[e];
        acc += d * d;
    }
    double tot;
    if (finish_sum(acc, sc, tot)) *loss = sqrt(tot / (double)V + 1.0e-6);
}

__global__ void pos_rec_bwd_kernel(const float* __restrict__ pos, const double* __restrict__ tgt,
                                   const double* __restrict__ loss, const double* __restrict__ gout,
                                   float* __restrict__ gpos, int64_t V) {
    const double k = *gout / ((double)V * *loss);
    GRID_STRIDE(e, 3 * V) gpos[e] = (float)(k * ((double)pos[e] - tgt[e]));
}

// ---- uniform Laplacian (reference util/loss.py:37-53 "rmse") -----------------------------------------------------
__global__ void __launch_bounds__(kLossThreads)
lap_fwd_kernel(const float* __restrict__ pos, const int* __restrict__ rowptr, const int* __restrict__ col,
               float* __restrict__ d, float* loss, LossScratch* sc, int64_t V) {
    double acc = 0.0;
    GRID_STRIDE(i, V) {
        const int s = rowptr[i], e = rowptr[i + 1];
        float sx = 0.f, sy = 0.f, sz = 0.f;
        for (int k = s; k < e; ++k) {
            const int64_t j = col[k];
            sx += __ldg(pos + 3 * j); sy += __ldg(pos + 3 * j + 1); sz += __ldg(pos + 3 * j + 2);
        }
        const float deg = (float)(e - s);      // deg == 0 -> 0/0 = NaN, like the reference (unreferenced vertex)
        const float dx = pos[3 * i] - sx / deg, dy = pos[3 * i + 1] - sy / deg, dz = pos[3 * i + 2] - sz / deg;
        d[3 * i] = dx; d[3 * i + 1] = dy; d[3 * i + 2] = dz;
        acc += (double)(dx * dx + dy * dy + dz * dz);
    }
    double tot;
    if (finish_sum(acc, sc, tot)) *loss = (float)sqrt(tot / (double)V + 1.0e-12);
}

__global__ void lap_bwd_kernel(const float* __restrict__ d, const int* __restrict__ rowptr,
                               const int* __restrict__ col, const float* __restrict__ loss,
                               const float* __restrict__ gout, float* __restrict__ gpos, int64_t V) {
    const float k = *gout / ((float)V * *loss);
    GRID_STRIDE(i, V) {
        const int s = rowptr[i], e = rowptr[i + 1];
        float gx = d[3 * i], gy = d[3 * i + 1], gz = d[3 * i + 2];
        for (int kk = s; kk < e; ++kk) {
            const int64_t j = col[kk];
            const float inv = 1.0f / (float)(rowptr[j + 1] - rowptr[j]);
            gx -= __ldg(d + 3 * j) * inv; gy -= __ldg(d + 3 * j + 1) * inv; gz -= __ldg(d + 3 * j + 2) * inv;
        }
        gpos[3 * i] = k * gx; gpos[3 * i + 1] = k * gy; gpos[3 * i + 2] = k * gz;
    }
}

// ---- norm_rec (reference util/loss.py:55-84 "l1mae"; float64) ----------------------------------------------------
__global__ void __launch_bounds__(kLossThreads)
norm_rec_fwd_kernel(const float* __restrict__ nrm, const double* __restrict__ tgt, double* loss, LossScratch* sc,
                    int64_t F) {
    double acc = 0.0;
    GRID_STRIDE(e, 3 * F) acc += fabs((double)nrm[e] - tgt[e]);
    double tot;
    if (finish_sum(acc, sc, tot)) *loss = tot / (double)F;
}

__global__ void norm_rec_bwd_kernel(const float* __restrict__ nrm, const double* __restrict__ tgt,
                                    const double* __restrict__ gout, float* __restrict__ gnrm, int64_t F) {
    const double k = *gout / (double)F;
    GRID_STRIDE(e, 3 * F) {
        const double d = (double)nrm[e] - tgt[e];
        gnrm[e] = (float)(d > 0.0 ? k : (d < 0.0 ? -k : 0.0));
    }
}

// ---- pos_norm (reference util/loss.py:140-160 "mae") ---------------------------------------------------------------
struct Tri { float p[3][3]; };
__device__ __forceinline__ Tri load_tri(const float* __restrict__ pos, const int* __restrict__ faces, int64_t f) {
    Tri t;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int64_t v = faces[3 * f + k];
        t.p[k][0] = __ldg(pos + 3 * v); t.p[k][1] = __ldg(pos + 3 * v + 1); t.p[k][2] = __ldg(pos + 3 * v + 2);
    }
    return t;
}
__device__ __forceinline__ float sgn(float x) { return x > 0.f ? 1.f : (x < 0.f ? -1.f : 0.f); }

__global__ void __launch_bounds__(kLossThreads)
pos_norm_fwd_kernel(const float* __restrict__ pos, const float* __restrict__ nrm, const int* __restrict__ faces,
                    float* loss, LossScratch* sc, int64_t V, int64_t F) {
    double acc = 0.0;
    GRID_STRIDE(f, F) {
        const Tri t = load_tri(pos, faces, f);
        const float nx = nrm[3 * f], ny = nrm[3 * f + 1], nz = nrm[3 * f + 2];
        const float cx = (t.p[0][0] + t.p[1][0] + t.p[2][0]) / 3.0f;
        const float cy = (t.p[0][1] + t.p[1][1] + t.p[2][1]) / 3.0f;
        const float cz = (t.p[0][2] + t.p[1][2] + t.p[2][2]) / 3.0f;
        float s = 0.f;
#pragma unroll
        for (int k = 0; k < 3; ++k)
            s += fabsf((t.p[k][0] - cx) * nx + (t.p[k][1] - cy) * ny + (t.p[k][2] - cz) * nz);
        acc += (double)s;
    }
    double tot;
    if (finish_sum(acc, sc, tot)) *loss = (float)(tot / (double)V);
}

__global__ void pos_norm_bwd_face_kernel(const float* __restrict__ pos, const float* __restrict__ nrm,
                                         const int* __restrict__ faces, const float* __restrict__ gout,
                                         float* __restrict__ face_tmp, float* __restrict__ gnrm, int64_t V,
                                         int64_t F) {
    const float k = *gout / (float)V;
    GRID_STRIDE(f, F) {
        const Tri t = load_tri(pos, faces, f);
        const float n[3] = {nrm[3 * f], nrm[3 * f + 1], nrm[3 * f + 2]};
        float c[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) c[a] = (t.p[0][a] + t.p[1][a] + t.p[2][a]) / 3.0f;
        float s[3], S = 0.f, gn[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            const float dot = (t.p[m][0] - c[0]) * n[0] + (t.p[m][1] - c[1]) * n[1] + (t.p[m][2] - c[2]) * n[2];
            s[m] = sgn(dot);
            S += s[m];
#pragma unroll
            for (int a = 0; a < 3; ++a) gn[a] += s[m] * (t.p[m][a] - c[a]);
        }
#pragma unroll
        for (int m = 0; m < 3; ++m) {
            const float coef = k * (s[m] - S / 3.0f);
#pragma unroll
            for (int a = 0; a < 3; ++a) face_tmp[9 * f + 3 * m + a] = coef * n[a];
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) gnrm[3 * f + a] = k * gn[a];
    }
}

// vertex <- sum of per-corner 3-vectors (deterministic replacement of the scatter-add backward of pos[faces])
__global__ void corner_gather_kernel(const float* __restrict__ face_tmp, const int* __restrict__ corner_ptr,
                                     const int* __restrict__ corner_slot, float* __restrict__ gpos, int64_t V) {
    GRID_STRIDE(v, V) {
        float x = 0.f, y = 0.f, z = 0.f;
        for (int k = corner_ptr[v]; k < corner_ptr[v + 1]; ++k) {
            const int64_t sl = corner_slot[k];
            x += __ldg(face_tmp + 3 * sl); y += __ldg(face_tmp + 3 * sl + 1); z += __ldg(face_tmp + 3 * sl + 2);
        }
        gpos[3 * v] = x; gpos[3 * v + 1] = y; gpos[3 * v + 2] = z;
    }
}

// ---- bilateral normal filtering (reference util/loss.py:86-138 "l1mae") ----------------------------------------
__global__ void bnf_geom_kernel(const float* __restrict__ pos, const int* __restrict__ faces,
                                float* __restrict__ fc, float* __restrict__ fa, int64_t F) {
    GRID_STRIDE(f, F) {
        const Tri t = load_tri(pos, faces, f);
#pragma unroll
        for (int a = 0; a < 3; ++a) fc[3 * f + a] = (t.p[0][a] + t.p[1][a] + t.p[2][a]) / 3.0f;
        const float ax = t.p[1][0] - t.p[0][0], ay = t.p[1][1] - t.p[0][1], az = t.p[1][2] - t.p[0][2];
        const float bx = t.p[2][0] - t.p[0][0], by = t.p[2][1] - t.p[0][1], bz = t.p[2][2] - t.p[0][2];
        const float cx = ay * bz - az * by, cy = az * bx - ax * bz, cz = ax * by - ay * bx;
        fa[f] = 0.5f * sqrtf(cx * cx + cy * cy + cz * cz + 1.0e-12f);
    }
}

__global__ void __launch_bounds__(kLossThreads)
bnf_dist_kernel(const float* __restrict__ fc, const int* __restrict__ f2f, float* __restrict__ dist,
                float* sigma_c, LossScratch* sc, int64_t F) {
    double acc = 0.0;
    GRID_STRIDE(f, F) {
        const float cx = fc[3 * f], cy = fc[3 * f + 1], cz = fc[3 * f + 2];
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int nb = f2f[3 * f + s];
            const int64_t j = nb < 0 ? (F - 1) : nb;       // python negative index: -1 is the LAST face
            const float dx = __ldg(fc + 3 * j) - cx, dy = __ldg(fc + 3 * j + 1) - cy, dz = __ldg(fc + 3 * j + 2) - cz;
            const float d2 = dx * dx + dy * dy + dz * dz;
            dist[3 * f + s] = d2;
            acc += (double)sqrtf(d2 + 1.0e-12f);
        }
    }
    double tot;
    if (finish_sum(acc, sc, tot)) *sigma_c = (float)(tot / (double)(3 * F));
}

__global__ void bnf_wca_kernel(const float* __restrict__ fa, const int* __restrict__ f2f,
                               const float* __restrict__ sigma_c, float* __restrict__ wca, int64_t F) {
    const float sg = *sigma_c;
    const float den = 2.0f * (sg * sg);
    GRID_STRIDE(i, 3 * F) {
        const int nb = f2f[i];
        const float d2 = wca[i];
        wca[i] = (nb < 0) ? 0.f : expf(-1.0f * d2 / den) * __ldg(fa + nb);
    }
}

constexpr float kTwoSigmaS2 = 0.18f;   // 2 * 0.3^2  (reference util/loss.py:110-112)
constexpr float kSigmaS2 = 0.09f;

__global__ void bnf_iter_fwd_kernel(const float* __restrict__ n_in, const int* __restrict__ f2f,
                                    const float* __restrict__ wca, float* __restrict__ n_out, int64_t F) {
    GRID_STRIDE(f, F) {
        const float nx = n_in[3 * f], ny = n_in[3 * f + 1], nz = n_in[3 * f + 2];
        float ax = 0.f, ay = 0.f, az = 0.f;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int nb = f2f[3 * f + s];
            const int64_t j = nb < 0 ? (F - 1) : nb;
            const float jx = __ldg(n_in + 3 * j), jy = __ldg(n_in + 3 * j + 1), jz = __ldg(n_in + 3 * j + 2);
            const float dx = jx - nx, dy = jy - ny, dz = jz - nz;
            const float W = wca[3 * f + s] * expf(-1.0f * (dx * dx + dy * dy + dz * dz) / kTwoSigmaS2);
            ax = fmaf(W, jx, ax); ay = fmaf(W, jy, ay); az = fmaf(W, jz, az);
        }
        const float r = sqrtf(ax * ax + ay * ay + az * az + 1.0e-12f) + 1.0e-12f;
        n_out[3 * f] = ax / r; n_out[3 * f + 1] = ay / r; n_out[3 * f + 2] = az / r;
    }
}

__global__ void __launch_bounds__(kLossThreads)
l1_mean_fwd_kernel(const float* __restrict__ a, const float* __restrict__ b, float* loss, LossScratch* sc,
                   int64_t F) {
    double acc = 0.0;
    GRID_STRIDE(e, 3 * F) acc += (double)fabsf(a[e] - b[e]);
    double tot;
    if (finish_sum(acc, sc, tot)) *loss = (float)(tot / (double)F);
}

__global__ void l1_mean_bwd_kernel(const float* __restrict__ a, const float* __restrict__ b,
                                   const float* __restrict__ gout, float* __restrict__ ga, int64_t F) {
    const float k = *gout / (float)F;
    GRID_STRIDE(e, 3 * F) ga[e] = k * sgn(a[e] - b[e]);
}

// backward of one filter iteration, phase A (per centre face): messages to the three neighbours + centre term
__global__ void bnf_iter_bwd_face_kernel(const float* __restrict__ n_in, const float* __restrict__ g_out,
                                         const int* __restrict__ f2f, const float* __restrict__ wca,
                                         float* __restrict__ msg, float* __restrict__ g_in, int64_t F) {
    GRID_STRIDE(f, F) {
        const float n[3] = {n_in[3 * f], n_in[3 * f + 1], n_in[3 * f + 2]};
        float nj[3][3], W[3], acc[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int nb = f2f[3 * f + s];
            const int64_t j = nb < 0 ? (F - 1) : nb;
#pragma unroll
            for (int a = 0; a < 3; ++a) nj[s][a] = __ldg(n_in + 3 * j + a);
            const float dx = nj[s][0] - n[0], dy = nj[s][1] - n[1], dz = nj[s][2] - n[2];
            W[s] = wca[3 * f + s] * expf(-1.0f * (dx * dx + dy * dy + dz * dz) / kTwoSigmaS2);
#pragma unroll
            for (int a = 0; a < 3; ++a) acc[a] = fmaf(W[s], nj[s][a], acc[a]);
        }
        const float r = sqrtf(acc[0] * acc[0] + acc[1] * acc[1] + acc[2] * acc[2] + 1.0e-12f);
        const float re = r + 1.0e-12f;
        const float g[3] = {g_out[3 * f], g_out[3 * f + 1], g_out[3 * f + 2]};
        const float gd = g[0] * acc[0] + g[1] * acc[1] + g[2] * acc[2];
        const float k2 = gd / (re * re * r);
        float ga[3];
#pragma unroll
        for (int a = 0; a < 3; ++a) ga[a] = g[a] / re - acc[a] * k2;
        float ctr[3] = {0.f, 0.f, 0.f};
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const float dotg = ga[0] * nj[s][0] + ga[1] * nj[s][1] + ga[2] * nj[s][2];
            const float q = dotg * W[s] / kSigmaS2;
#pragma unroll
            for (int a = 0; a < 3; ++a) {
                const float diff = nj[s][a] - n[a];
                msg[9 * f + 3 * s + a] = W[s] * ga[a] - q * diff;
                ctr[a] = fmaf(q, diff, ctr[a]);
            }
        }
#pragma unroll
        for (int a = 0; a < 3; ++a) g_in[3 * f + a] = ctr[a];
    }
}

// phase B (per face j): collect the messages its neighbours addressed to it (reverse-slot map, no atomics)
__global__ void bnf_iter_bwd_gather_kernel(const int* __restrict__ f2f, const int* __restrict__ rslot,
                                           const float* __restrict__ msg, const float* __restrict__ g_sub,
                                           float* __restrict__ g_in, int64_t F) {
    GRID_STRIDE(j, F) {
        float x = g_in[3 * j], y = g_in[3 * j + 1], z = g_in[3 * j + 2];
        if (g_sub) { x -= g_sub[3 * j]; y -= g_sub[3 * j + 1]; z -= g_sub[3 * j + 2]; }
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            const int f = f2f[3 * j + s];
            if (f >= 0) {
                const int64_t o = 9 * (int64_t)f + 3 * rslot[3 * j + s];
                x += __ldg(msg + o); y += __ldg(msg + o + 1); z += __ldg(msg + o + 2);
            }
        }
        g_in[3 * j] = x; g_in[3 * j + 1] = y; g_in[3 * j + 2] = z;
    }
}

// ---- geometry / evaluation (reference util/models.py, util/loss.py:261-272) ---------------------------------------
__global__ void face_normals_fwd_kernel(const float* __restrict__ pos, const int* __restrict__ faces,
                                        float* __restrict__ fn, int64_t F) {
    GRID_STRIDE(f, F) {
        const Tri t = load_tri(pos, faces, f);
        const float ax = t.p[1][0] - t.p[0][0], ay = t.p[1][1] - t.p[0][1], az = t.p[1][2] - t.p[0][2];
        const float bx = t.p[2][0] - t.p[0][0], by = t.p[2][1] - t.p[0][1], bz = t.p[2][2] - t.p[0][2];
        const float cx = ay * bz - az * by, cy = az * bx - ax * bz, cz = ax * by - ay * bx;
        const float nr = sqrtf(cx * cx + cy * cy + cz * cz);
        fn[3 * f] = cx / nr; fn[3 * f + 1] = cy / nr; fn[3 * f + 2] = cz / nr;
    }
}

__global__ void face_normals_bwd_face_kernel(const float* __restrict__ pos, const int* __restrict__ faces,
                                             const float* __restrict__ gfn, float* __restrict__ face_tmp,
                                             int64_t F) {
    GRID_STRIDE(f, F) {
        const Tri t = load_tri(pos, faces, f);
        const float a[3] = {t.p[1][0] - t.p[0][0], t.p[1][1] - t.p[0][1], t.p[1][2] - t.p[0][2]};
        const float b[3] = {t.p[2][0] - t.p[0][0], t.p[2][1] - t.p[0][1], t.p[2][2] - t.p[0][2]};
        const float c[3] = {a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]};
        const float nr = sqrtf(c[0] * c[0] + c[1] * c[1] + c[2] * c[2]);
        const float u[3] = {c[0] / nr, c[1] / nr, c[2] / nr};
        const float g[3] = {gfn[3 * f], gfn[3 * f + 1], gfn[3 * f + 2]};
        const float ug = u[0] * g[0] + u[1] * g[1] + u[2] * g[2];
        const float gc[3] = {(g[0] - u[0] * ug) / nr, (g[1] - u[1] * ug) / nr, (g[2] - u[2] * ug) / nr};
        const float ga[3] = {b[1] * gc[2] - b[2] * gc[1], b[2] * gc[0] - b[0] * gc[2], b[0] * gc[1] - b[1] * gc[0]};
        const float gb[3] = {gc[1] * a[2] - gc[2] * a[1], gc[2] * a[0] - gc[0] * a[2], gc[0] * a[1] - gc[1] * a[0]};
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            face_tmp[9 * f + 0 + k] = -ga[k] - gb[k];
            face_tmp[9 * f + 3 + k] = ga[k];
            face_tmp[9 * f + 6 + k] = gb[k];
        }
    }
}

__global__ void __launch_bounds__(kLossThreads)
mad_kernel(const float* __restrict__ n1, const float* __restrict__ n2, double* out, LossScratch* sc, int64_t F) {
    double acc = 0.0;
    GRID_STRIDE(f, F) {
        double inner = (double)n1[3 * f] * n2[3 * f] + (double)n1[3 * f + 1] * n2[3 * f + 1] +
                       (double)n1[3 * f + 2] * n2[3 * f + 2];
        inner = inner < -1.0 ? -1.0 : (inner > 1.0 ? 1.0 : inner);
        acc += acos(inner) * (180.0 / 3.14159265358979323846);
    }
    double tot;
    if (finish_sum(acc, sc, tot)) *out = tot / (double)F;
}

__global__ void vertex_normals_kernel(const float* __restrict__ fn, const int* __restrict__ corner_ptr,
                                      const int* __restrict__ corner_slot, float* __restrict__ vn, int64_t V) {
    GRID_STRIDE(v, V) {
        float x = 0.f, y = 0.f, z = 0.f;
        for (int k = corner_ptr[v]; k < corner_ptr[v + 1]; ++k) {
            const int64_t f = corner_slot[k] / 3;
            x += __ldg(fn + 3 * f); y += __ldg(fn + 3 * f + 1); z += __ldg(fn + 3 * f + 2);
        }
        const float nr = sqrtf(x * x + y * y + z * z);
        vn[3 * v] = x / nr; vn[3 * v + 1] = y / nr; vn[3 * v + 2] = z / nr;
    }
}

__global__ void vertex_update_kernel(const float* __restrict__ pos_in, const float* __restrict__ fc,
                                     const float* __restrict__ nrm, const int* __restrict__ corner_ptr,
                                     const int* __restrict__ corner_slot, float* __restrict__ pos_out, int64_t V) {
    GRID_STRIDE(v, V) {
        const float px = pos_in[3 * v], py = pos_in[3 * v + 1], pz = pos_in[3 * v + 2];
        float dx = 0.f, dy = 0.f, dz = 0.f;
        const int s = corner_ptr[v], e = corner_ptr[v + 1];
        for (int k = s; k < e; ++k) {
            const int64_t f = corner_slot[k] / 3;
            const float nx = __ldg(nrm + 3 * f), ny = __ldg(nrm + 3 * f + 1), nz = __ldg(nrm + 3 * f + 2);
            const float pr = nx * (__ldg(fc + 3 * f) - px) + ny * (__ldg(fc + 3 * f + 1) - py) +
                             nz * (__ldg(fc + 3 * f + 2) - pz);
            dx = fmaf(pr, nx, dx); dy = fmaf(pr, ny, dy); dz = fmaf(pr, nz, dz);
        }
        const float cnt = (float)(e - s);
        pos_out[3 * v] = px + dx / cnt; pos_out[3 * v + 1] = py + dy / cnt; pos_out[3 * v + 2] = pz + dz / cnt;
    }
}

__global__ void face_centroids_kernel(const float* __restrict__ pos, const int* __restrict__ faces,
                                      float* __restrict__ fc, int64_t F) {
    GRID_STRIDE(f, F) {
        const Tri t = load_tri(pos, faces, f);
#pragma unroll
        for (int a = 0; a < 3; ++a) fc[3 * f + a] = (t.p[0][a] + t.p[1][a] + t.p[2][a]) / 3.0f;
    }
}

// ---- step glue (reference main.py:108-110) ---------------------------------------------------------------------------
__global__ void __launch_bounds__(kLossThreads)
grad_norm_kernel(const float* __restrict__ g, float* norm_out, LossScratch* sc, int64_t count) {
    double acc = 0.0;
    GRID_STRIDE(i, count) acc += (double)g[i] * (double)g[i];
    double tot;
    if (finish_sum(acc, sc, tot)) *norm_out = (float)sqrt(tot);
}

__global__ void counter_increment_kernel(int64_t* counter) { *counter += 1; }

__device__ __forceinline__ void adam_bias_corrections(const int64_t* step_dev, float beta1, float beta2, float& bc1,
                                                      float& bc2_sqrt) {
    const double t = (double)*step_dev;
    bc1 = (float)(1.0 - pow((double)beta1, t));
    bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, t));
}

__device__ __forceinline__ float clip_coef(float norm, float max_norm) {
    const float coef = max_norm / (norm + 1.0e-6f);
    return coef > 1.f ? 1.f : coef;
}

__device__ __forceinline__ void adam_element(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                             float* __restrict__ v, int64_t i, float coef, float beta1, float beta2,
                                             float eps, float step_size, float bc2_sqrt) {
    const float gi = g[i] * coef;
    const float mi = m[i] + (gi - m[i]) * (1.f - beta1);      // torch lerp_
    const float vi = beta2 * v[i] + (1.f - beta2) * gi * gi;
    m[i] = mi; v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= step_size * (mi / denom);
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, const float* __restrict__ clip_norm, float max_norm, float lr,
                            float beta1, float beta2, float eps, float bc1, float bc2_sqrt,
                            const int64_t* __restrict__ step_dev, int64_t count) {
    // step count lives on the device (CUDA-graph replay: kernel arguments are frozen)
    if (step_dev) adam_bias_corrections(step_dev, beta1, beta2, bc1, bc2_sqrt);
    const float coef = clip_norm ? clip_coef(*clip_norm, max_norm) : 1.f;
    const float step_size = lr / bc1;
    GRID_STRIDE(i, count) adam_element(p, g, m, v, i, coef, beta1, beta2, eps, step_size, bc2_sqrt);
}

// ---- the optimizer of many networks over one flat buffer (ddmp_*_segments) -------------------------------------------
// Segment s (a network) is row s of the table: DDMP_SEGMENT_WORDS int64 words, see include/ddmp_b200.h.  blockIdx.y is
// the segment; a segment uses the blocks x < loss_grid(count) -- the grid its stand-alone call would launch -- and the
// other blocks of its row return at once.
struct Segment {
    int64_t off, count;
    bool clip;
    float lr, max_norm;
};
__device__ __forceinline__ Segment load_segment(const int64_t* __restrict__ table, int s) {
    const int64_t* w = table + (int64_t)s * DDMP_SEGMENT_WORDS;
    Segment g;
    g.off = w[0]; g.count = w[1]; g.clip = w[2] != 0;
    g.lr = __uint_as_float((unsigned)(w[3] & 0xffffffffll));
    g.max_norm = __uint_as_float((unsigned)(w[4] & 0xffffffffll));
    return g;
}
__device__ __forceinline__ unsigned loss_grid_dev(int64_t count) {
    int64_t g = (count + kLossThreads - 1) / kLossThreads;
    if (g > 4 * kNumSMs) g = 4 * kNumSMs;
    if (g < 1) g = 1;
    return (unsigned)g;
}

__global__ void __launch_bounds__(kLossThreads)
grad_norm_segments_kernel(const float* __restrict__ flat, const int64_t* __restrict__ table, float* norms,
                          LossScratch* sc) {
    const Segment sg = load_segment(table, blockIdx.y);
    const unsigned nblk = loss_grid_dev(sg.count);
    if (!sg.clip || blockIdx.x >= nblk) return;
    const float* __restrict__ g = flat + sg.off;
    double acc = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * kLossThreads + threadIdx.x; i < sg.count; i += (int64_t)nblk * kLossThreads)
        acc += (double)g[i] * (double)g[i];
    double tot;
    if (finish_sum_of(acc, sc + blockIdx.y, tot, blockIdx.x, nblk)) norms[blockIdx.y] = (float)sqrt(tot);
}

__global__ void adam_segments_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                     float* __restrict__ v, const int64_t* __restrict__ table,
                                     const float* __restrict__ norms, float beta1, float beta2, float eps,
                                     const int64_t* __restrict__ step_dev) {
    const Segment sg = load_segment(table, blockIdx.y);
    const unsigned nblk = loss_grid_dev(sg.count);
    if (blockIdx.x >= nblk) return;
    float bc1, bc2_sqrt;
    adam_bias_corrections(step_dev, beta1, beta2, bc1, bc2_sqrt);
    const float coef = sg.clip ? clip_coef(norms[blockIdx.y], sg.max_norm) : 1.f;
    const float step_size = sg.lr / bc1;
    for (int64_t i = sg.off + (int64_t)blockIdx.x * kLossThreads + threadIdx.x; i < sg.off + sg.count;
         i += (int64_t)nblk * kLossThreads)
        adam_element(p, g, m, v, i, coef, beta1, beta2, eps, step_size, bc2_sqrt);
}

// row s of the table: (source address, destination offset, count); blockIdx.y is the row
__global__ void __launch_bounds__(256) gather_table_kernel(const int64_t* __restrict__ table, float* __restrict__ dst) {
    const int64_t* w = table + 3 * (int64_t)blockIdx.y;
    const float* __restrict__ src = reinterpret_cast<const float*>(w[0]);
    float* __restrict__ out = dst + w[1];
    const int64_t cnt = w[2];
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * 256) out[i] = src[i];
}

// see ddmp_gather_flat
constexpr int kGatherMax = 80;
struct GatherArgs {
    const float* src[kGatherMax];
    int64_t off[kGatherMax];
    int64_t cnt[kGatherMax];
    int n;
};
__global__ void __launch_bounds__(256) gather_flat_kernel(const GatherArgs a, float* __restrict__ dst) {
    const int s = blockIdx.y;
    const float* __restrict__ src = a.src[s];
    float* __restrict__ out = dst + a.off[s];
    const int64_t cnt = a.cnt[s];
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < cnt; i += (int64_t)gridDim.x * 256) out[i] = src[i];
}

}  // namespace ddmp

#define LAUNCH_1D(kernel, count, st, ...) \
    kernel<<<ddmp::loss_grid(count), ddmp::kLossThreads, 0, st>>>(__VA_ARGS__)

extern "C" {

int64_t ddmp_loss_scratch_bytes(void) { return (int64_t)sizeof(ddmp::LossScratch); }

int ddmp_loss_pos_rec_fwd(const float* pos, const double* target, double* loss, void* scratch, int64_t V,
                          void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos && target && loss && scratch && V > 0, "loss_pos_rec_fwd: bad arguments");
    LAUNCH_1D(pos_rec_fwd_kernel, 3 * V, as_stream(stream), pos, target, loss, (LossScratch*)scratch, V);
    return check_launch("loss_pos_rec_fwd");
}

int ddmp_loss_pos_rec_bwd(const float* pos, const double* target, const double* loss, const double* gout,
                          float* gpos, int64_t V, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos && target && loss && gout && gpos && V > 0, "loss_pos_rec_bwd: bad arguments");
    LAUNCH_1D(pos_rec_bwd_kernel, 3 * V, as_stream(stream), pos, target, loss, gout, gpos, V);
    return check_launch("loss_pos_rec_bwd");
}

int ddmp_loss_lap_fwd(const float* pos, const int32_t* rowptr, const int32_t* col, float* d, float* loss,
                      void* scratch, int64_t V, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos && rowptr && col && d && loss && scratch && V > 0, "loss_lap_fwd: bad arguments");
    LAUNCH_1D(lap_fwd_kernel, V, as_stream(stream), pos, rowptr, col, d, loss, (LossScratch*)scratch, V);
    return check_launch("loss_lap_fwd");
}

int ddmp_loss_lap_bwd(const float* d, const int32_t* rowptr, const int32_t* col, const float* loss,
                      const float* gout, float* gpos, int64_t V, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(d && rowptr && col && loss && gout && gpos && V > 0, "loss_lap_bwd: bad arguments");
    LAUNCH_1D(lap_bwd_kernel, V, as_stream(stream), d, rowptr, col, loss, gout, gpos, V);
    return check_launch("loss_lap_bwd");
}

int ddmp_loss_norm_rec_fwd(const float* nrm, const double* target, double* loss, void* scratch, int64_t F,
                           void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(nrm && target && loss && scratch && F > 0, "loss_norm_rec_fwd: bad arguments");
    LAUNCH_1D(norm_rec_fwd_kernel, 3 * F, as_stream(stream), nrm, target, loss, (LossScratch*)scratch, F);
    return check_launch("loss_norm_rec_fwd");
}

int ddmp_loss_norm_rec_bwd(const float* nrm, const double* target, const double* gout, float* gnrm, int64_t F,
                           void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(nrm && target && gout && gnrm && F > 0, "loss_norm_rec_bwd: bad arguments");
    LAUNCH_1D(norm_rec_bwd_kernel, 3 * F, as_stream(stream), nrm, target, gout, gnrm, F);
    return check_launch("loss_norm_rec_bwd");
}

int ddmp_loss_pos_norm_fwd(const float* pos, const float* nrm, const int32_t* faces, float* loss, void* scratch,
                           int64_t V, int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos && nrm && faces && loss && scratch && V > 0 && F > 0, "loss_pos_norm_fwd: bad arguments");
    LAUNCH_1D(pos_norm_fwd_kernel, F, as_stream(stream), pos, nrm, faces, loss, (LossScratch*)scratch, V, F);
    return check_launch("loss_pos_norm_fwd");
}

int ddmp_loss_pos_norm_bwd(const float* pos, const float* nrm, const int32_t* faces, const int32_t* corner_ptr,
                           const int32_t* corner_slot, const float* gout, float* face_tmp, float* gpos,
                           float* gnrm, int64_t V, int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos && nrm && faces && corner_ptr && corner_slot && gout && face_tmp && gpos && gnrm && V > 0 &&
                     F > 0, "loss_pos_norm_bwd: bad arguments");
    cudaStream_t st = as_stream(stream);
    LAUNCH_1D(pos_norm_bwd_face_kernel, F, st, pos, nrm, faces, gout, face_tmp, gnrm, V, F);
    int rc = check_launch("loss_pos_norm_bwd(face)");
    if (rc) return rc;
    LAUNCH_1D(corner_gather_kernel, V, st, face_tmp, corner_ptr, corner_slot, gpos, V);
    return check_launch("loss_pos_norm_bwd(gather)");
}

int ddmp_bnf_setup(const float* pos, const int32_t* faces, const int32_t* f2f, float* fc, float* fa, float* wca,
                   float* sigma_c, void* scratch, int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos && faces && f2f && fc && fa && wca && sigma_c && scratch && F > 0, "bnf_setup: bad arguments");
    cudaStream_t st = as_stream(stream);
    LAUNCH_1D(bnf_geom_kernel, F, st, pos, faces, fc, fa, F);
    int rc = check_launch("bnf_setup(geom)");
    if (rc) return rc;
    LAUNCH_1D(bnf_dist_kernel, F, st, fc, f2f, wca, sigma_c, (LossScratch*)scratch, F);
    rc = check_launch("bnf_setup(dist)");
    if (rc) return rc;
    LAUNCH_1D(bnf_wca_kernel, 3 * F, st, fa, f2f, sigma_c, wca, F);
    return check_launch("bnf_setup(wca)");
}

int ddmp_bnf_iter_fwd(const float* n_in, const int32_t* f2f, const float* wca, float* n_out, int64_t F,
                      void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(n_in && f2f && wca && n_out && F > 0 && n_in != n_out, "bnf_iter_fwd: bad arguments");
    LAUNCH_1D(bnf_iter_fwd_kernel, F, as_stream(stream), n_in, f2f, wca, n_out, F);
    return check_launch("bnf_iter_fwd");
}

int ddmp_bnf_loss_fwd(const float* n_last, const float* n_first, float* loss, void* scratch, int64_t F,
                      void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(n_last && n_first && loss && scratch && F > 0, "bnf_loss_fwd: bad arguments");
    LAUNCH_1D(l1_mean_fwd_kernel, 3 * F, as_stream(stream), n_last, n_first, loss, (LossScratch*)scratch, F);
    return check_launch("bnf_loss_fwd");
}

int ddmp_bnf_loss_bwd(const float* n_last, const float* n_first, const float* gout, float* g_last, int64_t F,
                      void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(n_last && n_first && gout && g_last && F > 0, "bnf_loss_bwd: bad arguments");
    LAUNCH_1D(l1_mean_bwd_kernel, 3 * F, as_stream(stream), n_last, n_first, gout, g_last, F);
    return check_launch("bnf_loss_bwd");
}

int ddmp_bnf_iter_bwd(const float* n_in, const float* g_out, const int32_t* f2f, const int32_t* rslot,
                      const float* wca, const float* g_sub, float* msg, float* g_in, int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(n_in && g_out && f2f && rslot && wca && msg && g_in && F > 0 && g_in != g_out,
                 "bnf_iter_bwd: bad arguments");
    cudaStream_t st = as_stream(stream);
    LAUNCH_1D(bnf_iter_bwd_face_kernel, F, st, n_in, g_out, f2f, wca, msg, g_in, F);
    int rc = check_launch("bnf_iter_bwd(face)");
    if (rc) return rc;
    LAUNCH_1D(bnf_iter_bwd_gather_kernel, F, st, f2f, rslot, msg, g_sub, g_in, F);
    return check_launch("bnf_iter_bwd(gather)");
}

int ddmp_face_normals_fwd(const float* pos, const int32_t* faces, float* fn, int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos && faces && fn && F > 0, "face_normals_fwd: bad arguments");
    LAUNCH_1D(face_normals_fwd_kernel, F, as_stream(stream), pos, faces, fn, F);
    return check_launch("face_normals_fwd");
}

int ddmp_face_normals_bwd(const float* pos, const int32_t* faces, const int32_t* corner_ptr,
                          const int32_t* corner_slot, const float* gfn, float* face_tmp, float* gpos, int64_t V,
                          int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos && faces && corner_ptr && corner_slot && gfn && face_tmp && gpos && V > 0 && F > 0,
                 "face_normals_bwd: bad arguments");
    cudaStream_t st = as_stream(stream);
    LAUNCH_1D(face_normals_bwd_face_kernel, F, st, pos, faces, gfn, face_tmp, F);
    int rc = check_launch("face_normals_bwd(face)");
    if (rc) return rc;
    LAUNCH_1D(corner_gather_kernel, V, st, face_tmp, corner_ptr, corner_slot, gpos, V);
    return check_launch("face_normals_bwd(gather)");
}

int ddmp_mad(const float* n1, const float* n2, double* out, void* scratch, int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(n1 && n2 && out && scratch && F > 0, "mad: bad arguments");
    LAUNCH_1D(mad_kernel, F, as_stream(stream), n1, n2, out, (LossScratch*)scratch, F);
    return check_launch("mad");
}

int ddmp_vertex_normals(const float* fn, const int32_t* corner_ptr, const int32_t* corner_slot, float* vn,
                        int64_t V, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(fn && corner_ptr && corner_slot && vn && V > 0, "vertex_normals: bad arguments");
    LAUNCH_1D(vertex_normals_kernel, V, as_stream(stream), fn, corner_ptr, corner_slot, vn, V);
    return check_launch("vertex_normals");
}

int ddmp_vertex_update_sweep(const float* pos_in, const float* fc, const float* nrm, const int32_t* corner_ptr,
                             const int32_t* corner_slot, float* pos_out, int64_t V, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos_in && fc && nrm && corner_ptr && corner_slot && pos_out && V > 0 && pos_in != pos_out,
                 "vertex_update_sweep: bad arguments");
    LAUNCH_1D(vertex_update_kernel, V, as_stream(stream), pos_in, fc, nrm, corner_ptr, corner_slot, pos_out, V);
    return check_launch("vertex_update_sweep");
}

int ddmp_face_centroids(const float* pos, const int32_t* faces, float* fc, int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(pos && faces && fc && F > 0, "face_centroids: bad arguments");
    LAUNCH_1D(face_centroids_kernel, F, as_stream(stream), pos, faces, fc, F);
    return check_launch("face_centroids");
}

int ddmp_grad_norm(const float* grad, float* norm_out, void* scratch, int64_t count, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(grad && norm_out && scratch && count > 0, "grad_norm: bad arguments");
    LAUNCH_1D(grad_norm_kernel, count, as_stream(stream), grad, norm_out, (LossScratch*)scratch, count);
    return check_launch("grad_norm");
}

int ddmp_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, const float* clip_norm,
                   float max_norm, float lr, float beta1, float beta2, float eps, int64_t step, int64_t count,
                   void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(param && grad && exp_avg && exp_avg_sq && count > 0 && step >= 1, "adam_step: bad arguments");
    const double bc1 = 1.0 - pow((double)beta1, (double)step);
    const double bc2 = 1.0 - pow((double)beta2, (double)step);
    LAUNCH_1D(adam_kernel, count, as_stream(stream), param, grad, exp_avg, exp_avg_sq, clip_norm, max_norm, lr,
              beta1, beta2, eps, (float)bc1, (float)sqrt(bc2), (const int64_t*)nullptr, count);
    return check_launch("adam_step");
}

int ddmp_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, const float* clip_norm,
                       float max_norm, float lr, float beta1, float beta2, float eps, int64_t* step_counter,
                       int64_t count, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(param && grad && exp_avg && exp_avg_sq && step_counter && count > 0, "adam_step_dev: bad arguments");
    counter_increment_kernel<<<1, 1, 0, as_stream(stream)>>>(step_counter);
    int rc = check_launch("adam_step_dev(counter)");
    if (rc) return rc;
    LAUNCH_1D(adam_kernel, count, as_stream(stream), param, grad, exp_avg, exp_avg_sq, clip_norm, max_norm, lr,
              beta1, beta2, eps, 1.f, 1.f, (const int64_t*)step_counter, count);
    return check_launch("adam_step_dev");
}

// Flat gradient of a network: the gradient tensors autograd hands back (one per parameter) copied into one buffer in
// parameter order by ONE launch.  The (pointer, offset, count) triples travel as a kernel argument, so a CUDA-graph
// replay needs no pointer table in memory (graph-captured allocations keep their addresses).
int ddmp_gather_flat(const void* const* srcs, const int64_t* offsets, const int64_t* counts, int32_t n_src, float* dst,
                     void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(srcs && offsets && counts && dst && n_src >= 0, "gather_flat: bad arguments");
    cudaStream_t st = as_stream(stream);
    for (int base = 0; base < n_src; base += kGatherMax) {
        GatherArgs a{};
        a.n = (n_src - base < kGatherMax) ? (n_src - base) : kGatherMax;
        int64_t longest = 0;
        for (int i = 0; i < a.n; ++i) {
            DDMP_REQUIRE(srcs[base + i] != nullptr && counts[base + i] >= 0 && offsets[base + i] >= 0, "gather_flat: bad segment");
            a.src[i] = static_cast<const float*>(srcs[base + i]);
            a.off[i] = offsets[base + i];
            a.cnt[i] = counts[base + i];
            if (a.cnt[i] > longest) longest = a.cnt[i];
        }
        if (longest == 0) continue;
        int64_t bx = ceil_div(longest, 256 * 4);
        if (bx > 64) bx = 64;
        gather_flat_kernel<<<dim3((unsigned)bx, (unsigned)a.n), 256, 0, st>>>(a, dst);
        int rc = check_launch("gather_flat");
        if (rc != DDMP_OK) return rc;
    }
    return DDMP_OK;
}

int ddmp_gather_table(const int64_t* table, int32_t n_src, int64_t longest, float* dst, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(table && dst && n_src >= 0 && n_src <= 65535 && longest >= 0, "gather_table: bad arguments");
    if (n_src == 0 || longest == 0) return DDMP_OK;
    int64_t bx = ceil_div(longest, 256 * 4);
    if (bx > 64) bx = 64;
    gather_table_kernel<<<dim3((unsigned)bx, (unsigned)n_src), 256, 0, as_stream(stream)>>>(table, dst);
    return check_launch("gather_table");
}

int ddmp_grad_norm_segments(const float* flat, const int64_t* table, int32_t n_seg, int64_t longest, float* norms,
                            void* scratch, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(flat && table && norms && scratch && n_seg > 0 && n_seg <= 65535 && longest > 0,
                 "grad_norm_segments: bad arguments");
    grad_norm_segments_kernel<<<dim3(loss_grid(longest), (unsigned)n_seg), kLossThreads, 0, as_stream(stream)>>>(
        flat, table, norms, (LossScratch*)scratch);
    return check_launch("grad_norm_segments");
}

int ddmp_adam_segments(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, const int64_t* table,
                       int32_t n_seg, int64_t longest, const float* norms, float beta1, float beta2, float eps,
                       int64_t* step_counter, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(param && grad && exp_avg && exp_avg_sq && table && norms && step_counter && n_seg > 0 &&
                     n_seg <= 65535 && longest > 0, "adam_segments: bad arguments");
    counter_increment_kernel<<<1, 1, 0, as_stream(stream)>>>(step_counter);
    int rc = check_launch("adam_segments(counter)");
    if (rc) return rc;
    adam_segments_kernel<<<dim3(loss_grid(longest), (unsigned)n_seg), kLossThreads, 0, as_stream(stream)>>>(
        param, grad, exp_avg, exp_avg_sq, table, norms, beta1, beta2, eps, step_counter);
    return check_launch("adam_segments");
}

}  // extern "C"
