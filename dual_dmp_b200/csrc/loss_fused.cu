// The loss phase of a Dual-DMP iteration as ONE cooperative kernel (reference main.py:94-106 + the backward of it):
//     total = k1*pos_rec + k2*laplacian + k3*norm_rec + k4*(bnf * bnf_scale) + k5*pos_norm
// and d(total)/d(pos), d(total)/d(norm), with the arithmetic of the stand-alone kernels of loss.cu (same expressions,
// float64 where the reference promotes: util/loss.py:27,67).  The phases that depend on a mesh-wide scalar (sigma_c of
// the bilateral filter) or on neighbour values of the previous phase are separated by grid-wide barriers instead of
// kernel boundaries: 2 + 2*loop - 1 barriers replace ~25 launches, and every intermediate stays in L2.
//
//   P1  vertices: pos_rec partial, Laplacian residual d + partial       faces: centroid/area, norm_rec, pos_norm
//       (+ their gradients: both are piecewise linear, so no loss value is needed), per-corner messages for dpos
//   --- barrier: loss values l1, l2, l3, l5
//   P2  vertices: dpos = pos_rec' + Laplacian' + corner gather          faces: centroid distances, sigma_c partial
//   --- barrier: sigma_c
//   P3  faces: spatial weights wc*area, filter iteration 1 ... (barrier between iterations) ... last iteration also
//       takes the L1 partial of the bnf loss and its gradient
//   P4  backward of the iterations, newest first: per-face messages -> barrier -> gather through the reverse-slot map
//   end block 0 writes the five loss values and the weighted total
//
// Deterministic: grid size is a function of the device only, partials are combined in block order, no atomics on data.
// Roofline: HBM / L2 (the working set fits L2); algorithmic bytes: SURVEY.md §8d.
#include <cooperative_groups.h>

#include "common.cuh"

namespace cg = cooperative_groups;

namespace ddmp {
namespace fusedloss {

constexpr int kT = 256;
constexpr int kMaxBlocks = 2048;
constexpr int kSlots = 6;               // pos_rec, lap, norm_rec, pos_norm, sigma_c, bnf

struct Args {
    // inputs
    const float* pos;        // [V,3]
    const float* nrm;        // [F,3]
    const double* tgt_vs;    // [V,3]
    const double* tgt_fn;    // [F,3]
    const int* faces;        // [F,3]
    const int* f2f;          // [F,3]
    const int* rslot;        // [F,3]
    const int* lap_rowptr;   // [V+1]
    const int* lap_col;
    const int* corner_ptr;   // [V+1]
    const int* corner_slot;  // [3F]
    // workspace
    float* d;                // [V,3]
    float* ds;               // [V,4]  residual / degree (16-byte records)
    float* fc;               // [F,3]
    float* fa;               // [F]
    float* wca;              // [F,3]
    float* normals;          // [loop][F,3]   (iteration outputs 1..loop)
    float* g_last;           // [F,3]
    float* g;                // [F,3]
    float* face_tmp;         // [F,3,4]  per-corner messages of pos_norm (16-byte records)
    float* msg;              // [2][F,9]
    double* partials;        // [kSlots][kMaxBlocks]
    // outputs
    float* gpos;             // [V,3]
    float* gnrm;             // [F,3]
    double* losses;          // [6]: l1..l5 (as the reference computes them), weighted total
    int64_t V, F;
    int loop;
    float k[5];
    float bnf_scale;
};

__device__ __forceinline__ float sgnf(float x) { return x > 0.f ? 1.f : (x < 0.f ? -1.f : 0.f); }

struct Tri3 { float p[3][3]; };
__device__ __forceinline__ Tri3 load_tri3(const float* __restrict__ pos, const int* __restrict__ faces, int64_t f) {
    Tri3 t;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int64_t v = faces[3 * f + k];
        t.p[k][0] = __ldg(pos + 3 * v); t.p[k][1] = __ldg(pos + 3 * v + 1); t.p[k][2] = __ldg(pos + 3 * v + 2);
    }
    return t;
}

// block partial of `local` -> partials[slot][blk]  (blk: the block's index among the blocks of its mesh)
__device__ __forceinline__ void publish(double local, double* partials, int slot, double* sm, unsigned blk) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) local += __shfl_down_sync(0xffffffffu, local, o);
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = local;
    __syncthreads();
    if (threadIdx.x == 0) {
        double r = 0.0;
#pragma unroll
        for (int i = 0; i < kT / 32; ++i) r += sm[i];
        partials[slot * kMaxBlocks + blk] = r;
    }
    __syncthreads();
}

// sum of all blocks' partials of `slot`, identical in every thread of every block: lane l of warp 0 adds the partials
// l, l+32, l+64, ... in ascending order, the 32 lane sums are folded by a fixed shuffle tree.  (One thread adding the
// ~600 partials in a dependent chain of L2 loads and DADDs took ~15 us per scalar -- six scalars = 30 % of the kernel.)
__device__ __forceinline__ double total(const double* partials, int slot, double* sm, unsigned nblk) {
    if (threadIdx.x < 32) {
        const double* p = partials + slot * kMaxBlocks;
        double r = 0.0;
        for (unsigned i = threadIdx.x; i < nblk; i += 32) r += __ldcg(p + i);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) r += __shfl_xor_sync(0xffffffffu, r, o);
        if (threadIdx.x == 0) sm[0] = r;
    }
    __syncthreads();
    const double r = sm[0];
    __syncthreads();
    return r;
}

// Phase trace (ddmp_dual_loss_trace): block 0 / thread 0 stamps %globaltimer at the phase boundaries of the last launch.
__device__ unsigned long long g_trace[16];
__device__ __forceinline__ void stamp(int i) {
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        unsigned long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_trace[i] = t;
    }
}

constexpr float kTwoSigmaS2 = 0.18f;   // 2 * 0.3^2  (reference util/loss.py:110-112)
constexpr float kSigmaS2 = 0.09f;

#define STRIDE_LOOP(i, count) for (int64_t i = tid; i < (count); i += nth)

// The loss phase of one mesh, run by `nblk` blocks of a cooperative grid; `blk` is the block's index among them.  The
// stand-alone kernel gives a mesh the whole grid; the batched kernel gives each mesh the block range its stand-alone
// launch would have, so the arithmetic, the grid-stride partition and the order of every sum are the same.  Every block
// of the grid calls grid.sync() the same number of times (it depends on `loop` only).
// `Range` supplies blk() / nblk(); both are re-read where used (special registers, shared memory) rather than kept live.
struct WholeGrid {
    __device__ __forceinline__ unsigned blk() const { return blockIdx.x; }
    __device__ __forceinline__ unsigned nblk() const { return gridDim.x; }
};
__shared__ unsigned s_range[2];          // batched kernel: the block's index within its mesh, the mesh's block count
struct MeshRange {
    __device__ __forceinline__ unsigned blk() const { return s_range[0]; }
    __device__ __forceinline__ unsigned nblk() const { return s_range[1]; }
};

// ArgT: `const Args` (the stand-alone kernel's parameter, read in place) or `const Args&` (the batched kernel's copy in
// shared memory).
template <class Range, class ArgT>
__device__ __forceinline__ void dual_loss_body(ArgT a, cg::grid_group& grid, const Range rg, double* sm) {
#define blk rg.blk()
#define nblk rg.nblk()
    const int64_t tid = (int64_t)blk * kT + threadIdx.x;
    const int64_t nth = (int64_t)nblk * kT;
    const int64_t V = a.V, F = a.F;
    const int loop = a.loop;

    // ================= P1 =================================================================================
    stamp(0);
    {
        double acc_pr = 0.0, acc_lap = 0.0;
        STRIDE_LOOP(i, V) {
            float p[3], sx = 0.f, sy = 0.f, sz = 0.f;
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                p[c] = a.pos[3 * i + c];
                const double dd = a.tgt_vs[3 * i + c] - (double)p[c];
                acc_pr += dd * dd;
            }
            const int s = a.lap_rowptr[i], e = a.lap_rowptr[i + 1];
            for (int k0 = s; k0 < e; k0 += 8) {
                int jj[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) jj[u] = (k0 + u < e) ? a.lap_col[k0 + u] : -1;
                float vx[8], vy[8], vz[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) {
                    const int64_t j = jj[u] >= 0 ? jj[u] : i;
                    vx[u] = __ldg(a.pos + 3 * j); vy[u] = __ldg(a.pos + 3 * j + 1); vz[u] = __ldg(a.pos + 3 * j + 2);
                }
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    if (jj[u] >= 0) { sx += vx[u]; sy += vy[u]; sz += vz[u]; }
            }
            const float deg = (float)(e - s);
            const float dx = p[0] - sx / deg, dy = p[1] - sy / deg, dz = p[2] - sz / deg;
            a.d[3 * i] = dx; a.d[3 * i + 1] = dy; a.d[3 * i + 2] = dz;
            // residual / degree, 16-byte records: what the NEIGHBOURS gather in the backward (one 128-bit load each
            // instead of two rowptr lookups + three scalar loads)
            const float inv = 1.0f / deg;
            reinterpret_cast<float4*>(a.ds)[i] = make_float4(dx * inv, dy * inv, dz * inv, 0.f);
            acc_lap += (double)(dx * dx + dy * dy + dz * dz);
        }
        stamp(1);
        double acc_nr = 0.0, acc_pn = 0.0;
        const float kpn = a.k[4] / (float)V;                       // gout / V of pos_norm
        const double knr = (double)a.k[2] / (double)F;             // gout / F of norm_rec
        STRIDE_LOOP(f, F) {
            const Tri3 t = load_tri3(a.pos, a.faces, f);
            const float n[3] = {a.nrm[3 * f], a.nrm[3 * f + 1], a.nrm[3 * f + 2]};
            float c[3];
#pragma unroll
            for (int x = 0; x < 3; ++x) c[x] = (t.p[0][x] + t.p[1][x] + t.p[2][x]) / 3.0f;
            // geometry of the bilateral filter (bnf_geom)
            a.fc[3 * f] = c[0]; a.fc[3 * f + 1] = c[1]; a.fc[3 * f + 2] = c[2];
            {
                const float ax = t.p[1][0] - t.p[0][0], ay = t.p[1][1] - t.p[0][1], az = t.p[1][2] - t.p[0][2];
                const float bx = t.p[2][0] - t.p[0][0], by = t.p[2][1] - t.p[0][1], bz = t.p[2][2] - t.p[0][2];
                const float cx = ay * bz - az * by, cy = az * bx - ax * bz, cz = ax * by - ay * bx;
                a.fa[f] = 0.5f * sqrtf(cx * cx + cy * cy + cz * cz + 1.0e-12f);
            }
            // pos_norm forward + backward pieces
            float sg[3], S = 0.f, gn[3] = {0.f, 0.f, 0.f}, ssum = 0.f;
#pragma unroll
            for (int m = 0; m < 3; ++m) {
                const float dot = (t.p[m][0] - c[0]) * n[0] + (t.p[m][1] - c[1]) * n[1] + (t.p[m][2] - c[2]) * n[2];
                ssum += fabsf(dot);
                sg[m] = sgnf(dot);
                S += sg[m];
#pragma unroll
                for (int x = 0; x < 3; ++x) gn[x] += sg[m] * (t.p[m][x] - c[x]);
            }
            acc_pn += (double)ssum;
#pragma unroll
            for (int m = 0; m < 3; ++m) {
                const float coef = kpn * (sg[m] - S / 3.0f);
                reinterpret_cast<float4*>(a.face_tmp)[3 * f + m] = make_float4(coef * n[0], coef * n[1], coef * n[2], 0.f);
            }
            // norm_rec forward + backward
#pragma unroll
            for (int x = 0; x < 3; ++x) {
                const double dd = (double)n[x] - a.tgt_fn[3 * f + x];
                acc_nr += fabs(dd);
                const float g_nr = (float)(dd > 0.0 ? knr : (dd < 0.0 ? -knr : 0.0));
                a.gnrm[3 * f + x] = g_nr + kpn * gn[x];
            }
        }
        stamp(2);
        publish(acc_pr, a.partials, 0, sm, blk);
        publish(acc_lap, a.partials, 1, sm, blk);
        publish(acc_nr, a.partials, 2, sm, blk);
        publish(acc_pn, a.partials, 3, sm, blk);
    }
    grid.sync();
    stamp(3);
    const double l1 = sqrt(total(a.partials, 0, sm, nblk) / (double)V + 1.0e-6);
    const float l2 = (float)sqrt(total(a.partials, 1, sm, nblk) / (double)V + 1.0e-12);
    const double l3 = total(a.partials, 2, sm, nblk) / (double)F;
    const float l5 = (float)(total(a.partials, 3, sm, nblk) / (double)V);

    // ================= P2 =================================================================================
    stamp(4);
    {
        const double kpr = (double)a.k[0] / ((double)V * l1);
        const float klap = a.k[1] / ((float)V * l2);
        STRIDE_LOOP(i, V) {
            // Laplacian backward (transpose of the row-normalised adjacency: neighbours' residuals / their degree)
            const int s = a.lap_rowptr[i], e = a.lap_rowptr[i + 1];
            float gx = a.d[3 * i], gy = a.d[3 * i + 1], gz = a.d[3 * i + 2];
            // neighbour lists in batches of 8 (predicated): all index loads of a batch, then all gathers, are in flight
            // together; the sums keep the CSR order
            for (int k0 = s; k0 < e; k0 += 8) {
                int jj[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) jj[u] = (k0 + u < e) ? a.lap_col[k0 + u] : -1;
                float4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    v[u] = (jj[u] >= 0) ? __ldcg(reinterpret_cast<const float4*>(a.ds) + jj[u]) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    if (jj[u] >= 0) { gx -= v[u].x; gy -= v[u].y; gz -= v[u].z; }
            }
            // corner gather of the pos_norm messages
            float cx = 0.f, cy = 0.f, cz = 0.f;
            const int cs = a.corner_ptr[i], ce = a.corner_ptr[i + 1];
            for (int k0 = cs; k0 < ce; k0 += 8) {
                int sl[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) sl[u] = (k0 + u < ce) ? a.corner_slot[k0 + u] : -1;
                float4 v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    v[u] = (sl[u] >= 0) ? __ldcg(reinterpret_cast<const float4*>(a.face_tmp) + sl[u]) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                for (int u = 0; u < 8; ++u)
                    if (sl[u] >= 0) { cx += v[u].x; cy += v[u].y; cz += v[u].z; }
            }
            const float g3[3] = {klap * gx, klap * gy, klap * gz};
            const float c3[3] = {cx, cy, cz};
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float g_pr = (float)(kpr * ((double)a.pos[3 * i + c] - a.tgt_vs[3 * i + c]));
                a.gpos[3 * i + c] = (g_pr + g3[c]) + c3[c];
            }
        }
        stamp(5);
        double acc_sig = 0.0;
        if (loop > 0) {
            STRIDE_LOOP(f, F) {
                const float cx = a.fc[3 * f], cy = a.fc[3 * f + 1], cz = a.fc[3 * f + 2];
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const int nb = a.f2f[3 * f + s];
                    const int64_t j = nb < 0 ? (F - 1) : nb;       // python negative index: -1 is the LAST face
                    const float dx = __ldcg(a.fc + 3 * j) - cx, dy = __ldcg(a.fc + 3 * j + 1) - cy,
                                dz = __ldcg(a.fc + 3 * j + 2) - cz;
                    const float d2 = dx * dx + dy * dy + dz * dz;
                    a.wca[3 * f + s] = d2;
                    acc_sig += (double)sqrtf(d2 + 1.0e-12f);
                }
            }
        }
        stamp(6);
        publish(acc_sig, a.partials, 4, sm, blk);
    }
    float l4 = 0.f;
    if (loop > 0) {
        grid.sync();
        stamp(7);
        const float sg = (float)(total(a.partials, 4, sm, nblk) / (double)(3 * F));
        const float den = 2.0f * (sg * sg);
        const float kb = (a.k[3] * a.bnf_scale) / (float)F;        // gout / F of the bnf L1 term

        // ================= P3: filter iterations =======================================================
        double acc_bnf = 0.0;
        for (int t = 1; t <= loop; ++t) {
            const float* n_in = (t == 1) ? a.nrm : a.normals + (int64_t)(t - 2) * 3 * F;
            float* n_out = a.normals + (int64_t)(t - 1) * 3 * F;
            if (t > 1) grid.sync();
            STRIDE_LOOP(f, F) {
                float wc[3];
                if (t == 1) {
#pragma unroll
                    for (int s = 0; s < 3; ++s) {
                        const int nb = a.f2f[3 * f + s];
                        wc[s] = (nb < 0) ? 0.f : expf(-1.0f * a.wca[3 * f + s] / den) * __ldcg(a.fa + nb);
                        a.wca[3 * f + s] = wc[s];
                    }
                } else {
#pragma unroll
                    for (int s = 0; s < 3; ++s) wc[s] = a.wca[3 * f + s];
                }
                const float nx = __ldcg(n_in + 3 * f), ny = __ldcg(n_in + 3 * f + 1), nz = __ldcg(n_in + 3 * f + 2);
                float ax = 0.f, ay = 0.f, az = 0.f;
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const int nb = a.f2f[3 * f + s];
                    const int64_t j = nb < 0 ? (F - 1) : nb;
                    const float jx = __ldcg(n_in + 3 * j), jy = __ldcg(n_in + 3 * j + 1), jz = __ldcg(n_in + 3 * j + 2);
                    const float dx = jx - nx, dy = jy - ny, dz = jz - nz;
                    const float W = wc[s] * expf(-1.0f * (dx * dx + dy * dy + dz * dz) / kTwoSigmaS2);
                    ax = fmaf(W, jx, ax); ay = fmaf(W, jy, ay); az = fmaf(W, jz, az);
                }
                const float r = sqrtf(ax * ax + ay * ay + az * az + 1.0e-12f) + 1.0e-12f;
                const float o[3] = {ax / r, ay / r, az / r};
                n_out[3 * f] = o[0]; n_out[3 * f + 1] = o[1]; n_out[3 * f + 2] = o[2];
                if (t == loop) {                               // L1 term against the unfiltered prediction
#pragma unroll
                    for (int x = 0; x < 3; ++x) {
                        const float df = o[x] - a.nrm[3 * f + x];
                        acc_bnf += (double)fabsf(df);
                        a.g_last[3 * f + x] = kb * sgnf(df);
                    }
                }
            }
        }
        stamp(8);
        publish(acc_bnf, a.partials, 5, sm, blk);

        // ================= P4: backward of the iterations ===================================================
        for (int t = loop - 1; t >= 0; --t) {
            const float* n_in = (t == 0) ? a.nrm : a.normals + (int64_t)(t - 1) * 3 * F;
            const float* g_out = (t == loop - 1) ? a.g_last : a.g;
            float* msg = a.msg + (int64_t)(t & 1) * 9 * F;
            STRIDE_LOOP(f, F) {
                const float n[3] = {__ldcg(n_in + 3 * f), __ldcg(n_in + 3 * f + 1), __ldcg(n_in + 3 * f + 2)};
                float nj[3][3], W[3], acc[3] = {0.f, 0.f, 0.f};
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const int nb = a.f2f[3 * f + s];
                    const int64_t j = nb < 0 ? (F - 1) : nb;
#pragma unroll
                    for (int x = 0; x < 3; ++x) nj[s][x] = __ldcg(n_in + 3 * j + x);
                    const float dx = nj[s][0] - n[0], dy = nj[s][1] - n[1], dz = nj[s][2] - n[2];
                    W[s] = a.wca[3 * f + s] * expf(-1.0f * (dx * dx + dy * dy + dz * dz) / kTwoSigmaS2);
#pragma unroll
                    for (int x = 0; x < 3; ++x) acc[x] = fmaf(W[s], nj[s][x], acc[x]);
                }
                const float r = sqrtf(acc[0] * acc[0] + acc[1] * acc[1] + acc[2] * acc[2] + 1.0e-12f);
                const float re = r + 1.0e-12f;
                const float go[3] = {g_out[3 * f], g_out[3 * f + 1], g_out[3 * f + 2]};
                const float gd = go[0] * acc[0] + go[1] * acc[1] + go[2] * acc[2];
                const float k2 = gd / (re * re * r);
                float ga[3];
#pragma unroll
                for (int x = 0; x < 3; ++x) ga[x] = go[x] / re - acc[x] * k2;
                float ctr[3] = {0.f, 0.f, 0.f};
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const float dotg = ga[0] * nj[s][0] + ga[1] * nj[s][1] + ga[2] * nj[s][2];
                    const float q = dotg * W[s] / kSigmaS2;
#pragma unroll
                    for (int x = 0; x < 3; ++x) {
                        const float diff = nj[s][x] - n[x];
                        msg[9 * f + 3 * s + x] = W[s] * ga[x] - q * diff;
                        ctr[x] = fmaf(q, diff, ctr[x]);
                    }
                }
#pragma unroll
                for (int x = 0; x < 3; ++x) a.g[3 * f + x] = ctr[x];
            }
            if (t == 0) stamp(9);
            grid.sync();
            if (t == 0) stamp(10);
            STRIDE_LOOP(j, F) {
                float x = a.g[3 * j], y = a.g[3 * j + 1], z = a.g[3 * j + 2];
                if (t == 0) { x -= a.g_last[3 * j]; y -= a.g_last[3 * j + 1]; z -= a.g_last[3 * j + 2]; }
#pragma unroll
                for (int s = 0; s < 3; ++s) {
                    const int f = a.f2f[3 * j + s];
                    if (f >= 0) {
                        const int64_t o = 9 * (int64_t)f + 3 * a.rslot[3 * j + s];
                        x += __ldcg(msg + o); y += __ldcg(msg + o + 1); z += __ldcg(msg + o + 2);
                    }
                }
                if (t == 0) {
                    a.gnrm[3 * j] += x; a.gnrm[3 * j + 1] += y; a.gnrm[3 * j + 2] += z;
                } else {
                    a.g[3 * j] = x; a.g[3 * j + 1] = y; a.g[3 * j + 2] = z;
                }
            }
        }
        stamp(11);
        l4 = (float)(total(a.partials, 5, sm, nblk) / (double)F);
    }
    stamp(12);
    if (blk == 0 && threadIdx.x == 0) {
        const float l4s = l4 * a.bnf_scale;                      // `loss_norm2 * 0.0` while epoch <= 100 (main.py:101)
        a.losses[0] = l1; a.losses[1] = (double)l2; a.losses[2] = l3; a.losses[3] = (double)l4s; a.losses[4] = (double)l5;
        // python: k1*l1 (f64) + k2*l2 (f32) + k3*l3 (f64) + k4*l4 (f32) + k5*l5 (f32), left to right
        double tot = (double)a.k[0] * l1;
        tot += (double)(a.k[1] * l2);
        tot += (double)a.k[2] * l3;
        tot += (double)(a.k[3] * l4s);
        tot += (double)(a.k[4] * l5);
        a.losses[5] = tot;
    }
#undef blk
#undef nblk
}

__global__ void __launch_bounds__(kT, 4)
dual_loss_kernel(const Args a) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double sm[kT / 32];
    dual_loss_body<WholeGrid, const Args>(a, grid, WholeGrid{}, sm);
}

// Workspace layout of one mesh (ddmp_dual_loss_workspace_bytes): the same for the stand-alone and the batched kernel.
__host__ __device__ inline void carve_workspace(Args& a, void* workspace, int64_t V, int64_t F, int loop) {
    float* w = static_cast<float*>(workspace);
    w += (4 - ((reinterpret_cast<uintptr_t>(w) / 4) & 3)) & 3;       // 16-byte records first
    a.ds = w; w += 4 * V;
    a.face_tmp = w; w += 12 * F;
    a.d = w; w += 3 * V;
    a.fc = w; w += 3 * F;
    a.fa = w; w += F;
    a.wca = w; w += 3 * F;
    a.normals = w; w += (int64_t)(loop > 0 ? loop : 1) * 3 * F;
    a.g_last = w; w += 3 * F;
    a.g = w; w += 3 * F;
    a.msg = w; w += 18 * F;
    const int64_t off = (((w - static_cast<float*>(workspace)) * 4 + 15) / 16) * 16;
    a.partials = reinterpret_cast<double*>(static_cast<char*>(workspace) + off);
}

__host__ __device__ inline int64_t mesh_blocks(int64_t V, int64_t F, int g_single) {
    const int64_t want = (((V > F) ? V : F) + kT - 1) / kT;
    return want < g_single ? want : g_single;
}

// B meshes in one cooperative grid: mesh m owns mesh_blocks(V_m, F_m) consecutive blocks, in table order.  Thread 0 of
// each block finds its mesh and unpacks the descriptor (include/ddmp_b200.h, DDMP_DUAL_LOSS_DESC_WORDS) into shared
// memory; the meshes share the barriers, which is what makes one launch of all of them possible.
__global__ void __launch_bounds__(kT, 4)
dual_loss_multi_kernel(const int64_t* __restrict__ table, int n_mesh, int g_single, float bnf_scale, int loop) {
    cg::grid_group grid = cg::this_grid();
    __shared__ double sm[kT / 32];
    __shared__ Args sa;
    if (threadIdx.x == 0) {
        int start = 0, m = 0, b = 0;
        for (; m < n_mesh; ++m) {
            const int64_t* d = table + (int64_t)m * DDMP_DUAL_LOSS_DESC_WORDS;
            b = (int)mesh_blocks(d[15], d[16], g_single);
            if ((int)blockIdx.x < start + b) break;
            start += b;
        }
        const int64_t* d = table + (int64_t)m * DDMP_DUAL_LOSS_DESC_WORDS;
        Args a{};
        a.pos = reinterpret_cast<const float*>(d[0]);
        a.nrm = reinterpret_cast<const float*>(d[1]);
        a.tgt_vs = reinterpret_cast<const double*>(d[2]);
        a.tgt_fn = reinterpret_cast<const double*>(d[3]);
        a.faces = reinterpret_cast<const int*>(d[4]);
        a.f2f = reinterpret_cast<const int*>(d[5]);
        a.rslot = reinterpret_cast<const int*>(d[6]);
        a.lap_rowptr = reinterpret_cast<const int*>(d[7]);
        a.lap_col = reinterpret_cast<const int*>(d[8]);
        a.corner_ptr = reinterpret_cast<const int*>(d[9]);
        a.corner_slot = reinterpret_cast<const int*>(d[10]);
        a.V = d[15]; a.F = d[16];
        carve_workspace(a, reinterpret_cast<void*>(d[11]), a.V, a.F, loop);
        a.gpos = reinterpret_cast<float*>(d[12]);
        a.gnrm = reinterpret_cast<float*>(d[13]);
        a.losses = reinterpret_cast<double*>(d[14]);
#pragma unroll
        for (int i = 0; i < 5; ++i) a.k[i] = __uint_as_float((unsigned)(d[17 + i] & 0xffffffffll));
        a.loop = loop;
        a.bnf_scale = bnf_scale;
        sa = a;
        s_range[0] = blockIdx.x - (unsigned)start;
        s_range[1] = b;
    }
    __syncthreads();
    dual_loss_body<MeshRange, const Args&>(sa, grid, MeshRange{}, sm);
}

static int occupancy_blocks(const void* kernel) {
    int per_sm = 0, sms = 0, dev = 0;
    cudaGetDevice(&dev);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, kT, 0);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int v = per_sm * sms;
    if (v > kMaxBlocks) v = kMaxBlocks;
    return v > 0 ? v : 1;
}

// blocks per cooperative launch: of the stand-alone kernel (batched = 0) and of the batched kernel (batched = 1)
static int grid_blocks(int batched = 0) {
    static int cached[2][64] = {{0}};
    int dev = 0;
    cudaGetDevice(&dev);
    int& g = cached[batched ? 1 : 0][dev & 63];
    if (g == 0) g = occupancy_blocks(batched ? (const void*)dual_loss_multi_kernel : (const void*)dual_loss_kernel);
    return g;
}

}  // namespace fusedloss
}  // namespace ddmp

extern "C" {

int64_t ddmp_dual_loss_workspace_bytes(int64_t V, int64_t F, int32_t loop) {
    if (V <= 0 || F <= 0 || loop < 0) return 0;
    const int64_t floats = 4 + 4 * V + 12 * F + 3 * V + 3 * F + F + 3 * F + (int64_t)(loop > 0 ? loop : 1) * 3 * F + 3 * F + 3 * F + 18 * F;
    return ((floats * 4 + 15) / 16) * 16 + (int64_t)ddmp::fusedloss::kSlots * ddmp::fusedloss::kMaxBlocks * 8;
}

int ddmp_dual_loss_trace(uint64_t* out16) {
    DDMP_REQUIRE(out16, "dual_loss_trace: null pointer");
    cudaError_t e = cudaMemcpyFromSymbol(out16, ddmp::fusedloss::g_trace, 16 * sizeof(unsigned long long));
    if (e != cudaSuccess) {
        ddmp::set_error("dual_loss_trace: %s", cudaGetErrorString(e));
        return DDMP_ERR_CUDA;
    }
    return DDMP_OK;
}

int ddmp_dual_loss(const float* pos, const float* nrm, const double* tgt_vs, const double* tgt_fn,
                   const int32_t* faces, const int32_t* f2f, const int32_t* rslot, const int32_t* lap_rowptr,
                   const int32_t* lap_col, const int32_t* corner_ptr, const int32_t* corner_slot, float k1, float k2,
                   float k3, float k4, float k5, float bnf_scale, int32_t loop, void* workspace,
                   int64_t workspace_bytes, float* gpos, float* gnrm, double* losses, int64_t V, int64_t F,
                   void* stream) {
    using namespace ddmp;
    using namespace ddmp::fusedloss;
    DDMP_REQUIRE(pos && nrm && tgt_vs && tgt_fn && faces && f2f && rslot && lap_rowptr && lap_col && corner_ptr &&
                     corner_slot && workspace && gpos && gnrm && losses, "dual_loss: null pointer");
    DDMP_REQUIRE(V > 0 && F > 0 && loop >= 0, "dual_loss: bad shape V=%lld F=%lld loop=%d", (long long)V, (long long)F,
                 loop);
    DDMP_REQUIRE(workspace_bytes >= ddmp_dual_loss_workspace_bytes(V, F, loop), "dual_loss: workspace too small");
    Args a{};
    a.pos = pos; a.nrm = nrm; a.tgt_vs = tgt_vs; a.tgt_fn = tgt_fn; a.faces = faces; a.f2f = f2f; a.rslot = rslot;
    a.lap_rowptr = lap_rowptr; a.lap_col = lap_col; a.corner_ptr = corner_ptr; a.corner_slot = corner_slot;
    carve_workspace(a, workspace, V, F, loop);
    a.gpos = gpos; a.gnrm = gnrm; a.losses = losses;
    a.V = V; a.F = F; a.loop = loop;
    a.k[0] = k1; a.k[1] = k2; a.k[2] = k3; a.k[3] = k4; a.k[4] = k5;
    a.bnf_scale = bnf_scale;
    const int blocks = (int)mesh_blocks(V, F, grid_blocks());
    void* params[] = {&a};
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)dual_loss_kernel, dim3((unsigned)blocks), dim3(kT), params, 0,
                                                as_stream(stream));
    if (e != cudaSuccess) {
        set_error("dual_loss: cooperative launch failed: %s", cudaGetErrorString(e));
        return DDMP_ERR_CUDA;
    }
    return check_launch("dual_loss");
}

int64_t ddmp_dual_loss_grid(int32_t batched) { return ddmp::fusedloss::grid_blocks(batched); }

int ddmp_dual_loss_multi(const int64_t* table, const int64_t* vf, int32_t n_mesh, float bnf_scale, int32_t loop,
                         void* stream) {
    using namespace ddmp;
    using namespace ddmp::fusedloss;
    DDMP_REQUIRE(table && vf && n_mesh > 0 && loop >= 0, "dual_loss_multi: bad arguments n_mesh=%d loop=%d", n_mesh,
                 loop);
    const int g_single = grid_blocks(0);
    int64_t blocks = 0;
    for (int m = 0; m < n_mesh; ++m) {
        DDMP_REQUIRE(vf[2 * m] > 0 && vf[2 * m + 1] > 0, "dual_loss_multi: mesh %d has V=%lld F=%lld", m,
                     (long long)vf[2 * m], (long long)vf[2 * m + 1]);
        blocks += mesh_blocks(vf[2 * m], vf[2 * m + 1], g_single);
    }
    DDMP_REQUIRE(blocks <= grid_blocks(1), "dual_loss_multi: %lld blocks exceed one cooperative launch (%d)",
                 (long long)blocks, grid_blocks(1));
    int n = n_mesh, gs = g_single;
    void* params[] = {(void*)&table, &n, &gs, &bnf_scale, &loop};
    cudaError_t e = cudaLaunchCooperativeKernel((const void*)dual_loss_multi_kernel, dim3((unsigned)blocks), dim3(kT),
                                                params, 0, as_stream(stream));
    if (e != cudaSuccess) {
        set_error("dual_loss_multi: cooperative launch failed: %s", cudaGetErrorString(e));
        return DDMP_ERR_CUDA;
    }
    return check_launch("dual_loss_multi");
}

}  // extern "C"
