// Point-to-surface distance on the device: a linear BVH over the target triangles (Karras 2012, "Maximizing Parallelism
// in the Construction of BVHs, Octrees, and k-d Trees"), one nearest-triangle traversal per query point, and a
// fixed-order reduction of the per-point distances into (min, max, sum, sum of squares).
//
//   keys   : 63-bit Morton code of each face centroid, 21 bits per axis, quantised in the scene box (ddmp_prep_bbox)
//            like graph.morton_order; the host sorts them (torch.sort, stable).
//   build  : one thread per internal node finds its range and split (Karras); sorted keys that are equal are told
//            apart by their position, so coincident centroids still give a valid binary tree.  Then a bottom-up refit,
//            one thread per leaf, with an integer arrival counter per internal node: the second arrival merges both
//            child boxes (min / max: the result does not depend on which child arrived first) and zeroes the counter.
//   query  : depth-first, nearer child first, pruned with the best squared distance found so far.
//
// Precision: triangle tests and distances are float64.  Node boxes are float32, rounded outward, and the box test is a
// lower bound in round-down float arithmetic, compared with a threshold slightly above the current best (DESIGN.md
// "Point-to-mesh distance": the leaf routine's rounding cannot make a pruned face the winner).  Therefore the BVH
// query returns bit for bit what an exhaustive scan with the same leaf routine returns.  This file is compiled with
// -fmad=false (Makefile) so the leaf routine rounds identically in every kernel it is inlined into.
#include <limits.h>
#include <math_constants.h>

#include "common.cuh"

namespace ddmp {
namespace dist {

constexpr int kT = 256;
constexpr int kMaxBlocks = 1024;
static_assert(kT == DDMP_DISTANCE_THREADS && kMaxBlocks == DDMP_DISTANCE_MAX_BLOCKS, "batched block counts (header)");
// A root-to-leaf path visits internal nodes whose split prefix lengths strictly increase.  Keys use 63 of 64 bits (the
// root's prefix is >= 1) and a tie between equal keys adds 64 + clz32(i ^ j) <= 95, so a path holds at most 95
// internal nodes and a stack of 96 entries cannot overflow.
constexpr int kStack = 96;

// Internal node, 64 bytes: the boxes of BOTH children inline (one 64-byte load decides both), then the children.
// box[c] = (lo.x, lo.y, lo.z, hi.x, hi.y, hi.z); child >= 0: internal node, child < 0: leaf ~child (sorted position).
struct __align__(64) Node {
    float box[2][6];
    int child[2];
    int pad[2];
};
static_assert(sizeof(Node) == 64, "node layout");

struct Scratch {
    unsigned int ticket;
    unsigned int pad[63];
    double partials[4][kMaxBlocks];
};

static inline unsigned grid_for(int64_t count) {
    int64_t g = ceil_div(count, kT);
    if (g > kMaxBlocks) g = kMaxBlocks;
    return (unsigned)(g < 1 ? 1 : g);
}

__device__ __forceinline__ uint64_t part1by2(uint64_t x) {
    x &= 0x1fffffull;
    x = (x | x << 32) & 0x1f00000000ffffull;
    x = (x | x << 16) & 0x1f0000ff0000ffull;
    x = (x | x << 8) & 0x100f00f00f00f00full;
    x = (x | x << 4) & 0x10c30c30c30c30c3ull;
    x = (x | x << 2) & 0x1249249249249249ull;
    return x;
}

__global__ void __launch_bounds__(kT)
keys_kernel(const double* __restrict__ vs, const int* __restrict__ faces, const double* __restrict__ bbox,
            int64_t* __restrict__ keys, int64_t F) {
    const int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= F) return;
    uint64_t code = 0;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double c = (vs[3 * (int64_t)faces[3 * f] + a] + vs[3 * (int64_t)faces[3 * f + 1] + a] +
                          vs[3 * (int64_t)faces[3 * f + 2] + a]) / 3.0;
        const double lo = bbox[a], hi = bbox[3 + a];
        const double span = hi > lo ? hi - lo : 1.0;
        double q = floor((c - lo) / span * (double)((1 << 21) - 1));
        q = fmin(fmax(q, 0.0), (double)((1 << 21) - 1));
        code |= part1by2((uint64_t)q) << a;
    }
    keys[f] = (int64_t)code;
}

// length of the common prefix of sorted keys i and j (-1 outside [0, n)); equal keys continue with their positions
__device__ __forceinline__ int delta(const int64_t* __restrict__ k, int64_t n, int64_t i, int64_t j) {
    if (j < 0 || j >= n) return -1;
    const uint64_t a = (uint64_t)k[i], b = (uint64_t)k[j];
    if (a == b) return 64 + __clz((unsigned)i ^ (unsigned)j);
    return __clzll(a ^ b);
}

// internal node i of F-1; parent[] entries are (parent << 1 | slot), internal nodes at [0, F-1), leaves at F-1 + leaf
__global__ void __launch_bounds__(kT)
topology_kernel(const int64_t* __restrict__ keys, const int64_t* __restrict__ order, const int* __restrict__ faces,
                Node* __restrict__ nodes, int4* __restrict__ leaves, int* __restrict__ parent, int64_t F) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < F) {   // leaf payload: the face's corners and its id, in sorted order
        const int64_t f = order[i];
        leaves[i] = make_int4(faces[3 * f], faces[3 * f + 1], faces[3 * f + 2], (int)f);
    }
    if (i >= F - 1) return;
    const int d = delta(keys, F, i, i + 1) > delta(keys, F, i, i - 1) ? 1 : -1;
    const int dmin = delta(keys, F, i, i - d);
    int64_t lmax = 2;
    while (delta(keys, F, i, i + lmax * d) > dmin) lmax <<= 1;
    int64_t l = 0;
    for (int64_t t = lmax >> 1; t >= 1; t >>= 1)
        if (delta(keys, F, i, i + (l + t) * d) > dmin) l += t;
    const int64_t j = i + l * d;
    const int dnode = delta(keys, F, i, j);
    int64_t s = 0;
    for (int64_t div = 2;; div <<= 1) {
        const int64_t t = (l + div - 1) / div;
        if (delta(keys, F, i, i + (s + t) * d) > dnode) s += t;
        if (t <= 1) break;
    }
    const int64_t gamma = i + s * d + (d < 0 ? -1 : 0);
    const int64_t lo = i < j ? i : j, hi = i < j ? j : i;
    const int c0 = lo == gamma ? ~(int)gamma : (int)gamma;
    const int c1 = hi == gamma + 1 ? ~(int)(gamma + 1) : (int)(gamma + 1);
    nodes[i].child[0] = c0;
    nodes[i].child[1] = c1;
    parent[c0 < 0 ? F - 1 + ~c0 : c0] = (int)(i << 1);
    parent[c1 < 0 ? F - 1 + ~c1 : c1] = (int)(i << 1 | 1);
}

// Where a kernel body reads its block range.  A stand-alone kernel gives its one input the whole grid; a batched kernel
// (one launch over the rows of a descriptor table) gives each row the blocks its stand-alone launch would have, and the
// body sees row-local block ids and block count, so every partition and every order of summation stays the same.
struct WholeGrid {
    __device__ __forceinline__ unsigned blk() const { return blockIdx.x; }
    __device__ __forceinline__ unsigned nblk() const { return gridDim.x; }
};
__shared__ unsigned s_range[2];          // batched kernels: the block's index within its row, the row's block count
struct RowRange {
    __device__ __forceinline__ unsigned blk() const { return s_range[0]; }
    __device__ __forceinline__ unsigned nblk() const { return s_range[1]; }
};

// Batched kernels: rows of W int64 words in block order, word 0 = the row's first block, word 1 = its block count (a
// row may own no block).  Thread 0 finds the row that owns this block (the last one whose first block is <= it) and
// fills s_range; every thread gets the row after the barrier.
template <int W>
__device__ __forceinline__ const int64_t* claim_row(const int64_t* __restrict__ table, int n) {
    __shared__ int s_row;
    if (threadIdx.x == 0) {
        int m = 0;
        while (m + 1 < n && table[(int64_t)(m + 1) * W] <= (int64_t)blockIdx.x) ++m;
        s_row = m;
        s_range[0] = blockIdx.x - (unsigned)table[(int64_t)m * W];
        s_range[1] = (unsigned)table[(int64_t)m * W + 1];
    }
    __syncthreads();
    return table + (int64_t)s_row * W;
}
template <class T>
__device__ __forceinline__ T* word_ptr(const int64_t* row, int k) { return reinterpret_cast<T*>(row[k]); }

// bottom-up refit, one thread per leaf; counters [F-1] are zero on entry and zero again on exit.  Only the boxes change:
// the leaves hold corner ids, so a tree built once refits to any new positions of the same mesh.
template <class Range>
__device__ __forceinline__ void refit_body(const Range rg, const double* __restrict__ vs, const int4* __restrict__ leaves,
                                           Node* nodes, const int* __restrict__ parent, unsigned* counters, int64_t F) {
    const int64_t i = (int64_t)rg.blk() * blockDim.x + threadIdx.x;
    if (i >= F) return;
    const int4 lf = leaves[i];
    float b[6];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const double x0 = vs[3 * (int64_t)lf.x + a], x1 = vs[3 * (int64_t)lf.y + a], x2 = vs[3 * (int64_t)lf.z + a];
        b[a] = __double2float_rd(fmin(x0, fmin(x1, x2)));
        b[3 + a] = __double2float_ru(fmax(x0, fmax(x1, x2)));
    }
    int p = parent[F - 1 + i];
    while (true) {
        Node* n = nodes + (p >> 1);
#pragma unroll
        for (int k = 0; k < 6; ++k) n->box[p & 1][k] = b[k];
        __threadfence();
        if (atomicAdd(&counters[p >> 1], 1u) == 0u) return;   // first arrival: the sibling finishes this node
        counters[p >> 1] = 0u;
        __threadfence();
        const float* o = n->box[(p & 1) ^ 1];
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            b[a] = fminf(b[a], __ldcg(o + a));
            b[3 + a] = fmaxf(b[3 + a], __ldcg(o + 3 + a));
        }
        if ((p >> 1) == 0) return;   // root: its own box is never read
        p = parent[p >> 1];
    }
}

__global__ void __launch_bounds__(kT)
refit_kernel(const double* __restrict__ vs, const int4* __restrict__ leaves, Node* nodes, const int* __restrict__ parent,
             unsigned* counters, int64_t F) {
    refit_body(WholeGrid{}, vs, leaves, nodes, parent, counters, F);
}

__global__ void __launch_bounds__(kT)
refit_multi_kernel(const int64_t* __restrict__ table, int n) {
    const int64_t* r = claim_row<DDMP_BVH_REFIT_DESC_WORDS>(table, n);
    refit_body(RowRange{}, word_ptr<const double>(r, 2), word_ptr<const int4>(r, 3), word_ptr<Node>(r, 4),
               word_ptr<const int>(r, 5), word_ptr<unsigned>(r, 6), r[7]);
}

struct V3 {
    double x, y, z;
};
__device__ __forceinline__ V3 sub(V3 a, V3 b) { return {a.x - b.x, a.y - b.y, a.z - b.z}; }
__device__ __forceinline__ double dot(V3 a, V3 b) { return a.x * b.x + a.y * b.y + a.z * b.z; }
__device__ __forceinline__ V3 axpy(V3 a, double s, V3 d) { return {a.x + s * d.x, a.y + s * d.y, a.z + s * d.z}; }
__device__ __forceinline__ V3 load3(const double* __restrict__ vs, int v) {
    const double* q = vs + 3 * (int64_t)v;
    return {__ldg(q), __ldg(q + 1), __ldg(q + 2)};
}

// squared distance from p to segment [a, b]; a zero-length segment is the point a
__device__ __forceinline__ double seg_d2(V3 p, V3 a, V3 b) {
    const V3 ab = sub(b, a);
    const double l2 = dot(ab, ab);
    double t = l2 > 0.0 ? dot(sub(p, a), ab) / l2 : 0.0;
    t = fmin(fmax(t, 0.0), 1.0);
    const V3 d = sub(p, axpy(a, t, ab));
    return dot(d, d);
}

// Squared distance from p to triangle (a, b, c): Voronoi-region classification of Ericson, "Real-Time Collision
// Detection" §5.1.5.  Every closest point it forms is a convex combination of the corners (weights in [0, 1]).  A
// triangle whose corner angle at `a` has a sine below 1e-10 (zero area: collinear or coincident corners) is the union
// of its three edges.
__device__ __forceinline__ double tri_d2(V3 p, V3 a, V3 b, V3 c) {
    const V3 ab = sub(b, a), ac = sub(c, a), ap = sub(p, a);
    const V3 n = {ab.y * ac.z - ab.z * ac.y, ab.z * ac.x - ab.x * ac.z, ab.x * ac.y - ab.y * ac.x};
    if (!(dot(n, n) > 1e-20 * dot(ab, ab) * dot(ac, ac)))
        return fmin(seg_d2(p, a, b), fmin(seg_d2(p, b, c), seg_d2(p, c, a)));
    V3 q;
    const double d1 = dot(ab, ap), d2 = dot(ac, ap);
    const V3 bp = sub(p, b);
    const double d3 = dot(ab, bp), d4 = dot(ac, bp);
    const V3 cp = sub(p, c);
    const double d5 = dot(ab, cp), d6 = dot(ac, cp);
    const double vc = d1 * d4 - d3 * d2, vb = d5 * d2 - d1 * d6, va = d3 * d6 - d5 * d4;
    if (d1 <= 0.0 && d2 <= 0.0) {
        q = a;
    } else if (d3 >= 0.0 && d4 <= d3) {
        q = b;
    } else if (vc <= 0.0 && d1 >= 0.0 && d3 <= 0.0) {
        const double den = d1 - d3;
        q = axpy(a, den > 0.0 ? d1 / den : 0.0, ab);
    } else if (d6 >= 0.0 && d5 <= d6) {
        q = c;
    } else if (vb <= 0.0 && d2 >= 0.0 && d6 <= 0.0) {
        const double den = d2 - d6;
        q = axpy(a, den > 0.0 ? d2 / den : 0.0, ac);
    } else if (va <= 0.0 && d4 - d3 >= 0.0 && d5 - d6 >= 0.0) {
        const double den = (d4 - d3) + (d5 - d6);
        q = axpy(b, den > 0.0 ? (d4 - d3) / den : 0.0, sub(c, b));
    } else {
        const double den = va + vb + vc;   // > 0 in exact arithmetic; rounding may break that near an edge
        if (!(va >= 0.0 && vb >= 0.0 && vc >= 0.0 && den > 0.0))
            return fmin(seg_d2(p, a, b), fmin(seg_d2(p, b, c), seg_d2(p, c, a)));
        q = axpy(axpy(a, vb / den, ab), vc / den, ac);
    }
    const V3 d = sub(p, q);
    return dot(d, d);
}

__device__ __forceinline__ void leaf_test(V3 p, const double* __restrict__ vs, int4 lf, double& best, int& best_f) {
    const double d2 = tri_d2(p, load3(vs, lf.x), load3(vs, lf.y), load3(vs, lf.z));
    if (d2 < best || (d2 == best && lf.w < best_f)) {
        best = d2;
        best_f = lf.w;
    }
}

// lower bound of the squared distance from p (given as the float interval [plo, phi] per axis) to a box, round-down
__device__ __forceinline__ float box_lb2(const float* plo, const float* phi, const float* b) {
    float s = 0.f;
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float d = fmaxf(fmaxf(__fsub_rd(b[a], phi[a]), __fsub_rd(plo[a], b[3 + a])), 0.f);
        s = __fadd_rd(s, __fmul_rd(d, d));
    }
    return s;
}

template <class Range>
__device__ __forceinline__ void query_body(const Range rg, const double* __restrict__ pts, int64_t P,
                                           const double* __restrict__ vs, const Node* __restrict__ nodes,
                                           const int4* __restrict__ leaves, int64_t F, double* __restrict__ dist,
                                           int* __restrict__ face) {
    const int64_t i = (int64_t)rg.blk() * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const V3 p = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    double best = CUDART_INF;   // +inf
    int best_f = INT_MAX;
    if (F == 1) {
        leaf_test(p, vs, __ldg(leaves), best, best_f);
    } else {
        const float plo[3] = {__double2float_rd(p.x), __double2float_rd(p.y), __double2float_rd(p.z)};
        const float phi[3] = {__double2float_ru(p.x), __double2float_ru(p.y), __double2float_ru(p.z)};
        // Absolute slack of the pruning threshold: 1e-10 of the largest coordinate magnitude of the target (from
        // the root's child boxes), far above the leaf routine's rounding of a few ulps of that magnitude.
        float S = 0.f;
#pragma unroll
        for (int k = 0; k < 6; ++k) S = fmaxf(S, fmaxf(fabsf(__ldg(&nodes[0].box[0][k])), fabsf(__ldg(&nodes[0].box[1][k]))));
        const double m2 = (1e-10 * (double)S) * (1e-10 * (double)S);
        int stack[kStack];
        float stack_lb[kStack];
        int sp = 0;
        int node = 0;
        float thr = __double2float_ru(best);
        while (true) {
            const float4* q = reinterpret_cast<const float4*>(nodes + node);
            const float4 r0 = __ldg(q), r1 = __ldg(q + 1), r2 = __ldg(q + 2), r3 = __ldg(q + 3);
            const float b0[6] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y};
            const float b1[6] = {r1.z, r1.w, r2.x, r2.y, r2.z, r2.w};
            const int c0 = __float_as_int(r3.x), c1 = __float_as_int(r3.y);
            const float l0 = box_lb2(plo, phi, b0), l1 = box_lb2(plo, phi, b1);
            int next = -1;
            // nearer child first; a leaf is tested on the spot
            const bool first1 = l1 < l0;
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const bool one = (k == 0) == first1;
                const int c = one ? c1 : c0;
                const float lb = one ? l1 : l0;
                if (!(lb <= thr)) continue;
                if (c < 0) {
                    leaf_test(p, vs, __ldg(leaves + ~c), best, best_f);
                    thr = __double2float_ru(best + 1e-6 * best + m2);
                } else if (next < 0) {
                    next = c;
                } else {
                    stack[sp] = c;
                    stack_lb[sp] = lb;
                    ++sp;
                }
            }
            if (next >= 0) {
                node = next;
                continue;
            }
            node = -1;
            while (sp > 0) {
                --sp;
                if (stack_lb[sp] <= thr) {
                    node = stack[sp];
                    break;
                }
            }
            if (node < 0) break;
        }
    }
    dist[i] = sqrt(best);
    face[i] = best_f;
}

__global__ void __launch_bounds__(kT)
query_kernel(const double* __restrict__ pts, int64_t P, const double* __restrict__ vs, const Node* __restrict__ nodes,
             const int4* __restrict__ leaves, int64_t F, double* __restrict__ dist, int* __restrict__ face) {
    query_body(WholeGrid{}, pts, P, vs, nodes, leaves, F, dist, face);
}

__global__ void __launch_bounds__(kT)
query_multi_kernel(const int64_t* __restrict__ table, int n) {
    const int64_t* r = claim_row<DDMP_DISTANCE_DESC_WORDS>(table, n);
    query_body(RowRange{}, word_ptr<const double>(r, 2), r[3], word_ptr<const double>(r, 4), word_ptr<const Node>(r, 5),
               word_ptr<const int4>(r, 6), r[7], word_ptr<double>(r, 8), word_ptr<int>(r, 9));
}

__global__ void __launch_bounds__(kT)
exhaustive_kernel(const double* __restrict__ pts, int64_t P, const double* __restrict__ vs, const int* __restrict__ faces,
                  int64_t F, double* __restrict__ dist, int* __restrict__ face) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= P) return;
    const V3 p = {pts[3 * i], pts[3 * i + 1], pts[3 * i + 2]};
    double best = CUDART_INF;
    int best_f = INT_MAX;
    for (int64_t f = 0; f < F; ++f)
        leaf_test(p, vs, make_int4(__ldg(faces + 3 * f), __ldg(faces + 3 * f + 1), __ldg(faces + 3 * f + 2), (int)f),
                  best, best_f);
    dist[i] = sqrt(best);
    face[i] = best_f;
}

// (min, max, sum, sum of squares) of dist[0..P); per-block partials, the last block combines them in block order
template <class Range>
__device__ __forceinline__ void stats_body(const Range rg, const double* __restrict__ d, int64_t P, double* out,
                                           Scratch* sc, double (*sm)[kT / 32]) {
    double lo = CUDART_INF, hi = -CUDART_INF, s = 0.0, s2 = 0.0;
    for (int64_t i = (int64_t)rg.blk() * blockDim.x + threadIdx.x; i < P; i += (int64_t)rg.nblk() * blockDim.x) {
        const double x = d[i];
        lo = fmin(lo, x);
        hi = fmax(hi, x);
        s += x;
        s2 += x * x;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo = fmin(lo, __shfl_xor_sync(0xffffffffu, lo, o));
        hi = fmax(hi, __shfl_xor_sync(0xffffffffu, hi, o));
        s += __shfl_xor_sync(0xffffffffu, s, o);
        s2 += __shfl_xor_sync(0xffffffffu, s2, o);
    }
    if ((threadIdx.x & 31) == 0) {
        const int w = threadIdx.x >> 5;
        sm[0][w] = lo; sm[1][w] = hi; sm[2][w] = s; sm[3][w] = s2;
    }
    __syncthreads();
    if (threadIdx.x < 4) {
        const int q = threadIdx.x;
        double r = sm[q][0];
        for (int w = 1; w < kT / 32; ++w) r = q == 0 ? fmin(r, sm[q][w]) : q == 1 ? fmax(r, sm[q][w]) : r + sm[q][w];
        sc->partials[q][rg.blk()] = r;
    }
    if (publish_and_am_last(&sc->ticket, rg.nblk()) && threadIdx.x < 4) {
        const int q = threadIdx.x;
        double r = __ldcg(&sc->partials[q][0]);
        for (unsigned b = 1; b < rg.nblk(); ++b) {
            const double x = __ldcg(&sc->partials[q][b]);
            r = q == 0 ? fmin(r, x) : q == 1 ? fmax(r, x) : r + x;
        }
        out[q] = r;
    }
}

__global__ void __launch_bounds__(kT)
stats_kernel(const double* __restrict__ d, int64_t P, double* out, Scratch* sc) {
    __shared__ double sm[4][kT / 32];
    stats_body(WholeGrid{}, d, P, out, sc, sm);
}

__global__ void __launch_bounds__(kT)
stats_multi_kernel(const int64_t* __restrict__ table, int n) {
    __shared__ double sm[4][kT / 32];
    const int64_t* r = claim_row<DDMP_DISTANCE_STATS_DESC_WORDS>(table, n);
    stats_body(RowRange{}, word_ptr<const double>(r, 2), r[3], word_ptr<double>(r, 4), word_ptr<Scratch>(r, 5), sm);
}

// Evaluation of one fit's positions (float32 [V,3]) against its clean mesh, run by the row's blocks:
//   vs64 = the positions widened to float64 (the points and the vertex array of the fit's output tree);
//   mad  = mean over faces of the angle in degrees between the face normal of the positions and the clean normal.
// The face normal is the float32 arithmetic of util/mesh.py compute_face_normals on float32 positions: np.cross,
// np.linalg.norm (squares summed in axis order, sqrt) + 1e-24, division; this file is compiled without multiply-add
// contraction, so each product and difference rounds on its own as in numpy.  The angle is util/loss.py mad's float64
// clip / arccos / rad2deg; the per-block partial sums are combined by the row's last block in block order.
__global__ void __launch_bounds__(kT)
eval_multi_kernel(const int64_t* __restrict__ table, int n) {
    const int64_t* r = claim_row<DDMP_EVAL_DESC_WORDS>(table, n);
    const float* __restrict__ pos = word_ptr<const float>(r, 2);
    const int* __restrict__ faces = word_ptr<const int>(r, 3);
    const double* __restrict__ gt_fn = word_ptr<const double>(r, 4);
    double* __restrict__ vs64 = word_ptr<double>(r, 5);
    Scratch* sc = word_ptr<Scratch>(r, 7);
    const int64_t V = r[8], F = r[9];
    const RowRange rg;
    const int64_t tid = (int64_t)rg.blk() * kT + threadIdx.x, nth = (int64_t)rg.nblk() * kT;
    for (int64_t e = tid; e < 3 * V; e += nth) vs64[e] = (double)pos[e];
    double acc = 0.0;
    for (int64_t f = tid; f < F; f += nth) {
        float p[3][3];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const int64_t v = faces[3 * f + c];
#pragma unroll
            for (int a = 0; a < 3; ++a) p[c][a] = pos[3 * v + a];
        }
        const float u[3] = {p[1][0] - p[0][0], p[1][1] - p[0][1], p[1][2] - p[0][2]};
        const float w[3] = {p[2][0] - p[0][0], p[2][1] - p[0][1], p[2][2] - p[0][2]};
        const float cx = u[1] * w[2] - u[2] * w[1], cy = u[2] * w[0] - u[0] * w[2], cz = u[0] * w[1] - u[1] * w[0];
        const float len = sqrtf(cx * cx + cy * cy + cz * cz) + 1e-24f;
        const float nx = cx / len, ny = cy / len, nz = cz / len;
        double inner = (double)nx * gt_fn[3 * f] + (double)ny * gt_fn[3 * f + 1] + (double)nz * gt_fn[3 * f + 2];
        inner = inner < -1.0 ? -1.0 : (inner > 1.0 ? 1.0 : inner);
        acc += acos(inner) * (180.0 / 3.14159265358979323846);
    }
    __shared__ double sm[kT / 32];
    const double b = block_sum<kT>(acc, sm);
    if (threadIdx.x == 0) sc->partials[0][rg.blk()] = b;
    if (publish_and_am_last(&sc->ticket, rg.nblk()) && threadIdx.x == 0) {
        double t = 0.0;
        for (unsigned k = 0; k < rg.nblk(); ++k) t += __ldcg(&sc->partials[0][k]);
        *word_ptr<double>(r, 6) = t / (double)F;
    }
}

// ---- area-weighted surface samples and the normal angle across a correspondence (DESIGN.md §4.9) ----------------
// w_f = |(b-a) x (c-a)| (twice the area), float64, the cross product in tri_d2's component order, squares summed in
// axis order.  q_f = rint(w_f / w_max * 2^32) as int64 (0 where that is not positive, NaN included) and P_f its
// inclusive prefix.  Integer sums are exact in any order, so the prefix does not depend on the block partition.
constexpr int kScanItems = 4;                    // consecutive faces per thread in the prefix kernels
constexpr int kScanTile = kT * kScanItems;       // faces per block
constexpr uint64_t kGolden = 0x9E3779B97F4A7C15ull;

__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t z) {   // the output function of splitmix64
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__device__ __forceinline__ V3 cross3(V3 u, V3 w) {
    return {u.y * w.z - u.z * w.y, u.z * w.x - u.x * w.z, u.x * w.y - u.y * w.x};
}

__device__ __forceinline__ V3 face_cross(const double* __restrict__ vs, const int* __restrict__ faces, int64_t f) {
    const V3 a = load3(vs, __ldg(faces + 3 * f));
    return cross3(sub(load3(vs, __ldg(faces + 3 * f + 1)), a), sub(load3(vs, __ldg(faces + 3 * f + 2)), a));
}

__device__ __forceinline__ double face_weight(const double* __restrict__ vs, const int* __restrict__ faces, int64_t f) {
    const V3 n = face_cross(vs, faces, f);
    return sqrt(dot(n, n));
}

// exclusive prefix of v over the block's threads in thread order; total = the block's sum
__device__ __forceinline__ long long block_excl_scan(long long v, long long& total) {
    __shared__ long long warp_total[kT / 32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    long long incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += y;
    }
    if (lane == 31) warp_total[w] = incl;
    __syncthreads();
    long long off = 0;
    total = 0;
#pragma unroll
    for (int k = 0; k < kT / 32; ++k) {
        const long long t = warp_total[k];
        if (k < w) off += t;
        total += t;
    }
    return off + incl - v;
}

// *wmax = bits of max_f w_f (zero on entry; non-negative doubles order like their bit patterns)
__global__ void __launch_bounds__(kT)
weight_max_kernel(const double* __restrict__ vs, const int* __restrict__ faces, int64_t F,
                  unsigned long long* wmax) {
    double m = 0.0;
    for (int64_t f = (int64_t)blockIdx.x * kT + threadIdx.x; f < F; f += (int64_t)gridDim.x * kT)
        m = fmax(m, face_weight(vs, faces, f));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.0) atomicMax(wmax, (unsigned long long)__double_as_longlong(m));
}

// prefix[f] = q_f; tile_sum[block] = the sum of the block's q_f
__global__ void __launch_bounds__(kT)
weight_quant_kernel(const double* __restrict__ vs, const int* __restrict__ faces, int64_t F,
                    const unsigned long long* __restrict__ wmax, int64_t* __restrict__ prefix,
                    int64_t* __restrict__ tile_sum) {
    const double wm = __longlong_as_double((long long)*wmax);
    const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
    long long s = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
        if (base + k >= F) break;
        const double x = rint(face_weight(vs, faces, base + k) / wm * 4294967296.0);
        const long long q = x > 0.0 ? (long long)x : 0;
        prefix[base + k] = q;
        s += q;
    }
    long long total;
    block_excl_scan(s, total);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = total;
}

// tile_sum[0..nb) -> its exclusive prefix, one block; thread t scans the contiguous run [t*per, (t+1)*per)
__global__ void __launch_bounds__(kT)
tile_scan_kernel(int64_t* __restrict__ tile_sum, int64_t nb) {
    const int64_t per = (nb + kT - 1) / kT, lo = (int64_t)threadIdx.x * per, hi = lo + per < nb ? lo + per : nb;
    long long s = 0;
    for (int64_t k = lo; k < hi; ++k) s += tile_sum[k];
    long long total;
    long long run = block_excl_scan(s, total);
    for (int64_t k = lo; k < hi; ++k) {
        const long long x = tile_sum[k];
        tile_sum[k] = run;
        run += x;
    }
}

// prefix[f] = q_f -> P_f, the block's inclusive scan plus the tiles before it
__global__ void __launch_bounds__(kT)
prefix_apply_kernel(int64_t* __restrict__ prefix, const int64_t* __restrict__ tile_off, int64_t F) {
    const int64_t base = (int64_t)blockIdx.x * kScanTile + (int64_t)threadIdx.x * kScanItems;
    long long q[kScanItems], s = 0;
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
        q[k] = base + k < F ? prefix[base + k] : 0;
        s += q[k];
    }
    long long total;
    long long run = block_excl_scan(s, total) + tile_off[blockIdx.x];
#pragma unroll
    for (int k = 0; k < kScanItems; ++k) {
        run += q[k];
        if (base + k < F) prefix[base + k] = run;
    }
}

// Sample i: words k = 0, 1, 2 are splitmix64(key + (3i + k + 1) * golden); u0 = word 0 >> 32, r = (word >> 11) * 2^-53.
// Target T = ((i * 2^32 + u0) * Q) div (n * 2^32) < Q, face = the first f with P_f > T (a face with q_f = 0 is never
// first), point = (1 - s) a + s (1 - r2) b + s r2 c with s = sqrt(r1), per component ((wa a + wb b) + wc c).
__global__ void __launch_bounds__(kT)
sample_kernel(const double* __restrict__ vs, const int* __restrict__ faces, const int64_t* __restrict__ prefix,
              int64_t F, int64_t n, uint64_t key, double* __restrict__ pts, int* __restrict__ face) {
    const int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x;
    if (i >= n) return;
    const uint64_t Q = (uint64_t)__ldg(prefix + F - 1);
    const uint64_t w0 = key + (uint64_t)(3 * i + 1) * kGolden;
    const uint64_t u0 = splitmix64(w0) >> 32;
    // s = sqrt(r1) first: sqrt's slow path is a called routine, and taken here no value lives across the call (taken
    // after the search, it costs a spill)
    const double s = sqrt((double)(splitmix64(w0 + kGolden) >> 11) * 0x1p-53);
    const double r2 = (double)(splitmix64(w0 + 2 * kGolden) >> 11) * 0x1p-53;
    // T = ((i * 2^32 + u0) * Q) div (n * 2^32): the product is below 2^125
    const unsigned __int128 x = (unsigned __int128)(((uint64_t)i << 32) | u0);
    const uint64_t T = (uint64_t)(x * Q / ((unsigned __int128)(uint64_t)n << 32));
    int64_t lo = 0, hi = F - 1;
    while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if ((uint64_t)__ldg(prefix + mid) > T) hi = mid;
        else lo = mid + 1;
    }
    const V3 a = load3(vs, __ldg(faces + 3 * lo)), b = load3(vs, __ldg(faces + 3 * lo + 1)),
             c = load3(vs, __ldg(faces + 3 * lo + 2));
    const double wa = 1.0 - s, wb = s * (1.0 - r2), wc = s * r2;
    pts[3 * i] = (wa * a.x + wb * b.x) + wc * c.x;
    pts[3 * i + 1] = (wa * a.y + wb * b.y) + wc * c.y;
    pts[3 * i + 2] = (wa * a.z + wb * b.z) + wc * c.z;
    face[i] = (int)lo;
}

// deg[i] = rad2deg(arccos(clip(n_A(fa[i]) . n_B(fb[i]), -1, 1))), n = cross / (|cross| + 1e-24) as
// Mesh.compute_face_normals computes it in float64
__device__ __forceinline__ V3 unit_normal(const double* __restrict__ vs, const int* __restrict__ faces, int64_t f) {
    const V3 n = face_cross(vs, faces, f);
    const double len = sqrt(dot(n, n)) + 1e-24;
    return {n.x / len, n.y / len, n.z / len};
}

__global__ void __launch_bounds__(kT)
normal_angle_kernel(const double* __restrict__ vs_a, const int* __restrict__ faces_a, const int* __restrict__ fa,
                    const double* __restrict__ vs_b, const int* __restrict__ faces_b, const int* __restrict__ fb,
                    int64_t n, double* __restrict__ deg) {
    const int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x;
    if (i >= n) return;
    const V3 na = unit_normal(vs_a, faces_a, __ldg(fa + i)), nb = unit_normal(vs_b, faces_b, __ldg(fb + i));
    double c = dot(na, nb);
    c = c < -1.0 ? -1.0 : (c > 1.0 ? 1.0 : c);
    deg[i] = acos(c) * (180.0 / 3.14159265358979323846);
}

}  // namespace dist
}  // namespace ddmp

extern "C" {

int64_t ddmp_distance_scratch_bytes(void) { return (int64_t)sizeof(ddmp::dist::Scratch); }

int ddmp_bvh_keys(const double* vs, const int32_t* faces, const double* bbox6, int64_t* keys, int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(vs && faces && bbox6 && keys && F > 0, "bvh_keys: bad arguments");
    dist::keys_kernel<<<(unsigned)ceil_div(F, dist::kT), dist::kT, 0, as_stream(stream)>>>(vs, faces, bbox6, keys, F);
    return check_launch("bvh_keys");
}

int ddmp_bvh_build(const double* vs, const int32_t* faces, const int64_t* sorted_keys, const int64_t* order,
                   void* nodes, int32_t* leaves, int32_t* parent, int32_t* counters, int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(vs && faces && sorted_keys && order && nodes && leaves && parent && counters && F > 0 &&
                     F < ((int64_t)1 << 30),
                 "bvh_build: bad arguments");
    DDMP_REQUIRE(((uintptr_t)nodes & 63) == 0 && ((uintptr_t)leaves & 15) == 0, "bvh_build: nodes / leaves misaligned");
    const cudaStream_t st = as_stream(stream);
    const unsigned g = (unsigned)ceil_div(F, dist::kT);
    dist::topology_kernel<<<g, dist::kT, 0, st>>>(sorted_keys, order, faces, (dist::Node*)nodes, (int4*)leaves, parent, F);
    int rc = check_launch("bvh_build topology");
    if (rc != 0 || F == 1) return rc;
    dist::refit_kernel<<<g, dist::kT, 0, st>>>(vs, (const int4*)leaves, (dist::Node*)nodes, parent,
                                               (unsigned*)counters, F);
    return check_launch("bvh_build refit");
}

int ddmp_point_mesh_distance(const double* points, int64_t P, const double* vs, const void* nodes,
                             const int32_t* leaves, int64_t F, double* dist, int32_t* face, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(points && vs && nodes && leaves && dist && face && P > 0 && F > 0, "point_mesh_distance: bad arguments");
    dist::query_kernel<<<(unsigned)ceil_div(P, dist::kT), dist::kT, 0, as_stream(stream)>>>(
        points, P, vs, (const dist::Node*)nodes, (const int4*)leaves, F, dist, face);
    return check_launch("point_mesh_distance");
}

int ddmp_point_mesh_distance_exhaustive(const double* points, int64_t P, const double* vs, const int32_t* faces,
                                        int64_t F, double* dist, int32_t* face, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(points && vs && faces && dist && face && P > 0 && F > 0, "point_mesh_distance_exhaustive: bad arguments");
    dist::exhaustive_kernel<<<(unsigned)ceil_div(P, dist::kT), dist::kT, 0, as_stream(stream)>>>(points, P, vs, faces,
                                                                                                  F, dist, face);
    return check_launch("point_mesh_distance_exhaustive");
}

int ddmp_distance_stats(const double* dist, int64_t P, double* out, void* scratch, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(dist && out && scratch && P > 0, "distance_stats: bad arguments");
    dist::stats_kernel<<<dist::grid_for(P), dist::kT, 0, as_stream(stream)>>>(dist, P, out, (dist::Scratch*)scratch);
    return check_launch("distance_stats");
}

int ddmp_bvh_refit(const double* vs, const int32_t* leaves, void* nodes, const int32_t* parent, int32_t* counters,
                   int64_t F, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(vs && leaves && nodes && parent && counters && F > 0 && F < ((int64_t)1 << 30),
                 "bvh_refit: bad arguments");
    DDMP_REQUIRE(((uintptr_t)nodes & 63) == 0 && ((uintptr_t)leaves & 15) == 0, "bvh_refit: nodes / leaves misaligned");
    if (F == 1) return DDMP_OK;   // a single leaf: no internal node holds a box
    dist::refit_kernel<<<(unsigned)ceil_div(F, dist::kT), dist::kT, 0, as_stream(stream)>>>(
        vs, (const int4*)leaves, (dist::Node*)nodes, parent, (unsigned*)counters, F);
    return check_launch("bvh_refit");
}

static int launch_multi(void (*kernel)(const int64_t*, int), const int64_t* table, int32_t n, int64_t blocks,
                        void* stream, const char* what) {
    using namespace ddmp;
    DDMP_REQUIRE(table && n > 0 && blocks > 0 && blocks < ((int64_t)1 << 31), "%s: bad arguments", what);
    kernel<<<(unsigned)blocks, dist::kT, 0, as_stream(stream)>>>(table, n);
    return check_launch(what);
}

int ddmp_bvh_refit_multi(const int64_t* table, int32_t n, int64_t blocks, void* stream) {
    return launch_multi(ddmp::dist::refit_multi_kernel, table, n, blocks, stream, "bvh_refit_multi");
}

int ddmp_point_mesh_distance_multi(const int64_t* table, int32_t n, int64_t blocks, void* stream) {
    return launch_multi(ddmp::dist::query_multi_kernel, table, n, blocks, stream, "point_mesh_distance_multi");
}

int ddmp_distance_stats_multi(const int64_t* table, int32_t n, int64_t blocks, void* stream) {
    return launch_multi(ddmp::dist::stats_multi_kernel, table, n, blocks, stream, "distance_stats_multi");
}

int ddmp_eval_mad_multi(const int64_t* table, int32_t n, int64_t blocks, void* stream) {
    return launch_multi(ddmp::dist::eval_multi_kernel, table, n, blocks, stream, "eval_mad_multi");
}

int64_t ddmp_surface_prefix_workspace_bytes(int64_t F) {
    return 8 * (1 + ddmp::ceil_div(F > 0 ? F : 1, ddmp::dist::kScanTile));
}

int ddmp_surface_prefix(const double* vs, const int32_t* faces, int64_t F, int64_t* prefix, void* workspace,
                        void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(vs && faces && prefix && workspace && F > 0 && F < ((int64_t)1 << 30), "surface_prefix: bad arguments");
    const cudaStream_t st = as_stream(stream);
    unsigned long long* wmax = (unsigned long long*)workspace;
    int64_t* tile = (int64_t*)workspace + 1;
    const unsigned nb = (unsigned)ceil_div(F, dist::kScanTile);
    DDMP_REQUIRE(cudaMemsetAsync(wmax, 0, sizeof(*wmax), st) == cudaSuccess, "surface_prefix: memset failed");
    dist::weight_max_kernel<<<dist::grid_for(F), dist::kT, 0, st>>>(vs, faces, F, wmax);
    int rc = check_launch("surface_prefix max");
    if (rc != 0) return rc;
    dist::weight_quant_kernel<<<nb, dist::kT, 0, st>>>(vs, faces, F, wmax, prefix, tile);
    if ((rc = check_launch("surface_prefix quantise")) != 0) return rc;
    dist::tile_scan_kernel<<<1, dist::kT, 0, st>>>(tile, nb);
    if ((rc = check_launch("surface_prefix tiles")) != 0) return rc;
    dist::prefix_apply_kernel<<<nb, dist::kT, 0, st>>>(prefix, tile, F);
    return check_launch("surface_prefix scan");
}

int ddmp_surface_sample(const double* vs, const int32_t* faces, const int64_t* prefix, int64_t F, int64_t n,
                        int64_t seed, int32_t side, double* points, int32_t* face, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(vs && faces && prefix && points && face && F > 0 && F < ((int64_t)1 << 30) && n > 0 &&
                     n < ((int64_t)1 << 31) && seed >= 0 && side >= 0,
                 "surface_sample: bad arguments");
    using dist::kGolden;
    using dist::splitmix64;
    const uint64_t key = splitmix64(splitmix64((uint64_t)seed + kGolden) + ((uint64_t)side + 1) * kGolden);
    dist::sample_kernel<<<(unsigned)ceil_div(n, dist::kT), dist::kT, 0, as_stream(stream)>>>(vs, faces, prefix, F, n,
                                                                                           key, points, face);
    return check_launch("surface_sample");
}

int ddmp_normal_angle(const double* vs_a, const int32_t* faces_a, const int32_t* face_a, const double* vs_b,
                      const int32_t* faces_b, const int32_t* face_b, int64_t n, double* deg, void* stream) {
    using namespace ddmp;
    DDMP_REQUIRE(vs_a && faces_a && face_a && vs_b && faces_b && face_b && deg && n > 0, "normal_angle: bad arguments");
    dist::normal_angle_kernel<<<(unsigned)ceil_div(n, dist::kT), dist::kT, 0, as_stream(stream)>>>(
        vs_a, faces_a, face_a, vs_b, faces_b, face_b, n, deg);
    return check_launch("normal_angle");
}

}  // extern "C"
