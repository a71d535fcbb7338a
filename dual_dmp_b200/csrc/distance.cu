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

// bottom-up refit, one thread per leaf; counters [F-1] are zero on entry and zero again on exit
__global__ void __launch_bounds__(kT)
refit_kernel(const double* __restrict__ vs, const int4* __restrict__ leaves, Node* nodes, const int* __restrict__ parent,
             unsigned* counters, int64_t F) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
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

__global__ void __launch_bounds__(kT)
query_kernel(const double* __restrict__ pts, int64_t P, const double* __restrict__ vs, const Node* __restrict__ nodes,
             const int4* __restrict__ leaves, int64_t F, double* __restrict__ dist, int* __restrict__ face) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
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
__global__ void __launch_bounds__(kT)
stats_kernel(const double* __restrict__ d, int64_t P, double* out, Scratch* sc) {
    __shared__ double sm[4][kT / 32];
    double lo = CUDART_INF, hi = -CUDART_INF, s = 0.0, s2 = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P; i += (int64_t)gridDim.x * blockDim.x) {
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
        sc->partials[q][blockIdx.x] = r;
    }
    if (publish_and_am_last(&sc->ticket, gridDim.x) && threadIdx.x < 4) {
        const int q = threadIdx.x;
        double r = __ldcg(&sc->partials[q][0]);
        for (unsigned b = 1; b < gridDim.x; ++b) {
            const double x = __ldcg(&sc->partials[q][b]);
            r = q == 0 ? fmin(r, x) : q == 1 ? fmax(r, x) : r + x;
        }
        out[q] = r;
    }
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

}  // extern "C"
