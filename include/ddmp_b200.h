/* libddmp_b200 — C ABI of the B200-native Dual-DMP training hot path.
 *
 * The reference (astaka-pe/Dual-DMP) is pure Python and has no FFI; every entry point below replaces a LIBRARY
 * call site of its hot path (torch_geometric.GCNConv / torch_scatter / torch.nn / torch ops).  The reference
 * location each one replaces is cited as  [ref: file:line].  The Python binding is dual_dmp_b200/_lib.py (ctypes);
 * INTEGRATION.md shows the reference-side change.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer owned by the caller (PyTorch allocates everything); the library never
 *     allocates, frees or keeps device memory, and holds no mutable global state;
 *   - tensors are contiguous row-major float32 unless stated; indices are int32; `n` rows are int64;
 *   - `stream` is a cudaStream_t (torch.cuda.current_stream().cuda_stream); all work is enqueued on it and no
 *     call synchronises the host;
 *   - return value 0 = ok, <0 = error (DDMP_ERR_*); ddmp_last_error() returns a thread-local message;
 *   - entry points are re-entrant (autograd runs backward on another thread); call ddmp_set_device() on the
 *     calling thread first when more than one GPU is visible;
 *   - results are deterministic: no floating-point atomics anywhere; reductions combine partials in a fixed
 *     order.
 */
#ifndef DDMP_B200_H
#define DDMP_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DDMP_OK 0
#define DDMP_ERR_INVALID (-1)
#define DDMP_ERR_CUDA (-2)
#define DDMP_ERR_UNSUPPORTED (-3)

#define DDMP_GEMM_AUTO 0
#define DDMP_GEMM_FFMA 1  /* fp32 FFMA kernel                                  */
#define DDMP_GEMM_TC 2    /* tcgen05 tensor cores, 3xTF32 split, fp32 accumulate */

#define DDMP_HEAD_POS 0
#define DDMP_HEAD_NORM 1

/* ---- library ------------------------------------------------------------------------------------------- */
int ddmp_version(void);
const char* ddmp_last_error(void);
int ddmp_set_device(int device);
/* number of CUDA kernels this library has launched in this process (bench.py reports the per-step count). */
int64_t ddmp_launch_count(void);
/* sm count / compute capability of the current device; fails (DDMP_ERR_CUDA) when no CUDA device is usable. */
int ddmp_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* rows covered by one partial-statistics block for channel width C (all *_partials arguments below are
 * [ddmp_num_row_blocks(n, C)][sets][C] float32). */
int ddmp_rows_per_block(int32_t C);
int64_t ddmp_num_row_blocks(int64_t n, int32_t C);
/* row block of the element-wise kernels (ddmp_bn_bwd_reduce / ddmp_bn_bwd_apply / ddmp_colsum_partials): their partials
 * are [ddmp_num_elem_blocks(n, C)][sets][C] */
int ddmp_elem_rows_per_block(int32_t C);
int64_t ddmp_num_elem_blocks(int64_t n, int32_t C);

/* ---- graph --------------------------------------------------------------------------------------------- */
/* GCN symmetric normalisation, hoisted out of the step.  CSR rows are TARGET nodes and already contain exactly
 * one self loop per node:  w[k] = deg(row)^-1/2 * deg(col[k])^-1/2, deg(i) = rowptr[i+1]-rowptr[i].
 * [ref: torch_geometric gcn_norm, recomputed 24x per step at util/networks.py:51-62,112-123] */
int ddmp_gcn_edge_weights(const int32_t* rowptr, const int32_t* col, float* w, int64_t n, void* stream);

/* ---- GCN aggregation ------------------------------------------------------------------------------------ */
/* Y[i,:] = sum_k w[k] * H[col[k],:] (+ bias).  Optional epilogue statistics: stats_partials[b][0][c] = sum of
 * Y[:,c] over row block b, [b][1][c] = sum of Y^2 (BatchNorm partials).  The same call is the backward pass
 * (A_hat is symmetric): dH = spmm(dY) with bias = stats = NULL.  C must be a multiple of 4.
 * amax_blocks (optional, [ddmp_spmm_amax_len(n,C)]): max |Y| of every (row block, channel slice) a CTA produced, the
 * `amax` input of the dense transforms that consume Y.
 * Mesh widths (32, 64, multiples of 128 up to 512) run the tile-staged kernel: the row block's own rows of H arrive in
 * shared memory by one TMA tensor copy, its (rowptr, col, w) stream by coalesced loads (csrc/spmm_tile.cu).
 * [ref: GCNConv.propagate + bias at util/networks.py:51-62,112-123; torch_scatter.scatter_add] */
int ddmp_spmm_gcn(const int32_t* rowptr, const int32_t* col, const float* w, const float* H, const float* bias,
                  float* Y, float* stats_partials, float* amax_blocks, int64_t n, int32_t C, void* stream);
/* number of floats ddmp_spmm_gcn writes to amax_blocks for this shape */
int64_t ddmp_spmm_amax_len(int64_t n, int32_t C);
/* Kernel choice of ddmp_spmm_gcn (environment DDMP_SPMM_TILE, default 225).  setting = mode | flags << 4.
 * mode: 0 = gather-only kernel for every width, 1 = tile-staged kernel for C <= 128 (where it measures faster on B200),
 * 2 = tile-staged kernel for every mesh width (A/B measurements, bit-exactness test between the two kernels).
 * flags: 2 = streaming stores of Y in the gather kernel; 4 = forward flavour (bias + BatchNorm moments) at C = 512 with the
 * per-warp Welford state in tensor memory instead of shared memory (bitwise-equal results); 8 = the same at C = 256.
 * Returns the previous setting. */
int ddmp_spmm_use_tile_kernel(int mode);

/* Backward aggregation fused with ddmp_bn_bwd_apply:  dH = A_hat * dY  with dY recomputed on the fly from the gathered
 * rows of gX and Y (dY is never materialised); optional colsum_partials[b][0][c] = column sums of dY (conv bias
 * gradient).  Symmetric graphs only (the CSR is used as its own transpose); C in {32,64,128,256,512}. */
int ddmp_spmm_bn_bwd(const int32_t* rowptr, const int32_t* col, const float* w, const float* gX, const float* Y,
                     const float* mean, const float* rstd, const float* scale, const float* shift, const float* c1,
                     const float* c2, float slope, float* dH, float* colsum_partials, int64_t n, int32_t C,
                     void* stream);

/* The same fusion on the tile-staged kernel (csrc/spmm_tile.cu): the row block's own rows of gX and Y arrive by two TMA
 * tensor copies, dY of those rows is formed once in shared memory and gathered from there; only references that leave
 * the block recompute dY from global rows.  Per layer the backward pass then moves 3 tensor passes (+ halo) instead of 5
 * (ddmp_bn_bwd_apply: read gX, Y, write dY; ddmp_spmm_gcn: read dY, write dH).  colsum_partials (optional):
 * [ddmp_spmm_bn_bwd_tile_blocks(n,C)][C] column sums of dY per row block (conv-bias gradient); amax_blocks (optional):
 * [ddmp_spmm_bn_bwd_tile_amax_len(n,C)] max |dH| per CTA.  n may be smaller than the row count of gX / Y (partitioned
 * mode: [owned | halo] rows, only owned rows are produced).  Symmetric graphs only.
 * [ref: autograd of nn.BatchNorm1d + nn.LeakyReLU + GCNConv.propagate, util/networks.py:51-62,112-123] */
int ddmp_spmm_bn_bwd_tile(const int32_t* rowptr, const int32_t* col, const float* w, const float* gX, const float* Y,
                          const float* mean, const float* rstd, const float* scale, const float* shift,
                          const float* c1, const float* c2, float slope, float* dH, float* colsum_partials,
                          float* amax_blocks, int64_t n, int32_t C, void* stream);
int64_t ddmp_spmm_bn_bwd_tile_blocks(int64_t n, int32_t C);
int64_t ddmp_spmm_bn_bwd_tile_amax_len(int64_t n, int32_t C);

/* ---- BatchNorm1d (training mode) + LeakyReLU ------------------------------------------------------------ */
/* partials [nblk][2][C] = per row block (sum of y, M2 = sum of (y - block mean)^2), as ddmp_spmm_gcn's epilogue emits
 * them (Welford per thread, Chan merge per block; nblk = ddmp_num_row_blocks(n, C)) -> batch mean / biased var, combined
 * in float64 in block order; rstd = 1/sqrt(var+eps); scale = gamma*rstd; shift = beta - mean*scale; running stats
 * updated in place when non-NULL (momentum, unbiased var).
 * The normalise + LeakyReLU itself is applied lazily by the consumer (GEMM / head prologue).
 * bound (optional, [C]): |gamma|*sqrt(n-1)+|beta| >= |scale*y+shift| for every row of the batch (the `amax` input
 * of the dense transforms).
 * [ref: nn.BatchNorm1d at util/networks.py:31-42,51-62] */
int ddmp_bn_stats_finalize(const float* partials, int64_t nblk, int64_t n, int32_t C, const float* gamma,
                           const float* beta, float eps, float momentum, float* running_mean, float* running_var,
                           float* mean, float* rstd, float* scale, float* shift, float* bound, void* stream);
/* eval mode: the [mean, rstd, scale, shift] table from the running statistics. [ref: nn.BatchNorm1d.eval()] */
int ddmp_bn_eval_stats(const float* running_mean, const float* running_var, const float* gamma, const float* beta,
                       float eps, int32_t C, float* mean, float* rstd, float* scale, float* shift, void* stream);
/* Partitioned mode: this rank's (sum y, sum y^2) per channel in float64 [2][C] from the same partials (all-reduced over
 * the ranks, then ddmp_bn_stats_finalize_sums with the global row count). */
int ddmp_bn_stats_rank_sums(const float* partials, int64_t nblk, int64_t n, int32_t C, double* sums, void* stream);
int ddmp_bn_stats_finalize_sums(const double* sums, int64_t n, int32_t C, const float* gamma, const float* beta,
                                float eps, float momentum, float* running_mean, float* running_var, float* mean,
                                float* rstd, float* scale, float* shift, float* bound, void* stream);
/* Backward of LeakyReLU(BN(Y)) given gX = dL/d(activated output):  gZ = gX * lrelu'(scale*Y+shift),
 * xhat = (Y-mean)*rstd;  partials[b][0][c] = sum gZ, [b][1][c] = sum gZ*xhat. */
int ddmp_bn_bwd_reduce(const float* gX, const float* Y, const float* mean, const float* rstd, const float* scale,
                       const float* shift, float slope, float* partials, int64_t n, int32_t C, void* stream);
/* dgamma = sum gZ*xhat, dbeta = sum gZ, c1 = dbeta/n, c2 = dgamma/n. */
int ddmp_bn_bwd_finalize(const float* partials, int64_t nblk, int64_t n, int32_t C, float* dgamma, float* dbeta,
                         float* c1, float* c2, void* stream);
/* dY = scale * (gZ - c1 - xhat*c2);  optional colsum_partials[b][0][c] = sum of dY (the conv bias gradient). */
int ddmp_bn_bwd_apply(const float* gX, const float* Y, const float* mean, const float* rstd, const float* scale,
                      const float* shift, float slope, const float* c1, const float* c2, float* dY,
                      float* colsum_partials, int64_t n, int32_t C, void* stream);
/* out[s][c] = sum_b partials[b][s][c]  (fixed order, float64 accumulate). */
int ddmp_colsum_finalize(const float* partials, int64_t nblk, int32_t sets, int32_t C, float* out, void* stream);
/* partials[b][0][c] = sum over row block b of X[:,c]  (bias gradients of the heads). */
int ddmp_colsum_partials(const float* X, float* partials, int64_t n, int32_t C, void* stream);

/* dst[i,:] = src[idx[i],:], C a multiple of 4: packs the boundary rows a peer rank needs before the NCCL exchange
 * of the partitioned mode (SURVEY.md §8e mode B: per-layer halo exchange). */
int ddmp_gather_rows(const float* src, const int32_t* idx, float* dst, int64_t m, int32_t C, void* stream);

/* ---- dense feature transform ------------------------------------------------------------------------------ */
/* H[n,Cout] = act(X)[n,Cin] * W[Cout,Cin]^T.   act(x)[i,k] = lrelu(scale[k]*X[r,k]+shift[k]) when scale != NULL
 * (the previous layer's BatchNorm+LeakyReLU applied on load), r = row_map[i] when row_map != NULL (first-layer
 * gather from the caller's numbering into the space-filling-curve order).
 * [ref: GCNConv.lin at util/networks.py:51-62 — cuBLAS SGEMM] */
int ddmp_gemm_xw(const float* X, const int32_t* row_map, const float* scale, const float* shift, float slope,
                 const float* W, float* H, void* workspace, int64_t workspace_bytes, int64_t n, int32_t Cin,
                 int32_t Cout, const float* amax, int64_t amax_len, int backend, void* stream);
/* `amax` (optional, device, amax_len floats): max |amax[i]| is an upper bound of the magnitude of the left operand
 * (act(X) resp. dH).  With a bound the tensor-core path multiplies with three fp16 MMAs per product (operands
 * scaled by powers of two into the fp16 range, fp32 accumulation, accuracy of an fp32 product sum) at twice the
 * rate of the bound-free 3xTF32 kernels; results are wrong only if the bound is violated by more than 2x. */
/* scratch the tensor-core path of gemm_xw / gemm_dx needs for the pre-split, pre-swizzled weight image (0 when the
 * shape runs on the FFMA kernel; with workspace == NULL the FFMA kernel is used). */
int64_t ddmp_gemm_workspace_bytes(int64_t n, int32_t Cin, int32_t Cout);
/* A/B switches of the fp16-split tcgen05 kernels behind ddmp_gemm_xw / ddmp_gemm_dx (environment DDMP_TC_F16_FLAGS,
 * default 0): bit 0 = prefetch the next tile's rows into L2, bit 3 = unstaged epilogue, bit 4 = staged ld.shared +
 * st.global epilogue instead of TMA tensor stores.  flags < 0 only queries.  Returns the previous value. */
int ddmp_gemm_tc_flags(int flags);
/* gX[n,Cin] = dH[n,Cout] * W[Cout,Cin]. */
int ddmp_gemm_dx(const float* dH, const float* W, float* gX, void* workspace, int64_t workspace_bytes, int64_t n,
                 int32_t Cin, int32_t Cout, const float* amax, int64_t amax_len, int backend, void* stream);
/* dW[Cout,Cin] = dH[n,Cout]^T * act(X)[n,Cin]; deterministic split-K over rows through `workspace`.
 * amax_dh / amax_x (optional, both or neither): bounds of |dH| and |act(X)| as for ddmp_gemm_xw. */
int64_t ddmp_gemm_dw_workspace_bytes(int64_t n, int32_t Cin, int32_t Cout);
int ddmp_gemm_dw(const float* dH, const float* X, const int32_t* row_map, const float* scale, const float* shift,
                 float slope, float* dW, void* workspace, int64_t workspace_bytes, int64_t n, int32_t Cin,
                 int32_t Cout, const float* amax_dh, int64_t amax_dh_len, const float* amax_x, int64_t amax_x_len,
                 int backend, void* stream);

/* ---- network heads (32 -> 16 -> 3) ------------------------------------------------------------------------ */
/* x = lrelu(scale*Y12+shift); h = lrelu(W1 x + b1); o = W2 h + b2;
 * POS : out[p] = x_pos[p] + o                      [ref: util/networks.py:64-67]
 * NORM: t = tanh(o); out[p] = t / (||t|| + 1e-12)   [ref: util/networks.py:125-129]
 * p = perm[i] (row i of the reordered graph is node perm[i] of the caller) or i when perm == NULL.
 * h_save [n,16] and t_save [n,4] = (t, ||t||) (NORM only) are kept for the backward pass. */
int ddmp_head_fwd(int kind, const float* Y12, const float* scale, const float* shift, float slope, const float* W1,
                  const float* b1, const float* W2, const float* b2, const int32_t* perm, const float* x_pos,
                  float* out, float* h_save, float* t_save, int64_t n, void* stream);
/* g_out [n,3] in the caller's numbering ->  go [n,4] = (dL/do, 0), gh [n,16] = dL/d(pre-activation of linear1),
 * gX12 [n,32] = dL/dx (input of linear1, i.e. the activated trunk output); all three in reordered rows. */
int ddmp_head_bwd(int kind, const float* g_out, const int32_t* perm, const float* W1, const float* W2,
                  const float* h_save, const float* t_save, float slope, float* go, float* gh, float* gX12,
                  int64_t n, void* stream);

/* ---- losses ---------------------------------------------------------------------------------------------- */
/* Scalar results are written to device memory; `scratch` is a caller-provided zero-initialised buffer of at
 * least ddmp_loss_scratch_bytes() bytes that the kernels leave zeroed again (ticket counter + partials). */
int64_t ddmp_loss_scratch_bytes(void);
/* sqrt(mean_v ||pos-target||^2 + 1e-6), float64 like the reference's promotion. [ref: util/loss.py:16-35] */
int ddmp_loss_pos_rec_fwd(const float* pos, const double* target, double* loss, void* scratch, int64_t V,
                          void* stream);
int ddmp_loss_pos_rec_bwd(const float* pos, const double* target, const double* loss, const double* gout,
                          float* gpos, int64_t V, void* stream);
/* uniform Laplacian: d_i = pos_i - mean_{j in N(i)} pos_j; sqrt(mean ||d||^2 + 1e-12).  (rowptr, col) is the
 * unweighted vertex adjacency WITHOUT self loops.  d [V,3] is kept for backward. [ref: util/loss.py:37-53] */
int ddmp_loss_lap_fwd(const float* pos, const int32_t* rowptr, const int32_t* col, float* d, float* loss,
                      void* scratch, int64_t V, void* stream);
int ddmp_loss_lap_bwd(const float* d, const int32_t* rowptr, const int32_t* col, const float* loss,
                      const float* gout, float* gpos, int64_t V, void* stream);
/* mean_f ||norm - target||_1, float64. [ref: util/loss.py:55-84 "l1mae"] */
int ddmp_loss_norm_rec_fwd(const float* nrm, const double* target, double* loss, void* scratch, int64_t F,
                           void* stream);
int ddmp_loss_norm_rec_bwd(const float* nrm, const double* target, const double* gout, float* gnrm, int64_t F,
                           void* stream);
/* sum_f sum_k |(p_fk - c_f).n_f| / V.  Backward: gnrm per face; gpos through the corner CSR (corner_ptr [V+1],
 * corner_slot [3F] = 3*f+k of every corner incident to a vertex), deterministic gather instead of scatter-add;
 * face_tmp is [F,9] scratch. [ref: util/loss.py:140-160 "mae"] */
int ddmp_loss_pos_norm_fwd(const float* pos, const float* nrm, const int32_t* faces, float* loss, void* scratch,
                           int64_t V, int64_t F, void* stream);
int ddmp_loss_pos_norm_bwd(const float* pos, const float* nrm, const int32_t* faces, const int32_t* corner_ptr,
                           const int32_t* corner_slot, const float* gout, float* face_tmp, float* gpos,
                           float* gnrm, int64_t V, int64_t F, void* stream);
/* Bilateral normal filtering loss [ref: util/loss.py:86-138 "l1mae"].
 * setup: from (detached) pos: centroid / area / centroid distance per slot, global sigma_c, then
 *        wca[f,s] = exp(-dist/(2 sigma_c^2)) * area[f2f[f,s]] * (f2f[f,s] != -1); a -1 slot reads face F-1
 *        (Python negative indexing) and still counts in sigma_c, exactly like the reference (:99-103).
 * iter_fwd: n_out = normalise(sum_s wca*exp(-||n_j-n_i||^2/(2*0.3^2)) n_j)
 * loss: mean_f ||n_L - n_0||_1 ; iter_bwd: gradient through one iteration via the reverse-slot map rslot[f,s]
 *        (position of f in the row of its s-th neighbour), no atomics; msg is [F,9] scratch. */
int ddmp_bnf_setup(const float* pos, const int32_t* faces, const int32_t* f2f, float* fc, float* fa, float* wca,
                   float* sigma_c, void* scratch, int64_t F, void* stream);
int ddmp_bnf_iter_fwd(const float* n_in, const int32_t* f2f, const float* wca, float* n_out, int64_t F,
                      void* stream);
int ddmp_bnf_loss_fwd(const float* n_last, const float* n_first, float* loss, void* scratch, int64_t F,
                      void* stream);
/* g_last = gout*sign(n_last-n_first)/F ; g_first_direct = -g_last */
int ddmp_bnf_loss_bwd(const float* n_last, const float* n_first, const float* gout, float* g_last, int64_t F,
                      void* stream);
/* g_in = d(loss)/d(n_in) through one iteration, minus g_sub when g_sub != NULL (the direct -sign/F term of the
 * loss with respect to the unfiltered normals, folded into the first iteration's backward). */
int ddmp_bnf_iter_bwd(const float* n_in, const float* g_out, const int32_t* f2f, const int32_t* rslot,
                      const float* wca, const float* g_sub, float* msg, float* g_in, int64_t F, void* stream);

/* ---- geometry / evaluation ---------------------------------------------------------------------------------- */
/* fn = cross(p1-p0, p2-p0) / ||.||  (no epsilon) [ref: util/models.py:5-10]; backward through the corner CSR. */
int ddmp_face_normals_fwd(const float* pos, const int32_t* faces, float* fn, int64_t F, void* stream);
int ddmp_face_normals_bwd(const float* pos, const int32_t* faces, const int32_t* corner_ptr,
                          const int32_t* corner_slot, const float* gfn, float* face_tmp, float* gpos, int64_t V,
                          int64_t F, void* stream);
/* Point-to-surface distance (csrc/distance.cu), float64.  For a query point p and a target mesh (vs [V,3], faces [F,3]):
 *   dist(p) = min over faces f of |p - closest_point(p, triangle f)|  (exact Euclidean distance, no cutoff),
 *   face(p) = the face attaining it, the lowest face id on an exact tie.
 * A zero-area face (collinear or coincident corners) is the segment or point it spans; no input gives NaN or inf.
 * Linear BVH (Karras 2012): 64-byte internal nodes holding both children's float32 boxes (rounded outward) and ids.
 * The BVH query returns bit for bit the distance and face id of ddmp_point_mesh_distance_exhaustive.
 * [ref: util/loss.py:279-284 distance_from_reference_mesh and check/hausdorff_checker.py, both pymeshlab] */
/* keys [F] = 63-bit Morton code of each face centroid, 21 bits per axis quantised in bbox6 (ddmp_prep_bbox of vs),
 * to be sorted stably by the caller -> sorted_keys, order (order[k] = face at sorted position k). */
int ddmp_bvh_keys(const double* vs, const int32_t* faces, const double* bbox6, int64_t* keys, int64_t F, void* stream);
/* nodes: max(F-1,1) x 64 bytes, 64-byte aligned; leaves [F][4] int32 = (v0, v1, v2, face) in sorted order; parent
 * [2F-1] int32 scratch; counters [max(F-1,1)] int32, zero on entry and left zeroed.  F < 2^30. */
int ddmp_bvh_build(const double* vs, const int32_t* faces, const int64_t* sorted_keys, const int64_t* order,
                   void* nodes, int32_t* leaves, int32_t* parent, int32_t* counters, int64_t F, void* stream);
/* points [P,3]; dist [P] float64, face [P] int32 (ids of the caller's face numbering) */
int ddmp_point_mesh_distance(const double* points, int64_t P, const double* vs, const void* nodes,
                             const int32_t* leaves, int64_t F, double* dist, int32_t* face, void* stream);
/* the same outputs by scanning every face with the same leaf routine (reference for tests and benchmarks) */
int ddmp_point_mesh_distance_exhaustive(const double* points, int64_t P, const double* vs, const int32_t* faces,
                                        int64_t F, double* dist, int32_t* face, void* stream);
/* out [4] = (min, max, sum, sum of squares) of dist [P], float64, fixed combination order; scratch: zeroed buffer of
 * ddmp_distance_scratch_bytes() bytes, left zeroed. */
int64_t ddmp_distance_scratch_bytes(void);
int ddmp_distance_stats(const double* dist, int64_t P, double* out, void* scratch, void* stream);
/* ---- partitioned mode: BatchNorm reductions over NVLink peer memory (csrc/comm.cu) ------------------------- */
/* Every rank owns one exchange buffer (ddmp_comm_buffer_bytes() bytes, allocated and zeroed by ddmp_comm_alloc) that all
 * peers of the box map through CUDA IPC (ddmp_comm_ipc_handle on the owner -> 64 opaque bytes -> ddmp_comm_ipc_open on
 * each peer).  peer_buffers is a HOST array of `world` device pointers, entry r = rank r's buffer as mapped in this
 * process (own entry = the local pointer).  seq = 1, 2, 3, ... must advance by one per call, identically on all ranks.
 * ddmp_bn_stats_finalize_peer = this rank's float64 reduction of the aggregation partials + one-shot all-reduce through
 * the peers' buffers (P2P stores, sequence flags, sum in rank order: bit-identical on every rank) + the BatchNorm table
 * for the GLOBAL batch of n_global rows, in ONE kernel; replaces ddmp_bn_stats_rank_sums + an NCCL all-reduce +
 * ddmp_bn_stats_finalize_sums.  ddmp_bn_bwd_finalize_peer does the same for the two BatchNorm-backward sums
 * (partials [nblk][2][C] of ddmp_bn_bwd_reduce).  Waits are bounded; ddmp_comm_error reports a peer that never arrived.
 * [ref: nn.BatchNorm1d over the whole batch, util/networks.py:31-42,51-62; no counterpart in the reference (single GPU)] */
int64_t ddmp_comm_buffer_bytes(void);
int ddmp_comm_alloc(void** out);
int ddmp_comm_free(void* p);
int ddmp_comm_ipc_handle(void* p, void* handle64);
int ddmp_comm_ipc_open(const void* handle64, void** out);
int ddmp_comm_ipc_close(void* p);
int ddmp_comm_error(const void* p, int32_t* out);
int ddmp_bn_stats_finalize_peer(const float* partials, int64_t nblk, int64_t n_local, int32_t C,
                                const void* const* peer_buffers, int32_t rank, int32_t world, int64_t seq,
                                int64_t n_global, const float* gamma, const float* beta, float eps, float momentum,
                                float* running_mean, float* running_var, float* mean, float* rstd, float* scale,
                                float* shift, float* bound, void* stream);
int ddmp_bn_bwd_finalize_peer(const float* partials, int64_t nblk, int32_t C, const void* const* peer_buffers,
                              int32_t rank, int32_t world, int64_t seq, int64_t n_global, float* dgamma, float* dbeta,
                              float* c1, float* c2, void* stream);

/* ---- mesh preprocessing on the device, float64 (SURVEY.md §8f N3) ------------------------------------------ */
/* Conventions of the reference's offline tools, which need pymeshlab: uniform Laplacian smoothing x30 for the *_smooth
 * mesh, Gaussian noise along the vertex normal, unit-box normalisation, rescale to mean edge length 1.
 * (rowptr, col) = unweighted vertex adjacency CSR without self loops; (corner_ptr, corner_slot) = corner CSR.
 * [ref: preprocess/noisemaker.py:25-42, preprocess/preprocess.py:22-28,68-72; util/mesh.py:87-107] */
int64_t ddmp_prep_scratch_bytes(void);
/* one Jacobi sweep  x_i <- (x_i + sum_{j in N(i)} x_j) / (deg_i + 1) */
int ddmp_prep_smooth_sweep(const double* pos_in, const int32_t* rowptr, const int32_t* col, double* pos_out, int64_t V,
                           void* stream);
/* float64 face normals (n / (|n| + 1e-24)), areas, centroids; any output may be NULL */
int ddmp_prep_face_geometry(const double* vs, const int32_t* faces, double* fn, double* fa, double* fc, int64_t F,
                            void* stream);
/* vn = normalise(sum of incident face normals); all-zero rows stay zero */
int ddmp_prep_vertex_normals(const double* fn, const int32_t* corner_ptr, const int32_t* corner_slot, double* vn,
                             int64_t V, void* stream);
/* out[v,:] = (a[v,:] + b[v,:]*t[v] + shift[:]) * scale;  b/t and shift optional (noise along the normal; recentre+rescale) */
int ddmp_prep_affine_rows(const double* a, const double* b, const double* t, const double* shift, double scale,
                          double* out, int64_t V, void* stream);
/* sum over edges [E,2] of |v_a - v_b| (mean edge length = out / E) */
int ddmp_prep_edge_length_sum(const double* vs, const int32_t* edges, double* out, void* scratch, int64_t E,
                              void* stream);
/* out6 = (min x, min y, min z, max x, max y, max z) */
int ddmp_prep_bbox(const double* vs, double* out6, void* scratch, int64_t V, void* stream);

/* The whole loss phase of one iteration as ONE cooperative launch (csrc/loss_fused.cu): the five losses with the
 * reference's weights, total = k1*pos_rec + k2*laplacian + k3*norm_rec + k4*(bnf*bnf_scale) + k5*pos_norm, and its
 * gradients gpos [V,3] = d total / d pos, gnrm [F,3] = d total / d norm (for an upstream gradient of 1).  bnf_scale is
 * the reference's `loss_norm2 * 0.0` while epoch <= 100 (1.0 afterwards): the term is still evaluated and its
 * gradient multiplied by it.  losses [6] (float64): the five terms as the reference computes them (float64 for
 * pos_rec / norm_rec, float32 values for the others) and the weighted total.  Same arithmetic as the stand-alone
 * kernels above; phases that need a mesh-wide scalar or neighbour values of the previous phase are separated by
 * grid-wide barriers instead of kernel boundaries.  rslot [F,3]: position of face f in the f2f row of its neighbour.
 * workspace: ddmp_dual_loss_workspace_bytes(V, F, loop) bytes, contents irrelevant on entry.
 * [ref: main.py:94-106 (loss calls, warm-up switch, weighted sum) + loss.backward() at :107; util/loss.py:16-160] */
int64_t ddmp_dual_loss_workspace_bytes(int64_t V, int64_t F, int32_t loop);
int ddmp_dual_loss(const float* pos, const float* nrm, const double* tgt_vs, const double* tgt_fn,
                   const int32_t* faces, const int32_t* f2f, const int32_t* rslot, const int32_t* lap_rowptr,
                   const int32_t* lap_col, const int32_t* corner_ptr, const int32_t* corner_slot, float k1, float k2,
                   float k3, float k4, float k5, float bnf_scale, int32_t loop, void* workspace,
                   int64_t workspace_bytes, float* gpos, float* gnrm, double* losses, int64_t V, int64_t F,
                   void* stream);
/* Phase trace of the most recent ddmp_dual_loss launch on the current device: 13 %globaltimer stamps (ns) taken by block
 * 0 at the phase boundaries (start | P1 vertices | P1 faces | publish + barrier | totals | P2 vertices | P2 faces |
 * publish + barrier | total + filter | publish + filter backward: messages | barrier | gather | final total),
 * out16[13..15] unused (scripts/bench_loss.py prints the differences).  Synchronises the device. */
int ddmp_dual_loss_trace(uint64_t* out16);

/* ddmp_dual_loss for n_mesh independent meshes as ONE cooperative launch.  Mesh m gets the min(G, ceil(max(V,F)/256))
 * blocks its stand-alone launch would use (G = ddmp_dual_loss_grid(0)) and runs the stand-alone arithmetic on them, so
 * its losses, gpos and gnrm equal a ddmp_dual_loss call bit for bit.  bnf_scale and loop are shared by the batch.
 * table: DEVICE array of n_mesh descriptors of DDMP_DUAL_LOSS_DESC_WORDS 8-byte words each:
 *   0 pos   1 nrm   2 tgt_vs   3 tgt_fn   4 faces   5 f2f   6 rslot   7 lap_rowptr   8 lap_col   9 corner_ptr
 *   10 corner_slot   11 workspace (ddmp_dual_loss_workspace_bytes(V, F, loop) bytes, its own per mesh)
 *   12 gpos   13 gnrm   14 losses[6]   (device addresses, as int64)
 *   15 V   16 F   (int64)
 *   17..21 k1..k5   (IEEE float32 in the low 4 bytes of the word, upper 4 bytes zero)
 * vf: HOST array [n_mesh][2] of the same V, F (the launch size is computed from it; it must match the table).
 * The sum of the meshes' blocks must not exceed ddmp_dual_loss_grid(1), the co-resident blocks of the batched kernel;
 * callers split larger batches into consecutive launches on one stream. */
#define DDMP_DUAL_LOSS_DESC_WORDS 22
int64_t ddmp_dual_loss_grid(int32_t batched);
int ddmp_dual_loss_multi(const int64_t* table, const int64_t* vf, int32_t n_mesh, float bnf_scale, int32_t loop,
                         void* stream);

/* mean angular distance in degrees between two sets of unit normals, float64 [ref: util/loss.py:261-272]. */
int ddmp_mad(const float* n1, const float* n2, double* out, void* scratch, int64_t F, void* stream);
/* vertex normals: normalise(sum of incident face normals) through the corner CSR [ref: util/models.py:12-29]. */
int ddmp_vertex_normals(const float* fn, const int32_t* corner_ptr, const int32_t* corner_slot, float* vn,
                        int64_t V, void* stream);
/* One Jacobi sweep of the normal-guided vertex update [ref: util/models.py:31-44]: fc is the centroid array of
 * the sweep's input positions. */
int ddmp_vertex_update_sweep(const float* pos_in, const float* fc, const float* nrm, const int32_t* corner_ptr,
                             const int32_t* corner_slot, float* pos_out, int64_t V, void* stream);
int ddmp_face_centroids(const float* pos, const int32_t* faces, float* fc, int64_t F, void* stream);

/* ---- step glue ----------------------------------------------------------------------------------------------- */
/* Global L2 norm of a flat gradient buffer (float64 accumulate) -> norm_out[0]; then the Adam update with the
 * clip coefficient min(1, max_norm/(norm+1e-6)) folded in (clip_norm == NULL: no clipping).
 * [ref: main.py:108-110 clip_grad_norm_ + torch.optim.Adam(lr, betas=(0.9,0.999), eps=1e-8)] */
int ddmp_grad_norm(const float* grad, float* norm_out, void* scratch, int64_t count, void* stream);
int ddmp_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, const float* clip_norm,
                   float max_norm, float lr, float beta1, float beta2, float eps, int64_t step, int64_t count,
                   void* stream);

/* Same update with the step count kept in device memory (incremented by the call): what a CUDA-graph-replayed
 * iteration needs, since kernel arguments are frozen at capture. */
int ddmp_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, const float* clip_norm,
                       float max_norm, float lr, float beta1, float beta2, float eps, int64_t* step_counter,
                       int64_t count, void* stream);

/* The gradients of one network (n_src device tensors of counts[i] floats each) copied to dst + offsets[i] by one launch
 * per 80 tensors: the flat gradient ddmp_grad_norm / ddmp_adam_step_dev consume.  srcs / offsets / counts are HOST arrays;
 * they travel as kernel arguments (frozen at CUDA-graph capture together with the -- stable -- addresses).
 * [ref: main.py:107-110: loss.backward() leaves one .grad per parameter; the optimizer walks them] */
int ddmp_gather_flat(const void* const* srcs, const int64_t* offsets, const int64_t* counts, int32_t n_src, float* dst,
                     void* stream);

/* ---- the optimizer of many networks at once (a batch of fits), one launch per stage ------------------------------ */
/* ddmp_gather_flat from a DEVICE table of n_src rows (source address, destination offset, count), 3 int64 words each,
 * in one launch (n_src <= 65535); `longest` is the largest count. */
int ddmp_gather_table(const int64_t* table, int32_t n_src, int64_t longest, float* dst, void* stream);
/* Segment table: DEVICE array of n_seg rows of DDMP_SEGMENT_WORDS int64 words, one row per network:
 *   0 offset into the flat buffers   1 count   2 clip (0 / 1)   3 lr   4 max_norm
 *   (lr, max_norm: IEEE float32 in the low 4 bytes of the word, upper 4 bytes zero).  `longest` is the largest count.
 * ddmp_grad_norm_segments: norms[s] = ddmp_grad_norm of segment s, for every segment with clip = 1, bit for bit (the
 * same block partition and summation order).  scratch: n_seg * ddmp_loss_scratch_bytes() bytes, zeroed once.
 * ddmp_adam_segments: increments *step_counter, then the update of ddmp_adam_step_dev on every segment with its lr
 * and, where clip = 1, the clip coefficient min(1, max_norm/(norms[s]+1e-6)). */
#define DDMP_SEGMENT_WORDS 5
int ddmp_grad_norm_segments(const float* flat, const int64_t* table, int32_t n_seg, int64_t longest, float* norms,
                            void* scratch, void* stream);
int ddmp_adam_segments(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, const int64_t* table,
                       int32_t n_seg, int64_t longest, const float* norms, float beta1, float beta2, float eps,
                       int64_t* step_counter, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DDMP_B200_H */
