/*
 * pglb.h -- C-ABI of libpglb.so: the B200 (sm_100a) send/recv message-passing path
 * behind PGL's Graph.send/recv API.
 *
 * The reference (PaddlePaddle/PGL @ 6dbb47c) has no native boundary of its own on this
 * path: it is Python over Paddle's operator API plus one Cython module.  Every entry point
 * below therefore names the reference call site(s) it replaces (paths relative to the
 * reference root).  See INTEGRATION.md for the reference-side binding.
 *
 * Conventions
 *  - extern "C", plain pointers and sizes; no torch / CUDA C++ types.  `stream` is a
 *    cudaStream_t passed as void* (NULL = legacy default stream).
 *  - All device entry points are asynchronous on `stream`, re-entrant and thread-safe; the
 *    library never allocates or frees device memory and keeps no pointer past the call.
 *    Scratch space is caller-owned: query with the matching *_ws() and pass (ws, ws_bytes).
 *  - Index tensors are int64 (PGL mandates int64 edges: pgl/graph.py:130-135), features
 *    are float32 row-major with an explicit leading dimension where noted.
 *  - Return value: 0 = PGLB_OK; <0 = argument error (no device work was enqueued);
 *    >= PGLB_CUDA_ERR_BASE = PGLB_CUDA_ERR_BASE + cudaError_t.  pglb_last_error() returns a
 *    thread-local, human-readable description of the last non-zero return.
 *  - No C++ exception crosses this boundary.
 */
#ifndef PGLB_H_
#define PGLB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PGLB_VERSION 100 /* 0.1.0 */

#define PGLB_OK 0
#define PGLB_EINVAL (-1)    /* null pointer / negative size / unknown enum */
#define PGLB_ESHAPE (-2)    /* inconsistent sizes */
#define PGLB_EWORKSPACE (-3) /* workspace too small or misaligned */
#define PGLB_EUNSUPPORTED (-4)
#define PGLB_ENOLIB (-5)    /* optional host dependency (METIS) not loadable */
#define PGLB_CUDA_ERR_BASE 1000

/* reduce_op of send_u_recv / send_ue_recv / segment_* (pgl/graph.py:856-857, pgl/math.py:34-46) */
#define PGLB_REDUCE_SUM 0
#define PGLB_REDUCE_MEAN 1
#define PGLB_REDUCE_MAX 2
#define PGLB_REDUCE_MIN 3

/* message_op of send_ue_recv / send_uv (pgl/graph.py:923-927,958-962); COPY = no edge operand */
#define PGLB_MSG_COPY 0
#define PGLB_MSG_ADD 1
#define PGLB_MSG_SUB 2
#define PGLB_MSG_MUL 3
#define PGLB_MSG_DIV 4

/* how the second operand's row broadcasts against the D = H*Dh output columns */
#define PGLB_BCAST_FULL 0   /* y row has D values                      */
#define PGLB_BCAST_HEAD 1   /* y row has H values, y[c / Dh]  ([E,H,1] against [N,H,Dh]) */
#define PGLB_BCAST_SCALAR 2 /* y row has 1 value   ([E] or [E,1])       */

int pglb_version(void);
const char *pglb_last_error(void);
/* number of kernels this library has launched in the calling process (bench "gpu_launches") */
int64_t pglb_launch_count(void);

/* ------------------------------------------------------------------------------------
 * CSR build on the device.  Replaces EdgeIndex.from_edges (pgl/utils/edge_index.py:38-58;
 * tensor branch :43-54 = scatter-count + argsort + 2 gathers + cumsum) and is bit-identical
 * to the numpy branch's graph_kernel.build_index (pgl/graph_kernel.pyx:59-88): stable, i.e.
 * ascending edge id inside every bucket.
 *   u, v         : int64 device pointers, element i at u[i*u_stride] (so edges[:,1] of an
 *                  [E,2] array is (edges+1, stride 2) -- no strided copies as in
 *                  pgl/graph.py:859)
 *   degree[N], indptr[N+1], sorted_u[E], sorted_v[E], sorted_eid[E] : int64 outputs
 * ---------------------------------------------------------------------------------- */
int pglb_csr_build_ws(int64_t num_edges, int64_t num_nodes, size_t *ws_bytes);
int pglb_csr_build(const int64_t *u, int64_t u_stride, const int64_t *v, int64_t v_stride,
                   int64_t num_edges, int64_t num_nodes, int64_t *degree, int64_t *indptr,
                   int64_t *sorted_u, int64_t *sorted_v, int64_t *sorted_eid, void *ws,
                   size_t ws_bytes, void *stream);

/* Host twin of the above for numpy-mode graphs (EdgeIndex numpy branch,
 * pgl/utils/edge_index.py:56-57 -> pgl/graph_kernel.pyx:59-88).  Blocking, host pointers. */
int pglb_build_index_host(const int64_t *u, int64_t u_stride, const int64_t *v,
                          int64_t v_stride, int64_t num_edges, int64_t num_nodes,
                          int64_t *degree, int64_t *indptr, int64_t *sorted_u,
                          int64_t *sorted_v, int64_t *sorted_eid);

/* segment ids of a CSR: replaces Graph.get_segment_ids -> unique_segment
 * (pgl/graph.py:1397-1407, pgl/utils/helper.py:156-160; paddle.unique(return_inverse)).
 *   uniq_ind[K]   = rows with degree > 0 (ascending), segment_ids[E] = dense id per slot.
 *   num_uniq      : device int64 scalar that receives K.
 *   ws >= pglb_segment_ids_ws bytes. */
int pglb_segment_ids_ws(int64_t num_nodes, size_t *ws_bytes);
int pglb_segment_ids(const int64_t *indptr, int64_t num_nodes, int64_t num_edges,
                     int64_t *uniq_ind, int64_t *segment_ids, int64_t *num_uniq, void *ws,
                     size_t ws_bytes, void *stream);

/* sorted segment ids [E] -> indptr[K+1] (used by segment_* below; K = ids[E-1]+1, caller-known) */
int pglb_segment_indptr(const int64_t *segment_ids, int64_t num_edges, int64_t num_segments,
                        int64_t *indptr, void *stream);

/* ------------------------------------------------------------------------------------
 * Node-parallel CSR aggregation  out[d] = reduce_{slot j in row d} msg(j)   (K1/K2/K4)
 *   msg(j) = x[cols[j]]                       (msg_op = COPY)
 *          = x[cols[j]] (op) y[eid[j]]        (ADD/SUB/MUL/DIV, y broadcast per y_bcast)
 * Replaces paddle.geometric.send_u_recv / send_ue_recv as called at pgl/graph.py:860,886,
 * 930 (COO + atomics in the reference; here a cached dst-CSR, one writer per row,
 * summation in ascending edge id = the reference CPU loop's order), the legacy
 * helper.graph_send_recv (pgl/utils/helper.py:163-210) and, with cols == NULL (slot j
 * reads row j), paddle.geometric.segment_{sum,mean,max,min} (pgl/math.py:36-42).
 *   indptr[n_dst+1], cols[E] (nullable), eid[E] (nullable: y indexed by slot)
 *   x  [n_src, ldx] (first D columns used), y per y_bcast (nullable iff COPY), row stride ldy
 *   out[n_dst, ldo]; rows without a message are 0 for every reduce_op; MEAN divides by the
 *   row's slot count.
 *   scale_src[n_src] / scale_dst[n_dst] (nullable): msg *= scale_src[cols[j]] before the
 *   reduce, out[d] *= scale_dst[d] after it (GCNConv's two norm multiplies, conv.py:242,250)
 *   D = H * Dh output columns; head_dim = Dh (only used by PGLB_BCAST_HEAD).
 *   cols_packed[E] (nullable, uint32): a packed copy of cols made by pglb_pack_cols() (needs
 *   n_src < 2^31).  Halves the index traffic of the wide-row kernel; with PGLB_SPMM_L2_HINTS in
 *   flags, bit 31 marks sources worth keeping in L2 (evict_last, all other rows evict_first).
 *   Pure performance hints: results do not depend on them.
 *   max_degree_hint : max row length if the caller knows it (skips the hub pass when
 *   small), or -1.
 * ---------------------------------------------------------------------------------- */
int pglb_spmm_csr_ws(int64_t n_dst, int64_t num_edges, int64_t D, size_t *ws_bytes);
int pglb_spmm_csr_f32(const int64_t *indptr, const int64_t *cols, const int64_t *eid,
                      const float *x, int64_t ldx, const float *y, int64_t ldy, int y_bcast,
                      float *out, int64_t ldo, int64_t n_dst, int64_t n_src,
                      int64_t num_edges, int64_t D, int64_t head_dim, int msg_op,
                      int reduce_op, const float *scale_src, const float *scale_dst,
                      const uint32_t *cols_packed, int64_t max_degree_hint, int flags, void *ws,
                      size_t ws_bytes, void *stream);
/* flags of pglb_spmm_csr_f32 */
#define PGLB_SPMM_ACCUMULATE 1 /* SUM only: out[d] = (out[d] + sum of messages) * scale_dst[d];
                                  lets a caller aggregate one edge subset while the feature rows of
                                  another subset (halo rows) are still in flight */
#define PGLB_SPMM_L2_HINTS 2   /* bit 31 of cols_packed carries an L2 residency hint */

/* Packed column ids for pglb_spmm_csr_f32: count[n_src] (int32, zeroed by the call) receives how
 * often every source occurs in cols[E]; packed[j] = cols[j] | (count[cols[j]] >= min_count) << 31.
 * Pass min_count = INT64_MAX for plain 32-bit ids without hints. */
int pglb_pack_cols(const int64_t *cols, int64_t num_edges, int64_t n_src, int32_t *count,
                   int64_t min_count, uint32_t *packed, void *stream);

/* Narrow-row copy aggregation (sum / mean, D = 4..64 floats, D % 4 == 0): the same send_u_recv
 * (pgl/graph.py:860,886) for the 16..256-byte rows of a COLUMN-sharded feature matrix (every GPU holds the whole
 * CSR and D/R columns; reference precedent for the layout: examples/.../dist_feat.py:31-49).
 * pglb_narrow_plan builds, once per graph, what the kernel streams instead of cols/indptr:
 *   plan[E]        uint32: cols[j] | (slot j is the first of its row) << 30   (needs n_src < 2^30)
 *   nz_row[n_dst+2] int32: ids of the non-empty rows in order, padded with two copies of the last one
 *   blk_k[ceil(E/32)] int32: index into nz_row of the row that owns slot 32 b - 1 (-1 for b = 0)
 * ws: pglb_narrow_plan_ws(n_dst) / pglb_spmm_narrow_ws(E, D).  x and out rows 16-byte aligned (ldx, ldo % 4 == 0).
 * Row sums are formed in slot order inside 32-slot ranges and the ranges of a row added left to right:
 * deterministic, equal to the sequential loop up to fp32 rounding of the regrouping. */
int pglb_narrow_plan_ws(int64_t n_dst, size_t *ws_bytes);
/* cols_packed (nullable): the uint32 ids of pglb_pack_cols; its bit 31 (L2 residency hint) is carried into the plan */
int pglb_narrow_plan(const int64_t *indptr, const int64_t *cols, const uint32_t *cols_packed, int64_t n_dst,
                     int64_t n_src, int64_t num_edges, uint32_t *plan, int32_t *nz_row, int32_t *blk_k, void *ws,
                     size_t ws_bytes, void *stream);
int pglb_spmm_narrow_ws(int64_t num_edges, int64_t D, size_t *ws_bytes);
/* scale_src[n_src] (nullable): gathered per slot.  scale_slot[E] (nullable, wins over scale_src): the same values
 * already laid out per CSR slot (scale_slot[j] = scale_src[cols[j]], i.e. the edge values of the normalised adjacency),
 * streamed with the plan instead of gathered.  flags: PGLB_SPMM_L2_HINTS = honour bit 31 of the plan. */
int pglb_spmm_narrow_f32(const uint32_t *plan, const int32_t *nz_row, const int32_t *blk_k, const int64_t *indptr,
                         const float *x, int64_t ldx, float *out, int64_t ldo, int64_t n_dst, int64_t n_src,
                         int64_t num_edges, int64_t D, int reduce_op, const float *scale_src, const float *scale_slot,
                         const float *scale_dst, int flags, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------
 * Edge-parallel ops
 * ---------------------------------------------------------------------------------- */
/* out[e] = x[src[e]] (op) y[dst[e]] ; replaces paddle.geometric.send_uv (pgl/graph.py:965).
 * src/dst strided like pglb_csr_build.  x [n_src, D], y [n_dst, D], out [E, D]. */
int pglb_send_uv_f32(const float *x, const float *y, const int64_t *src, int64_t src_stride,
                     const int64_t *dst, int64_t dst_stride, int64_t num_edges, int64_t D,
                     int msg_op, float *out, void *stream);

/* out[i] = x[index[i]] ; paddle.gather(axis=0) at pgl/utils/op.py:45, pgl/message.py:157,
 * pgl/math.py:219,223.  index strided. */
int pglb_gather_rows_f32(const float *x, int64_t ldx, const int64_t *index,
                         int64_t index_stride, int64_t num_rows, int64_t D, float *out,
                         int64_t ldo, void *stream);
/* out[index[i]] = x[i] (unique indices) ; paddle.scatter(overwrite=True) at
 * pgl/graph.py:830, pgl/nn/functional/graph_op.py:122. */
int pglb_scatter_rows_f32(const float *x, int64_t ldx, const int64_t *index,
                          int64_t num_rows, int64_t D, float *out, int64_t ldo,
                          void *stream);

/* Per-row softmax over CSR rows, H columns; replaces pgl.math.segment_softmax
 * (pgl/math.py:216-224: 7 ops) and, with eid != NULL, GF.edge_softmax
 * (pgl/nn/functional/graph_op.py:117-123): slot j reads logits[eid[j]] and writes
 * out[eid[j]] (original edge order).  exp(x - rowmax) / rowsum, true division. */
int pglb_edge_softmax_csr_ws(int64_t num_edges, size_t *ws_bytes);
int pglb_edge_softmax_csr_f32(const int64_t *indptr, const int64_t *eid, const float *logits,
                              float *out, int64_t n_rows, int64_t num_edges, int64_t H,
                              void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------
 * Backward kernels.  The reference gets every gradient from Paddle autograd through the ops
 * above; sum / mean aggregation backward is pglb_spmm_csr_f32 on the reverse CSR, the rest:
 * ---------------------------------------------------------------------------------- */
/* out[e,h] = <a[ia[e],h,:], b[ib[e],h,:]>  (a, b rows of H*Dh floats; ia/ib strided like
 * pglb_csr_build).  Gradient of send_ue_recv(mul) wrt the edge operand [E,H,1] (pgl/graph.py:930
 * as used by GATConv, pgl/nn/conv.py:339) and of send_uv(mul). */
int pglb_sddmm_dot_f32(const float *a, const float *b, const int64_t *ia, int64_t ia_stride,
                       const int64_t *ib, int64_t ib_stride, int64_t num_edges, int64_t H,
                       int64_t Dh, float *out, void *stream);
/* gradient of pglb_edge_softmax_csr_f32: grad_logits = alpha * (grad - rowsum(alpha * grad)),
 * same row / eid convention as the forward (pgl/math.py:216-224 differentiated). */
int pglb_edge_softmax_bwd_csr_f32(const int64_t *indptr, const int64_t *eid, const float *alpha,
                                  const float *grad, float *grad_logits, int64_t n_rows,
                                  int64_t num_edges, int64_t H, void *stream);
/* gradient of send_u_recv(max|min) wrt x on the reverse (src-keyed) CSR: every source entry that
 * equals the reduced output receives the output's gradient (Paddle's send_u_recv grad contract).
 *   src_indptr[n_src+1], dst_of_slot[E]; x [n_src, D], out / grad_out [n_dst, D], grad_x [n_src, D] */
int pglb_maxmin_bwd_f32(const int64_t *src_indptr, const int64_t *dst_of_slot, const float *x,
                        const float *out, const float *grad_out, float *grad_x, int64_t n_src,
                        int64_t D, void *stream);

/* GAT attention in one launch (inference path of GATConv, pgl/nn/conv.py:333-335): for every dst row
 * d and head h, alpha[j,h] = softmax_j( leaky_relu(attn_src[cols[j],h] + attn_dst[d,h]) ) over the
 * row's slots j -- send_uv(add) + LeakyReLU + edge_softmax without materialising the [E,H] logits.
 * alpha_slots is in CSR SLOT order (row-contiguous), which is what pglb_spmm_csr_f32 reads
 * sequentially when eid == NULL.  ws as pglb_edge_softmax_csr_ws. */
int pglb_gat_attention_csr_f32(const int64_t *indptr, const int64_t *cols, const float *attn_src,
                               const float *attn_dst, float negative_slope, float *alpha_slots,
                               int64_t n_rows, int64_t num_edges, int64_t H, void *ws,
                               size_t ws_bytes, void *stream);

/* The whole GAT aggregation in ONE pass (inference path of GATConv, pgl/nn/conv.py:333-339):
 *   out[d,h,:] = sum_j softmax_j( leaky_relu(attn_src[cols[j],h] + attn_dst[d,h]) ) * f[cols[j],h,:]
 * send_uv + LeakyReLU + edge_softmax + send_ue_recv(mul,sum) with an online softmax inside the
 * wide-row aggregation kernel: neither the logits nor alpha are ever written.  f rows of
 * H*head_dim <= 128 floats (head_dim % 4 == 0, 16-byte aligned); ws as pglb_spmm_csr_ws(D = H*head_dim). */
int pglb_gat_fused_csr_f32(const int64_t *indptr, const int64_t *cols, const float *f, int64_t ldf,
                           const float *attn_src, const float *attn_dst, float negative_slope,
                           float *out, int64_t ldo, int64_t n_dst, int64_t n_src, int64_t num_edges,
                           int64_t H, int64_t head_dim, void *ws, size_t ws_bytes, void *stream);

/* GATConv's attention projections (pgl/nn/conv.py:323-326: paddle.sum(feature * weight_src, -1) and the same with
 * weight_dst -- two multiplies, two reductions, two [N, H, head_dim] temporaries) in one pass over f:
 *   attn_src[n,h] = <f[n,h,:], w_src[h,:]>,  attn_dst[n,h] = <f[n,h,:], w_dst[h,:]>.
 * f rows of H*head_dim <= 128 floats, 16-byte aligned; head_dim in {4, 8, ..., 128}. */
int pglb_head_dots_f32(const float *f, int64_t ldf, int64_t n, int64_t H, int64_t head_dim, const float *w_src,
                       const float *w_dst, float *attn_src, float *attn_dst, void *stream);

/* Training forward of the same layer (GATConv under autograd, pgl/nn/conv.py:333-339; the reference gets the
 * backward from Paddle autograd over four ops): the same single launch, which also leaves
 *   lse[d,h] = log sum_j exp(leaky_relu(attn_src[cols[j],h] + attn_dst[d,h]))
 * for every row with at least one in-edge (other rows of lse are not written).  PGLB_EUNSUPPORTED when the shape is
 * outside the TMA kernel (H % 4 != 0, slope outside [0, 1], rows not 16-byte aligned): the caller keeps the
 * op-by-op path, every op of which has a backward. */
int pglb_gat_fused_train_csr_f32(const int64_t *indptr, const int64_t *cols, const float *f, int64_t ldf,
                                 const float *attn_src, const float *attn_dst, float negative_slope,
                                 float *out, int64_t ldo, float *lse, int64_t n_dst, int64_t n_src,
                                 int64_t num_edges, int64_t H, int64_t head_dim, void *ws, size_t ws_bytes,
                                 void *stream);

/* Per-edge part of that layer's backward.  rows[j] / cols[j] / eid[j] = destination, source and original edge id
 * of dst-CSR slot j (EdgeIndex.triples(); eid NULL = identity).  With z = attn_src[src,h] + attn_dst[dst,h]:
 *   alpha_e[e,h] = exp(leaky_relu(z) - lse[dst,h])                                   (the attention weight, rebuilt)
 *   dz_e[e,h]    = alpha * (<grad_out[dst,h,:], f[src,h,:]> - <grad_out[dst,h,:], out[dst,h,:]>) * leaky_relu'(z)
 * both [num_edges, H] in ORIGINAL edge order.  The caller finishes with reverse-CSR aggregations:
 * grad f = send_ue_recv(grad_out, alpha_e, mul, sum) over the src-keyed CSR, grad attn_src / grad attn_dst = segment
 * sums of dz_e over the src- / dst-keyed CSR.  head_dim in {4, 8, 16, 32, 64, 128}, H*head_dim <= 128. */
int pglb_gat_bwd_edge_f32(const int64_t *rows, const int64_t *cols, const int64_t *eid, const float *f,
                          int64_t ldf, const float *grad_out, int64_t ldg, const float *out, int64_t ldo,
                          const float *attn_src, const float *attn_dst, const float *lse,
                          float negative_slope, int64_t num_edges, int64_t H, int64_t head_dim,
                          float *alpha_e, float *dz_e, void *stream);

/* out[M, N] = act(x[M, K] @ w[K, N] + bias[N]) -- the dense transform of the conv layers
 * (pgl/nn/conv.py:238-251 GCNConv: `self.linear(...)`, `+ self.bias`, activation; the same Linear in
 * GATConv :321 / GraphSageConv :107-108) on the tensor cores with 3xTF32 error compensation (fp32-level
 * accuracy, fp32 accumulate), bias and ReLU fused into the single write of out.
 * w is contiguous [K, N] (paddle.nn.Linear layout); K % 4 == 0, 4 <= K <= 128; N in {64, 128};
 * ldx % 4 == 0, x 16-byte aligned; bias may be NULL; act: 0 none, 1 relu. */
int pglb_linear_tf32x3_f32(const float *x, int64_t ldx, const float *w, const float *bias, float *out,
                           int64_t ldo, int64_t M, int64_t K, int64_t N, int act, void *stream);

/* ------------------------------------------------------------------------------------
 * Neighbour sampling + reindex for mini-batch GraphSAGE (SURVEY 8f rank 4).  Replace
 * paddle.geometric.sample_neighbors / reindex_graph as called by NeighborSampler.sample_neighbors
 * (pgl/sampling/sage.py:130-155) on the cached dst-CSR (row = adj_dst_index._sorted_v,
 * colptr = adj_dst_index._indptr).  Validated on hardware in round 2 (tests/test_gpu_sampling.py).
 * ---------------------------------------------------------------------------------- */
/* count[i] = min(deg(nodes[i]), sample_size)  (all neighbours when sample_size < 0);
 * offsets[0..n] = exclusive scan of count, offsets[n] = total (n + 1 entries). */
int pglb_sample_count(const int64_t *indptr, const int64_t *nodes, int64_t n, int64_t sample_size,
                      int64_t *count, int64_t *offsets, void *stream);
/* out_neighbors[offsets[i] + j] = j-th sampled in-neighbour of nodes[i]: the whole list in CSR order
 * when deg <= sample_size, else a uniform subset without replacement (Floyd), a pure function of
 * (seed, i).  out_eids (may be NULL) receives eid[slot] (or the CSR slot when eid is NULL).
 * sample_size <= 4096; degrees < 2^31. */
int pglb_sample_fill(const int64_t *indptr, const int64_t *row, const int64_t *eid, const int64_t *nodes,
                     int64_t n, int64_t sample_size, uint64_t seed, const int64_t *offsets,
                     int64_t *out_neighbors, int64_t *out_eids, void *stream);
/* Dense lookup table for pglb_reindex_graph: num_nodes int64, filled with INT64_MAX ("empty"). */
int pglb_reindex_table_init(int64_t *table, int64_t num_nodes, void *stream);
int pglb_reindex_graph_ws(int64_t num_neighbors, size_t *ws_bytes);
/* paddle.geometric.reindex_graph(x, neighbors, count): out_nodes = x followed by the new ids among
 * neighbors in first-appearance order; reindex_src[p] = position of neighbors[p] in out_nodes;
 * reindex_dst[p] = i for the slots of x[i] (offsets as produced by pglb_sample_count, n + 1 entries).
 * x must hold distinct ids.  *num_out (device scalar) = number of entries written to out_nodes
 * (capacity n + m).  table: see pglb_reindex_table_init; left all-empty again on return. */
int pglb_reindex_graph(const int64_t *x, int64_t n, const int64_t *neighbors, const int64_t *offsets,
                       int64_t m, int64_t *table, int64_t *reindex_src, int64_t *reindex_dst,
                       int64_t *out_nodes, int64_t *num_out, void *ws, size_t ws_bytes, void *stream);

/* ------------------------------------------------------------------------------------
 * Random walks and skip-gram pairs (csrc/walk.cu): pgl.sampling.random_walk / node2vec_walk /
 * node2vec_walk_plus (pgl/sampling/walk.py:23-183, the per-step pgl/graph_kernel.pyx:142-224) and
 * graph_kernel.skip_gram_gen_pair (pgl/graph_kernel.pyx:343-364) over a whole batch of walks.
 *
 * indptr[N+1], cols[E]: the successor CSR with every row's columns in ascending order.
 * out[n, ldo] (ldo >= steps + 1): out[i, 0] = nodes[i], out[i, t+1] = the node reached by step t; a walk
 * ends at the first node without successors and the rest of its row is -1.
 *
 * RNG, a pure function of (seed, i) whatever the launch geometry (all arithmetic mod 2^64):
 *   mix64(z):  z += 0x9e3779b97f4a7c15; z = (z ^ z >> 30) * 0xbf58476d1ce4e5b9;
 *              z = (z ^ z >> 27) * 0x94d049bb133111eb; return z ^ z >> 31
 *   word(t, k) = mix64(mix64(seed ^ mix64(i)) + PGLB_WALK_WORDS_PER_STEP * t + k)
 * Step t from node c with d > 0 successors cols[s .. s+d):
 *   uniform mode, and step 0 of every mode: next = cols[s + umul64hi(word(t, 0), d)]
 *   node2vec / node2vec+, t >= 1: the weight class of a candidate x is 0 when x is the previous node,
 *     1 when x is in the seen set (node2vec: successors of the previous node; node2vec+: successors of
 *     every earlier node of the walk), 2 otherwise.  With w = (1/p, 1, 1/q), M = max(w) (double):
 *       T[c] = max(1, floor(w[c] / M * 2^32))
 *     draw k = 0 .. PGLB_WALK_MAX_REJECT-1: x = cols[s + umul64hi(word(t, 2k), d)], accepted when
 *       (word(t, 2k+1) >> 32) < T[class(x)];
 *     when no draw is accepted: S = sum over the row's slots j of T[class(cols[s+j])],
 *       r = umul64hi(word(t, 2 PGLB_WALK_MAX_REJECT), S), next = cols[s + first j whose inclusive prefix
 *       sum of T exceeds r]  (exact inverse CDF; on the device one warp per such step).
 * Both entries produce the same walks bit for bit.
 * ---------------------------------------------------------------------------------- */
#define PGLB_WALK_UNIFORM 0
#define PGLB_WALK_NODE2VEC 1
#define PGLB_WALK_NODE2VEC_PLUS 2
#define PGLB_WALK_MAX_REJECT 32
#define PGLB_WALK_WORDS_PER_STEP 128
/* Device.  Ids of `nodes` outside [0, N) give a row of -1 (callers are expected to reject them first). */
int pglb_random_walk(const int64_t *indptr, const int64_t *cols, int64_t N, const int64_t *nodes, int64_t n,
                     int64_t steps, int mode, double p, double q, uint64_t seed, int64_t *out, int64_t ldo,
                     void *stream);
/* Host twin: the same arguments on host pointers, blocking.  An id outside [0, N) is PGLB_ESHAPE. */
int pglb_random_walk_host(const int64_t *indptr, const int64_t *cols, int64_t N, const int64_t *nodes, int64_t n,
                          int64_t steps, int mode, double p, double q, uint64_t seed, int64_t *out, int64_t ldo);
/* Skip-gram pairs of walks[n, W] (row stride ldw; a walk is the entries before its row's first -1).
 * Position i of walk w < n draws r = 1 + umul64hi(mix64(mix64(seed ^ mix64(w)) + i), win_size) and pairs
 * (walk[i], walk[j]) for every j in [i - r, i + r] inside the walk with walk[j] != walk[i], in that order.
 *   count: offsets[n*W + 1]; offsets[p + 1] - offsets[p] = pairs of position p = w*W + i, offsets[n*W] = total.
 *   fill : src[total], dst[total] in walk, position, j order.
 * ws: pglb_skip_gram_ws bytes, the same buffer passed to both calls, untouched between them. */
int pglb_skip_gram_ws(int64_t n, int64_t W, size_t *ws_bytes);
int pglb_skip_gram_count(const int64_t *walks, int64_t n, int64_t W, int64_t ldw, int64_t win_size, uint64_t seed,
                         int64_t *offsets, void *ws, size_t ws_bytes, void *stream);
int pglb_skip_gram_fill(const int64_t *walks, int64_t n, int64_t W, int64_t ldw, int64_t win_size, uint64_t seed,
                        const int64_t *offsets, int64_t *src, int64_t *dst, void *ws, size_t ws_bytes,
                        void *stream);

/* Same contract as pglb_memcpy2d_async, but the copy is done by a kernel through the unified address
 * space (zero-copy loads / stores across PCIe; the host side must be pinned memory).  For narrow column
 * blocks, where the copy engine's 2-D transfers run at about half the PCIe rate.  width, pitches and both
 * pointers multiples of 16 bytes; ctas <= 0 -> 16.  Opt-in (PGLB_HOST_COPY=kernel) and unmeasured: the cross-call
 * pipeline of Graph.host_aggregator removed the need for narrow 2-D copies (DESIGN.md section 4.8). */
int pglb_copy2d_kernel_async(void *dst, size_t dpitch, const void *src, size_t spitch, size_t width_bytes,
                             int64_t height, int ctas, void *stream);

/* norm[i] = clip(float(degree[i]), 1)^-0.5 ; GF.degree_norm (graph_op.py:46-55) */
int pglb_degree_norm_f32(const int64_t *degree, int64_t n, float *norm, void *stream);

/* Strided host<->device copy on `stream` (cudaMemcpy2DAsync): moves a column block of a row-major
 * matrix without staging.  kind: 1 = host->device, 2 = device->host.  Used by the host-buffer
 * entry of the aggregation (features in pinned host memory): column chunks are independent for a
 * copy-message aggregation, so chunk c+1's upload, chunk c's kernel and chunk c-1's download
 * overlap (PCIe is full duplex). */
int pglb_memcpy2d_async(void *dst, size_t dst_pitch, const void *src, size_t src_pitch,
                        size_t width_bytes, size_t height, int kind, void *stream);

/* ------------------------------------------------------------------------------------
 * Peer-mappable device buffers for the multi-GPU halo pull (NVLink P2P, one process per GPU).
 * The only place the library allocates: cudaMalloc'ed buffers whose CUDA IPC handle (64 bytes)
 * other ranks open under THEIR device with pglb_ipc_open; kernels such as pglb_gather_rows_f32
 * then read the owner's HBM directly.  No reference counterpart (the reference replicates all
 * features on every GPU, pgl/graph.py:1410-1553).
 * ---------------------------------------------------------------------------------- */
int pglb_ipc_alloc(size_t bytes, void **dev_ptr, void *handle64);
int pglb_ipc_free(void *dev_ptr);
int pglb_ipc_open(const void *handle64, void **peer_ptr);
int pglb_ipc_close(void *peer_ptr);

/* Debug aid (scripts/task_trace.py): while `buffer` (device, capacity_tasks x 4 int64) is armed, the wide-row
 * aggregation kernels record (start ns, end ns, SM id, warp slot) for every task of a launch with at most
 * capacity_tasks tasks.  buffer = NULL disarms.  Process-global; not for concurrent use. */
int pglb_debug_task_trace(void *buffer, int64_t capacity_tasks);

/* ------------------------------------------------------------------------------------
 * Partition -> local-graph pipeline on the device (SURVEY.md section 8f rank 3; csrc/localgraph.cu).
 * ---------------------------------------------------------------------------------- */
/* graph_kernel.map_nodes(nodes, reindex) (pgl/graph_kernel.pyx:123-138) with the dict as a dense table
 * new_id[old_id] (table_size entries): out[i] = table[nodes[i]].  An id outside [0, table_size) gives -1 and
 * sets *bad_flag (device int, may be NULL; the caller zeroes it) -- the reference's unordered_map would
 * silently insert 0. */
int pglb_map_nodes(const int64_t *nodes, int64_t n, const int64_t *table, int64_t table_size,
                   int64_t *out, int32_t *bad_flag, void *stream);
/* graph_kernel.map_edges(eid, edges, reindex) (pgl/graph_kernel.pyx:104-120): out[i, :] = table[edges[eid[i], :]];
 * eid NULL = all edges in order.  edges / out contiguous [*, 2] int64. */
int pglb_map_edges(const int64_t *eid, int64_t n, const int64_t *edges, int64_t num_edges,
                   const int64_t *table, int64_t table_size, int64_t *out, int32_t *bad_flag, void *stream);
/* inverse[perm[j]] = j.  With perm = sorted_eid of pglb_csr_build(u = part) -- the stable sort of the nodes by
 * part -- inverse is the `new id of every node` of apps/GNNAutoScale/graph_partition.py:94-101 and the build's
 * indptr is its offsets array. */
int pglb_invert_perm(const int64_t *perm, int64_t n, int64_t *inverse, void *stream);
/* One rank's local graph of a 1-D node partition whose parts are contiguous id ranges (this rank owns
 * [lo, hi)).  Two calls, because the output sizes are data dependent:
 *   count: counts[0] = E_local (edges whose destination is owned), counts[1] = H (distinct remote sources);
 *          *bad_flag (device int, zeroed by the caller) is set when an endpoint lies outside [0, num_nodes).
 *   fill : eid[E_local]       ascending global edge ids of the local edges,
 *          dst_local[E_local] destination - lo,
 *          col_local[E_local] source - lo when owned, else (hi - lo) + position of the source in halo_ids,
 *          halo_ids[H]        ascending distinct remote source ids (= grouped by owner),
 *          recv_counts[K]     how many of them lie in [offsets[p], offsets[p+1])  (offsets: device, K + 1 entries).
 * The same workspace (pglb_halo_plan_ws bytes, 256-byte aligned) must be passed to both calls, untouched between. */
int pglb_halo_plan_ws(int64_t num_edges, int64_t num_nodes, size_t *ws_bytes);
int pglb_halo_plan_count(const int64_t *edges, int64_t num_edges, int64_t num_nodes, int64_t lo, int64_t hi,
                         int64_t *counts, int32_t *bad_flag, void *ws, size_t ws_bytes, void *stream);
int pglb_halo_plan_fill(const int64_t *edges, int64_t num_edges, int64_t num_nodes, int64_t lo, int64_t hi,
                        const int64_t *offsets, int64_t num_parts, int64_t *eid, int64_t *dst_local,
                        int64_t *col_local, int64_t *halo_ids, int64_t *recv_counts, void *ws, size_t ws_bytes,
                        void *stream);

/* ------------------------------------------------------------------------------------
 * Host: METIS K-way behind the same call shape as graph_kernel.metis_partition
 * (pgl/graph_kernel.pyx:434-472 <- pgl/partition.py:83-90).  libmetis (IDXTYPEWIDTH 64) is
 * dlopen()ed from `libmetis_path` (NULL = default search); returns PGLB_ENOLIB if absent.
 * ---------------------------------------------------------------------------------- */
int pglb_metis_partition(const char *libmetis_path, int64_t num_nodes, const int64_t *indptr,
                         const int64_t *adjncy, int64_t nparts, const int64_t *node_weights,
                         const int64_t *edge_weights, int recursive, int64_t *part);

#ifdef __cplusplus
}
#endif
#endif /* PGLB_H_ */
