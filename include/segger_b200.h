/*
 * libsegger_b200 -- C ABI of the B200-native segger hot path.
 *
 * Every entry point (82) is `extern "C"`, takes plain device pointers and sizes (no torch types),
 * enqueues its work on the `stream` passed in (a cudaStream_t) and returns 0 on success or a
 * negative SGB_ERR_* code; the message is available from sgb_last_error() (thread-local).
 * The library never allocates, frees or retains device memory: outputs and workspaces are
 * caller-owned (torch caching allocator / RMM compatible, CUDA-graph capturable).
 *
 * Each function cites the reference interface (file:line under /root/reference/src/segger) it
 * replaces.  Where the arithmetic lives in a third-party dependency of the reference
 * (torch_geometric 2.7.0, torch_scatter 2.1.2, scipy cKDTree) the citation is segger's call site.
 */
#ifndef SEGGER_B200_H_
#define SEGGER_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SGB_VERSION 202

#if defined(__GNUC__)
#define SGB_API __attribute__((visibility("default")))
#else
#define SGB_API
#endif

#define SGB_OK 0
#define SGB_ERR_ARG -1
#define SGB_ERR_ALIGN -2
#define SGB_ERR_RANGE -3
#define SGB_ERR_WORKSPACE -4
#define SGB_ERR_CUDA -5

/* activation selectors for the fused GEMM epilogues */
#define SGB_ACT_NONE 0
#define SGB_ACT_GELU 1 /* exact erf GELU (F.gelu default, models/ist_encoder.py:320,325) */
#define SGB_ACT_SILU 2 /* torch.nn.SiLU (models/ist_encoder.py:45) */

SGB_API int sgb_version(void);
SGB_API const char* sgb_last_error(void);

/* ------------------------------------------------------------------------------------------
 * Graph layout: COO edge_index -> dst-sorted CSR (+ src-sorted transposed CSR).
 * Replaces the per-call gather/scatter indexing of PyG MessagePassing.propagate reached from
 * models/ist_encoder.py:183-189.  edge_index is [2,E] int32 or int64 (idx_bytes 4|8) with
 * arbitrary element strides (row_stride between the two rows, col_stride between edges), so
 * `.T` views (data/utils/neighbors.py:196) are accepted without a copy.
 * Stable: edges of a row keep their original order.  status (optional int32 on device) gets bit 0
 * set if any index was out of range (indices are clamped so the call never faults).
 * Transposed outputs may be NULL (inference).  src_pos[k] = position of that edge in the dst CSR.
 * ---------------------------------------------------------------------------------------- */
SGB_API size_t sgb_csr_workspace_bytes(int64_t E);
SGB_API int sgb_csr_build(const void* edge_index, int idx_bytes, int64_t row_stride, int64_t col_stride,
                  int64_t E, int64_t n_src, int64_t n_dst,
                  int32_t* dst_rowptr /*[n_dst+1]*/, int32_t* dst_col /*[E] source ids*/,
                  int32_t* dst_eid /*[E] original edge ids*/,
                  int32_t* src_rowptr /*[n_src+1] or NULL*/, int32_t* src_dst /*[E]*/,
                  int32_t* src_pos /*[E]*/, int32_t* status, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Fused GATv2 attention + aggregation (everything in GATv2Conv.forward after lin_l/lin_r):
 *   e_ij = att . leaky_relu(x_l[j] + x_r[i]);  alpha = segment softmax over edges into i (+1e-16);
 *   dropout(alpha);  out_i = sum_j alpha_ij x_l[j] + bias.
 * Replaces torch_geometric GATv2Conv edge_updater/softmax/propagate as configured at
 * models/ist_encoder.py:111-131 (SURVEY Appendix A.1).  One pass, no per-edge tensors.
 * x_l [n_src, H*C] / x_r [n_dst, H*C] fp32 with leading dimensions ld_* (floats, multiple of 4 for
 * the vector path), so column slices of a concatenated projection buffer can be passed directly.
 * out = pre-activation (o + bias); out_act (optional) = GELU(out) (fuses ist_encoder.py:325).
 * out may be NULL when out_act is given (inference: only the activated output is written).
 * stat_max/stat_den [n_dst,H] are saved for the backward.  seed/p_drop/training drive the
 * counter-based dropout keyed on (seed, original edge id, head).  seed_dev (or NULL) points to one device-resident
 * 64-bit word that is ADDED to seed when the kernel runs: a captured CUDA graph freezes by-value arguments, so a
 * replayed training step advances that word to draw a fresh mask (forward and backward read the same word).
 * e_logit (optional, [E, H]): where the sub-warp kernels run (sgb_gatv2_quad_supported, 16-byte aligned operands) the
 * forward leaves the raw logit of every (edge, head) there, in dst-CSR order, and a backward that is handed the same
 * buffer reads it back instead of re-evaluating att . leaky_relu(x_l[j] + x_r[i]) (4H bytes per edge against ~3
 * instructions per edge and feature).  The other kernel paths neither write nor read it: passing it to them is an
 * error (SGB_ERR_ARG), not a silent no-op.
 * ---------------------------------------------------------------------------------------- */
SGB_API int sgb_gatv2_fwd(const float* x_l, int64_t ld_l, const float* x_r, int64_t ld_r, const float* att,
                  const float* bias /*or NULL*/, const int32_t* dst_rowptr, const int32_t* dst_col,
                  const int32_t* dst_eid, int64_t n_dst, int64_t E, int H, int C, float negative_slope,
                  float p_drop, uint64_t seed, const uint64_t* seed_dev /*or NULL*/, int training,
                  float* out /*or NULL*/, int64_t ld_out,
                  float* out_act /*or NULL*/, int64_t ld_act, float* stat_max, float* stat_den,
                  float* e_logit /*or NULL: [E, H] raw logits e_ij in dst-CSR order, for sgb_gatv2_bwd*/,
                  void* stream);

/* 1 iff (H, C) is covered by the sub-warp-per-row kernels (needed for the one-source-per-edge form of sgb_gatv2_bwd:
 * src_rowptr == NULL, n_src == E, dst_col a permutation of [0, E) -- grad_x_l is then written by the dst pass). */
SGB_API int sgb_gatv2_quad_supported(int H, int C);

/* attention coefficients alpha [E,H] in ORIGINAL edge order (return_attention_weights=True path of
 * GATv2Conv; SkipGAT.attention_weights, models/ist_encoder.py:192-211).  Pre-dropout alpha. */
SGB_API int sgb_gatv2_alpha(const float* x_l, int64_t ld_l, const float* x_r, int64_t ld_r, const float* att,
                    const int32_t* dst_rowptr, const int32_t* dst_col, const int32_t* dst_eid,
                    int64_t n_dst, int64_t E, int H, int C, float negative_slope,
                    const float* stat_max, const float* stat_den, float* alpha, void* stream);

/* Deterministic backward of sgb_gatv2_fwd (autograd of the PyG ops above, SURVEY Appendix D).
 * grad_out: dL/d(out) -- or, if gelu_fused != 0, dL/d(out_act); then g = grad_out * gelu'(out) is
 * formed in-kernel and written to g_buf [n_dst, ld_g] (g_buf may alias grad_out; required when
 * gelu_fused).  Two passes: dst-CSR (grad_x_r, grad_att, grad_bias, per-edge scalars) and src-CSR
 * (grad_x_l); both row-owner reductions, no atomics.  grad_att/grad_bias are [H*C], overwritten.
 * n_src rows of grad_x_l are all written (zeros for sources without edges). */
SGB_API size_t sgb_gatv2_bwd_workspace_bytes(int64_t n_dst, int64_t E, int H, int C);
SGB_API int sgb_gatv2_bwd(const float* x_l, int64_t ld_l, const float* x_r, int64_t ld_r, const float* att,
                  const float* bias /*or NULL*/, const float* out, int64_t ld_out,
                  const float* grad_out, int64_t ld_g, int gelu_fused, float* g_buf,
                  const int32_t* dst_rowptr, const int32_t* dst_col, const int32_t* dst_eid,
                  const int32_t* src_rowptr, const int32_t* src_dst, const int32_t* src_pos,
                  int64_t n_src, int64_t n_dst, int64_t E, int H, int C, float negative_slope,
                  float p_drop, uint64_t seed, const uint64_t* seed_dev /*or NULL*/, int training,
                  const float* stat_max, const float* stat_den,
                  const float* e_logit /*or NULL: what sgb_gatv2_fwd left there for the same graph and inputs*/,
                  float* grad_x_l, int64_t ld_gl, float* grad_x_r,
                  int64_t ld_gr, float* grad_att, float* grad_bias /*or NULL*/, void* ws,
                  size_t ws_bytes, void* stream);

/* The keep mask the kernels use, [E,H] uint8 in ORIGINAL edge order (test hook: lets the oracle
 * replay the identical dropout realisation). */
SGB_API int sgb_dropout_mask(uint64_t seed, int64_t E, int H, float p_drop, uint8_t* mask, void* stream);

/* ------------------------------------------------------------------------------------------
 * Dense projections y = x W^T + b (PyG Linear / HeteroDictLinear / GATv2Conv.lin_l, lin_r /
 * torch.nn.Linear of the positional MLP; models/ist_encoder.py:43-47,261,282-286 and the
 * GATv2Conv constructors at :111-131).  x [M,K] ldx, w [N,K] ldw, y [M,N] ldy, fp32 in/out.
 * Error-compensated split-TF32 on tcgen05 when the tile is a real dense GEMM, fp32 SIMT otherwise.
 * The tensor core accumulates in fp32 with round-toward-zero, a biased error that the attention
 * backward amplifies (d_e - c_i cancellation), so the reduction is cut into chunks whose TMEM
 * partials are added in registers with round-to-nearest (DESIGN.md, "GEMM precision"):
 *   exact = 0  3 products, 32-deep chunks (gradients, inference)
 *   exact = 1  4 products (fp32-exact operand products), 32-deep chunks: for projections that a
 *              following GATv2 layer will be differentiated through
 *   exact = 2  force the fp32 SIMT kernel
 * y_act (optional) receives act(y).  ws: sgb_linear_workspace_bytes(N, K) bytes of device scratch
 * (the split + swizzled copy of the weights); fwd and dgrad of the same weights need the same size.
 * ---------------------------------------------------------------------------------------- */
SGB_API size_t sgb_linear_workspace_bytes(int64_t N, int64_t K);
SGB_API int sgb_linear_fwd(const float* x, int64_t ldx, const float* w, int64_t ldw, const float* b /*or NULL*/,
                   int64_t M, int64_t N, int64_t K, float* y, int64_t ldy, int act,
                   float* y_act /*or NULL*/, int64_t ldya, int exact, void* ws, size_t ws_bytes, void* stream);
/* y = x W^T + b + table[ids]: forward projection of an input whose leading columns are a row of a small table
 * selected by an integer id -- ISTEncoder's first layer input is cat(GELU(Embedding[gene]), GELU(pos MLP))
 * (models/ist_encoder.py:312-320), so that half of the product is table = GELU(Embedding) W_first^T (n_genes rows,
 * computed once per step) looked up per transcript in the GEMM epilogue instead of K more columns of GEMM.
 * x [M,K] = the remaining dense columns, w [N,K] the matching weight columns, ids [M] int32|int64, table [*,N]. */
SGB_API int sgb_linear_fwd_gather(const float* x, int64_t ldx, const float* w, int64_t ldw, const float* b /*or NULL*/,
                          int64_t M, int64_t N, int64_t K, float* y, int64_t ldy, const void* ids, int idx_bytes,
                          const float* table, int64_t ld_table, int exact, void* ws, size_t ws_bytes, void* stream);
/* dx = dy W (+ dx if accumulate) ; if act_pre != NULL: dx *= act'(act_pre) (GELU/SiLU backward
 * fused as epilogue).  dy [M,N], w [N,K], dx [M,K]. */
SGB_API int sgb_linear_dgrad(const float* dy, int64_t ldy, const float* w, int64_t ldw, int64_t M, int64_t N,
                     int64_t K, float* dx, int64_t ldx, int accumulate, int act,
                     const float* act_pre /*or NULL*/, int64_t ld_pre, void* ws, size_t ws_bytes, void* stream);
/* dw = dy^T x (+ dw if accumulate), db = column sums of dy (+ db if accumulate); deterministic split-K. */
SGB_API size_t sgb_linear_wgrad_workspace_bytes(int64_t M, int64_t N, int64_t K);
SGB_API int sgb_linear_wgrad(const float* dy, int64_t ldy, const float* x, int64_t ldx, int64_t M, int64_t N,
                     int64_t K, float* dw, int64_t lddw, float* db /*or NULL*/, int accumulate,
                     void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Element-wise / row-wise pieces of ISTEncoder.forward (models/ist_encoder.py:312-333).
 * ---------------------------------------------------------------------------------------- */
/* y = act(x) and dx = dy * act'(x) over [M,N] with leading dimensions. */
SGB_API int sgb_act_fwd(const float* x, int64_t ldx, int64_t M, int64_t N, int act, float* y, int64_t ldy, void* stream);
SGB_API int sgb_act_bwd(const float* dy, int64_t ldy, const float* x, int64_t ldx, int64_t M, int64_t N, int act,
                float* dx, int64_t lddx, void* stream);
/* Embedding gather (lin_first['tx'], ist_encoder.py:260,312): out[i, 0:D] = table[ids[i], :];
 * optional fused GELU into out_act.  ids int32 or int64. */
SGB_API int sgb_embedding_fwd(const float* table, int64_t n_rows, int D, const void* ids, int idx_bytes, int64_t N,
                      float* out, int64_t ldo, float* out_act, int64_t lda, int act, void* stream);
/* grad_table[n_rows,D] = segment sum of dy rows by id (deterministic: sort by id + row-owner sum).
 * If table != NULL the rows are first multiplied by act'(table[id]) (backward of the fused
 * activation of sgb_embedding_fwd's out_act). */
SGB_API size_t sgb_embedding_bwd_workspace_bytes(int64_t N, int D, int64_t n_rows);
SGB_API int sgb_embedding_bwd(const float* dy, int64_t ldy, const void* ids, int idx_bytes, int64_t N, int D,
                      int64_t n_rows, const float* table /*or NULL*/, int act, float* grad_table,
                      void* ws, size_t ws_bytes, void* stream);
/* Positional2dEmbedder front end (ist_encoder.py:22-31,57-79): per-tile min/max normalisation of
 * pos [N,2] by batch id (NULL batch = one global tile without the 1e-8 eps, :63-65), then the
 * sinusoid cos(p*freqs) | sin(p*freqs) per coordinate -> feat [2][N][dim] (coordinate-major: the
 * x features of all nodes, then the y features).  freqs [dim/2] is the frequency table of
 * sinusoidal_embedding (computed once on the host with the reference's own formula). */
SGB_API size_t sgb_posfreq_workspace_bytes(int64_t n_batches);
SGB_API int sgb_posfreq_fwd(const float* pos, int64_t N, const void* batch, int idx_bytes, int64_t n_batches,
                    int dim, const float* freqs, float* feat, int64_t ldf, void* ws, size_t ws_bytes,
                    void* stream);
/* Same front end, low-rank form: out[2N, deg] (ld ldo) = Chebyshev basis T_0..T_{deg-1}(2p - 1) of the normalised
 * coordinates p (x rows of all nodes, then y rows).  The 256 sinusoid columns of sgb_posfreq_fwd equal
 * out @ M to fp32 rounding for a constant [deg, dim] matrix M (deg = 12 suffices: f_k <= 1, p in [0,1]), so the
 * first Linear of the positional MLP (ist_encoder.py:43-47,76-79) contracts over deg instead of dim columns and
 * the [2N, dim] feature matrix is never written.  deg % 4 == 0; workspace as sgb_posfreq_workspace_bytes. */
SGB_API int sgb_poscheb_fwd(const float* pos, int64_t N, const void* batch, int idx_bytes, int64_t n_batches,
                    int deg, float* out, int64_t ldo, void* ws, size_t ws_bytes, void* stream);
/* Row-subset helpers for the tx-belongs-bd conv (HeteroConv fan-out, ist_encoder.py:118-124,183-189): only the
 * transcripts that are sources of a belongs edge need the conv's lin_l projection.  When the edge list's source row
 * is strictly increasing (each source once, as setup_heterodata emits it, data/utils/heterodata.py:147) the layer
 * gathers those rows (sgb_embedding_fwd with the feature matrix as table), projects E rows instead of N, and adds
 * the input gradient back with sgb_rows_add.
 * sgb_index_strictly_increasing: flag[0] = 1 iff ids[0] < ids[1] < ... (device flag, int32).
 * sgb_rows_add: dst[ids[k], 0:D] += src[k, 0:D], ids unique (no atomics needed), D % 4 == 0. */
SGB_API int sgb_index_strictly_increasing(const void* ids, int idx_bytes, int64_t n, int32_t* flag, void* stream);
SGB_API int sgb_rows_add(float* dst, int64_t ldd, int64_t n_dst_rows, const void* ids, int idx_bytes, int64_t n, int D,
                 const float* src, int64_t lds, void* stream);
/* F.normalize(x, dim=-1, eps=1e-12) forward / backward (ist_encoder.py:331-332). */
SGB_API int sgb_l2norm_fwd(const float* x, int64_t ldx, int64_t M, int D, float eps, float* y, int64_t ldy,
                   float* norm /*[M]*/, void* stream);
SGB_API int sgb_l2norm_bwd(const float* dy, int64_t ldy, const float* y, int64_t ldyy, const float* norm, int64_t M,
                   int D, float eps, float* dx, int64_t lddx, void* stream);

/* ------------------------------------------------------------------------------------------
 * tx<->cell scoring: cosine similarity over candidate edges + per-transcript max / arg-max +
 * cell-id lookup.  Replaces torch.cosine_similarity + torch_scatter.scatter_max + the index
 * plumbing of LitISTEncoder.predict_step (models/lightning_model.py:275-293).
 * Candidates come as a CSR over transcripts (sgb_csr_build with dst := transcript, i.e. call it
 * with the edge_index rows swapped; cand_eid = original edge ids).  Ties -> lowest original edge
 * id.  Transcripts without candidates: max_sim = 0, arg_edge = E, seg = -1 (SURVEY Appendix A.7).
 * min_similarity: NaN disables the filter.
 * ---------------------------------------------------------------------------------------- */
SGB_API int sgb_score_argmax(const float* emb_tx, int64_t ld_tx, const float* emb_bd, int64_t ld_bd, int D,
                     const int32_t* cand_rowptr, const int32_t* cand_col, const int32_t* cand_eid,
                     int64_t n_tx, int64_t E, float eps, const void* bd_index, int bd_index_bytes,
                     float min_similarity, float* max_sim, int64_t* arg_edge, int64_t* seg_idx,
                     void* stream);

/* ------------------------------------------------------------------------------------------
 * 2-D k-nearest-neighbour graph with radius cap: replaces scipy cKDTree.query as called from
 * kdtree_neighbors (data/utils/neighbors.py:139-150) and knn_to_edge_index (:54-92).
 * Uniform grid (cell >= max_dist), float64 distances of the float32/float64 coordinates,
 * neighbour accepted iff d < max_dist (strict), rows ordered by (d^2, index), padded with n_points.
 * sgb_knn2d_plan computes the bounding box on the device and synchronises the stream once to
 * size the grid; the plan is a small host struct.
 * ---------------------------------------------------------------------------------------- */
typedef struct sgb_knn_plan {
  double xmin, ymin, cell; /* cell edge (>= max_dist) */
  int64_t nx, ny;          /* grid dimensions */
  int64_t n_points, n_query;
  int k;
  double max_dist;
} sgb_knn_plan;
SGB_API int sgb_knn2d_plan(const void* points, int is_f64, int64_t n_points, const void* query /*or NULL*/,
                   int64_t n_query, int k, double max_dist, sgb_knn_plan* plan, void* ws64 /*>=64 B device*/,
                   void* stream);
SGB_API size_t sgb_knn2d_workspace_bytes(const sgb_knn_plan* plan);
SGB_API int sgb_knn2d(const sgb_knn_plan* plan, const void* points, int is_f64, const void* query /*or NULL*/,
              int64_t* table /*[n_query,k]*/, int32_t* count /*[n_query]*/, void* ws, size_t ws_bytes,
              void* stream);
/* The same search for any 1 <= k <= 1024 and any max_dist in (0, +inf] (+inf: no radius cap), with the same
 * outputs, arithmetic and order: KDTree(points).query(q, k, distance_upper_bound) for every k and bound scipy
 * accepts, and the k nearest transcripts of every boundary centroid of setup_prediction_graph(mode='uniform')
 * (data/utils/neighbors.py:200-238).  The grid spans the points only and its cell is sized from their density
 * (no larger than max_dist); a warp per query visits square rings of cells around the query's cell, keeps the
 * top-k in shared memory and stops once no unscanned point can enter it.  ws64 >= 64 B device; the plan
 * synchronises the stream once.  k or max_dist out of range -> SGB_ERR_ARG before any CUDA call. */
SGB_API int sgb_knn2d_ring_plan(const void* points, int is_f64, int64_t n_points, const void* query /*or NULL*/,
                        int64_t n_query, int k, double max_dist, sgb_knn_plan* plan, void* ws64 /*>=64 B device*/,
                        void* stream);
SGB_API size_t sgb_knn2d_ring_workspace_bytes(const sgb_knn_plan* plan);
SGB_API int sgb_knn2d_ring(const sgb_knn_plan* plan, const void* points, int is_f64, const void* query /*or NULL*/,
                   int64_t* table /*[n_query,k]*/, int32_t* count /*[n_query]*/, void* ws, size_t ws_bytes,
                   void* stream);
/* padded table -> COO (query-major) with offsets = exclusive scan of count: edge_index [2,E] int64
 * contiguous, index_ptr [n_query+1] int64 (knn_to_edge_index, neighbors.py:54-92), summed in int64 so it
 * stays exact past 2^31 edges. total E is returned through *n_edges_host after a stream synchronise when n_edges_host != NULL. */
SGB_API int sgb_knn_count_valid(const int64_t* table, int64_t n, int k, int64_t pad_value, int32_t* count, void* stream);
SGB_API size_t sgb_knn_coo_workspace_bytes(int64_t n_query);
SGB_API int sgb_knn_count_edges(const int32_t* count, int64_t n_query, int64_t* index_ptr, int64_t* n_edges_host,
                        void* ws, size_t ws_bytes, void* stream);
SGB_API int sgb_knn_table_to_coo(const int64_t* table, const int64_t* index_ptr, int64_t n_query, int k,
                         int64_t pad_value, int64_t row_offset, int64_t E, int64_t* edge_index /*[2,E]*/,
                         void* stream);

/* ------------------------------------------------------------------------------------------
 * Training losses (SURVEY 8f, row N1).  All index arrays are int64 device arrays; a NULL index means
 * "row i of the table".  Means are reduced in a fixed order (bit-reproducible); backward kernels write
 * per-item row gradients [T,D] which the caller segment-sums by target row with sgb_embedding_bwd.
 * `grad` is a device scalar (dL/dloss).  Workspace: sgb_loss_workspace_bytes(T).
 * ---------------------------------------------------------------------------------------- */
/* FastTripletSelector.sample_triplets (models/triplet_loss.py:88-125) given the index built by _build_index
 * (:27-86: counts/offsets/sorted_idx by cluster, present clusters, row-wise CDFs of the (dis)similarity among
 * present clusters) and the four uniform vectors the reference draws with torch.rand (:93,:99,:105,:112). */
SGB_API int sgb_triplet_sample(const int64_t* labels, int64_t N, int C, int P, const int64_t* present_idx,
                       const int64_t* present, const int64_t* counts, const int64_t* offsets,
                       const int64_t* sorted_idx, const float* cdf_pos /*[P,P]*/, const float* cdf_neg /*[P,P]*/,
                       const float* similarity /*[C,C]*/, const float* u_pos, const float* u2, const float* u_neg,
                       const float* u3, int64_t* positives, int64_t* negatives, float* dists_pos, float* dists_neg,
                       void* stream);
SGB_API size_t sgb_loss_workspace_bytes(int64_t T);
/* torch.nn.TripletMarginLoss(margin, p=2, eps, reduction='mean') over gathered rows
 * (triplet_loss.py:128-160; lightning_model.py:116,181-186): loss = mean(max(margin + |a-p+eps| - |a-n+eps|, 0)). */
SGB_API int sgb_triplet_margin_fwd(const float* ta, int64_t lda, const int64_t* ia, const float* tp, int64_t ldp,
                           const int64_t* ip, const float* tn, int64_t ldn, const int64_t* in_, int64_t T, int D,
                           float margin, float eps, float* d_ap /*[T]*/, float* d_an /*[T]*/, float* loss /*scalar*/,
                           void* ws, size_t ws_bytes, void* stream);
SGB_API int sgb_triplet_margin_bwd(const float* ta, int64_t lda, const int64_t* ia, const float* tp, int64_t ldp,
                           const int64_t* ip, const float* tn, int64_t ldn, const int64_t* in_, int64_t T, int D,
                           float margin, float eps, const float* d_ap, const float* d_an, const float* grad,
                           float* ga /*[T,D]*/, float* gp /*[T,D]*/, float* gn /*[T,D]*/, void* stream);
/* The same backward for TripletLoss's own call shape (triplet_loss.py:150-160: anchors = all T rows of `emb`, positives /
 * negatives = sampled rows of the SAME matrix), as ONE row-owner pass: gout[r] = d loss / d emb[r], the anchor term of
 * triplet r plus the terms of every triplet that sampled r, summed in a fixed order.  p_rowptr/p_tid (n_*): CSR over
 * ip (in_) -- p_tid[p_rowptr[r] .. p_rowptr[r+1]) = the triplets t with ip[t] == r, t increasing (sgb_csr_build of the
 * edge list (t -> ip[t])).  D in {32, 64, 128} (sgb_triplet_self_bwd_supported). */
SGB_API int sgb_triplet_self_bwd_supported(int D);
SGB_API int sgb_triplet_self_bwd(const float* emb, int64_t ld, const int64_t* ip, const int64_t* in_, int64_t T, int D,
                         float margin, float eps, const float* d_ap, const float* d_an, const float* grad,
                         const int32_t* p_rowptr, const int32_t* p_tid, const int32_t* n_rowptr, const int32_t* n_tid,
                         float* gout /*[T, D]*/, int64_t ldg, void* stream);
/* mode 0: mse_loss(cosine_similarity(a, b, eps), target, 'mean') -- MetricLoss (triplet_loss.py:193-204);
 * mode 1: BCEWithLogitsLoss()(sum(a * b, -1), target) -- segmentation BCE (lightning_model.py:188-205).
 * val [T] receives the cosine / the logit (saved for the backward). */
SGB_API int sgb_pair_loss_fwd(const float* ta, int64_t lda, const int64_t* ia, const float* tb, int64_t ldb,
                      const int64_t* ib, const float* target, int64_t T, int D, int mode, float eps, float* val,
                      float* loss /*scalar*/, void* ws, size_t ws_bytes, void* stream);
SGB_API int sgb_pair_loss_bwd(const float* ta, int64_t lda, const int64_t* ia, const float* tb, int64_t ldb,
                      const int64_t* ib, const float* target, int64_t T, int D, int mode, float eps,
                      const float* val, const float* grad, float* gA /*[T,D]*/, float* gB /*[T,D]*/, void* stream);

/* ------------------------------------------------------------------------------------------
 * Points-in-polygons spatial join (SURVEY 8f, row N2): the tx-neighbors-bd candidate edges.
 * Replaces cuspatial.quadtree_point_in_polygon behind points_in_polygons(predicate='contains')
 * (geometry/query.py:21-100) as called by setup_prediction_graph (data/utils/neighbors.py:226-238).
 * points [N,2] fp32 or fp64; polygons = one ring each: verts [V,2] fp64, ring_off [n_poly+1] int64
 * (a closing duplicate of the first vertex is tolerated).  Inside = even-odd crossing rule in fp64.
 * The uniform grid (xmin, ymin, cell, nx, ny) must cover the bounding box of all polygons.
 * Two passes over one workspace: sgb_pip_count -> total[0] (device int32, read it back to allocate),
 * then sgb_pip_fill -> edge_index [2,E] int32 (row 0 = point, row 1 = polygon; point-major, polygons
 * ascending per point; rows ld apart).
 * ---------------------------------------------------------------------------------------- */
SGB_API size_t sgb_pip_workspace_bytes(int64_t n_points, int64_t n_poly, int nx, int ny);
SGB_API int sgb_pip_count(const void* points, int points_f64, int64_t n_points, const double* verts, const int64_t* ring_off,
                  int64_t n_poly, double xmin, double ymin, double cell, int nx, int ny, int32_t* total, void* ws,
                  size_t ws_bytes, void* stream);
SGB_API size_t sgb_pip_fill_scratch_bytes(int64_t E);
SGB_API int sgb_pip_fill(const double* verts, const int64_t* ring_off, int64_t n_points, int64_t n_poly, double xmin, double ymin,
                 double cell, int nx, int ny, int64_t E, int32_t* edge_index, int64_t ld, void* ws, size_t ws_bytes,
                 void* scratch, size_t scratch_bytes, void* stream);
/* Buffered outlines (data/utils/neighbors.py:229-231, geopandas .buffer(sqrt(area / pi) * buffer_ratio) then the join):
 * per-ring area (signed shoelace, fp64, x relative to the first vertex), area-weighted centroid [n_poly,2] (triangle
 * fan from the first vertex), box [n_poly,4] = (xmin, ymin, xmax, ymax) and dist = sqrt(|area| / pi) * ratio; each
 * output may be NULL.  Fixed operation order, so a numpy evaluation gives the same doubles. */
SGB_API int sgb_polygon_props(const double* verts, const int64_t* ring_off, int64_t n_poly, double ratio, double* area,
                      double* centroid, double* box, double* dist, void* stream);
/* neighbors.py:229-231: the join of sgb_pip_count / sgb_pip_fill (same workspace and scratch sizes, same output) against
 * every ring grown by dist[poly] (device fp64): d > 0 keeps points inside the ring or at squared distance < d^2 from it
 * (the exact Minkowski sum with a disc), d < 0 keeps points inside and at squared distance > d^2, d == 0 is the plain
 * test.  The grid must cover the union of the polygon boxes grown by |d| (1 + 2^-20). */
SGB_API int sgb_pip_buffered_count(const void* points, int points_f64, int64_t n_points, const double* verts,
                      const int64_t* ring_off, const double* dist, int64_t n_poly, double xmin, double ymin, double cell,
                      int nx, int ny, int32_t* total, void* ws, size_t ws_bytes, void* stream);
SGB_API int sgb_pip_buffered_fill(const double* verts, const int64_t* ring_off, const double* dist, int64_t n_points,
                      int64_t n_poly, double xmin, double ymin, double cell, int nx, int ny, int64_t E, int32_t* edge_index,
                      int64_t ld, void* ws, size_t ws_bytes, void* scratch, size_t scratch_bytes, void* stream);
/* Outlines with holes and several parts (the GeoArrow / cuSpatial polygon layout the reference's GeoSeries carries):
 * ring_off [R+1] = vertices of ring r, part_off [Q+1] = rings of part q (the first its exterior, the rest its holes),
 * geom_off [n_geom+1] = parts of geometry g (one boundary row, one polygon id of the output).  Per geometry: area =
 * sum of |ring area| over exteriors minus holes, centroid = the area-weighted mean of the ring centroids, box = union
 * of the ring boxes, dist = sqrt(|area| / pi) * ratio; a geometry of one ring gives |area| and the centroid, box and
 * dist of sgb_polygon_props bit for bit.  Each output may be NULL. */
SGB_API int sgb_polygon_props_multi(const double* verts, const int64_t* ring_off, const int64_t* part_off,
                      const int64_t* geom_off, int64_t n_geom, double ratio, double* area, double* centroid, double* box,
                      double* dist, void* stream);
/* The join of sgb_pip_count / _fill (same grid, workspace, scratch and output, geometries in place of rings) against
 * that layout: p is in geometry g iff the even-odd rule over all rings of g says so (the XOR of the single-ring
 * decisions; for valid geometry the union of the parts minus their holes), listed once per geometry.  dist [n_geom]
 * device fp64 or NULL (the plain join): geometry g grown by dist[g] as sgb_pip_buffered_count grows one ring, the
 * distance taken to the nearest edge of any of its rings; the grid must cover the geometry boxes grown by
 * |dist| (1 + 2^-20). */
SGB_API int sgb_pip_multi_count(const void* points, int points_f64, int64_t n_points, const double* verts,
                      const int64_t* ring_off, const int64_t* part_off, const int64_t* geom_off, const double* dist,
                      int64_t n_geom, double xmin, double ymin, double cell, int nx, int ny, int32_t* total, void* ws,
                      size_t ws_bytes, void* stream);
SGB_API int sgb_pip_multi_fill(const double* verts, const int64_t* ring_off, const int64_t* part_off, const int64_t* geom_off,
                      const double* dist, int64_t n_points, int64_t n_geom, double xmin, double ymin, double cell, int nx,
                      int ny, int64_t E, int32_t* edge_index, int64_t ld, void* ws, size_t ws_bytes, void* scratch,
                      size_t scratch_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Device-side tile slicing and batch assembly (SURVEY 8f rows N2/N3) and the masked compaction that ends
 * predict_step.  All selections are order-preserving (flags -> exclusive scan -> scatter), i.e. they equal
 * torch.nonzero / boolean-mask indexing element for element.  Positions and counts are int32 (n < 2^31).
 * Workspace for a selection over n items: sgb_select_workspace_bytes(n).  `count` is a device int32.
 * ---------------------------------------------------------------------------------------- */
SGB_API size_t sgb_select_workspace_bytes(int64_t n);
/* sel[0..count) = indices with mask != 0 (ascending); map[i] = rank of i in sel or -1 (either may be NULL). */
SGB_API int sgb_mask_select(const uint8_t* mask, int64_t n, int32_t* sel, int32_t* map, int32_t* count, void* ws,
                    size_t ws_bytes, void* stream);
/* TilePredictDataset._subset (data/tile_dataset.py:218-246): nodes with outer[0] <= x < outer[2] and
 * outer[1] <= y < outer[3] (the tile grown by the margin), plus predict_mask = inside the closed inner box for the
 * selected nodes.  pos [n,2] fp32 (bounds are rounded to fp32 first, as torch does) or fp64. */
SGB_API int sgb_box_select(const void* pos, int pos_f64, int64_t n, const double* outer, const double* inner /*or NULL*/,
                   int32_t* sel, int32_t* map, uint8_t* inner_mask /*[count]*/, int32_t* count, void* ws,
                   size_t ws_bytes, void* stream);
/* map[sel[k]] = k (fill_mode 0) or = fill (fill_mode 1) for k < *count (count == NULL: k < m): maintains the
 * global -> tile-local node numbering of a tile subset in a persistent array (set before the edge pass, cleared after). */
SGB_API int sgb_scatter_rank(int32_t* map, const int32_t* sel, const int32_t* count, int64_t m, int fill_mode, int32_t fill,
                     void* stream);
/* dst[k,:] = src[sel[k],:] for k < *count (count == NULL: k < m), rows of row_bytes bytes of any dtype: the node /
 * edge attribute slicing of HeteroData.subgraph and PartitionDataset._index_select. */
SGB_API int sgb_gather_rows_bytes(const void* src, int64_t row_bytes, const int32_t* sel, const int32_t* count, int64_t m,
                          void* dst, void* stream);
/* PyG bipartite_subgraph(relabel_nodes=True) as HeteroData.subgraph applies it per edge type: keep edges whose
 * endpoints are both selected (map_* >= 0), relabel them, keep their order; kept_eid (optional) = original edge ids. */
SGB_API int sgb_edge_subset(const void* edge_index, int idx_bytes, int64_t row_stride, int64_t col_stride, int64_t E,
                    const int32_t* map_src, int64_t n_src, const int32_t* map_dst, int64_t n_dst, void* out_edge_index,
                    int64_t ld_out, int32_t* kept_eid, int32_t* count, void* ws, size_t ws_bytes, void* stream);
/* PartitionDataset._get_permutation (data/partition/dataset.py:375-401): perm = stable argsort of the node labels
 * (the reference's torch.argsort is not stable; stable = members of a partition keep their original order) and
 * rowptr[range+1] = the partition pointers (indptr).  status bit 0: a label was outside [0, range). */
SGB_API size_t sgb_argsort_workspace_bytes(int64_t n);
SGB_API int sgb_argsort_stable(const void* labels, int idx_bytes, int64_t n, int64_t range, int32_t* perm, int32_t* rowptr,
                       int32_t* status, void* ws, size_t ws_bytes, void* stream);
SGB_API int sgb_invert_permutation(const int32_t* perm, int64_t n, int32_t* inv, void* stream);
/* PartitionDataset._permute_edge_store (:440-506): edges renumbered through the node permutations, stably sorted by the
 * partition of their source, edges between different partitions DROPPED (:483-494).  lab_* = labels of the ORIGINAL
 * node ids, inv_* = inverse node permutations.  edge_rowptr[P+2]: [0..P] partition pointers of the kept edges
 * (edge_rowptr[P] = number kept).  ws: sgb_argsort_workspace_bytes(E) + 4E bytes. */
SGB_API int sgb_partition_edges(const void* edge_index, int idx_bytes, int64_t row_stride, int64_t col_stride, int64_t E,
                        const void* lab_src, const void* lab_dst, int lab_bytes, int64_t n_src, int64_t n_dst, int64_t P,
                        const int32_t* inv_src, const int32_t* inv_dst, void* out_edge_index, int64_t ld_out,
                        int32_t* kept_eid, int32_t* edge_rowptr, int32_t* status, void* ws, size_t ws_bytes, void* stream);
/* PartitionDataset.__getitem__ (data/partition/dataset.py:512-579) for K tiles + the DataLoader collate: rows
 * [starts[k], starts[k] + out_off[k+1] - out_off[k]) of src land at out_off[k] of dst (device int64 arrays). */
SGB_API int sgb_ranges_gather(const void* src, int64_t row_bytes, const int64_t* starts, const int64_t* out_off, int K,
                      int64_t total_rows, void* dst, void* stream);
/* same for edge_index [2, *] (rows ld_in apart): each tile's edges are shifted from tile-local node numbering
 * (global id - *_starts[k]) to batch numbering (+ *_out_off[k]) for the source and destination node types. */
SGB_API int sgb_edges_collate(const void* edge_index, int idx_bytes, int64_t ld_in, const int64_t* e_starts,
                      const int64_t* e_out_off, const int64_t* src_starts, const int64_t* src_out_off,
                      const int64_t* dst_starts, const int64_t* dst_out_off, int K, int64_t total_edges, void* out,
                      int64_t ld_out, void* stream);
/* Batched prediction-tile cut: TilePredictDataset._subset (data/tile_dataset.py:218-246) for T tiles ("slots") at once,
 * producing the collated batch of data_module.py:333-344 directly.  Candidates are contiguous ranges of an id array
 * sorted by grid cell (rng_start[R], rng_off[R+1] = exclusive prefix sum of the range lengths, rng_slot[R]; C = total
 * candidates); boxes [T][8] = (outer x0,y0,x1,y1 half-open; inner x0,y0,x1,y1 closed) per slot.
 * nodes: mask[c] = candidate inside its slot's outer box; keys[c] = slot << 40 | id << 1 | inside-inner (written where
 *        mask is set); slot_counts[T] = kept per slot.  Sorting the kept keys gives the collated node order.
 * edges: (edge ids sorted by the cell of their source) kept iff both endpoints are among the slot's nodes -- binary search
 *        in the slot's segment [ptr[slot], ptr[slot+1]) of the SORTED node keys of the source / destination node type;
 *        pu/pv = positions found (= collated node numbers), ekeys[c] = slot << 40 | edge id. */
SGB_API int sgb_tilecut_nodes(const int32_t* perm, const void* pos, int pos_f64, const int64_t* rng_start, const int64_t* rng_off,
                      const int32_t* rng_slot, int R, int64_t C, const double* boxes, int T, int64_t* keys, uint8_t* mask,
                      int32_t* slot_counts, void* stream);
SGB_API int sgb_tilecut_edges(const int32_t* eperm, const void* edge_index, int idx_bytes, int64_t row_stride, int64_t col_stride,
                      const int64_t* rng_start, const int64_t* rng_off, const int32_t* rng_slot, int R, int64_t C,
                      const void* src_pos, int pos_f64, const double* boxes, int T, const int64_t* src_keys,
                      const int64_t* src_ptr, const int64_t* dst_keys, const int64_t* dst_ptr, int64_t* ekeys, int32_t* pu,
                      int32_t* pv, uint8_t* mask, int32_t* slot_counts, void* stream);
/* Quadtree tiling: QuadTreeTiling (data/tiling.py:198-235, cuSpatial leaves of <= max_tile_size points over all node
 * positions) and TileFitDataset's tile label / training mask (data/tile_dataset.py:13-153).  Rules (oracle/quadtree_ref.py):
 * root = (xmin, ymin, scale = max(x range, y range, or 1 if 0) / 2^D), D = max_depth in 1..15; every cell edge is
 * xmin + c * scale in fp64; a point's cell is floor((x - xmin) / scale) corrected by +-1 so that the point lies in
 * [edge(c), edge(c+1)), clamped to [0, 2^D - 1]; a quadrant at level L < D holding > max_tile_size points is split;
 * tiles = non-empty unsplit quadrants in Morton order (x in the even key bits).
 * sgb_quadtree_build: labels[n] = tile of each point; root[3] = (xmin, ymin, scale); per tile leaf_meta[3] = (Morton
 *   prefix of 2*level bits, level, point count) and leaf_box[4] = (x0, y0, x1, y1); *n_leaves = tile count (leaf_cap >=
 *   sgb_quadtree_max_leaves(n, max_tile_size, max_depth) rows are caller-allocated).
 * sgb_quadtree_label: labels[n] = tile whose quadrant contains the point's cell (points outside the root clamp to the rim
 *   cells), -1 when that cell lies in an empty quadrant.
 * sgb_quadtree_fit_mask: mask[n] = point inside its own tile's box shrunk by margins[label] on every side (closed); 0 for
 *   labels outside [0, n_leaves). */
SGB_API int64_t sgb_quadtree_max_leaves(int64_t n, int64_t max_tile_size, int max_depth);
SGB_API size_t sgb_quadtree_workspace_bytes(int64_t n, int64_t max_tile_size, int max_depth);
SGB_API int sgb_quadtree_build(const void* pos, int pos_f64, int64_t n, int64_t max_tile_size, int max_depth, int32_t* labels,
                       double* root, int32_t* leaf_meta, double* leaf_box, int64_t leaf_cap, int32_t* n_leaves, void* ws,
                       size_t ws_bytes, void* stream);
SGB_API int sgb_quadtree_label(const void* pts, int pos_f64, int64_t n, const double* root, int max_depth, const int32_t* leaf_meta,
                       int n_leaves, int32_t* labels, void* stream);
SGB_API int sgb_quadtree_fit_mask(const void* pos, int pos_f64, int64_t n, const int32_t* labels, const double* leaf_box,
                          const double* margins, int n_leaves, uint8_t* mask, void* stream);
/* batch[r] = k for out_off[k] <= r < out_off[k+1] (the PyG Batch.batch vector). */
SGB_API int sgb_batch_vector(const int64_t* out_off, int K, int64_t total_rows, int64_t* batch, void* stream);
/* `src_idx[mask], seg_idx[mask], max_sim[mask], gen_idx[mask]` of LitISTEncoder.predict_step
 * (models/lightning_model.py:294-298) in one pass; outputs sized n, *count rows valid. */
SGB_API int sgb_compact_predictions(const uint8_t* mask, int64_t n, const int64_t* src_idx, const int64_t* seg_idx,
                            const float* max_sim, const void* gene, int gene_bytes, int64_t* out_src, int64_t* out_seg,
                            float* out_sim, void* out_gene, int32_t* count, void* ws, size_t ws_bytes, void* stream);

/* ------------------------------------------------------------------------------------------
 * Writer post-processing (SURVEY 8f row N4): ISTSegmentationWriter.assign_transcripts_to_cells
 * (data/writer.py:132-253, data/utils/threshold.py:3-11).
 * sgb_dedupe_max: one row per transcript, the prediction with the highest similarity (writer.py:199-203; exact ties ->
 * lowest cell id).  row_bits = number of significant bits of the row indices.  order[0..count) = indices of the kept
 * predictions, ascending in row index.
 * sgb_gene_thresholds: per gene, over its ASSIGNED transcripts (seg >= 0): scikit-image's threshold_yen and the
 * threshold_li iteration bounded by max_iter callbacks (li_iters = -1: not converged -> the writer back-fills with the
 * median of the others, writer.py:242-246); counts[g] = assigned transcripts of gene g (0: thresholds are NaN).
 * ---------------------------------------------------------------------------------------- */
SGB_API size_t sgb_dedupe_workspace_bytes(int64_t n);
SGB_API int sgb_dedupe_max(const int64_t* row, const int64_t* seg, const float* sim, int64_t n, int row_bits, int32_t* order,
                   int32_t* count, void* ws, size_t ws_bytes, void* stream);
SGB_API size_t sgb_gene_threshold_workspace_bytes(int64_t n, int n_genes);
SGB_API int sgb_gene_thresholds(const void* gene, int gene_bytes, const int64_t* seg, const float* sim, int64_t n, int n_genes,
                        int max_iter, double* thr_yen, double* thr_li, int32_t* li_iters, int32_t* counts, void* ws,
                        size_t ws_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SEGGER_B200_H_ */
