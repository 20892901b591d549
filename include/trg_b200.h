/* trg_b200.h -- C ABI of the B200-native (sm_100a) hetero-SAGE hot path.
 *
 * The reference (ramkp990/Truth_Recommendation_GNN) is pure Python and has no FFI layer; its
 * seam is the PyG operator API used by the scripts.  Each entry point below names the
 * reference lines it replaces.  The Python binding a maintainer adds is in INTEGRATION.md; the
 * host-side mirror of the reference interface lives in truth_recommendation_gnn_b200/.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless marked host;
 *  - int return: 0 = ok, non-zero = TRG_E_*; trg_last_error() returns a thread-local message;
 *  - no ownership transfer: all buffers including workspaces are allocated by the caller;
 *  - stateless, asynchronous on the given stream (a cudaStream_t passed as void*), no host
 *    synchronisation inside, re-entrant across streams and threads;
 *  - dtype: TRG_F32 (fp32 storage) or TRG_BF16 (bf16 storage, fp32 accumulation); TRG_F8E4M3 (e4m3
 *    bytes, fp32 accumulation) is accepted by trg_score_topk / trg_score_topk_excluding only;
 *  - row widths (F, H) must make a row a multiple of 16 bytes (F % 4 == 0 for fp32,
 *    F % 8 == 0 for bf16) and tables must be 16-byte aligned;
 *  - edge counts must be < 2^31 per relation; node ids are stored as int32 in the CSR.
 */
#ifndef TRG_B200_H
#define TRG_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TRG_ABI_VERSION 4

enum { TRG_F32 = 0, TRG_BF16 = 1, TRG_F8E4M3 = 2 /* trg_score_topk(_excluding) only */ };
enum {
  TRG_OK = 0,
  TRG_E_ARG = 1,        /* bad argument (null pointer, unsupported width, size overflow) */
  TRG_E_WORKSPACE = 2,  /* workspace too small */
  TRG_E_CUDA = 3,       /* a CUDA runtime call failed (message has the CUDA error string) */
  TRG_E_UNSUPPORTED = 4
};

/* ---- library ---------------------------------------------------------------------------- */
int trg_abi_version(void);
const char* trg_last_error(void);
/* Number of kernels this library has launched in the calling process (all threads). */
int64_t trg_launch_count(void);

/* ---- A0 / K0: destination-sorted CSR ---------------------------------------------------------
 * Replaces the implicit COO->dense scatter PyG performs on the reference's edge_index tensors
 * (build_graph.py:387,394,402; local ids train_gnn.py:128-133; .flip(0) train_gnn.py:142).
 * Stable LSD radix sort by key: bit-exact with
 *     perm = argsort(key, stable); rowptr = [0, cumsum(bincount(key, N))]; col = other[perm]; eid = perm
 * Call with (other = src, key = dst) for the forward CSR and (other = dst, key = src) for the
 * transposed one.  Keys must lie in [0, n_key) (the caller validates).  col / eid may be NULL. */
size_t trg_csr_workspace_bytes(int64_t n_edges, int64_t n_key);
int trg_csr_build(const int64_t* other, const int64_t* key, int64_t n_edges, int64_t n_key,
                  int32_t* rowptr /* [n_key+1] */, int32_t* col /* [E] */, int32_t* eid /* [E] */,
                  void* workspace, size_t workspace_bytes, void* stream);

/* Stable range selection without host synchronisation (multi-GPU: the share of this step's sampled
 * negatives, train_gnn.py:272, whose post this rank owns).  key_out / other_out receive the pairs
 * (key - lo, other) with lo <= key < hi in input order, then (pad_key, pad_other) up to `capacity` entries;
 * count_out[0] = the number selected.  The consumers (trg_csr_build with n_key + 1 rows) take `capacity` as
 * their edge count, so no size ever travels to the host; the padding lands in the sentinel row.  More than
 * `capacity` selected entries abort the kernel (message + trap), never truncate silently. */
size_t trg_select_range_workspace_bytes(int64_t n);
int trg_select_range(const int64_t* key, const int64_t* other, int64_t n, int64_t lo, int64_t hi,
                     int64_t capacity, int64_t pad_key, int64_t pad_other,
                     int64_t* key_out /* [capacity] */, int64_t* other_out /* [capacity] */,
                     int32_t* count_out /* [1] */, void* workspace, size_t workspace_bytes, void* stream);

/* Long-row splitting for skewed degree distributions (all optional: pass NULL when no row is long).
 * Rows longer than the caller's threshold T are cut into <= T-edge slices ("virtual rows"); slices
 * accumulate raw fp32 partial sums which a second small kernel adds up in slice order, so the result
 * is deterministic (it equals the sequential sum to fp32 rounding, not bit for bit, for those rows).
 *   vrowptr[n_vrows+1]: edge offsets of the virtual rows (consecutive, covering every edge once);
 *   vinfo[n_vrows]    : >= 0 = the (short) row this virtual row is; < 0 = partial slot -(v+1);
 *   long_rows[n_long], long_ptr[n_long+1]: the long rows and their slot ranges;
 *   partial           : fp32 workspace [n_slots, feat]. */
typedef struct {
  const int32_t* vrowptr;
  const int32_t* vinfo;
  int64_t n_vrows;
  const int32_t* long_rows;
  const int32_t* long_ptr;
  int64_t n_long;
  float* partial;
} trg_long_rows;

/* ---- A1+A2 / K1: fused gather + segmented mean (SAGEConv propagate + MeanAggregation) ------------
 * Replaces x_j = x_src.index_select(0, src); scatter(x_j, dst, reduce='mean') inside the
 * SAGEConv calls at train_gnn.py:177-184,194-197.  mean[r] = (sum_{j in row r} x_src[col[j]]) /
 * max(deg r, 1), neighbours added in CSR order (== edge order), so fp32 results equal the CPU
 * scatter_add_ bit for bit.  inv_deg_out (nullable) receives 1 / max(deg, 1). */
int trg_sage_agg_fwd(const int32_t* rowptr, const int32_t* col, const void* x_src,
                     int64_t n_dst, int32_t feat, int dtype,
                     void* mean_out /* [n_dst, feat] dtype */, float* inv_deg_out /* [n_dst] */,
                     const trg_long_rows* long_rows /* host struct, nullable */, void* stream);

/* ---- A7 / K2: atomic-free backward of K1 w.r.t. the sources (layers >= 2) ----------------------
 * Replaces autograd of index_select + scatter-mean (index_add / gather).  Uses the transposed
 * CSR (rows = sources, col_t = destination of each edge):
 *     g_src[s] (+)= sum_{j in row s} g_mean[col_t[j]] * inv_deg[col_t[j]]   (inv_deg nullable)
 * accumulate != 0 adds to the rows already in g_src_out (autograd's gradient accumulation of a table
 * that feeds several relations, fused); relu_of (nullable, [n_src, feat] dtype) is the forward
 * activation the gradient belongs to: rows are finally gated by relu_of > 0, i.e. the ReLU backward
 * of train_gnn.py:187-198 (aten threshold_backward) fused into the last accumulating pass.
 * out_dtype = dtype, or TRG_F32 with dtype = TRG_BF16: the sums are written (and accumulated) as fp32
 * rows -- partial sums that a multi-GPU run reduces across ranks are rounded to bf16 once, after the
 * cross-rank add (trg_rows_finish), like the single-GPU kernel rounds once after its fp32 accumulation. */
int trg_sage_agg_bwd(const int32_t* rowptr_t, const int32_t* col_t, const float* inv_deg,
                     const void* g_mean, int64_t n_src, int32_t feat, int dtype,
                     void* g_src_out /* [n_src, feat] out_dtype */, int out_dtype, int accumulate,
                     const void* relu_of, const trg_long_rows* long_rows /* host struct, nullable */,
                     void* stream);

/* ---- generic weighted segmented gather-sum (used by the loss backward) ------------------------
 *     out[r] (+)= scale * sum_{j in row r} coef[eid[j]] * x[col[j]]
 * scale is a device scalar (nullable = 1); accumulate != 0 adds to out; relu_of and out_dtype as in
 * trg_sage_agg_bwd (relu_of applied after the accumulation). */
int trg_gather_wsum(const int32_t* rowptr, const int32_t* col, const int32_t* eid,
                    const float* coef, const float* scale, const void* x,
                    int64_t n_rows, int32_t feat, int dtype, void* out, int out_dtype, int accumulate,
                    const void* relu_of, const trg_long_rows* long_rows /* host struct, nullable */, void* stream);

/* ---- row-wise finish of a cross-GPU reduced table (multi-GPU only; no single-GPU counterpart) ---
 *     out[r, :] = gate( row_scale[r] * in[r, :] + add[r, :] )
 * in: [n_rows, feat] of in_dtype (TRG_F32 for fp32-transported partial sums); row_scale (nullable, fp32
 * [n_rows]) = 1 / max(global in-degree, 1) of a source-partitioned mean; add (nullable, dtype) = the local
 * gradient term of the same rows; gate: relu_of (nullable, dtype) > 0 ? value : 0 -- the ReLU backward of
 * train_gnn.py:187-198.  One pass over 1/G of a table instead of three element-wise torch kernels;
 * the arithmetic is fp32 and out is rounded to dtype once.  out may alias add. */
int trg_rows_finish(const void* in, int in_dtype, const float* row_scale, const void* add,
                    const void* relu_of, int64_t n_rows, int32_t feat, int dtype, void* out, void* stream);

/* ---- reduce-scatter FUSED with the row finish, over peer memory (multi-GPU only) ----------------
 *     out[r, :] = gate( row_scale[r] * sum_{g < n_peers} parts[g][row0 + r, :] + add[r, :] )
 * parts: HOST array of n_peers DEVICE pointers, one per rank in rank order, each the base of that rank's
 * full-height [>= row0 + n_rows, feat] table of partial sums (in_dtype: TRG_F32 or dtype), all addressable
 * from this device (cudaIpc / CUDA VMM peer mappings over NVLink; parts[own rank] is local memory).  The
 * caller owns the cross-rank ordering: every rank's table is complete before the call (a barrier on the
 * stream) and is not overwritten until every peer's call has finished.  The sum runs in rank order
 * (deterministic); row_scale / add / relu_of as in trg_rows_finish.  Replaces an NCCL reduce-scatter plus
 * trg_rows_finish: the rows cross NVLink inside the kernel's own loads and the reduced table is never
 * materialised.  ctas_per_sm (0 = default 2): CTAs of 256 threads per SM -- the kernel is latency-bound on
 * the links and is meant to run beside a compute kernel. */
int trg_peer_reduce_rows(const void* const* parts, int32_t n_peers, int64_t row0, int in_dtype,
                         const float* row_scale, const void* add, const void* relu_of, int64_t n_rows,
                         int32_t feat, int dtype, void* out, int32_t ctas_per_sm, void* stream);

/* ---- A5+A6 / K4: fused positive/negative edge score + BCE-with-logits -------------------------
 * Replaces train_gnn.py:259-281:  pos = <u[pos_u], p[pos_p]>, neg = <u[pos_u], p[neg_p]>,
 *     loss = wbar * mean(softplus(-pos)) + mean(softplus(neg)),   wbar = mean(w[pos_p + U])
 * (the reference's BCEWithLogitsLoss is a scalar mean, so its "weighted" loss is exactly this).
 * Positive edges are given grouped by user: rowptr_u/col_p/eid = trg_csr_build(other = pos_p,
 * key = pos_u).  neg_p is in ORIGINAL edge order (index it with eid).  The edges processed are
 * those of rowptr_u; n_edges is the E of the two means (the GLOBAL number of positives when the
 * caller holds one partition of them, so that partial losses and gradients add up).
 * Outputs: loss_out[1]; and when c_pos/c_neg/g_u are non-NULL the backward ingredients
 *     c_pos[e] = dloss/dpos_e,  c_neg[e] = dloss/dneg_e   (original edge order)
 *     g_u[r]   = sum_e c_pos[e] p[pos_p[e]] + c_neg[e] p[neg_p[e]]   (dloss/du, dtype rows)
 * dloss/dp is then two trg_gather_wsum calls over the post-grouped structures. */
size_t trg_edge_bce_workspace_bytes(int64_t n_users);
int trg_edge_bce_fwd(const int32_t* rowptr_u, const int32_t* col_p, const int32_t* eid,
                     const int64_t* neg_p, const void* u, const void* p,
                     int64_t n_users, int64_t n_edges, int32_t hidden, int dtype,
                     const float* wbar /* device scalar */, float* loss_out,
                     float* c_pos, float* c_neg, void* g_u,
                     void* workspace, size_t workspace_bytes, void* stream);

/* Multi-GPU form of K4: the loss terms are evaluated by the OWNER OF THE POST.  Rows = local posts
 * (anchor table), one gathered row per edge from the all-gathered user table (5x smaller than the
 * post table), one label per launch: label 1 = positive edges (loss += wbar * sum softplus(-x) / E),
 * label 0 = sampled negatives (loss += sum softplus(x) / E); E = n_edges_scale, the global positive
 * count.  loss_out[0] receives this launch's partial loss; coef_out[eid] = dloss/dx per edge (eid NULL:
 * coef_out is written in CSR edge order, i.e. sequentially -- no scattered 4-byte stores);
 * g_anchor (+)= sum_e coef_e * gathered[col_e] (accumulate != 0 adds to the rows already there);
 * relu_gate != 0 finally zeroes g_anchor where the anchor row itself is <= 0 (the anchor table is the
 * output of the last layer's ReLU, so this is that ReLU's backward, at no extra traffic). */
int trg_edge_anchor_loss(const int32_t* rowptr, const int32_t* col, const int32_t* eid,
                         const void* anchor, const void* gathered, int64_t n_rows,
                         int64_t n_edges_scale, int32_t hidden, int dtype, int label,
                         const float* wbar, float* loss_out, float* coef_out, void* g_anchor,
                         int accumulate, int relu_gate, void* workspace, size_t workspace_bytes,
                         void* stream);

/* ---- A3+A4 / K3: SAGE projections + relation combine + ReLU ---------------------------------
 * Replaces lin_l(mean) + lin_r(x_dst) of every SAGEConv and the combine of
 * train_gnn.py:187-198.  out = act( sum_i alpha_i * ( A_i[n, k_i] @ W_i[h, k_i]^T ) + bias ),
 * up to 4 (A, W) pairs (user rows: mean_direct, mean_social, x; post rows: mean, x).
 * fp32 inputs are multiplied as 3xTF32 split products on tcgen05 (fp32-accurate), bf16 inputs as
 * kind::f16 with fp32 TMEM accumulation (hidden in {64,128,256}, k_i a multiple of 128 bytes);
 * other shapes take a strict-fp32 FMA kernel.  The bf16 tensor-core path stores alpha_i * W_i as its
 * bf16 weight operand, so an alpha that is not a power of two rounds that product once (2^-9 relative).
 * Workspace: trg_sage_proj_workspace_bytes. */
typedef struct {
  const void* a;      /* [n_rows, k] dtype, row-major, 16B-aligned */
  const void* w;      /* [hidden, k] dtype, row-major (torch Linear.weight layout) */
  int32_t k;
  float alpha;
} trg_proj_term;
size_t trg_sage_proj_workspace_bytes(int32_t k_total, int32_t hidden, int dtype);
int trg_sage_proj_fwd(const trg_proj_term* terms /* host */, int32_t n_terms,
                      const float* bias /* [hidden] fp32, nullable; already alpha-combined */,
                      int64_t n_rows, int32_t hidden, int dtype, int relu,
                      void* out /* [n_rows, hidden] dtype */,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Input-gradient half of the backward of trg_sage_proj_fwd (autograd of F.linear at
 * train_gnn.py:283, needed for layers >= 2):  d_a_i = row_scale_i * ( alpha_i * dZ @ W_i ),
 * dZ[n_rows, hidden] = dOut masked by the ReLU.  row_scale (nullable, fp32 [n_rows]) fuses the
 * 1/deg of the mean aggregation so that K2 is a plain gather-sum.  All k_i must be equal for the
 * tensor-core path.  bf16 rounds alpha_i * W_i to bf16 once, as the forward's tensor-core path does. */
typedef struct {
  const void* w;          /* [hidden, k] dtype */
  int32_t k;
  float alpha;
  const float* row_scale; /* nullable */
  void* d_a;              /* [n_rows, k] dtype, out */
} trg_proj_bwd_term;
int trg_sage_proj_bwd_input(const void* dz, const trg_proj_bwd_term* terms /* host */, int32_t n_terms,
                            int64_t n_rows, int32_t hidden, int dtype,
                            void* workspace, size_t workspace_bytes, void* stream);

/* Weight-gradient half: dW_i = alpha_i * dZ^T @ A_i (reduction over the node rows) and
 * db = column sums of dZ (nullable).  Both operands are consumed MN-major from the row-major
 * tables by tcgen05 (3xTF32 for fp32); per-CTA partials are reduced in a fixed order
 * (deterministic).  n_rows = 0 writes dW = 0 and db = 0.  Workspace: trg_sage_proj_dw_workspace_bytes(). */
typedef struct {
  const void* a;   /* [n_rows, k] dtype */
  int32_t k;
  float alpha;
  void* d_w;       /* [hidden, k] dtype, out */
} trg_proj_dw_term;
size_t trg_sage_proj_dw_workspace_bytes(void);
int trg_sage_proj_bwd_weight(const void* dz, const trg_proj_dw_term* terms /* host */, int32_t n_terms,
                             float* d_bias /* [hidden] fp32, nullable */,
                             int64_t n_rows, int32_t hidden, int dtype,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ---- A9+A10 / K5: score contraction + top-k ---------------------------------------------------
 * Replaces scores = torch.mm(user_emb, known_post_emb.T); torch.topk(scores, min(K, n))
 * (inference.py:427-428; train_gnn.py:335-341).  Never materialises the score matrix.  Total
 * order: score descending, id ascending.  ids_out are global: local + id_offset (shards).
 * k_out = min(k, n_cat) columns are written; rows are q rows. */
size_t trg_score_topk_workspace_bytes(int64_t n_query, int64_t n_cat, int32_t hidden, int32_t k);
int trg_score_topk(const void* q /* [B, H] */, const void* cat /* [P, H] */,
                   int64_t n_query, int64_t n_cat, int32_t hidden, int dtype, int32_t k,
                   int64_t id_offset, float* vals_out /* [B, k_out] */, int64_t* ids_out /* [B, k_out] */,
                   void* workspace, size_t workspace_bytes, void* stream);
/* trg_score_topk with a per-query list of posts that must not be returned (e.g. the posts a user has
 * already engaged with).  The exclusion index is a CSR over "exclusion rows":
 *   excl_rowptr int32[R+1]; excl_ids int32[nnz] holding GLOBAL post ids (the id space of ids_out:
 *   local + id_offset), ascending within each row.  Duplicates are allowed, and so are ids outside the
 *   catalogue or shard (they never match).
 * Query b uses exclusion row query_rows[b], or row b when query_rows is NULL.  The result of query b is
 * the top k_out = min(k, n_cat) posts of the catalogue with that row's ids removed, under the same total
 * order (score desc, id asc).  A row with fewer than k_out admissible posts is padded at its tail with
 * (-inf, -1); the output stays [B, k_out].  An empty exclusion row gives exactly trg_score_topk's result.
 * excl_rowptr == NULL means no exclusions (then this is trg_score_topk); excl_ids must be non-NULL when
 * excl_rowptr is given.  The index is read on the device only (no host sync).  Same workspace as
 * trg_score_topk (trg_score_topk_workspace_bytes). */
int trg_score_topk_excluding(const void* q /* [B, H] */, const void* cat /* [P, H] */,
                             int64_t n_query, int64_t n_cat, int32_t hidden, int dtype, int32_t k,
                             int64_t id_offset, const int32_t* excl_rowptr /* [R+1] */,
                             const int32_t* excl_ids /* [nnz] */, const int64_t* query_rows /* [B], nullable */,
                             float* vals_out /* [B, k_out] */, int64_t* ids_out /* [B, k_out] */,
                             void* workspace, size_t workspace_bytes, void* stream);
/* Merge n_lists per-row sorted (vals, ids) lists of length k_in into the top k_out. */
int trg_topk_merge(const float* vals_in /* [B, n_lists*k_in] */, const int64_t* ids_in,
                   int64_t n_query, int32_t n_lists, int32_t k_in, int32_t k_out,
                   float* vals_out, int64_t* ids_out, void* stream);

/* Exact re-ranking of per-query candidate lists (the second stage of a top-k whose first stage ran on
 * TRG_F8E4M3 copies of the tables).  dtype TRG_F32 or TRG_BF16; q [B, H] and table [P, H] row-major and
 * 16-byte aligned; cand_ids int64 [B, n_cand] GLOBAL post ids (the id space of ids_out: local + id_offset).
 * Candidate g of query b, when id_offset <= g < id_offset + n_table, scores
 *     s = 0; for h = 0 .. H-1: s = fmaf(float(q[b][h]), float(table[g - id_offset][h]), s)
 * -- the order of trg_score_topk's fp32 kernel, so an fp32 table gives its scores bit for bit.  Candidates
 * with id -1 or outside that range are skipped (never read).  Candidates are expected to be distinct.
 * The top k_out = min(k, n_cand) <= 128 of each row under (score desc, id asc) are written to
 * vals_out / ids_out [B, k_out]; a row with fewer valid candidates is padded at its tail with (-inf, -1). */
size_t trg_rescore_topk_workspace_bytes(int64_t n_query, int32_t n_cand);
int trg_rescore_topk(const void* q /* [B, H] */, const void* table /* [P, H] */, int64_t n_query, int64_t n_table,
                     int32_t hidden, int dtype, const int64_t* cand_ids /* [B, n_cand] */, int32_t n_cand,
                     int64_t id_offset, int32_t k, float* vals_out /* [B, k_out] */,
                     int64_t* ids_out /* [B, k_out] */, void* workspace, size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* TRG_B200_H */
