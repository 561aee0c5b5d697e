/* gmlm_b200.h — C ABI of libgmlm_b200.so: B200 (sm_100a) kernels for the message-passing
 * hot path of chungimungi/GMLM (the GNN encoder of /root/reference/main.py:250-320).
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch/ATen types.
 *   - Every pointer is a DEVICE pointer unless the parameter name ends in `_host`.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - Row-major dense matrices with an explicit leading dimension in ELEMENTS.
 *   - Return value: 0 = ok; GMLM_ERR_* otherwise; gmlm_last_error() gives the thread-local
 *     message.  Kernels never allocate, free or retain memory; scratch is passed in as
 *     (ws, ws_bytes) and sized by the matching *_workspace_bytes() query.
 *   - Nothing here touches the host CPU for arithmetic: there is no CPU fallback.
 *
 * Each entry point names the reference interface it replaces (file:line in
 * /root/reference/main.py; [PyG] = the torch_geometric operator imported at main.py:6-7).
 */
#ifndef GMLM_B200_H_
#define GMLM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GMLM_OK 0
#define GMLM_ERR_INVALID 1   /* bad argument (shape / dtype / alignment / size limits) */
#define GMLM_ERR_CUDA 2      /* a CUDA runtime call or launch failed */
#define GMLM_ERR_INDEX 3     /* an index (node id / relation id) is out of range */
#define GMLM_ERR_WORKSPACE 4 /* workspace too small */

/* element types of dense feature matrices */
#define GMLM_F32 0
#define GMLM_BF16 1
#define GMLM_F16 2   /* GEMM operands only (torch.amp.autocast's matmul dtype) */

/* aggregation modes of gmlm_spmm_csr */
#define GMLM_AGG_SUM 0      /* out[r] = sum_e x[col[e]]                       */
#define GMLM_AGG_MEAN 1     /* out[r] = sum_e x[col[e]] / max(1, |row r|)     */
#define GMLM_AGG_WEIGHTED 2 /* out[r] = sum_e w[e] * x[col[e]]                */

int gmlm_abi_version(void);
const char* gmlm_last_error(void);
/* tuning knobs for A/B measurements: key in {"spmm_variant","spmm_unroll","spmm_overlap","halo_pull_ctas","halo_pull_threads"};
 * returns old value (halo_pull_*: launch shape of gmlm_gather_rows_ptr when a pull shares the GPU with an aggregation) */
int gmlm_set_tuning(const char* key, int value);

/* ---- A1  degree()  [PyG] torch_geometric.utils.degree, called main.py:65 and main.py:256 ----
 * deg[i] = |{e : index[e] == i}|.  int32 counts are exact; the f32 variant is what the
 * reference returns (float32[N]); identical bits while every degree < 2^24.
 * Out-of-range indices are skipped and make the call return GMLM_ERR_INDEX when
 * `check_host_sync` != 0 (costs one stream synchronisation). */
int gmlm_degree_i32(const int64_t* index, int64_t num_edges, int64_t num_nodes, int32_t* deg,
                    int check_host_sync, void* stream);
/* the same over the edges with keep[e] != 0 only (N3: the reference's 10 % edge dropout `augment_graph`,
 * main.py:832-837, fused into the histogram instead of materialising a filtered edge_index; keep NULL = all) */
int gmlm_degree_i32_masked(const int64_t* index, const uint8_t* keep, int64_t num_edges, int64_t num_nodes,
                           int32_t* deg, int check_host_sync, void* stream);
int gmlm_degree_f32(const int64_t* index, int64_t num_edges, int64_t num_nodes, float* deg,
                    int32_t* deg_i32_ws /* [num_nodes] scratch */, int check_host_sync, void* stream);

/* ---- A2  degree-bucket edge typing, the per-edge Python loop main.py:253-267 ----
 * edge_type[e] = #{k : deg[src[e]] > bounds_host[k]}   (bounds ascending; reference: {2,5,10}) */
int gmlm_edge_type_bucket(const int64_t* src, int64_t num_edges, const int32_t* deg, int64_t num_nodes,
                          const int32_t* bounds_host, int num_bounds, int64_t* edge_type, void* stream);

/* per-relation edge counts (host decides which relations are populated; SURVEY §0 fact 5) */
int gmlm_relation_histogram(const int64_t* edge_type, const uint8_t* keep /* NULL = all edges */, int64_t num_edges,
                            int num_relations, int64_t* counts /* [num_relations] */, void* stream);

/* ---- content key of an int64 index tensor (graph cache: the reference re-creates edge_type on every call,
 *      main.py:255, so tensor identity cannot key the cached CSR) ----
 * out2[0], out2[1] = two position-weighted 64-bit sums of x[0..n) (order-independent integer atomics). */
int gmlm_checksum_i64(const int64_t* x, int64_t n, uint64_t* out2, void* stream);

/* ---- A3  (dst,rel)-keyed CSR: replaces the per-relation boolean-mask compaction inside
 *          [PyG] RGCNConv.forward (called main.py:272,285,298,308) ----
 * Segment id s = dst*num_slots + slot_of_rel_host[edge_type[e]]  (edge_type may be NULL: slot 0).
 * Stable in original edge order.
 * dst in [0,num_dst), src in [0,num_src)  (equal for a whole graph; num_src > num_dst for a
 * destination-row partition whose columns include halo rows).  Outputs:
 *   rowptr int32[num_dst*num_slots+1], col int32[E] (= src), perm int32[E] (= original edge),
 *   seg_of_edge int32[E] (segment of ORIGINAL edge e; may be NULL).
 * Synchronises the stream once to report GMLM_ERR_INDEX. */
size_t gmlm_csr_workspace_bytes(int64_t num_edges, int64_t num_rows);
/* keep (N3, optional): uint8 [num_edges] edge-dropout mask (main.py:832-837 `augment_graph`) fused into the build: a
 * dropped edge is not counted and sorts behind every kept edge, so rowptr[num_dst*num_slots] = *nnz_host = the
 * number of kept edges and only the first nnz entries of col / perm are the CSR (seg_of_edge of a dropped edge is
 * num_dst*num_slots).  Equal, array for array, to building from edge_index[:, keep]. */
int gmlm_csr_build(const int64_t* src, const int64_t* dst, const int64_t* edge_type, const uint8_t* keep,
                   int64_t num_edges, int64_t num_dst, int64_t num_src, int num_relations,
                   const int32_t* slot_of_rel_host, int num_slots,
                   int32_t* rowptr, int32_t* col, int32_t* perm, int32_t* seg_of_edge, int64_t* nnz_host,
                   void* ws, size_t ws_bytes, void* stream);

/* ---- A14 transposed CSR for the backward gather (autograd of index_select/scatter_add in
 *          [PyG] MessagePassing.propagate) ----
 * rows = `row_of_edge` (e.g. src) in [0,num_rows); payload_t[i] = payload[perm_t[i]];
 * if fwd_rowptr != NULL: w_t[i] = 1 / (fwd_rowptr[p+1]-fwd_rowptr[p]) with p = payload_t[i]
 * (the mean divisor folded in); else if edge_w != NULL: w_t[i] = edge_w[perm_t[i]]; else w_t untouched. */
int gmlm_csr_transpose(const int64_t* row_of_edge, const int32_t* payload, const float* edge_w,
                       const int32_t* fwd_rowptr, const uint8_t* keep /* as in csr_build; NULL = all */,
                       int64_t num_edges, int64_t num_rows,
                       int32_t* rowptr_t, int32_t* payload_t, float* w_t, int32_t* perm_t,
                       void* ws, size_t ws_bytes, void* stream);

/* ---- transform-first plan (A5+A6 for layers whose output is narrower than their input) ----
 * [PyG] RGCNConv computes sum_r mean_r(x) @ W_r + x @ root (main.py:272); because the mean is linear this equals
 * sum_r mean_r(x @ W_r) + (x @ root), so when (S+1)*Fo < S*Fi the dense transform Z = x @ [W_0|..|W_{S-1}|root]
 * runs FIRST and the aggregation gathers Fo-wide slabs of Z; H [N, S*Fi] is never materialised.  This call
 * re-reads the (dst,rel) CSR as a dst-keyed CSR over the rows of Z viewed as [num_src*(S+1), Fo]:
 *   row i        = the edges of segments i*S .. i*S+S-1 in CSR order, then one self entry for the root slab
 *   col_d        = src*(S+1) + slot   (self entry: i*(S+1) + S)
 *   w_d          = 1/|segment|        (self entry: 1)         dst_d = i  (payload for gmlm_csr_transpose)
 * Sizes: rowptr_d [N+1], col_d / w_d / dst_d [E+N]. */
int gmlm_dst_plan(const int32_t* rowptr, const int32_t* col, int64_t num_dst, int num_slots, int64_t num_edges,
                  int64_t num_src, int32_t* rowptr_d, int32_t* col_d, float* w_d, int32_t* dst_d, void* stream);

/* ---- hub plan: rows longer than `thresh` are split into chunks of `thresh` edges so that the
 *      aggregation stays balanced AND deterministic on power-law graphs ----
 * count: counts_host[0] = #hub rows, counts_host[1] = #chunks (synchronises).
 * fill : hub_row[n_hub], hub_chunk_ptr[n_hub+1], chunk_beg[n_chunks], chunk_end[n_chunks]. */
int gmlm_hub_count(const int32_t* rowptr, int64_t num_rows, int32_t thresh, int64_t* counts_host,
                   void* ws, size_t ws_bytes, void* stream);
int gmlm_hub_fill(const int32_t* rowptr, int64_t num_rows, int32_t thresh, int64_t n_hub, int64_t n_chunks,
                  int32_t* hub_row, int32_t* hub_chunk_ptr, int32_t* chunk_beg, int32_t* chunk_end,
                  void* ws, size_t ws_bytes, void* stream);

/* ---- band-ordered hub plan (512-byte rows of gmlm_spmm_csr_banded) ----
 * The edges of every hub row sorted by source (stable: ties keep CSR order), so that the chunks gathering from one
 * band of 2^band_shift source rows can run together and find those rows in L2.
 * hub_off[n_hub+1]: hub_off[h] = edges of hub rows before h (exclusive scan of the hub row lengths).
 * band_sort : hub_col[n_hub_edges] (and hub_w, when w is given) = col / w of the hub rows, row by row, each row by
 *             source; band_chunk_ptr[n_hub+1] = the row -> chunk pointer of the band cuts; *n_band_host = #chunks.
 *             A band boundary inside a row is a cut when both sides hold >= min_run edges; pieces between cuts are
 *             cut every `thresh` edges.
 * band_order: band_plan = [band_chunk_ptr (n_hub+1, copied in by the caller) | cut (n_band+1) | chunk_order (n_band)];
 *             chunk c covers hub_col[cut[c], cut[c+1]); chunk_order = chunk ids stably sorted by the band of their
 *             first edge. */
size_t gmlm_hub_band_workspace_bytes(int64_t n_hub_edges);
int gmlm_hub_band_sort(const int32_t* rowptr, const int32_t* col, const float* w, int64_t n_hub, const int32_t* hub_row,
                       const int32_t* hub_off, int64_t n_hub_edges, int band_shift, int32_t thresh, int32_t min_run,
                       int32_t* hub_col, float* hub_w, int32_t* band_chunk_ptr, int64_t* n_band_host, void* ws,
                       size_t ws_bytes, void* stream);
int gmlm_hub_band_order(const int32_t* hub_col, const int32_t* hub_off, int64_t n_hub, int64_t n_hub_edges,
                        int64_t n_band, int band_shift, int32_t thresh, int32_t min_run, int32_t* band_plan, void* ws,
                        size_t ws_bytes, void* stream);

/* ---- cost-balanced group plan for gmlm_spmm_csr ----
 * Cuts the row sequence where (r + rowptr[r]) crosses multiples of `quantum`, so that every
 * group of lanes moves about `quantum` row-sized units (one per gathered edge + one per written
 * row) whatever the degree distribution.  n_groups = gmlm_group_plan_size(); grp_row has
 * n_groups+1 entries, grp_row[g] = first row of group g, grp_row[n_groups] = num_rows. */
int64_t gmlm_group_plan_size(int64_t num_rows, int64_t nnz, int64_t quantum);
int gmlm_group_plan(const int32_t* rowptr, int64_t num_rows, int64_t nnz, int64_t quantum,
                    int32_t* grp_row, void* stream);

/* ---- A5 / A14  aggregation: [PyG] RGCNConv.propagate + mean aggregation (forward) and the
 *      gather-form backward.  out[r, :] = reduce_{e in row r} w[e] * x[col[e], :] ----
 * x: [*, feat] dtype, leading dim ldx; out: [num_rows, feat] same dtype, leading dim ldo.
 * fp32 accumulation in CSR order (deterministic).  grp_row may be NULL (uniform 32-row groups).
 * w is [nnz, w_heads]: w_heads = 1 is one scalar per edge; w_heads = H > 1 (GAT attention, row A9)
 * gives head h its own weight column for the features [h*feat/H, (h+1)*feat/H).
 * Hub arrays may be NULL when n_hub == 0; hub_ws: float[n_chunks * feat] scratch. */
int gmlm_spmm_csr(const void* x, int dtype, int64_t feat, int64_t ldx,
                  const int32_t* rowptr, const int32_t* col, const float* w, int32_t w_heads,
                  int64_t num_rows, int mode, const int32_t* grp_row, int64_t n_groups,
                  int32_t hub_thresh, int64_t n_hub, int64_t n_chunks, const int32_t* hub_row,
                  const int32_t* hub_chunk_ptr, const int32_t* chunk_beg, const int32_t* chunk_end,
                  float* hub_ws, void* out, int64_t ldo, void* stream);
/* gmlm_spmm_csr with the band-ordered hub plan (gmlm_hub_band_sort / _order) of the same CSR: rows of exactly 512
 * bytes (F = 256 bf16 / 128 fp32, no head slabs, one weight column) gather their hub chunks from hub_col / hub_w in
 * chunk_order, so that one band of source rows is served from L2; other widths use the chunk plan above.  band_plan
 * NULL (or hub_w NULL in weighted mode) = the chunk plan above for every width.  hub_ws holds
 * max(n_chunks, n_band) * feat floats.  gmlm_spmm_csr is this call without a band plan. */
int gmlm_spmm_csr_banded(const void* x, int dtype, int64_t feat, int64_t ldx,
                         const int32_t* rowptr, const int32_t* col, const float* w, int32_t w_heads,
                         int64_t num_rows, int mode, const int32_t* grp_row, int64_t n_groups,
                         int32_t hub_thresh, int64_t n_hub, int64_t n_chunks, const int32_t* hub_row,
                         const int32_t* hub_chunk_ptr, const int32_t* chunk_beg, const int32_t* chunk_end,
                         int64_t n_band, const int32_t* band_plan, const int32_t* hub_col, const float* hub_w,
                         float* hub_ws, void* out, int64_t ldo, void* stream);

/* ---- A7  GraphNorm  [PyG] torch_geometric.nn.GraphNorm(batch=None), called main.py:273,286,299,309 ----
 * stats: colsum[c] = sum_i x[i,c], colsq[c] = sum_i x[i,c]^2 in fp64 (deterministic two-stage).
 * fwd  : mu = colsum/N; o = x - mu*mean_scale; var = E[o^2]; y = weight*o/sqrt(var+eps)+bias,
 *        optionally followed by exact-erf GELU (main.py:274) when fuse_gelu != 0.
 * bwd  : grads for x, weight, bias, mean_scale (through the optional GELU).
 * stat_rows: the row count the sums were taken over (the divisor of the statistics).  0 = num_rows.  A rank of
 *        a row partition passes the all-reduced WHOLE-GRAPH sums and stat_rows = N_global while num_rows is its
 *        own (possibly zero) row count; the parameter gradients that come out are then whole-graph values. */
size_t gmlm_colstats_workspace_bytes(int64_t num_rows, int64_t channels);
int gmlm_colstats(const void* x, int dtype, int64_t num_rows, int64_t channels, int64_t ldx,
                  double* colsum, double* colsq, void* ws, size_t ws_bytes, void* stream);
int gmlm_graphnorm_fwd(const void* x, int dtype, int64_t num_rows, int64_t channels, int64_t ldx,
                       const double* colsum, const double* colsq, const float* weight, const float* bias,
                       const float* mean_scale, float eps, int fuse_gelu, void* y, int64_t ldy,
                       float* mean_out /* [C] */, float* rstd_out /* [C] */, int64_t stat_rows, void* stream);
int gmlm_graphnorm_bwd_stats(const void* x, const void* gy, int dtype, int64_t num_rows, int64_t channels,
                             int64_t ldx, int64_t ldg, const float* mean, const float* rstd,
                             const float* weight, const float* bias, const float* mean_scale, int fuse_gelu,
                             double* sum_g /* [C] sum of dL/dn */, double* sum_go /* [C] sum dL/dn * ohat */,
                             void* ws, size_t ws_bytes, void* stream);
int gmlm_graphnorm_bwd_apply(const void* x, const void* gy, int dtype, int64_t num_rows, int64_t channels,
                             int64_t ldx, int64_t ldg, const float* mean, const float* rstd,
                             const float* weight, const float* bias, const float* mean_scale, int fuse_gelu,
                             const double* sum_g, const double* sum_go, void* gx, int64_t ldgx,
                             float* g_weight, float* g_bias, float* g_mean_scale, int64_t stat_rows,
                             void* stream);

/* ---- A11 soft node masking, soft_masking_gnn_input main.py:92-99 ----
 * fwd: y = x; y[m] = (1-beta)*x[m] + beta*token.   bwd: g_token = beta * sum_{m} gy[m]; gx (optional)
 * = gy * (m ? 1-beta : 1). */
int gmlm_soft_mask_fwd(const void* x, int dtype, int64_t num_rows, int64_t feat, int64_t ldx,
                       const uint8_t* mask, const float* token, float beta, void* y, int64_t ldy, void* stream);
size_t gmlm_soft_mask_bwd_workspace_bytes(int64_t num_rows, int64_t feat);
int gmlm_soft_mask_bwd(const void* gy, int dtype, int64_t num_rows, int64_t feat, int64_t ldg,
                       const uint8_t* mask, float beta, float* g_token /* [feat] */, void* gx /* may be NULL */,
                       int64_t ldgx, void* ws, size_t ws_bytes, void* stream);

/* ---- A13 LayerNorm closing MultiScaleFusion (main.py:171,180 `self.layer_norm(fused)`, the last op of
 *          get_graph_embeddings main.py:320) ----
 * fwd: y = (x - mean_row) * rstd_row * gamma + beta   (biased variance, eps inside the sqrt; nn.LayerNorm)
 * bwd: gx (may be NULL), g_gamma[c] = sum_i gy*xhat, g_beta[c] = sum_i gy  (either may be NULL).
 * channels: multiple of 4 (f32) / 8 (bf16), <= gmlm_layernorm_max_channels(dtype); 16-byte aligned rows. */
int64_t gmlm_layernorm_max_channels(int dtype);
int gmlm_layernorm_fwd(const void* x, int dtype, int64_t num_rows, int64_t channels, int64_t ldx,
                       const float* gamma, const float* beta, float eps, void* y, int64_t ldy,
                       float* mean_out /* [rows] */, float* rstd_out /* [rows] */, void* stream);
size_t gmlm_layernorm_bwd_workspace_bytes(int64_t num_rows, int64_t channels);
int gmlm_layernorm_bwd(const void* x, const void* gy, int dtype, int64_t num_rows, int64_t channels, int64_t ldx,
                       int64_t ldg, const float* gamma, const float* mean, const float* rstd, void* gx,
                       int64_t ldgx, float* g_gamma, float* g_beta, void* ws, size_t ws_bytes, void* stream);

/* ---- A4  basis composition: [PyG] RGCNConv.forward `weight = (comp @ weight.view(num_bases, -1)).view(R, Fi, Fo)`
 *          (modules built main.py:189,193,197,201; upstream recomputes it on every call) ----
 * W_s[i,o] = sum_b comp[rel_of_slot_host[s], b] * basis[b,i,o] for the `num_slots` populated relations
 * (comp NULL: W_s = basis[rel_of_slot_host[s]], the layer without basis decomposition), plus `root` as one more slab
 * (NULL: none).  ONE pass over the fp32 bases writes the result in the GEMM operand type `out_dtype`
 * (GMLM_F32 / GMLM_BF16 / GMLM_F16) and in up to two layouts (either pointer may be NULL):
 *   out_n[s*n_slot_stride + i*n_row_stride + o]   root at n_root_off   ("natural": B operand of [dH|dx] = g W^T)
 *   out_t[s*t_slot_stride + o*t_row_stride + i]   root at t_root_off   ("transposed": B operand of out = [H|x] W)
 * so that neither the index_select of the populated relations, nor the concatenation with root, nor the cast, nor
 * the transposition is a separate pass.  Strides and offsets in elements. */
int gmlm_basis_compose(const float* comp, const float* basis, const float* root, const int32_t* rel_of_slot_host,
                       int num_slots, int num_relations, int num_bases, int64_t in_channels, int64_t out_channels,
                       int out_dtype, void* out_n, int64_t n_slot_stride, int64_t n_row_stride, int64_t n_root_off,
                       void* out_t, int64_t t_slot_stride, int64_t t_row_stride, int64_t t_root_off, void* stream);
/* backward of the composition (autograd of the matmul above): dw = gradient of the composed weights in the natural
 * strided layout, fp32;  dbasis[b,i,o] = sum_s comp[rel_s,b] dw_s[i,o]  (NULL: skipped),
 * dcomp[r,b] = sum_{i,o} dw_{slot(r)}[i,o] basis[b,i,o], zero rows for relations without a slot (NULL: skipped).
 * One pass over the bases; per-CTA partials + fixed-order fp64 final sum (deterministic).  out_channels and the
 * strides must be multiples of 4; 1..8 slots, <= 64 relations. */
size_t gmlm_basis_compose_bwd_workspace_bytes(int num_slots, int num_relations, int num_bases, int64_t in_channels,
                                              int64_t out_channels);
int gmlm_basis_compose_bwd(const float* comp, const float* basis, const float* dw, int64_t slot_stride,
                           int64_t row_stride, const int32_t* rel_of_slot_host, int num_slots, int num_relations,
                           int num_bases, int64_t in_channels, int64_t out_channels, float* dbasis, float* dcomp,
                           void* ws, size_t ws_bytes, void* stream);

/* ---- A6  dense feature transform on tcgen05 tensor cores (TMA tiles, TMEM accumulator):
 *          [PyG] RGCNConv.forward `out += h @ W[r]` / `out += x @ root` / `+ bias`, main.py:272 ----
 * C[M,N] = [A1 | A2][M, K1+K2] * B[N, K1+K2]^T + bias[N];  A1, A2, B bf16 row-major (K contiguous),
 * fp32 accumulation, C bf16 or fp32.  Output columns [0,N1) go to C1 and [N1,N) to C2 (N1 <= 0 or
 * >= N: everything to C1).  Any K1, K2, N, N1: partial 64-column blocks of a source are zero-filled by the TMA,
 * partial output tiles are clipped by the TMA store; row pitches must be multiples of 16 bytes. */
int gmlm_gemm_nt_bf16(const void* A1, int64_t lda1, int64_t K1, const void* A2, int64_t lda2, int64_t K2,
                      const void* B, int64_t ldb, const float* bias, int64_t M, int64_t N, void* C1, int64_t ldc1,
                      int64_t N1, void* C2, int64_t ldc2, int out_dtype, void* stream);
/* the same with the operand type given: in_dtype = GMLM_BF16 or GMLM_F16 (fp16 is what torch.amp.autocast feeds
 * the reference's matmuls, main.py:446,543) */
int gmlm_gemm_nt(const void* A1, int64_t lda1, int64_t K1, const void* A2, int64_t lda2, int64_t K2,
                 const void* B, int64_t ldb, const float* bias, int64_t M, int64_t N, void* C1, int64_t ldc1,
                 int64_t N1, void* C2, int64_t ldc2, int in_dtype, int out_dtype, void* stream);
/* the general form: A = [A_0 | .. | A_{n-1}] from up to 4 sources (one tensor map each: the layer outputs that feed
 * MultiScaleFusion, main.py:176-180, are never concatenated), operands GMLM_BF16 / GMLM_F16 or GMLM_F32 (fp32 operands
 * run as 3xTF32: hi/lo split in shared memory, three tf32 MMAs per k-step; fp32 output), and an optional addend [M,N]
 * of the output type read in the epilogue: C = A B^T + bias + addend (the residual adds `x1 + residual_proj1(x_feat)`,
 * main.py:281-282, 294-295, folded into the projection; single output only).  The N = sum N_i output columns go to
 * `num_outputs` matrices: one, two with any split, or up to four cut at multiples of 64 columns (the input gradients of
 * the fusion land contiguous per layer).  A_host / lda_host / K_host / C_host / ldc_host / N_host are HOST arrays;
 * every source but the last must be a multiple of 16 bytes wide (its columns of B start on a 16-byte boundary). */
int gmlm_gemm_nt_multi(int num_sources, const void* const* A_host, const int64_t* lda_host, const int64_t* K_host,
                       const void* B, int64_t ldb, const float* bias, const void* addend, int64_t ld_add, int64_t M,
                       int num_outputs, void* const* C_host, const int64_t* ldc_host, const int64_t* N_host,
                       int in_dtype, int out_dtype, void* stream);

/* ---- A14 weight gradients on the tensor cores: D[sum K_i, N] (fp32) = [A_0 | A_1 | ..]^T . G, the reduction over all
 *      M rows (nodes) that autograd of [PyG] RGCNConv.forward's `h @ weight[r]`, `x @ root` (main.py:272) and of the
 *      residual / fusion linears (main.py:176-180, 205-207) needs: dW = H^T g, droot = x^T g, dWt = g^T x.
 * A_i [M, K_i] and G [M, N] are read as they lie in memory (row-major activations = MN-major tensor-core operands,
 * 64x64 TMA boxes), bf16 or fp16, fp32 accumulation in TMEM.  The M range is split over CTAs; partial sums go
 * through `ws` and are added in split order (deterministic).  Any sizes; row pitches multiples of 16 bytes. */
size_t gmlm_gemm_tn_workspace_bytes(int num_sources, const int64_t* K_host, int64_t M, int64_t N);
int gmlm_gemm_tn(int num_sources, const void* const* A_host, const int64_t* lda_host, const int64_t* K_host,
                 const void* G, int64_t ldg, int64_t M, int64_t N, float* D, int64_t ldd, int in_dtype, void* ws,
                 size_t ws_bytes, void* stream);

/* ---- A8 / A9 (extensions named by north_star; no counterpart in /root/reference: semantics = upstream GCNConv /
 *      GATConv defaults, restated in oracle/pyg_ref.py) on a dst-keyed CSR with upstream's self-loop handling ----
 * gcn_edge_weights: w[e] = deg[col[e]]^-1/2 * deg[row]^-1/2, deg = CSR row length (self-loops included); the GCN
 *                   aggregation itself is gmlm_spmm_csr in weighted mode.
 * segment_sum_f32 : out[r,h] = sum_{i in row r} vals[idx[i],h]  (idx NULL = identity; one warp per row)
 *
 * gat_fused_fwd   : out[i,h,:] = sum_{e->i} alpha[e,h] z[col[e],h,:],  alpha = softmax over the in-edges of i of
 *                   leaky_relu(a_src[col[e],h] + a_dst[i,h]) (+1e-16 in the denominator, as upstream), optional
 *                   attention dropout on alpha.  ONE pass with an online softmax: the score is computed where the
 *                   source row is gathered and alpha is never materialised; m_out / l_out [rows, H] keep each row's
 *                   maximum and normaliser for the backward.  Rows longer than hub_thresh use the CSR's hub plan
 *                   (chunk partials merged by the split-softmax identity, chunk order => deterministic).
 * gat_bwd_edges   : per edge alpha_eff[e,h] (alpha * keep / (1-p): the weights of the transposed aggregation of g),
 *                   d_score[e,h] (gradient of the raw score) and da_dst[i,h] = sum_e d_score;  t[i,h] must hold
 *                   <g[i,h,:], out[i,h,:]>.  da_src and dz are gathers over the transposed CSR (segment_sum_f32,
 *                   gmlm_spmm_csr with one weight column per head).
 * gat_dropout_mask: keep[i] of the counter-based hash both kernels use (index = CSR position * H + head).
 * gat_loop_fill   : per-edge scores alpha [E_in, H] (input order) -> a_edge [nnz, H] (forward-CSR order):
 *                   a_edge[k] = alpha[csr_src[k]] for every entry but the row's loop entry loop_csr[r], which gets
 *                   the mean of the row's other entries, 0 without any (upstream add_self_loops(fill_value="mean")).
 *                   One warp per row; deterministic.
 * gat_loop_fill_bwd: d_alpha[j] = g[in2csr[j]] + g[loop_csr[in_dst[j]]] / cnt(in_dst[j]), cnt = the row's entries
 *                   other than its loop clamped at 1; d_alpha[j] = 0 where in2csr[j] < 0 (an input self-loop).
 *
 * gat_fused_fwd_eattr / gat_bwd_edges_eattr: the same two passes with a per-edge score term (upstream GATConv with
 *                   edge_dim): a_edge [nnz, H] fp32 in CSR order, self-loop entries included, enters the score as
 *                   leaky_relu(a_src[col[e],h] + a_edge[e,h] + a_dst[i,h]) in the forward and in the backward's
 *                   recomputed score.  Its gradient is d_score.  a_edge = NULL is exactly gat_fused_fwd /
 *                   gat_bwd_edges, which forward to these with NULL. */
int gmlm_gcn_edge_weights(const int32_t* rowptr, const int32_t* col, int64_t num_rows, float* dis_ws /* [rows] */,
                          float* w /* [nnz] */, void* stream);
int gmlm_segment_sum_f32(const float* vals, const int64_t* idx, const int32_t* rowptr, int64_t num_rows,
                         int heads, float* out, void* stream);
size_t gmlm_gat_workspace_bytes(int64_t n_chunks, int heads, int head_dim);
int gmlm_gat_fused_fwd(const int32_t* rowptr, const int32_t* col, int64_t num_rows, const void* z, int dtype,
                       int64_t ldz, const float* a_src, const float* a_dst, int heads, int head_dim,
                       float negative_slope, float p_drop, uint64_t seed, int32_t hub_thresh, int64_t n_hub,
                       int64_t n_chunks, const int32_t* hub_row, const int32_t* hub_chunk_ptr,
                       const int32_t* chunk_beg, const int32_t* chunk_end, void* ws, size_t ws_bytes,
                       void* out, int64_t ldo, float* m_out, float* l_out, void* stream);
int gmlm_gat_bwd_edges(const int32_t* rowptr, const int32_t* col, int64_t num_rows, const void* z, int dtype,
                       int64_t ldz, const void* g, int64_t ldg, const float* a_src, const float* a_dst,
                       const float* m_in, const float* l_in, const float* t_in, int heads, int head_dim,
                       float negative_slope, float p_drop, uint64_t seed, int32_t hub_thresh, int64_t n_hub,
                       int64_t n_chunks, const int32_t* hub_row, const int32_t* hub_chunk_ptr,
                       const int32_t* chunk_beg, const int32_t* chunk_end, void* ws, size_t ws_bytes,
                       float* alpha_eff, float* d_score, float* da_dst, void* stream);
int gmlm_gat_fused_fwd_eattr(const int32_t* rowptr, const int32_t* col, int64_t num_rows, const void* z, int dtype,
                             int64_t ldz, const float* a_src, const float* a_dst, const float* a_edge /* [nnz, H] */,
                             int heads, int head_dim, float negative_slope, float p_drop, uint64_t seed,
                             int32_t hub_thresh, int64_t n_hub, int64_t n_chunks, const int32_t* hub_row,
                             const int32_t* hub_chunk_ptr, const int32_t* chunk_beg, const int32_t* chunk_end, void* ws,
                             size_t ws_bytes, void* out, int64_t ldo, float* m_out, float* l_out, void* stream);
int gmlm_gat_bwd_edges_eattr(const int32_t* rowptr, const int32_t* col, int64_t num_rows, const void* z, int dtype,
                             int64_t ldz, const void* g, int64_t ldg, const float* a_src, const float* a_dst,
                             const float* a_edge /* [nnz, H] */, const float* m_in, const float* l_in,
                             const float* t_in, int heads, int head_dim, float negative_slope, float p_drop,
                             uint64_t seed, int32_t hub_thresh, int64_t n_hub, int64_t n_chunks, const int32_t* hub_row,
                             const int32_t* hub_chunk_ptr, const int32_t* chunk_beg, const int32_t* chunk_end, void* ws,
                             size_t ws_bytes, float* alpha_eff, float* d_score, float* da_dst, void* stream);
int gmlm_gat_dropout_mask(uint64_t seed, int64_t n, float p_drop, uint8_t* keep, void* stream);
int gmlm_gat_loop_fill(const float* alpha, const int32_t* csr_src, const int32_t* loop_csr, const int32_t* rowptr,
                       int64_t num_rows, int heads, float* a_edge, void* stream);
int gmlm_gat_loop_fill_bwd(const float* g, const int32_t* in2csr, const int32_t* in_dst, const int32_t* loop_csr,
                           const int32_t* rowptr, int64_t num_edges, int heads, float* d_alpha, void* stream);

/* ---- halo pack / unpack for the destination-row partition (SURVEY §8e; the reference has no
 *      multi-GPU path) ----
 * gather_rows     : out[k,:]      = x[ids[k],:]
 * scatter_add_rows: dst[ids[k],:] += src[k,:]   ids unique within a call => no atomics, deterministic */
int gmlm_gather_rows(const void* x, int dtype, int64_t feat, int64_t ldx, const int64_t* ids, int64_t n,
                     void* out, int64_t ldo, void* stream);
int gmlm_scatter_add_rows(void* dst, int dtype, int64_t feat, int64_t ldd, const int64_t* ids, int64_t n,
                          const void* src, int64_t lds, void* stream);

/* ---- halo exchange over NVLink peer memory: every row carries its own 64-bit source address
 *      (a pointer into a peer-mapped symmetric buffer), so ONE launch moves rows from all peers ----
 * gather_rows_ptr : out[out_ids[k],:] = row_ptrs[k][0:feat]   (out_ids NULL = identity; callers list the
 *                   rows round-robin over the peers so that no peer's egress is hit by everyone at once)
 * reduce_rows_ptr : dst[row_ids[r],:] += sum over entries e of row r of entry_ptrs[e][0:feat]
 *                   (fp32 accumulation in entry order, one rounding; one owner per row => no atomics).
 * Rows must be multiples of 16 bytes and 16-byte aligned. */
int gmlm_gather_rows_ptr(const void* const* row_ptrs, const int64_t* out_ids, int dtype, int64_t feat,
                         int64_t n, void* out, int64_t ldo, void* stream);
int gmlm_reduce_rows_ptr(void* dst, int dtype, int64_t feat, int64_t ldd, const int64_t* row_ids,
                         const int32_t* rowptr, const void* const* entry_ptrs, int64_t n_rows, void* stream);
/* gather_rows_ptr moved by the bulk-copy engine (cp.async.bulk: peer memory -> shared-memory ring -> local HBM)
 * from `ctas` CTAs (0 = one per SM) of `warps` warps (0 = up to 3; each warp runs its own ring and moves
 * ~12 M rows/s) sharing `smem_kb` KiB (0 = 200): the transport that can run UNDER an aggregation kernel without
 * sharing its load queues.  Batches are `rows_per_batch` rows (0 = 32; 16 or 8 keep the ring -- and the bite out of
 * the SM's unified L1 / shared memory -- small); three batches per warp must fit the ring. */
int gmlm_gather_rows_ptr_tma(const void* const* row_ptrs, const int64_t* out_ids, int dtype, int64_t feat,
                             int64_t n, void* out, int64_t ldo, int ctas, int warps, int smem_kb,
                             int rows_per_batch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* GMLM_B200_H_ */
