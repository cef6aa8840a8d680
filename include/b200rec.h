/*
 * b200rec — C-ABI of the B200-native two-tower hot path (libb200rec.so, sm_100a).
 *
 * The reference (yxyxcyx/Real-Time-Recommendation-System-with-Feature-Store) is pure Python and has no FFI of its
 * own; each entry point below replaces the LIBRARY CALL the reference makes at the cited file:line (paths relative
 * to the reference root).  INTEGRATION.md shows the ctypes binding a maintainer would add on the reference side.
 * Conventions:
 *   - every pointer is a DEVICE pointer unless its name ends in _host; sizes are element counts;
 *   - `stream` is a cudaStream_t passed as void*; every launch is asynchronous on it;
 *   - nothing is allocated or freed inside; workspaces / scratch buffers are caller-owned;
 *   - return 0 on success, non-zero on argument / CUDA error; b200rec_last_error() explains (thread-local);
 *   - bf16 operands are raw 16-bit storage, row-major, leading dimension in ELEMENTS.
 */
#ifndef B200REC_H
#define B200REC_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

const char* b200rec_last_error(void);
int b200rec_version(void);
/* number of kernels launched by this library since load (bench.py's `gpu_launches`) */
int64_t b200rec_launch_count(void);

/* ---------------------------------------------------------------- operand preparation (csrc/prep.cu)
 * fp32 -> bf16 tensor-core operand [rows, terms*kpad] (zero padded to kpad columns per block).
 *   x = h + m + l exactly (h = bf16(x), m = bf16(x-h), l = bf16(x-h-m))
 *   terms 1: [h] | [h]                  plain bf16 (2e-2 budget of the bf16 mode)
 *   terms 3: [h m h] | [m h h]          (~2^-17 per product)
 *   terms 6: [m l h m h h] | [m h l h m h]   fp32-grade products (drops only m*l, l*m, l*l)
 *   (smallest piece products first: tcgen05 accumulates with truncation, late small addends would be lost)
 * side 0 = left operand pattern, side 1 = right operand pattern.  transpose != 0 reads src as [cols, rows].
 * Feeds the GEMM that replaces ATen addmm / matmul (src/models/two_tower.py:62,70,129,276,470). */
int b200rec_split_bf16(const float* src, int64_t rows, int64_t cols, int64_t ld_src, int transpose, void* dst,
                       int64_t kpad, int terms, int side, void* stream);

/* faiss.normalize_L2 (src/serving/retrieval.py:86,167,214; faiss_zero_rule=1: zero rows untouched) and
 * F.normalize(p=2, eps=1e-12) (src/models/two_tower.py:132,279; faiss_zero_rule=0), fused with the operand cast:
 * dst_f32 (nullable) gets the normalised fp32 rows, dst_bf16 (nullable) the operand as b200rec_split_bf16,
 * norms_out (nullable) the row norms (clamped to eps under the torch rule).  normalize == 0 only casts. */
int b200rec_normalize_rows(const float* src, int64_t rows, int64_t cols, int64_t ld_src, int normalize,
                           int faiss_zero_rule, float* dst_f32, int64_t ld_dst, float* norms_out, void* dst_bf16,
                           int64_t kpad, int terms, int side, void* stream);

/* ---------------------------------------------------------------- tensor-core GEMM (csrc/gemm.cu; tcgen05 + TMA)
 * C[M,N] (+)= alpha * A[M,K] . B[N,K]^T + bias[N];  A,B bf16 K-major (lda/ldb multiples of 8), C fp32 row-major.
 * k_splits > 1 splits K over CTAs and ACCUMULATES into C with fp32 atomics (caller pre-zeroes or pre-loads C);
 * k_splits < 0 means |k_splits| splits and accumulate even if only one split remains (C += ...).
 * Replaces nn.Linear forward/backward (two_tower.py:62,70) and torch.matmul (:470). */
int b200rec_gemm_bf16_tn(const void* A, int64_t lda, int64_t M, const void* B, int64_t ldb, int64_t N, int64_t K,
                         float* C, int64_t ldc, const float* bias, float alpha, int k_splits, void* stream);

/* ---------------------------------------------------------------- exact inner-product top-K (csrc/topk.cu)
 * Replaces faiss.IndexFlatIP.search(q, k) (src/serving/retrieval.py:171) and the np.dot + argsort twin
 * (scripts/evaluate_model.py:217-232, src/evaluation/metrics.py:381-396).
 * catalogue bf16 [N, ld], queries bf16 [Q, ld] (ld = padded dim, multiple of 64).  out_scores fp32 [Q,k] descending,
 * out_ids int64 [Q,k] = row + row_offset; unfilled slots -FLT_MAX / -1.  Total order: score desc, row asc.
 * exclude_* (nullable): CSR of per-query LOCAL rows (ascending) that must never be returned (the -inf mask of
 * evaluate_model.py:225-228).  k <= 2048, N < 2^32 - 1 per shard. */
size_t b200rec_topk_workspace_bytes(int64_t N, int64_t ld, int64_t Q, int k);
/* tau_init (nullable, device float[Q]): caller-supplied lower bounds of each query's FINAL k-th score; candidates below
 * them are never considered (a shard may then return fewer than k rows), and the internal sampling pass is skipped. */
int b200rec_flat_ip_topk(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k,
                         int64_t row_offset, const int64_t* exclude_indptr, const int32_t* exclude_rows,
                         const float* tau_init, float* out_scores, int64_t* out_ids, void* workspace,
                         size_t workspace_bytes, void* stream);
/* Filtered search: the exact top-k over the rows allowed by a row filter.  allow_bits is a bitmap over LOCAL rows in
 * faiss' IDSelectorBitmap layout (bit r = bit r&7 of byte r>>3, LSB first; equivalently bit r&31 of little-endian
 * uint32 word r>>5), allow_n its length in rows: rows >= allow_n are not allowed.  Same order, padding, workspace and
 * limits as b200rec_flat_ip_topk; disallowed rows are rejected where candidates enter the running lists, and the
 * internal sampling pass counts them as -inf.  Cost grows as the filter gets more selective (disallowed rows above the
 * running threshold still take the slow path): for selective filters search a compacted catalogue instead
 * (b200rec_gather_rows + b200rec_flat_ip_topk + b200rec_remap_ids). */
int b200rec_flat_ip_topk_filtered(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k,
                                  int64_t row_offset, const uint32_t* allow_bits, int64_t allow_n, float* out_scores,
                                  int64_t* out_ids, void* workspace, size_t workspace_bytes, void* stream);
/* Row filters (csrc/filter.cu).  bits [ceil(n_bits/32)] uint32 = the bitmap of the rows[0..n) that lie in [0, n_bits)
 * (out-of-range rows are ignored, duplicates are harmless; the bitmap is cleared first; rows may be NULL when n = 0).  b200rec_remap_ids maps the
 * ids of a search over a compacted catalogue (row j = catalogue row rows[j], rows ascending) back:
 * out[i] = rows[ids[i]] + row_offset, -1 stays -1 (in place allowed). */
int b200rec_rows_to_bitmap(const int64_t* rows, int64_t n, int64_t n_bits, uint32_t* bits, void* stream);
int b200rec_remap_ids(const int64_t* ids, int64_t n, const int64_t* rows, int64_t n_rows, int64_t row_offset,
                      int64_t* out, void* stream);
/* Sampling pass alone: out_vals [Q,k_out] = the k_out (<= k) largest group maxima (distinct sampled rows) of every
 * query, descending.  Row-sharded search exchanges these (all-gather) and starts every shard from the k-th best of the
 * union; `shards` (>= 1) says how many shards pool their samples, so each one samples 1/shards as densely.
 * b200rec_topk_has_sample says whether this shape runs a sampling pass at all (small shards do not). */
int b200rec_topk_sample(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k, int k_out,
                        int shards, float* out_vals, void* workspace, size_t workspace_bytes, void* stream);
int b200rec_topk_has_sample(int64_t N, int64_t ld, int64_t Q, int k);
/* out_kth[q] = k-th largest of the parts x k_in pooled sample maxima vals[parts][Q][k_in] of query q: the shared
 * starting threshold of row-sharded search (a lower bound of the global k-th score), in one launch. */
int b200rec_topk_pooled_kth(const float* vals, int parts, int64_t Q, int k_in, int k, float* out_kth, void* stream);
/* Fan-out variants for row-sharded search over NVLink peer memory: the select kernels store every result row to n_dst
 * (<= 16) destinations — dst_*[d] are device pointers to [Q,k] (resp. [Q,k_out]) arrays, typically this shard's slot in
 * each GPU's gather buffer (peer-mapped symmetric memory) — so the kernel that produces the local top-k is also the
 * all-gather.  The caller orders the exchange with a cross-GPU barrier on the same stream.  dst[0] may be local. */
int b200rec_flat_ip_topk_fanout(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k,
                                int64_t row_offset, const float* tau_init, int n_dst, void* const* dst_scores,
                                void* const* dst_ids, void* workspace, size_t workspace_bytes, void* stream);
int b200rec_topk_sample_fanout(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k,
                               int k_out, int shards, int n_dst, void* const* dst_vals, void* workspace,
                               size_t workspace_bytes, void* stream);
/* Filtered row-shard steps (row-sharded filtered search; every shard passes through both exchanges, so neither step
 * fails for lack of work: it stores padding rows to every destination instead).
 * b200rec_topk_sample_filtered[_fanout]: b200rec_topk_sample over the rows allowed by allow_bits (bitmap as in
 * b200rec_flat_ip_topk_filtered; disallowed sampled rows count as -inf), or over the whole catalogue when allow_bits is
 * NULL (a compacted catalogue).  When no row is allowed (N == 0 or allow_n == 0) or the shape has no sampling pass, every
 * destination gets -FLT_MAX rows, which bound nothing from below.
 * b200rec_flat_ip_topk_filtered_fanout: the local top-k of a row shard starting from tau_init (nullable), stored to the
 * n_dst destinations.  Exactly one of allow_bits (bitmap path; ids = row + row_offset) and remap_rows (compacted
 * catalogue path: N = n_remap compacted rows, row j is local row remap_rows[j], ids = remap_rows[j] + row_offset, mapped
 * inside the select kernel) is given.  No allowed row (N == 0 or allow_n == 0): -FLT_MAX / -1 rows everywhere. */
int b200rec_topk_sample_filtered(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q, int k,
                                 int k_out, int shards, const uint32_t* allow_bits, int64_t allow_n, float* out_vals,
                                 void* workspace, size_t workspace_bytes, void* stream);
int b200rec_topk_sample_filtered_fanout(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q,
                                        int k, int k_out, int shards, const uint32_t* allow_bits, int64_t allow_n,
                                        int n_dst, void* const* dst_vals, void* workspace, size_t workspace_bytes,
                                        void* stream);
int b200rec_flat_ip_topk_filtered_fanout(const void* catalogue, int64_t N, int64_t ld, const void* queries, int64_t Q,
                                         int k, int64_t row_offset, const uint32_t* allow_bits, int64_t allow_n,
                                         const int64_t* remap_rows, int64_t n_remap, const float* tau_init, int n_dst,
                                         void* const* dst_scores, void* const* dst_ids, void* workspace,
                                         size_t workspace_bytes, void* stream);
/* k-way merge of `parts` candidate lists [parts][Q][k_in] (id < 0 = empty, ids < 2^32) into the global top k_out under
 * the same order: the exchange step after the all-gather of per-GPU results.  *_part_stride = element distance
 * between consecutive parts (0 = dense, Q*k_in); non-dense strides let one all-gather carry scores and ids together. */
int b200rec_topk_merge(const float* scores, const int64_t* ids, int parts, int64_t Q, int k_in, int k_out,
                       int64_t scores_part_stride, int64_t ids_part_stride, float* out_scores, int64_t* out_ids,
                       void* stream);
/* Exact fp32 re-scoring of candidate rows (csrc/rescore.cu): scores[q, j] = <queries[q, :d], rows[ids[q, j] - row_offset, :d]>
 * with fp32 FMAs (-FLT_MAX where ids[q, j] < 0).  The "fp32" storage of the drop-in index (reference
 * src/serving/retrieval.py:171 on an fp32 IndexFlatIP) selects k + margin candidates with split-bf16 tensor-core
 * products (~2^-17) and re-scores them from the fp32 rows it keeps, so scores and order are those of an fp32 CPU search;
 * b200rec_topk_merge (parts = 1) then orders the candidates (score desc, id asc) and keeps k. */
int b200rec_rescore_fp32(const float* queries, int64_t ld_q, const float* rows, int64_t ld_rows, int64_t n_rows,
                         int64_t row_offset, int d, const int64_t* ids, int64_t Q, int k_in, float* scores,
                         void* stream);

/* ---------------------------------------------------------------- embedding bags (csrc/embedding.cu)
 * out[b, 0:num_cols] = numerical[b, :]; out[b, col_off[f] : +width[f]] = table_f[idx_f[b], :width[f]].
 * Replaces nn.Embedding forward + 2x torch.cat (two_tower.py:113-126, :254-273).  The *_host arrays are HOST arrays
 * of F entries (F <= 16).  err_flag (nullable device int) is set to 1+f when field f holds an out-of-range index. */
int b200rec_gather_concat(const float* numerical, int64_t num_cols, int64_t ld_num, const float* const* tables_host,
                          const int64_t* const* indices_host, const int64_t* table_rows_host,
                          const int32_t* widths_host, const int32_t* table_ld_host, const int32_t* col_off_host, int F,
                          int64_t B, float* out, int64_t ld_out, int32_t* err_flag, void* stream);
/* Sparse row gradient of one table: coalesced (unique_rows[U] ascending, grad_rows[U,width]), duplicates summed, the
 * padding row dropped — the non-zero rows of ATen embedding_dense_backward (nn.Embedding(padding_idx=0)).
 * n_unique_out is a device int32.  table_rows (> 0) bounds the sort key width. */
size_t b200rec_sparse_grad_workspace_bytes(int64_t B);
int b200rec_embedding_sparse_grad(const int64_t* idx, int64_t B, const float* dY, int64_t ld_dy, int width,
                                  int64_t padding_idx, int64_t table_rows, int64_t* unique_rows, float* grad_rows,
                                  int32_t* n_unique_out, void* workspace, size_t workspace_bytes, void* stream);
/* dense[rows[u], :width] (+)= grad_rows[u, :] for u < *n_rows (rows distinct) — materialises the dense gradient
 * the reference's optimizer expects. */
int b200rec_scatter_rows(const int64_t* rows, const float* grad_rows, const int32_t* n_rows, int64_t max_rows,
                         int width, float* dense, int64_t ld, int accumulate, void* stream);
/* dense[idx[b], :width] += dY[b, :width] (padding row and ids outside [0, table_rows) skipped): the dense gradient of
 * nn.Embedding accumulated in place with fp32 atomics, one launch (two_tower.py:116 under autograd). */
int b200rec_scatter_add_rows(const int64_t* idx, int64_t B, const float* dY, int64_t ld_dy, int width,
                             int64_t padding_idx, int64_t table_rows, float* dense, int64_t ld, void* stream);

/* ---------------------------------------------------------------- tower MLP pieces (csrc/tower_ops.cu)
 * act: 0 relu, 1 gelu(erf), 2 leaky_relu(0.1), 3 tanh, 4 sigmoid, 5 identity  (two_tower.py:77-86).
 * One hidden block after its Linear:  y = dropout(BatchNorm1d(act(z)))  (order of two_tower.py:56-72).
 * training != 0: batch statistics (biased variance), running stats updated with `momentum` (unbiased variance),
 * dropout mask = Philox(seed, element index).  training == 0: running statistics, no dropout.
 * mean / invstd [H] are outputs kept for the backward.  scratch: >= 3*H doubles. */
int b200rec_bn_forward(const float* z, int64_t B, int64_t H, int64_t ld, int act, int training, float eps,
                       float momentum, const float* gamma, const float* beta, float* running_mean,
                       float* running_var, float drop_p, uint64_t seed, float* mean, float* invstd, float* y,
                       int64_t ld_y, double* scratch, void* stream);
/* dz [B,H] from dy; dgamma, dbeta and (nullable) dbias = colsum(dz) are ACCUMULATED into their outputs. */
int b200rec_bn_backward(const float* dy, int64_t ld_dy, const float* z, int64_t ld_z, int64_t B, int64_t H, int act,
                        int training, const float* mean, const float* invstd, const float* gamma, float drop_p,
                        uint64_t seed, float* dz, int64_t ld_dz, float* dgamma, float* dbeta, float* dbias,
                        double* scratch, void* stream);
/* Data-parallel BatchNorm1d: batch statistics over the rows of ALL replicas (what a single process computes on the
 * global batch, trainers/two_tower.py:98-151 under one-process-per-GPU training).  Two phases around the caller's
 * all-reduce (sum) of the fp64 partial sums scratch[0, 2H): phase 0 accumulates the local sums (backward: also adds the
 * LOCAL dbeta / dgamma), phase 1 finishes with B_total = rows over all replicas.  scratch: >= 3*H doubles. */
int b200rec_bn_forward_dp(const float* z, int64_t B, int64_t H, int64_t ld, int act, float eps, float momentum,
                          const float* gamma, const float* beta, float* running_mean, float* running_var,
                          float drop_p, uint64_t seed, float* mean, float* invstd, float* y, int64_t ld_y,
                          double* scratch, int phase, int64_t B_total, void* stream);
int b200rec_bn_backward_dp(const float* dy, int64_t ld_dy, const float* z, int64_t ld_z, int64_t B, int64_t H, int act,
                           const float* mean, const float* invstd, const float* gamma, float drop_p, uint64_t seed,
                           float* dz, int64_t ld_dz, float* dgamma, float* dbeta, float* dbias, double* scratch,
                           int phase, int64_t B_total, void* stream);
/* y = dropout(act(z)) without BatchNorm (ItemTower.content_projection, two_tower.py:184-191) and its backward. */
int b200rec_act_dropout(const float* z, int64_t B, int64_t H, int64_t ld, int act, float drop_p, uint64_t seed,
                        float* y, int64_t ld_y, void* stream);
int b200rec_act_dropout_bwd(const float* dy, int64_t ld_dy, const float* z, int64_t ld_z, int64_t B, int64_t H,
                            int act, float drop_p, uint64_t seed, float* dz, int64_t ld_dz, void* stream);
/* out[h] (+)= sum_b x[b,h]  — Linear bias gradients.  scratch: >= H doubles. */
int b200rec_colsum(const float* x, int64_t B, int64_t H, int64_t ld, float* out, int accumulate, double* scratch,
                   void* stream);
/* F.normalize backward: dO = (dE - E * rowsum(E*dE)) / norm. */
int b200rec_normalize_bwd(const float* dE, const float* E, const float* norms, int64_t B, int64_t D, float* dO,
                          void* stream);

/* ---------------------------------------------------------------- fused tower-MLP layers (csrc/mlp_fused.cuh)
 * One launch per Linear and direction.  A hidden block [Linear -> activation -> BatchNorm1d -> Dropout] (reference
 * src/models/two_tower.py:60-66,200-206) is described by its tensors; the kernels apply the block's transform while
 * they BUILD the tensor-core operand of the next GEMM (no split-bf16 copies, no separate BN / activation / dropout
 * passes) and reduce the batch statistics the next launch needs in their epilogue.
 *   np = bf16 pieces per operand: 3 (6 piece products, fp32 grade), 2 (3 products, ~2^-17), 1 (plain bf16). */
typedef struct b200rec_bn_block {
  const float* z;                 /* [rows, H] pre-activations (output of the block's Linear) */
  int64_t ldz;
  int32_t H;                      /* <= 512 */
  int32_t act;                    /* 0 relu, 1 gelu, 2 leaky_relu(0.1), 3 tanh, 4 sigmoid, 5 identity */
  int32_t training;               /* batch statistics (sums) + dropout, or running statistics */
  int32_t update_running;         /* forward: apply the momentum update + count the batch (done once, by one CTA) */
  const double* sums;             /* training: [2H] sum act(z), sum act(z)^2 over B_stat rows */
  const float* gamma;
  const float* beta;
  float* running_mean;
  float* running_var;
  int64_t* num_batches_tracked;   /* may be NULL */
  float eps, momentum, drop_p;
  uint64_t seed;
  int64_t B_stat;                 /* rows the statistics cover (the global batch under data parallel) */
} b200rec_bn_block;
/* out[B,N] = input . w[N,K]^T + bias, input = x (lower == NULL) or Dropout(BN(act(lower->z))).
 * out_sums != NULL: [2N] += sum act_out(out), sum act_out(out)^2 (pre-zeroed; the statistics of this layer's own block).
 * normalize != 0 (last layer, N <= 128): out = F.normalize(out) (two_tower.py:132,279), norms[B] = max(||row||, 1e-12). */
int b200rec_mlp_forward(const float* x, int64_t ldx, const b200rec_bn_block* lower, const float* w, int64_t ldw,
                        const float* bias, int64_t B, int N, int K, int np, float* out, int64_t ldo, int out_act,
                        double* out_sums, int normalize, float* norms, void* stream);
/* dx[B,K] = dz . w, dz = dy (own == NULL: last layer) or the BatchNorm/activation/dropout backward of `own` applied to
 * dy with own_bsums = [2N] sum g, sum g*xhat.  lower_bsums != NULL: [2K] += the same two sums for the block below
 * (g = dx * its dropout mask), ready for the next launch. */
int b200rec_mlp_dgrad(const float* dy, int64_t lddy, const b200rec_bn_block* own, const double* own_bsums, const float* w,
                      int64_t ldw, int64_t B, int N, int K, int np, float* dx, int64_t lddx,
                      const b200rec_bn_block* lower, double* lower_bsums, void* stream);
/* dw[N,K] += dz^T . input, db[N] += colsum(dz) (fp32 atomics into pre-zeroed or accumulating buffers);
 * dgamma / dbeta [N] += own_bsums_local (NULL = own_bsums) halves. */
int b200rec_mlp_wgrad(const float* dy, int64_t lddy, const b200rec_bn_block* own, const double* own_bsums,
                      const double* own_bsums_local, const float* x, int64_t ldx, const b200rec_bn_block* lower,
                      int64_t B, int N, int K, int np, float* dw, int64_t lddw, float* db, float* dgamma, float* dbeta,
                      void* stream);

/* ---------------------------------------------------------------- losses (csrc/loss_ops.cu, csrc/inbatch_lse.cu)
 * In-batch softmax cross-entropy (two_tower.py:467-479), forward fused with the logits GEMM: the B x NI logits live
 * only in TMEM.  U_op [B, ld] / I_op [NI, ld] are split-bf16 operands (left / right patterns).  Output per row:
 * lse[b] = logsumexp_j(inv_T * <u_b, i_j>).  Under data parallelism I may hold more rows than U (all-gathered). */
size_t b200rec_inbatch_lse_workspace_bytes(int64_t B, int64_t NI, int64_t ld);
int b200rec_inbatch_lse(const void* U_op, const void* I_op, int64_t ld, int64_t B, int64_t NI, float inv_temperature,
                        float* lse_out, void* workspace, size_t workspace_bytes, void* stream);
/* Row-wise pieces used by the chunked backward (and by the unfused forward):
 * lse[r] = logsumexp_j(scale*S[r,j]); pos[r] (nullable) = scale*S[r, diag0 + r]. */
int b200rec_lse_rows(const float* S, int64_t ld, int64_t rows, int64_t cols, float scale, int64_t diag0, float* lse,
                     float* pos, void* stream);
/* G[r,j] = coef * (*coef_dev) * (exp(scale*S[r,j] - lse[r]) - [j == diag0 + r])   (in place allowed; coef_dev nullable) */
int b200rec_softmax_grad(const float* S, int64_t ld, int64_t rows, int64_t cols, float scale, const float* lse,
                         int64_t diag0, float coef, const float* coef_dev, float* G, int64_t ldg, void* stream);
/* *acc += sum_r (lse[r] - pos[r])   (pos nullable: plain sum) */
int b200rec_ce_sum(const float* lse, const float* pos, int64_t n, float* acc, void* stream);
/* Explicit-negative CE (two_tower.py:422-451): logits[b] = [<u,p>/T + ub + ib, <u,n_{b,0..R-1}>/T], label 0.
 * row_loss[b] is written; when dU != NULL the gradients scaled by grad_scale are written too
 * (dU, dP [B,E], dN [B*R,E], row_dbias[b] = grad_scale * dlogit_0). */
int b200rec_explicit_ce(const float* U, const float* P, const float* Nn, int64_t B, int64_t R, int64_t E,
                        float inv_temperature, const float* user_bias, const float* item_bias, float* row_loss,
                        float grad_scale, const float* grad_scale_dev, float* dU, float* dP, float* dN,
                        float* row_dbias, void* stream);
/* compute_similarity (two_tower.py:380-404): out[b] = <u_b, i_b> * scale + ub + ib, and its backward. */
int b200rec_rowdot(const float* U, const float* I, int64_t B, int64_t E, float scale, const float* user_bias,
                   const float* item_bias, float* out, void* stream);
int b200rec_rowdot_bwd(const float* g, const float* U, const float* I, int64_t B, int64_t E, float scale, float* dU,
                       float* dI, void* stream);

/* ---------------------------------------------------------------- optimiser (csrc/optim.cu)
 * clip_grad_norm_ (src/training/trainers/two_tower.py:144): *out += sum x^2 (fp64); coef = min(1, max/(norm+1e-6)). */
int b200rec_sumsq(const float* x, int64_t n, double* out, void* stream);
int b200rec_clip_coef(const double* sumsq, float max_norm, float* coef, float* norm_out, void* stream);
/* torch.optim.Adam with L2-coupled weight decay (trainers/two_tower.py:60-64,146) on a flat fp32 buffer;
 * clip_coef_dev (device float, nullable) scales g first.  bias_c1 = 1-beta1^t, bias_c2_sqrt = sqrt(1-beta2^t). */
/* clear_grad != 0: every gradient element that was non-zero is reset to zero after it was consumed (the next step's
 * zero_grad without a pass over the whole buffer). */
int b200rec_adam_dense(float* p, float* g, float* m, float* v, int64_t n, float lr, float beta1, float beta2,
                       float eps, float weight_decay, float bias_c1, float bias_c2_sqrt, const float* clip_coef_dev,
                       int clear_grad, void* stream);
/* Row-sparse Adam on the touched rows only (large embedding tables; no weight decay on untouched rows). */
int b200rec_sparse_adam(float* table, float* exp_avg, float* exp_avg_sq, int64_t ld, int width, const int64_t* rows,
                        const float* grad_rows, const int32_t* n_rows, int64_t max_rows, float lr, float beta1,
                        float beta2, float eps, float bias_c1, float bias_c2_sqrt, const float* clip_coef_dev,
                        void* stream);

/* ---- CUDA-graph training: per-step state in device memory ----
 * A captured step replays with the kernel arguments of the capture, so the step counter, Adam's bias corrections, the
 * learning rate and the dropout streams live on the device.  b200rec_train_step_begin (first node of the graph):
 * step = ++*step_dev; hyper_dev[0..2] = {*lr_dev, 1 - beta1^step, sqrt(1 - beta2^step)}; every dropout seed of the step
 * is XOR-ed with a hash of (salt_key, step) (salt_key 0 = no salt).  b200rec_adam_dense_dev / _sparse_adam_dev are
 * b200rec_adam_dense / _sparse_adam reading hyper_dev instead of host scalars.  One training stream per process. */
int b200rec_train_step_begin(int64_t* step_dev, const float* lr_dev, float beta1, float beta2, float* hyper_dev,
                             uint64_t salt_key, void* stream);
int b200rec_adam_dense_dev(float* p, float* g, float* m, float* v, int64_t n, float beta1, float beta2, float eps,
                           float weight_decay, const float* hyper_dev, const float* clip_coef_dev, int clear_grad,
                           void* stream);

/* ---- dense embedding tables under dense Adam (reference trainers/two_tower.py:60-64: Adam + weight decay over ALL
 * parameters moves every row each step, but a step's gradient is non-zero only on the rows the batch touched).
 * b200rec_scatter_add_rows_flagged = b200rec_scatter_add_rows that also sets row_flags[row] = 1; b200rec_table_sumsq adds
 * the squared gradient of the flagged rows to *out; b200rec_adam_table applies the Adam + weight-decay update to every
 * row, reading (and, with clear_grad, zeroing) the gradient of flagged rows only and clearing their flags: 24 B per
 * parameter instead of 32.  hyper_dev != NULL: {lr, 1 - beta1^t, sqrt(1 - beta2^t)} come from device memory
 * (b200rec_train_step_begin) and lr / bias_c1 / bias_c2_sqrt are ignored.  width <= 128. */
int b200rec_scatter_add_rows_flagged(const int64_t* idx, int64_t B, const float* dY, int64_t ld_dy, int width,
                                     int64_t padding_idx, int64_t table_rows, float* dense, int64_t ld, int32_t* row_flags,
                                     void* stream);
/* Row-sparse tables without a sort: acc [B, width] must be zero, slot [table_rows] int32 all zero (it is zero again on
 * return).  rows_out[b] = idx[b] for the first sample of every distinct valid row (its leader) and -1 otherwise; the
 * gradient rows of all samples of a row are summed into acc[leader].  Feed (rows_out, acc, n = B) to
 * b200rec_sparse_adam(_dev), which skips rows < 0, and acc to b200rec_sumsq.  Replaces b200rec_embedding_sparse_grad
 * (sort + segment sum) on the training path; that one stays for deterministic runs. */
int b200rec_sparse_claim_accumulate(const int64_t* idx, int64_t B, const float* dY, int64_t ld_dy, int width,
                                    int64_t padding_idx, int64_t table_rows, int32_t* slot, int64_t* rows_out, float* acc,
                                    void* stream);
int b200rec_table_sumsq(const float* g, int64_t ld, int64_t rows, int width, const int32_t* row_flags, double* out,
                        void* stream);
int b200rec_adam_table(float* p, float* g, float* m, float* v, int64_t ld, int64_t rows, int width, int32_t* row_flags,
                       float lr, float beta1, float beta2, float eps, float weight_decay, float bias_c1, float bias_c2_sqrt,
                       const float* hyper_dev, const float* clip_coef_dev, int clear_grad, void* stream);
int b200rec_sparse_adam_dev(float* table, float* exp_avg, float* exp_avg_sq, int64_t ld, int width, const int64_t* rows,
                            const float* grad_rows, const int32_t* n_rows, int64_t max_rows, float beta1, float beta2,
                            float eps, const float* hyper_dev, const float* clip_coef_dev, void* stream);

/* ---- device-side batch feed (replaces MovieLensDataset.__getitem__ + collate_fn, reference
 * src/training/datasets/movielens.py:86-162, and sample_negative_items, src/data/movielens.py:487-512) ----
 * out[b, :] = table[idx[b], :] (fp32 rows of `width` floats).  An index outside [0, n_rows) sets *err_flag = 1 (numpy's
 * fancy indexing raises IndexError there) and yields a zero row. */
int b200rec_gather_rows(const float* table, int64_t n_rows, int width, int64_t ld, const int64_t* idx, int64_t B,
                        float* out, int64_t ld_out, int* err_flag, void* stream);
/* out_items [B, num_negatives]: for every row, `num_negatives` DISTINCT items drawn uniformly from the items its user
 * has not interacted with (np.random.choice(list(all_items - positives), n, replace=False)).  Positives come as a CSR
 * over users (pos_indptr int64 [n_users + 1], pos_items int32 sorted ascending per user).  Deterministic in
 * (seed, row_base + row).  *err_flag = 2 when a user's pool is smaller than num_negatives (the reference then returns
 * a short list and collate_fn fails). */
int b200rec_sample_negatives(const int64_t* user_of_row, int64_t B, const int64_t* pos_indptr, const int32_t* pos_items,
                             int64_t n_users, int64_t num_items, int num_negatives, uint64_t seed, uint64_t row_base,
                             int64_t* out_items, int* err_flag, void* stream);

/* ---- fused in-batch loss backward (csrc/inbatch_grad.cu; flash-style: logits recomputed in TMEM, never in HBM) ----
 * dU[b,:] = sum_j G[b,j] V[j,:],  dV[j,:] = sum_b G[b,j] U[b,:],  G = coef * (*coef_dev) * (exp(<u_b,v_j>*inv_t - lse[b])
 * - [j == diag0 + b]) — the gradient of mean-CE(U V^T / T, arange) that autograd derives for reference
 * src/models/two_tower.py:470-477.  u_op / v_op: split-bf16 row operands as b200rec_split_bf16 writes them
 * ([B | NI, blocks * pad64(E)]); ut_op / vt_op / ld_ut / ld_vt / ut_pieces_host / vt_pieces_host are IGNORED (may be
 * NULL / 0): the gradient GEMMs read the row operands as MN-major tiles, no transposed copies are needed.
 * *_pieces_host[p]: block index of piece p (0 = h, 1 = m, 2 = l) inside an operand row.  nprod_s = 1 | 3 | 6 piece
 * products recompute the logits, nprod_g = 1 | 3 form the two gradient GEMMs.  E must be 64 or 128
 * (b200rec_inbatch_grad_supported tells; callers fall back to the chunked GEMM path otherwise).  dU / dV are written
 * completely (no accumulation), rows 16-byte aligned. */
int b200rec_inbatch_grad_supported(int64_t B, int64_t NI, int E, int nprod_s, int nprod_g);
int b200rec_inbatch_grad(const void* u_op, int64_t ld_u, const int32_t* u_pieces_host, const void* v_op, int64_t ld_v,
                         const int32_t* v_pieces_host, const void* ut_op, int64_t ld_ut, const int32_t* ut_pieces_host,
                         const void* vt_op, int64_t ld_vt, const int32_t* vt_pieces_host, int64_t B, int64_t NI, int E,
                         int nprod_s, int nprod_g, float inv_t, const float* lse, int64_t diag0, float coef,
                         const float* coef_dev, float* dU, int64_t ld_du, float* dV, int64_t ld_dv, void* stream);

/* ---- one-shot all-reduce of a small fp64 vector over NVLink peer memory (csrc/peer_reduce.cu): the synced BatchNorm
 * statistics and the loss share of exact data-parallel training (reference: none, the reference is single-process;
 * this keeps N replicas equal to its one process on the global batch, trainers/two_tower.py:98-151).
 * peer_buffers_host[r]: device address of rank r's symmetric buffer (b200rec_peer_allreduce_bytes(max_n) bytes, zeroed,
 * mapped on this device, e.g. by torch.distributed._symmetric_memory); data[0..n) is replaced by the sum over ranks taken
 * in rank order (bit-identical on every rank).  Every rank issues the same calls in the same order on one stream.
 * *status_dev is set to 1 when a peer did not answer within seconds (the kernel then returns instead of hanging). */
size_t b200rec_peer_allreduce_bytes(int max_n);
int b200rec_peer_allreduce_f64(double* data, int n, int rank, int world, const uint64_t* peer_buffers_host, int max_n,
                               int* status_dev, void* stream);

/* ---- on-device ranking metrics (csrc/eval_metrics.cu; replaces the per-user Python of Evaluator.evaluate,
 * reference src/evaluation/metrics.py:240-319 with helpers :74-231) ----
 * pred int64 [Q, K] (ld_pred): ranked item ROWS per user as the top-K kernel emits them (-1 = empty slot);
 * repeat uint8 [Q, K] (nullable): 1 where a position repeats an id seen earlier in its row (set semantics of
 * recall / precision / hit rate; the fused top-K never repeats); ground truth as a CSR over the Q users (gt_rows
 * ascending per user) with gt_count (nullable) = |ground truth| when it also holds items outside the catalogue.
 * inv_log2[i] = 1/log2(i+2) for i < K and idcg[n] = sum_{i<n} inv_log2[i] (n <= max k) come from the host so that the
 * fp64 results equal the reference's expressions bit for bit.  per_user fp64 [Q, 4*n_k + 2]: for each k
 * (recall, precision, ndcg, hit), then reciprocal rank and average precision; sums (nullable) fp64 [4*n_k + 2] =
 * column sums; coverage_bits (nullable, uint32 [ceil(n_items/32)]) / coverage_count: distinct rows recommended in the
 * first coverage_k positions (metrics.py:279,312-314). */
int b200rec_eval_metrics(const int64_t* pred, int64_t Q, int K, int64_t ld_pred, const uint8_t* repeat,
                         int64_t ld_repeat, const int64_t* gt_indptr, const int64_t* gt_rows, const int64_t* gt_count,
                         const int32_t* k_values_host, int n_k, const double* inv_log2, const double* idcg,
                         double* per_user, double* sums, uint32_t* coverage_bits, int64_t n_items, int coverage_k,
                         unsigned long long* coverage_count, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200REC_H */
