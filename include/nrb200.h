/*
 * nrb200.h -- C ABI of the B200-native embedding-and-scoring hot path.
 *
 * Drop-in boundary for AhmedFahim-git/news_recommendation_project_v2.  The
 * reference is pure Python on stock torch ops and has no FFI of its own
 * (SURVEY.md section 8b); each entry point below names the reference call
 * site(s) (file:line under src/news_rec_utils/) whose arithmetic it replaces.
 * INTEGRATION.md shows the ctypes binding a maintainer adds on the reference
 * side.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in `_host`;
 *   - matrices are row-major, `ld*` / `*_stride` are in ELEMENTS;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every call is asynchronous on `stream` and returns 0 on success or a
 *     negative NRB_E_* code; nrb_last_error() gives the message (thread local);
 *   - no call allocates device memory: callers pass a workspace sized by the
 *     matching *_workspace_bytes() query;
 *   - out-of-range row ids never fault: the kernels substitute row 0 and set
 *     bit 0 of `*err_flag` (device int32), which the host turns into an
 *     IndexError like torch indexing does.
 *   - there is NO CPU implementation behind this ABI.
 */
#ifndef NRB200_H_
#define NRB200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NRB_OK 0
#define NRB_E_INVALID (-1)   /* bad argument / unsupported shape            */
#define NRB_E_CUDA (-2)      /* CUDA runtime / driver error                 */
#define NRB_E_ARCH (-3)      /* device is not sm_100                        */
#define NRB_E_WORKSPACE (-4) /* workspace too small                         */

#define NRB_F32 0
#define NRB_BF16 1

/* user-encoder pooling applied to the gathered history rows */
#define NRB_POOL_FINAL_ATTENTION 0 /* u = sum(x*e) / (sum(e) + 1e-10); modeling_utils.py:224-228 */
#define NRB_POOL_MEAN_L2 1         /* u = normalize(mean(x));          latent_attention.py:165-170 */

/* epilogues of the dense row kernels (nrb_linear) */
#define NRB_EPI_NONE 0      /* y = acc (+ bias)                       */
#define NRB_EPI_RELU 1      /* y = relu(acc + bias)                   modeling_utils.py:218-221 */
#define NRB_EPI_EXP 2       /* y = exp(acc + bias)                    modeling_utils.py:224     */
#define NRB_EPI_RESIDUAL 3  /* y = acc + bias + res                   latent_attention.py:162-163 */
#define NRB_EPI_GEGLU 4     /* y[j] = a_j * gelu_erf(g_j), W rows interleaved in pairs (a0,a1,g0,g1,a2,a3,g2,g3..) latent_attention.py:24-27 */
#define NRB_EPI_SOFTMAX 5   /* y = softmax over each group of `group` columns (first `group_valid` valid); latent_attention.py:69-72 */
#define NRB_EPI_TOPK 6      /* internal to nrb_recommend: per-row top-k of acc * scale[col], no output tile */
#define NRB_EPI_TOPK_BLEND 7 /* internal to nrb_recommend_pool_blend: the same of acc * scale[col] blended with base[col] */

typedef void* nrb_stream_t;

const char* nrb_version(void);
const char* nrb_last_error(void);
/* 0 when `device` is a compute-capability 10.x GPU (B200). */
int nrb_check_device(int device);
int nrb_sm_count(int device);
/* cumulative number of kernels this library has launched in the process (bench.py's gpu_launches). */
long long nrb_kernel_launches(void);

/* ---- Stage C: per-impression dense rank -------------------------------------------
 * replaces data_utils.py:414-415 rank_group_preds = scipy.stats.rankdata(-x, "dense")
 * per group.  ranks[j] = 1 + #{distinct scores in the group that are > scores[j]};
 * a group containing a NaN gets rank 0 everywhere (host maps 0 -> NaN). */
int nrb_dense_rank(const float* scores, const int64_t* offsets, int64_t n_groups,
                   int32_t* ranks, nrb_stream_t stream);
/* the same for float64 scores: scipy ranks an array in its own dtype, so rank_group_preds on float64
 * input must not merge values that differ only below fp32 resolution. */
int nrb_dense_rank_f64(const double* scores, const int64_t* offsets, int64_t n_groups,
                       int32_t* ranks, nrb_stream_t stream);

/* int32 dense ranks -> int16 on the device, for hosts that want the ranks of a large evaluation over PCIe at 2
 * bytes per candidate (a dense rank never exceeds the candidate count of its impression).  A value above 32767
 * saturates and sets bit 1 of *err_flag. */
int nrb_narrow_ranks(const int32_t* ranks, int16_t* ranks16, int64_t n, int32_t* err_flag, nrb_stream_t stream);

/* ---- Stage C: per-impression top-k ordering --------------------------------------------------
 * the order evaluation.py:14,28 derives from the ranks (argsort of the scores, descending), made
 * explicit: out_idx[g, p] = position inside group g of the candidate at place p (p < k), equal scores in
 * their original order (np.argsort(-scores, kind="stable")[:k]), -1 where the group has fewer than k
 * candidates, NaN scores last.  out_idx is int32 [n_groups, k]. */
int nrb_topk_order(const float* scores, const int64_t* offsets, int64_t n_groups, int k,
                   int32_t* out_idx, nrb_stream_t stream);

/* ---- Stage B: padded history gather -----------------------------------------------
 * replaces data_utils.py:784-791 final_attention_eval_collate_fn (+ pad_to_maxlen
 * :723-750): emb_out[g, s, :] = table[idx[offsets[g]+s], :] for s < len_g else 0;
 * mask_out[g, s] = s < len_g.  emb_out has the table dtype. */
int nrb_gather_collate(const void* table, int dtype, int64_t n_rows, int dim, int64_t table_stride,
                       const int32_t* idx, const int64_t* offsets, int64_t n_groups, int max_len,
                       void* emb_out, int32_t* mask_out, int32_t* err_flag, nrb_stream_t stream);

/* attention_mask int32 [batch, seq] (any 0 / non-zero pattern) -> CSR form of the valid slots: idx_out[k] = flat
 * position b*seq + s of the k-th valid slot (int32, capacity batch*seq), off_out int64 [batch + 1].  This is the
 * mask handling of FinalAttention.forward / NewAttention.forward (modeling_utils.py:224, attention.py:270: weights
 * times mask) turned into the index form nrb_score_rank pools over.  workspace: int32 [2*batch + 2]. */
int nrb_mask_to_csr(const int32_t* mask, int64_t batch, int seq, int32_t* idx_out, int64_t* off_out,
                    int32_t* workspace, nrb_stream_t stream);

/* ---- Stage B+C fused: gather -> user vector -> cosine -> dense rank --------------------
 * replaces data_model_helper.py:112-131 (get_final_attention_eval: CPU gather in
 * DataLoader workers + user-encoder pooling), :200-230 (per-impression
 * F.cosine_similarity loop, eps 1e-8, normalise-first) and data_utils.py:414-415.
 *
 *   hist_x / hist_e : per-row tables the pooling reads (hist_e NULL for MEAN_L2);
 *                     for FINAL_ATTENTION they are the separable per-row outputs
 *                     x and exp(logit) of nrb_final_attention_rows.
 *   cand            : the table candidates are scored against (news_embeddings).
 *   cand_base/alpha : optional fp32 [n_rows] per-row baseline (the classification head's score) blended behind
 *                     the cosine like WeightedSumModel (modeling_utils.py:158-165): alpha*cos + (1-alpha)*base;
 *                     impressions with an empty history get `base` alone (data_model_helper.py:284-299).
 *                     NULL = pure cosine.
 *   *_off           : int64 CSR offsets [n_imp + 1] into hist_idx / cand_idx.
 *   user_out        : optional fp32 [n_imp, dim] (NULL to skip).
 *   scores          : fp32 [cand_off[n_imp]] (absolute candidate positions).
 *   ranks           : optional int32, same indexing.
 * dim * elemsize must be a multiple of 512 bytes and at most 4096. */
int nrb_score_rank(int pool_mode, int dtype, int dim, int64_t n_rows,
                   const void* hist_x, const void* hist_e, int64_t hist_stride,
                   const void* cand, int64_t cand_stride,
                   const float* cand_base, float blend_alpha,
                   const int32_t* hist_idx, const int64_t* hist_off,
                   const int32_t* cand_idx, const int64_t* cand_off, int64_t n_imp,
                   float* user_out, float* scores, int32_t* ranks, int32_t* err_flag,
                   nrb_stream_t stream);

/* ---- dense row kernels -------------------------------------------------------------
 * y[M,N] = epilogue(a[M,K] @ w[N,K]^T + bias[N]) -- the torch.nn.Linear contraction
 * (latent_attention.py:65-74,33-37; modeling_utils.py:218-222).
 *   precision NRB_BF16: a, w are bf16, tcgen05.mma (kind::f16) with fp32 TMEM accumulators,
 *                       operands staged by TMA; K % 64 == 0, N % 32 == 0.
 *   precision NRB_F32 : a, w are fp32, FFMA accumulation (the reference's own fp32 arithmetic).
 * out_dtype selects the dtype of y (and of `res` for NRB_EPI_RESIDUAL, which is fp32).
 * For GEGLU y has N/2 columns.  SOFTMAX (bf16 precision, bf16 output only): every `group` consecutive
 * columns (a power of two in [32, 1024], N % 256 == 0) form one softmax row of which the first
 * `group_valid` are real; groups wider than one 256-column tile are computed by a thread-block cluster
 * that exchanges the row statistics through distributed shared memory. */
int nrb_linear(int precision, int epilogue, int out_dtype,
               const void* a, int64_t lda, const void* w, int64_t ldw, const float* bias,
               const float* res, int64_t ldres, void* y, int64_t ldy,
               int64_t M, int N, int K, int group, int group_valid, nrb_stream_t stream);

/* dst[r, :] = (dst_dtype) src[r, :] for a [n_rows, dim] row block (strides in elements): the fp32 -> bf16 rounding
 * (round to nearest even, = torch .to(bfloat16)) of the cached table `embeddings/<dataset>.pt`
 * (components.py:199-214 writes fp32) on its way into HBM, and the fp32 view of bf16 rows. */
int nrb_convert_rows(const void* src, int src_dtype, int64_t src_stride, void* dst, int dst_dtype,
                     int64_t dst_stride, int64_t n_rows, int dim, nrb_stream_t stream);

/* y = LayerNorm(x) * gamma + beta over the last dimension (biased variance, eps inside the sqrt):
 * torch.nn.LayerNorm at latent_attention.py:10-19 (eps 1e-5) and attention.py:170-171,193 (eps 1e-12). */
int nrb_layer_norm(const void* x, int x_dtype, int64_t ldx, const float* gamma, const float* beta, float eps,
                   void* y, int y_dtype, int64_t ldy, int64_t rows, int dim, nrb_stream_t stream);

/* ---- FinalAttention per-row transform -------------------------------------------------
 * replaces the per-history-slot MLPs of modeling_utils.py:218-222 by one pass over the
 * table (they depend only on the news row; SURVEY.md 8a row a9):
 *   x = W3 relu(W2 relu(W1 e + b1) + b2) + b3 ; elog = exp(W5 relu(W4 x + b4)).
 * Weights are in `precision` dtype, row-major [out,in] (torch Linear layout), biases fp32.
 * x_out / e_out have `out_dtype`. */
size_t nrb_final_attention_rows_workspace_bytes(int precision, int64_t n_rows, int dim, int hidden);
int nrb_final_attention_rows(int precision, int out_dtype, const void* table, int64_t table_stride,
                             int64_t n_rows, int dim, int hidden,
                             const void* w1, const float* b1, const void* w2, const float* b2,
                             const void* w3, const float* b3, const void* w4, const float* b4,
                             const void* w5, void* x_out, void* e_out, int64_t out_stride,
                             void* workspace, size_t workspace_bytes, nrb_stream_t stream);

/* Split-bf16 tensor-core variant for fp32 tables (the rank-exact path): with hi = bf16(v), lo = bf16(v - hi),
 * nrb_split_rows writes [hi | hi | lo] (role 0, activations) or [hi | lo | hi] (role 1, weights) as bf16 rows of
 * 3*dim columns, so that ONE tcgen05 GEMM over K' = 3K accumulates a_hi w_hi + a_hi w_lo + a_lo w_hi in fp32
 * (~2^-17 relative per operand instead of bf16's 2^-9).  nrb_final_attention_rows_split runs the five Linear layers
 * of modeling_utils.py:218-224 that way: fp32 table in, fp32 x / exp(logit) out, weights pre-split with role 1. */
int nrb_split_rows(const float* src, int64_t src_stride, void* dst, int64_t dst_stride, int64_t n_rows, int dim,
                   int role, nrb_stream_t stream);
size_t nrb_final_attention_rows_split_workspace_bytes(int64_t n_rows, int dim, int hidden);
int nrb_final_attention_rows_split(const float* table, int64_t table_stride, int64_t n_rows, int dim, int hidden,
                                   const void* w1s, const float* b1, const void* w2s, const float* b2,
                                   const void* w3s, const float* b3, const void* w4s, const float* b4,
                                   const void* w5s, float* x_out, float* e_out, int64_t out_stride,
                                   void* workspace, size_t workspace_bytes, nrb_stream_t stream);

/* ---- Stage A: latent-attention pooling ---------------------------------------------------
 * replaces latent_attention.py:134-171 LatentAttentionModel.forward.
 *
 * nrb_latent_fold (once per weight set): K,V = to_kv(LN_ctx(latents)) are input independent
 * (latent_attention.py:161,67), so they are projected once and folded into the per-head
 * matrices  A[h*Lp + l, :] = (Wq_h^T k_{h,l}) * dim_head^-0.5   ([heads*Lp, dim])
 *           B[:, h*Lp + l] =  Wout_h v_{h,l}                    ([dim, heads*Lp])
 * so that logits = LN(x) A^T and attn_out = softmax(logits) B^T.  Lp = L rounded up to a
 * power of two (>= 32); padded latents get zero probability.  All inputs fp32; A,B written in `precision`.
 *
 * nrb_latent_forward: x[B,S,dim] (fp32 or bf16) + lengths -> pooled[B,dim] fp32 (masked mean,
 * L2-normalised), or un-pooled fp32 [B,S,dim] when pooled_out is NULL.  Padded tokens are never
 * computed (they cannot influence the output; SURVEY.md 3.2).  `token_mask` is the reference's
 * attention_mask int32 [B,S]; it may be any 0/1 pattern. */
size_t nrb_latent_fold_workspace_bytes(int dim, int heads, int dim_head, int num_latents);
int nrb_latent_fold(int precision, int dim, int heads, int dim_head, int num_latents,
                    const float* latents, const float* ln_ctx_w, const float* ln_ctx_b,
                    const float* w_q, const float* w_kv, const float* w_out,
                    void* a_out, void* b_out, void* workspace, size_t workspace_bytes,
                    nrb_stream_t stream);

typedef struct nrb_latent_weights {
  int precision;        /* NRB_BF16 | NRB_F32: dtype of a, b, w_ff1, w_ff2            */
  int dim, heads, num_latents, latents_padded;
  const void* a;        /* [heads*Lp, dim]   from nrb_latent_fold                     */
  const void* b;        /* [dim, heads*Lp]                                            */
  const float* ln1_w;   /* cross_attend_blocks.0.norm                                 */
  const float* ln1_b;
  const float* ln2_w;   /* cross_attend_blocks.1.norm                                 */
  const float* ln2_b;
  const void* w_ff1;    /* [8*dim, dim] rows interleaved in pairs (a0,a1,g0,g1,...)    */
  const float* b_ff1;   /* [8*dim] interleaved the same way                           */
  const void* w_ff2;    /* [dim, 4*dim]                                               */
  const float* b_ff2;   /* [dim]                                                      */
} nrb_latent_weights;

size_t nrb_latent_forward_workspace_bytes(const nrb_latent_weights* w, int64_t max_tokens);
int nrb_latent_forward(const nrb_latent_weights* w, const void* x, int x_dtype,
                       int64_t batch, int seq, const int32_t* token_mask,
                       float* pooled_out, float* unpooled_out,
                       void* workspace, size_t workspace_bytes, int64_t max_tokens,
                       int64_t* n_tokens_host, nrb_stream_t stream);

/* Varlen form of nrb_latent_forward: x_packed [n_tokens, dim] holds only real tokens, item_off (device int32
 * [batch+1]) their CSR offsets per item -- the layout a packed token store produces (the reference pads each
 * batch to its longest item and masks: data_utils.py:878-933, 753-781).  One chunk: the caller keeps
 * n_tokens <= the max_tokens the workspace was sized for. */
int nrb_latent_forward_packed(const nrb_latent_weights* w, const void* x_packed, int x_dtype,
                              int64_t n_tokens, const int32_t* item_off, int64_t batch,
                              float* pooled_out, void* workspace, size_t workspace_bytes,
                              nrb_stream_t stream);

/* ---- whole-table retrieval: the k best rows of the table for each user -------------------------------------
 * (no reference counterpart: the reference only scores candidate lists it is given.)
 *   score(u, r) = (u / max(|u|, 1e-8)) . c_r / max(|c_r|, 1e-8)    -- the cosine of nrb_score_rank
 * out_rows int32 [n_users, k] / out_scores fp32 [n_users, k]: score descending, equal scores by ascending row id
 * (-0.0 equals 0.0), NaN scores never returned, (-1, NaN) where a user has fewer than k eligible rows.
 *   precision NRB_BF16: `table` and `table_op` are the bf16 table (the same pointer); users are normalised in fp32
 *                       and rounded to bf16.
 *   precision NRB_F32 : `table` is the fp32 table (row norms), `table_op` its nrb_split_rows(role 1) copy [n_rows,
 *                       3*dim]; users are split with role 0, so ONE tensor-core GEMM over K' = 3*dim scores at ~2^-17
 *                       relative.  The FFMA GEMM has no top-k epilogue.
 *   users           : fp32 [n_users, dim] (e.g. nrb_score_rank's user_out).
 *   excl_idx / excl_off : optional CSR (int32 ids, int64 offsets [n_users + 1], n_excl = excl_off[n_users] or more)
 *                     of rows never returned for each user (their history); ids may repeat and need not be sorted.
 *                     An id outside [0, n_rows) sets bit 0 of *err_flag.  Both NULL: nothing excluded.
 * The scores are computed by one tcgen05 GEMM whose epilogue keeps each row's running top-k in shared memory: the
 * [n_users, n_rows] score matrix never exists in memory.  A user's result does not depend on the other users of the
 * call as long as the same GEMM configuration runs (n_users <= 128: single CTAs; more: CTA pairs).
 * Limits: 1 <= k <= 32, dim % 64 == 0, any n_users >= 1 and n_rows >= 1.  Invalid arguments are rejected before any
 * CUDA call (the workspace query then returns 0). */
size_t nrb_recommend_workspace_bytes(int precision, int dim, int64_t n_rows, int64_t n_users, int64_t n_excl, int k);
int nrb_recommend(int precision, int dim, int64_t n_rows, const void* table, int64_t table_stride,
                  const void* table_op, int64_t op_stride, const float* users, int64_t users_stride, int64_t n_users,
                  const int32_t* excl_idx, const int64_t* excl_off, int64_t n_excl, int k,
                  int32_t* out_rows, float* out_scores, int32_t* err_flag, void* workspace, size_t workspace_bytes,
                  nrb_stream_t stream);

/* nrb_recommend from a pool of the table's rows, with the classification-baseline blend of nrb_score_rank.
 * (nrb_recommend is this call with n_pool = -1 and cand_base = NULL.)  Arguments of nrb_recommend, plus:
 *   pool / n_pool   : int32 table row ids, strictly ascending, in [0, n_rows): only these rows are eligible, and the
 *                     GEMM runs over them alone (their rows of table_op are gathered into the workspace, so table_op
 *                     must then be 16-byte aligned with a 16-byte multiple row pitch).  A violation sets bit 0 of
 *                     *err_flag.  n_pool < 0: the whole table (pool ignored).  n_pool = 0: every list is padding and
 *                     no GEMM runs.  Returned ids are table row ids; excluded ids outside the pool are ignored but
 *                     still range-checked against n_rows.
 *   cand_base       : optional fp32 [n_rows] per-row baseline (NULL: pure cosine), blend_alpha its weight:
 *                       score = cos * blend_alpha + cand_base[r] * (1 - blend_alpha)   for users with a history,
 *                       score = cand_base[r]                                           for users without one
 *                     (the expression and the fallback of nrb_score_rank; the fallback is a select, so the NaN vector
 *                     a mean-pool encoder gives an empty history never scores).  A row whose baseline is NaN is never
 *                     returned.
 *   hist_off        : optional int64 [n_users + 1] history offsets; user u has no history when
 *                     hist_off[u + 1] == hist_off[u].  NULL: every user has one.  Separate from excl_off so that the
 *                     fallback holds when the history is not excluded.
 * Order, padding, limits and the dependence on the other users of the call are those of nrb_recommend, with the
 * GEMM configuration chosen by n_users alone. */
size_t nrb_recommend_pool_blend_workspace_bytes(int precision, int dim, int64_t n_rows, int64_t n_users,
                                                int64_t n_excl, int k, int64_t n_pool);
int nrb_recommend_pool_blend(int precision, int dim, int64_t n_rows, const void* table, int64_t table_stride,
                             const void* table_op, int64_t op_stride, const float* users, int64_t users_stride,
                             int64_t n_users, const int32_t* excl_idx, const int64_t* excl_off, int64_t n_excl, int k,
                             const int32_t* pool, int64_t n_pool, const float* cand_base, float blend_alpha,
                             const int64_t* hist_off, int32_t* out_rows, float* out_scores, int32_t* err_flag,
                             void* workspace, size_t workspace_bytes, nrb_stream_t stream);

/* ---- MIND metrics on device (consumer of the ranks; "next" row of the hot path) ---------------
 * replaces evaluation.py:34-98 (score_row per impression in a 4-process pool + mean):
 * per impression AUC (tie-aware, = sklearn roc_auc_score), MRR, nDCG@5, nDCG@10 from dense ranks and
 * integer labels with y_score = 1/rank and the reversed-stable-argsort order among tied ranks.
 * per_imp_out: optional double [n_imp, 4] (NaN for impressions with a single class or NaN ranks);
 * sums: double[5], ACCUMULATED (caller zeroes): sum of the four metrics over valid impressions and
 * their count. */
int nrb_mind_metrics(const int32_t* ranks, const int8_t* labels, const int64_t* offsets,
                     int64_t n_imp, double* per_imp_out, double* sums, nrb_stream_t stream);

/* ---- row-sharded table: all-gather by peer stores over NVLink -----------------------------------
 * (no reference counterpart: the reference is single GPU; BASELINE configs[4] / SURVEY.md 8e.)
 * Writes rows [0, n_rows) of the local chunk `src` into rows dst_row_offset + r of EVERY destination
 * in dst_ptrs_host[0..world) -- device pointers to each rank's copy of the full table, peer-mapped
 * (symmetric memory) -- optionally converting fp32 -> bf16 on the way.  `dst_ptrs_host` is a HOST array. */
int nrb_push_rows(const void* src, int src_dtype, int64_t src_stride, int64_t n_rows, int dim,
                  void* const* dst_ptrs_host, int world, int dst_dtype, int64_t dst_row_offset,
                  int64_t dst_stride, nrb_stream_t stream);

/* Copy-engine variant of the same all-gather step: `n_bytes` contiguous bytes at `src` are copied to
 * dst_ptrs_host[g] + dst_byte_offset for every g in [0, world) with one asynchronous peer copy each
 * (a destination equal to `src` -- the chunk already sits in the local table -- is skipped).  Unlike the
 * store kernel the DMA engines need no SM resources, so the transfer proceeds at NVLink rate even
 * while persistent GEMM CTAs own every SM's register file.  dst_ptrs_host is a HOST array. */
int nrb_push_bytes(const void* src, int64_t n_bytes, void* const* dst_ptrs_host, int world,
                   int64_t dst_byte_offset, nrb_stream_t stream);

/* Fused compute + collective variant: the all-gather rides INSIDE the tensor-core kernels.  nrb_push_attach
 * registers up to 3 row segments (finished rows of the previous chunk) whose destination `mc_dst` is the NVLink
 * MULTICAST address (NVLS) of the table every rank holds; the next `spread` tcgen05 GEMM launches issued by this
 * host thread (nrb_linear / nrb_final_attention_rows / nrb_latent_forward on the bf16 path) each carry
 * ceil(n_rows / spread) rows of every segment: the otherwise idle fourth control warp of each persistent GEMM CTA
 * streams them out with one multimem.st per 16 bytes (fp32 -> bf16 rounding on the way if asked) while the MMA and
 * epilogue warps work, so the transfer needs no extra SM, no copy engine and no second kernel.  nrb_push_flush
 * sends whatever no GEMM picked up with a small store-only kernel (also the way to push the last chunk). */
typedef struct nrb_push_seg {
  const void* src;         /* local rows [n_rows, dim]                                   */
  int src_dtype;           /* NRB_F32 | NRB_BF16                                         */
  int64_t src_stride;      /* elements                                                   */
  void* mc_dst;            /* multicast address of the destination table (row 0)         */
  int dst_dtype;           /* NRB_BF16 | NRB_F32 (same as src, or fp32 -> bf16)          */
  int64_t dst_stride;      /* elements                                                   */
  int64_t dst_row_offset;  /* first destination row                                      */
  int64_t n_rows;
  int dim;
} nrb_push_seg;
int nrb_push_attach(const nrb_push_seg* segs, int n_segs, int spread);
int nrb_push_flush(nrb_stream_t stream);
/* drop pending segments without sending them (error paths: nothing stale may ride in a later, unrelated GEMM).
 * Pending segments are per host thread AND per device: launches on another device never carry them. */
void nrb_push_cancel(void);

/* ---- behaviour log -> CSR index builder (host; the step in front of the hot path) ------------------
 * replaces data_utils.py:168-232 split_impressions_and_history.  `impressions` / `history` are
 * '\n'-separated UTF-8 buffers with one line per behaviour row (empty history line = no history).
 * Row ids are assigned in first-appearance order over history-then-impression tokens.  Returns an
 * opaque handle (NULL on error); query sizes, export into caller-owned HOST arrays, then free.
 * sizes[0..4] = {n_news, sum_history, n_history_rows, sum_candidates, label_present}. */
void* nrb_csr_build(const char* impressions, int64_t imp_bytes, const char* history, int64_t hist_bytes,
                    int64_t n_rows);
int nrb_csr_sizes(void* handle, int64_t* sizes);
int nrb_csr_export(void* handle, int32_t* hist_idx, int32_t* hist_owner, int32_t* hist_len,
                   int32_t* cand_idx, int32_t* cand_owner, int32_t* cand_len, int8_t* labels);
int64_t nrb_csr_news_ids(void* handle, char* out, int64_t cap);
void nrb_csr_free(void* handle);

/* ---- host staging for the packed token file (the data format in front of Stage A) -------------------------
 * (replaces the per-item sqlite read + torch.load + pad-to-batch-max of data_utils.py:878-933, 753-781: a chunk of
 * items is one contiguous byte range of the mmap'd file.)  memcpy of `n_bytes` HOST bytes split over `n_threads`
 * worker threads (page cache -> pinned staging buffer); blocks until done. */
int nrb_host_copy(void* dst_host, const void* src_host, int64_t n_bytes, int n_threads);

#ifdef __cplusplus
}
#endif
#endif /* NRB200_H_ */
