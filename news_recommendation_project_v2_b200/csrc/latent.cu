// Stage A: latent-attention pooling head (reference latent_attention.py:77-171).
//
//   nrb_latent_fold    : one-time weight preparation.  K,V = to_kv(LN_ctx(latents)) do not depend on
//                        the input (the reference recomputes them for every batch row, :161,:67), so they
//                        are projected once and folded through to_q / to_out into two per-head matrices
//                        A [heads*Lp, d] and B [d, heads*Lp]:  logits = LN(x) A^T, attn = softmax(logits) B^T.
//   nrb_latent_forward : varlen token packing (padded tokens are never computed) -> LN -> GEMM(A) ->
//                        per-head softmax -> GEMM(B)+residual -> LN -> GEMM(FF1)+bias+GEGLU ->
//                        GEMM(FF2)+bias+residual -> masked mean -> L2 normalise.
// All contractions go through nrb::linear (tcgen05 for bf16 weights, FFMA for fp32 weights).
#include "dense.cuh"

#include <algorithm>
#include <cmath>

namespace nrb {

// ---- varlen packing ----------------------------------------------------------------------
// counts[i] = number of non-zero mask entries of item i (one warp per item)
__global__ void __launch_bounds__(256)
count_valid_kernel(const int32_t* mask, int64_t items, int seq, int32_t* counts) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp_id; i < items; i += n_warps) {
    int c = 0;
    for (int s = lane; s < seq; s += 32) c += mask[i * seq + s] != 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(kFullMask, c, o);
    if (lane == 0) counts[i] = c;
  }
}

// exclusive scan of counts -> item_off[items+1]; total -> *m_dev.  Single CTA (items <= ~1e6).
__global__ void __launch_bounds__(1024)
scan_items_kernel(const int32_t* counts, int64_t items, int32_t* item_off, int32_t* m_dev) {
  __shared__ int32_t warp_tot[32];
  __shared__ int32_t carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) carry = 0;
  __syncthreads();
  for (int64_t base = 0; base < items; base += 1024) {
    const int64_t i = base + tid;
    const int32_t v = i < items ? counts[i] : 0;
    int32_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int32_t t = __shfl_up_sync(kFullMask, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_tot[warp] = incl;
    __syncthreads();
    if (warp == 0) {
      int32_t w = warp_tot[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int32_t t = __shfl_up_sync(kFullMask, w, o);
        if (lane >= o) w += t;
      }
      warp_tot[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const int32_t before = carry + (warp > 0 ? warp_tot[warp - 1] : 0) + incl - v;
    if (i < items) item_off[i] = before;
    __syncthreads();
    if (tid == 1023) carry = before + v;
    __syncthreads();
  }
  if (tid == 0) {
    item_off[items] = carry;
    *m_dev = carry;
  }
}

// row_map[item_off[i] + rank] = i*seq + s for every valid token (one warp per item)
__global__ void __launch_bounds__(256)
fill_row_map_kernel(const int32_t* mask, int64_t items, int seq, const int32_t* item_off, int32_t* row_map) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t i = warp_id; i < items; i += n_warps) {
    int32_t pos = item_off[i];
    for (int s0 = 0; s0 < seq; s0 += 32) {
      const int s = s0 + lane;
      const bool v = s < seq && mask[i * seq + s] != 0;
      const unsigned b = __ballot_sync(kFullMask, v);
      if (v) row_map[pos + __popc(b & ((1u << lane) - 1))] = (int32_t)(i * seq + s);
      pos += __popc(b);
    }
  }
}

// int32 item offsets -> int64 CSR offsets (the layout nrb_score_rank takes)
__global__ void widen_offsets_kernel(const int32_t* in, int64_t n, int64_t* out) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
    out[i] = in[i];
}

// pooled[i] = normalize(mean over the item's packed rows)  (latent_attention.py:165-170)
// one CTA per item; thread t owns float4 columns t, t+256, ...
template <int MAXV>
__global__ void __launch_bounds__(256)
pool_items_kernel(const float* h, int64_t ldh, const int32_t* item_off, int seq_if_dense, int64_t items, int dim,
                  float* out) {
  __shared__ float red[8];
  const int tid = threadIdx.x;
  const int nvec = dim / 4;
  for (int64_t i = blockIdx.x; i < items; i += gridDim.x) {
    const int64_t r0 = item_off != nullptr ? item_off[i] : i * seq_if_dense;
    const int64_t r1 = item_off != nullptr ? item_off[i + 1] : (i + 1) * seq_if_dense;
    const float cnt = (float)(r1 - r0);
    float4 acc[MAXV];
    float ss = 0.f;
#pragma unroll
    for (int k = 0; k < MAXV; ++k) {
      const int v = tid + k * 256;
      acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (v < nvec) {
        for (int64_t r = r0; r < r1; ++r) {
          const float4 t = *reinterpret_cast<const float4*>(h + r * ldh + (size_t)v * 4);
          acc[k].x += t.x;
          acc[k].y += t.y;
          acc[k].z += t.z;
          acc[k].w += t.w;
        }
        acc[k].x /= cnt;  // 0/0 -> NaN for an all-masked item, like the reference
        acc[k].y /= cnt;
        acc[k].z /= cnt;
        acc[k].w /= cnt;
        ss += acc[k].x * acc[k].x + acc[k].y * acc[k].y + acc[k].z * acc[k].z + acc[k].w * acc[k].w;
      }
    }
    ss = warp_sum(ss);
    if ((tid & 31) == 0) red[tid >> 5] = ss;
    __syncthreads();
    float tot = 0.f;
#pragma unroll
    for (int w = 0; w < 8; ++w) tot += red[w];
    const float nrm = fmaxf(sqrtf(tot), 1e-12f);  // F.normalize eps
#pragma unroll
    for (int k = 0; k < MAXV; ++k) {
      const int v = tid + k * 256;
      if (v < nvec)
        *reinterpret_cast<float4*>(out + i * (int64_t)dim + (size_t)v * 4) =
            make_float4(acc[k].x / nrm, acc[k].y / nrm, acc[k].z / nrm, acc[k].w / nrm);
    }
    __syncthreads();
  }
}

// padded latent count: a power of two >= 32 so that softmax groups tile the 256-column MMA tiles
static int pad_latents(int L) {
  int p = 32;
  while (p < L) p <<= 1;
  return p;
}

// latent rows of the fold's FFMA GEMMs: the B fold has N = latents, and that GEMM takes N in multiples of 4; the rows
// past L are zero, so they give zero rows of A and zero columns of B (L4 <= Lp)
static int fold_latents(int L) { return (L + 3) / 4 * 4; }

struct FoldWs {
  float *cn, *kv, *wqT, *a32, *b32;
  size_t bytes;
};
static FoldWs fold_ws(void* base, int dim, int heads, int dim_head, int L) {
  const int inner = heads * dim_head;
  const int Lp = pad_latents(L), L4 = fold_latents(L);
  Workspace ws(base, (size_t)-1);
  FoldWs f;
  f.cn = (float*)ws.take((size_t)L4 * dim * 4);
  f.kv = (float*)ws.take((size_t)L4 * 2 * inner * 4);
  f.wqT = (float*)ws.take((size_t)dim * inner * 4);
  f.a32 = (float*)ws.take((size_t)heads * Lp * dim * 4);
  f.b32 = (float*)ws.take((size_t)dim * heads * Lp * 4);
  f.bytes = ws.used + 256;
  return f;
}

struct FwdWs {
  int32_t *counts, *item_off, *m_dev, *row_map;
  void *xn, *p, *hn, *g;
  float *logits, *h1, *h2;
  size_t bytes;
};
// fused softmax epilogue (logits never leave TMEM): bf16, whole 256-column tiles, a softmax row within one cluster
static bool fused_softmax(const nrb_latent_weights* w) {
  return w->precision == NRB_BF16 && (w->heads * w->latents_padded) % 256 == 0 && w->latents_padded <= 1024;
}

static FwdWs fwd_ws(void* base, const nrb_latent_weights* w, int64_t cap_tokens, int64_t cap_items) {
  const size_t es = dtype_size(w->precision);
  const int64_t hl = (int64_t)w->heads * w->latents_padded;
  Workspace ws(base, (size_t)-1);
  FwdWs f;
  f.counts = (int32_t*)ws.take((size_t)cap_items * 4);
  f.item_off = (int32_t*)ws.take((size_t)(cap_items + 1) * 4);
  f.m_dev = (int32_t*)ws.take(16);
  f.row_map = (int32_t*)ws.take((size_t)cap_tokens * 4);
  f.xn = ws.take((size_t)cap_tokens * w->dim * es);
  f.logits = fused_softmax(w) ? nullptr : (float*)ws.take((size_t)cap_tokens * hl * 4);
  f.p = ws.take((size_t)cap_tokens * hl * es);
  f.h1 = (float*)ws.take((size_t)cap_tokens * w->dim * 4);
  f.hn = ws.take((size_t)cap_tokens * w->dim * es);
  f.g = ws.take((size_t)cap_tokens * 4 * w->dim * es);
  f.h2 = (float*)ws.take((size_t)cap_tokens * w->dim * 4);
  f.bytes = ws.used + 256;
  return f;
}

}  // namespace nrb

using namespace nrb;

extern "C" int nrb_mask_to_csr(const int32_t* mask, int64_t batch, int seq, int32_t* idx_out, int64_t* off_out,
                               int32_t* workspace, nrb_stream_t stream) {
  NRB_REQUIRE(batch >= 0 && seq > 0, "nrb_mask_to_csr: bad sizes");
  NRB_REQUIRE(batch * (int64_t)seq < (int64_t)1 << 31, "nrb_mask_to_csr: batch * seq must fit int32");
  NRB_REQUIRE(off_out != nullptr, "nrb_mask_to_csr: null pointer");
  cudaStream_t st = as_stream(stream);
  if (batch == 0) {
    NRB_CUDA_CHECK(cudaMemsetAsync(off_out, 0, 8, st));
    return NRB_OK;
  }
  NRB_REQUIRE(mask && idx_out && workspace, "nrb_mask_to_csr: null pointer");
  int32_t* counts = workspace;                // [batch]
  int32_t* item_off = workspace + batch;      // [batch + 1]
  int32_t* total = workspace + 2 * batch + 1;  // [1]
  const int g1 = (int)std::min<int64_t>((batch + 7) / 8, (int64_t)sm_count_cached() * 16);
  count_valid_kernel<<<g1, 256, 0, st>>>(mask, batch, seq, counts); note_launch();
  scan_items_kernel<<<1, 1024, 0, st>>>(counts, batch, item_off, total); note_launch();
  fill_row_map_kernel<<<g1, 256, 0, st>>>(mask, batch, seq, item_off, idx_out); note_launch();
  const int g2 = (int)std::min<int64_t>((batch + 1 + 255) / 256, (int64_t)sm_count_cached() * 4);
  widen_offsets_kernel<<<g2, 256, 0, st>>>(item_off, batch + 1, off_out); note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

extern "C" size_t nrb_latent_fold_workspace_bytes(int dim, int heads, int dim_head, int num_latents) {
  return fold_ws(nullptr, dim, heads, dim_head, num_latents).bytes;
}

extern "C" int nrb_latent_fold(int precision, int dim, int heads, int dim_head, int num_latents,
                               const float* latents, const float* ln_ctx_w, const float* ln_ctx_b,
                               const float* w_q, const float* w_kv, const float* w_out, void* a_out, void* b_out,
                               void* workspace, size_t workspace_bytes, nrb_stream_t stream) {
  NRB_REQUIRE(precision == NRB_F32 || precision == NRB_BF16, "nrb_latent_fold: bad precision");
  NRB_REQUIRE(dim > 0 && dim % 16 == 0, "nrb_latent_fold: dim must be a multiple of 16");
  NRB_REQUIRE(heads > 0 && dim_head > 0 && dim_head % 16 == 0, "nrb_latent_fold: dim_head must be a multiple of 16");
  NRB_REQUIRE(num_latents > 0, "nrb_latent_fold: num_latents must be positive");
  NRB_REQUIRE(precision != NRB_BF16 || heads * pad_latents(num_latents) % 64 == 0,
              "nrb_latent_fold: bf16 needs heads * latents_padded to be a multiple of 64 (got %d x %d)", heads,
              pad_latents(num_latents));
  NRB_REQUIRE(latents && ln_ctx_w && ln_ctx_b && w_q && w_kv && w_out && a_out && b_out && workspace,
              "nrb_latent_fold: null pointer");
  FoldWs f = fold_ws(workspace, dim, heads, dim_head, num_latents);
  if (workspace_bytes < f.bytes) {
    set_error("nrb_latent_fold: workspace too small (%zu < %zu)", workspace_bytes, f.bytes);
    return NRB_E_WORKSPACE;
  }
  cudaStream_t st = as_stream(stream);
  const int L = num_latents, L4 = fold_latents(L), Lp = pad_latents(L), inner = heads * dim_head, hl = heads * Lp;
  int rc;
  // context = LN_ctx(latents); kv = to_kv(context)            (latent_attention.py:18-19, 67)
  if (L4 > L) NRB_CUDA_CHECK(cudaMemsetAsync(f.cn + (size_t)L * dim, 0, (size_t)(L4 - L) * dim * 4, st));
  if ((rc = layer_norm_rows(latents, NRB_F32, dim, nullptr, ln_ctx_w, ln_ctx_b, f.cn, NRB_F32, dim, nullptr, 0, L,
                            nullptr, dim, st)) != NRB_OK)
    return rc;
  if ((rc = gemm_f32_simt(NRB_EPI_NONE, NRB_F32, f.cn, dim, w_kv, dim, nullptr, nullptr, 0, f.kv, 2 * inner, L4,
                          nullptr, 2 * inner, dim, st)) != NRB_OK)
    return rc;
  // fold the SDPA scale dim_head^-0.5 (:69-72) into K
  if ((rc = scale_cols_f32(f.kv, 2 * inner, L4, inner, 1.0f / sqrtf((float)dim_head), st)) != NRB_OK) return rc;
  if ((rc = transpose_f32(w_q, inner, dim, f.wqT, st)) != NRB_OK) return rc;
  NRB_CUDA_CHECK(cudaMemsetAsync(f.a32, 0, (size_t)hl * dim * 4, st));
  NRB_CUDA_CHECK(cudaMemsetAsync(f.b32, 0, (size_t)dim * hl * 4, st));
  for (int h = 0; h < heads; ++h) {
    // A_h[l, i] = sum_c K[l, h*dh+c] * Wq[h*dh+c, i]
    if ((rc = gemm_f32_simt(NRB_EPI_NONE, NRB_F32, f.kv + h * dim_head, 2 * inner, f.wqT + h * dim_head, inner,
                            nullptr, nullptr, 0, f.a32 + (size_t)h * Lp * dim, dim, L4, nullptr, dim, dim_head,
                            st)) != NRB_OK)
      return rc;
    // B[i, h*Lp + l] = sum_c Wout[i, h*dh+c] * V[l, h*dh+c]
    if ((rc = gemm_f32_simt(NRB_EPI_NONE, NRB_F32, w_out + h * dim_head, inner, f.kv + inner + h * dim_head,
                            2 * inner, nullptr, nullptr, 0, f.b32 + (size_t)h * Lp, hl, dim, nullptr, L4, dim_head,
                            st)) != NRB_OK)
      return rc;
  }
  if ((rc = convert_rows(f.a32, NRB_F32, dim, a_out, precision, dim, hl, dim, st)) != NRB_OK) return rc;
  if ((rc = convert_rows(f.b32, NRB_F32, hl, b_out, precision, hl, dim, hl, st)) != NRB_OK) return rc;
  return NRB_OK;
}

// LN -> logits GEMM + per-head softmax -> value GEMM + residual -> LN -> GEGLU GEMM -> output GEMM + residual for
// `rows_cap` packed token rows (effective count *m_dev when given); h2 receives the fp32 block output.
static int latent_block_rows(const nrb_latent_weights* w, const FwdWs& f, const void* xc, int x_dtype,
                             const int32_t* row_map, const int* m_dev, int64_t rows_cap, float* h2, cudaStream_t st) {
  const int d = w->dim, P = w->precision;
  const int hl = w->heads * w->latents_padded;
  int rc;
    // xn = LN1(x), gathered through the row map when tokens are packed      latent_attention.py:16
    if ((rc = layer_norm_rows(xc, x_dtype, d, row_map, w->ln1_w, w->ln1_b, f.xn, P, d, nullptr, 0, rows_cap, m_dev, d,
                              st)) != NRB_OK)
      return rc;
    // P = softmax_h(xn A^T)  (SDPA scale folded into A)            :65-72
    if (fused_softmax(w)) {
      // fused: logits never leave TMEM; row statistics exchanged across the cluster through DSMEM
      if ((rc = linear(P, NRB_EPI_SOFTMAX, P, f.xn, d, w->a, d, nullptr, nullptr, 0, f.p, hl, rows_cap, m_dev, hl, d,
                       st, w->latents_padded, w->num_latents)) != NRB_OK)
        return rc;
    } else {
      if ((rc = linear(P, NRB_EPI_NONE, NRB_F32, f.xn, d, w->a, d, nullptr, nullptr, 0, f.logits, hl, rows_cap,
                       m_dev, hl, d, st)) != NRB_OK)
        return rc;
      if ((rc = softmax_groups(f.logits, hl, f.p, P, hl, rows_cap, m_dev, w->heads, w->latents_padded,
                               w->num_latents, st)) != NRB_OK)
        return rc;
    }
    // h1 = P B^T + x                                               :74, :162
    // (the residual operand is the RAW input row, read in place through the same row map: no fp32 copy)
    if ((rc = linear(P, NRB_EPI_RESIDUAL, NRB_F32, f.p, hl, w->b, hl, nullptr, xc, d, f.h1, d, rows_cap, m_dev, d, hl,
                     st, 0, 0, x_dtype, row_map)) != NRB_OK)
      return rc;
    // hn = LN2(h1)                                                 :16 (second PreNorm)
    if ((rc = layer_norm_rows(f.h1, NRB_F32, d, nullptr, w->ln2_w, w->ln2_b, f.hn, P, d, nullptr, 0, rows_cap, m_dev,
                              d, st)) != NRB_OK)
      return rc;
    // g = GEGLU(hn W1^T + b1)                                      :33-35, 24-27
    if ((rc = linear(P, NRB_EPI_GEGLU, P, f.hn, d, w->w_ff1, d, w->b_ff1, nullptr, 0, f.g, 4 * d, rows_cap, m_dev,
                     8 * d, d, st)) != NRB_OK)
      return rc;
    // h2 = g W2^T + b2 + h1                                        :36, :163
    if ((rc = linear(P, NRB_EPI_RESIDUAL, NRB_F32, f.g, 4 * d, w->w_ff2, 4 * d, w->b_ff2, f.h1, d, h2, d, rows_cap,
                     m_dev, d, 4 * d, st)) != NRB_OK)
      return rc;
  return NRB_OK;
}

static int64_t chunk_items_for(int64_t max_tokens, int seq) { return std::max<int64_t>(1, max_tokens / seq); }

extern "C" size_t nrb_latent_forward_workspace_bytes(const nrb_latent_weights* w, int64_t max_tokens) {
  if (w == nullptr || max_tokens <= 0) return 0;
  // capacity in items is unknown here (depends on seq): bound it by max_tokens (seq >= 1)
  return fwd_ws(nullptr, w, max_tokens, max_tokens).bytes;
}

extern "C" int nrb_latent_forward(const nrb_latent_weights* w, const void* x, int x_dtype, int64_t batch, int seq,
                                  const int32_t* token_mask, float* pooled_out, float* unpooled_out,
                                  void* workspace, size_t workspace_bytes, int64_t max_tokens,
                                  int64_t* n_tokens_host, nrb_stream_t stream) {
  NRB_REQUIRE(w != nullptr, "nrb_latent_forward: null weights");
  NRB_REQUIRE(w->precision == NRB_F32 || w->precision == NRB_BF16, "nrb_latent_forward: bad precision");
  NRB_REQUIRE(x_dtype == NRB_F32 || x_dtype == NRB_BF16, "nrb_latent_forward: bad x dtype");
  NRB_REQUIRE(batch >= 0 && seq > 0, "nrb_latent_forward: bad batch/seq");
  NRB_REQUIRE((pooled_out != nullptr) != (unpooled_out != nullptr),
              "nrb_latent_forward: exactly one of pooled_out / unpooled_out must be given");
  NRB_REQUIRE(pooled_out == nullptr || token_mask != nullptr, "nrb_latent_forward: pooling needs token_mask");
  NRB_REQUIRE(w->dim % 64 == 0, "nrb_latent_forward: dim must be a multiple of 64 (got %d)", w->dim);
  NRB_REQUIRE(w->latents_padded >= 32 && (w->latents_padded & (w->latents_padded - 1)) == 0 &&
                  w->latents_padded >= w->num_latents,
              "nrb_latent_forward: latents_padded must be a power of two >= max(32, num_latents)");
  NRB_REQUIRE(max_tokens >= seq, "nrb_latent_forward: max_tokens (%lld) must be >= seq (%d)", (long long)max_tokens,
              seq);
  NRB_REQUIRE(w->dim <= 4096, "nrb_latent_forward: dim > 4096 unsupported");
  if (n_tokens_host) *n_tokens_host = -1;
  if (batch == 0) return NRB_OK;
  NRB_REQUIRE(x && workspace, "nrb_latent_forward: null pointer");
  const int64_t ib = std::min<int64_t>(batch, chunk_items_for(max_tokens, seq));
  const int64_t cap = ib * seq;
  FwdWs f = fwd_ws(workspace, w, cap, ib);
  if (workspace_bytes < f.bytes) {
    set_error("nrb_latent_forward: workspace too small (%zu < %zu)", workspace_bytes, f.bytes);
    return NRB_E_WORKSPACE;
  }
  cudaStream_t st = as_stream(stream);
  const int d = w->dim;
  const size_t xs = dtype_size(x_dtype);
  const bool packed = pooled_out != nullptr;
  const int sms = sm_count_cached();
  for (int64_t i0 = 0; i0 < batch; i0 += ib) {
    const int64_t items = std::min<int64_t>(ib, batch - i0);
    const int64_t rows_cap = items * seq;
    const void* xc = (const char*)x + (size_t)i0 * seq * d * xs;
    const int32_t* row_map = nullptr;
    const int* m_dev = nullptr;
    int rc;
    if (packed) {
      const int32_t* mk = token_mask + i0 * seq;
      const int g1 = (int)std::min<int64_t>((items + 7) / 8, (int64_t)sms * 16);
      count_valid_kernel<<<g1, 256, 0, st>>>(mk, items, seq, f.counts); note_launch();
      scan_items_kernel<<<1, 1024, 0, st>>>(f.counts, items, f.item_off, f.m_dev); note_launch();
      fill_row_map_kernel<<<g1, 256, 0, st>>>(mk, items, seq, f.item_off, f.row_map); note_launch();
      NRB_CUDA_CHECK(cudaGetLastError());
      row_map = f.row_map;
      m_dev = f.m_dev;
    }
    float* h2 = packed ? f.h2 : unpooled_out + (size_t)i0 * seq * d;
    if ((rc = latent_block_rows(w, f, xc, x_dtype, row_map, m_dev, rows_cap, h2, st)) != NRB_OK) return rc;
    if (packed) {
      const int gp = (int)std::min<int64_t>(items, (int64_t)sms * 16);
      pool_items_kernel<4><<<gp, 256, 0, st>>>(f.h2, d, f.item_off, seq, items, d, pooled_out + i0 * d); note_launch();
      NRB_CUDA_CHECK(cudaGetLastError());
    }
  }
  return NRB_OK;
}

// Varlen entry: tokens already packed [n_tokens, dim] with CSR item offsets (device int32 [batch+1]); this is the
// layout a packed token store hands over (the reference pads per batch: data_utils.py:878-933, 753-781).
extern "C" int nrb_latent_forward_packed(const nrb_latent_weights* w, const void* x_packed, int x_dtype,
                                         int64_t n_tokens, const int32_t* item_off, int64_t batch,
                                         float* pooled_out, void* workspace, size_t workspace_bytes,
                                         nrb_stream_t stream) {
  NRB_REQUIRE(w != nullptr, "nrb_latent_forward_packed: null weights");
  NRB_REQUIRE(w->precision == NRB_F32 || w->precision == NRB_BF16, "nrb_latent_forward_packed: bad precision");
  NRB_REQUIRE(x_dtype == NRB_F32 || x_dtype == NRB_BF16, "nrb_latent_forward_packed: bad x dtype");
  NRB_REQUIRE(n_tokens >= 0 && batch >= 0, "nrb_latent_forward_packed: bad sizes");
  NRB_REQUIRE(w->dim % 64 == 0 && w->dim <= 4096, "nrb_latent_forward_packed: unsupported dim %d", w->dim);
  if (batch == 0) return NRB_OK;
  if (n_tokens == 0) {
    // every item is empty: the reference's masked mean is 0/0 = NaN (latent_attention.py:165-168)
    NRB_REQUIRE(item_off && pooled_out, "nrb_latent_forward_packed: null pointer");
    const int gp0 = (int)std::min<int64_t>(batch, (int64_t)sm_count_cached() * 16);
    pool_items_kernel<4><<<gp0, 256, 0, as_stream(stream)>>>(nullptr, w->dim, item_off, 0, batch, w->dim, pooled_out);
    note_launch();
    NRB_CUDA_CHECK(cudaGetLastError());
    return NRB_OK;
  }
  NRB_REQUIRE(x_packed && item_off && pooled_out && workspace, "nrb_latent_forward_packed: null pointer");
  FwdWs f = fwd_ws(workspace, w, n_tokens, 1);
  if (workspace_bytes < f.bytes) {
    set_error("nrb_latent_forward_packed: workspace too small (%zu < %zu)", workspace_bytes, f.bytes);
    return NRB_E_WORKSPACE;
  }
  cudaStream_t st = as_stream(stream);
  int rc;
  if ((rc = latent_block_rows(w, f, x_packed, x_dtype, nullptr, nullptr, n_tokens, f.h2, st)) != NRB_OK) return rc;
  const int gp = (int)std::min<int64_t>(batch, (int64_t)sm_count_cached() * 16);
  pool_items_kernel<4><<<gp, 256, 0, st>>>(f.h2, w->dim, item_off, 0, batch, w->dim, pooled_out); note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}
