// Stage B + C: clicked-history gather -> user vector -> cosine scores -> dense rank.
//
// Replaces (reference, src/news_rec_utils/):
//   data_utils.py:784-791      final_attention_eval_collate_fn (CPU gather in DataLoader workers)
//   modeling_utils.py:224-228  FinalAttention pooling (exp-weights, masked normalise, weighted sum)
//   latent_attention.py:165-170 masked mean + F.normalize (LatentAttention as user encoder)
//   data_model_helper.py:200-230 per-impression F.cosine_similarity loop
//   data_utils.py:414-415      scipy.stats.rankdata(-x, "dense") per impression
//
// Bandwidth-bound design: ONE WARP PER IMPRESSION.  A table row is read with coalesced
// 128-bit loads (lane l owns 16-byte vectors l, l+32, ...), history rows are accumulated in
// fp32 registers, the user vector never leaves the register file, each candidate row is
// reduced with warp shuffles and the impression's scores are ranked in shared memory by the
// same warp.  Algorithmic bytes per impression: (r*H + C)*d*e + 4(H+C) + 8C  (SURVEY 8d).
#include "common.cuh"

#include <algorithm>

namespace nrb {

constexpr int kWarpsPerCta = 8;
// Fused score kernel: warps per CTA.  A CTA keeps its SM slot until its slowest warp is done and impressions
// differ widely in size (H 1..50, C 2..300), so with 8-warp CTAs ~25 % of the warp slots idled (ncu: 12.1 of 16
// resident warps active).  One-warp CTAs hand the load balancing to the hardware CTA scheduler: same-box A/B
// 6,175 -> 6,726 GB/s (FinalAttention pooling), 5,216 -> 5,743 GB/s (mean pooling); 2 / 4 warps land in between.
#ifndef NRB_SCORE_WARPS
#define NRB_SCORE_WARPS 1
#endif
#ifndef NRB_SCORE_GRID_MULT
#define NRB_SCORE_GRID_MULT 4
#endif
constexpr int kScoreWarps = NRB_SCORE_WARPS;
constexpr int kRankCap = 512;  // scores of one impression staged in smem (per warp)

// Dense rank (descending) of s[0..n) by one warp.  r is output AND scratch: bit 31 of r[k]
// temporarily holds "k is the first occurrence of its value".  rank_j = 1 + number of
// distinct values greater than s_j; equal scores (incl. -0.0 == 0.0) share a rank; any NaN
// makes the whole group rank 0 (scipy nan_policy 'propagate' -> host maps 0 to NaN).
template <typename V>
__device__ __forceinline__ void warp_dense_rank(const V* s, int32_t* r, int n, int lane) {
  bool has_nan = false;
  for (int k = lane; k < n; k += 32) has_nan |= (s[k] != s[k]);
  if (__any_sync(kFullMask, has_nan)) {
    for (int k = lane; k < n; k += 32) r[k] = 0;
    return;
  }
  for (int k = lane; k < n; k += 32) {
    const V v = s[k];
    int first = 1;
    for (int m = 0; m < k; ++m) first &= (s[m] != v);
    r[k] = first ? (int32_t)0x80000000 : 0;
  }
  __syncwarp();
  for (int j = lane; j < n; j += 32) {
    const V v = s[j];
    int cnt = 1;
    for (int k = 0; k < n; ++k) cnt += (int)(s[k] > v) & (int)((uint32_t)r[k] >> 31);
    r[j] = (r[j] & (int32_t)0x80000000) | cnt;
  }
  __syncwarp();
  for (int k = lane; k < n; k += 32) r[k] &= 0x7fffffff;
}

// Sums each of the N (power of two) values v[] over the 32 lanes with N-1 + log2(32/N) shuffles instead of
// 5*N: at every halving step a lane keeps one half of its values and hands the other half to its partner.
// Returns the total of value number (lane >> (5 - log2 N)); all lanes of that group hold identical bits.
template <int N>
__device__ __forceinline__ float warp_sum_transposed(float (&v)[N], int lane) {
  static_assert(N >= 1 && N <= 32 && (N & (N - 1)) == 0, "N must be a power of two");
  int o = 16;
#pragma unroll
  for (int n = N; n > 1; n >>= 1, o >>= 1) {
    const bool up = (lane & o) != 0;
#pragma unroll
    for (int j = 0; j < n / 2; ++j) {
      const float send = up ? v[j] : v[j + n / 2];
      const float keep = up ? v[j + n / 2] : v[j];
      v[j] = keep + __shfl_xor_sync(kFullMask, send, o);
    }
  }
  float r = v[0];
#pragma unroll
  for (int k = 16 / N; k > 0; k >>= 1) r += __shfl_xor_sync(kFullMask, r, k);
  return r;
}

struct ScoreRankParams {
  const char* hist_x;
  const char* hist_e;
  const char* cand;
  const float* cand_base;  // optional per-row baseline score blended into the cosine (NULL = pure cosine)
  float alpha;             // blended = alpha * cosine + (1 - alpha) * base; impressions without history: base
  int64_t hist_stride_bytes;
  int64_t cand_stride_bytes;
  const int32_t* hist_idx;
  const int64_t* hist_off;
  const int32_t* cand_idx;
  const int64_t* cand_off;
  int64_t n_imp;
  int64_t n_rows;
  int dim;
  float* user_out;
  float* scores;
  int32_t* ranks;
  int32_t* err_flag;
};

// Rows a warp will gather in its next load batches are requested into L2 ahead of time by the lanes that hold their
// indices (one bulk prefetch per row: no registers, no shared memory, no completion to wait for).  Without it a warp's
// DRAM requests stop while it computes on a batch it has received; with it the next batches are already on their way
// and are then read from L2.  Results do not depend on it.  Up to 148 SMs x 16 warps x kPrefetchBatches x 8 KB stay
// in L2 at a time (19 MB per batch of distance).  Same-box alternating A/B on one B200 (1,000 W), bench headline, bf16
// d=1024 FinalAttention: kernel 64.1 -> 59.6 ms at a distance of one batch, 60.3 at two, 60.7 at four
// (profiles/score_prefetch_ab_b200.txt).
#ifndef NRB_SCORE_PREFETCH
#define NRB_SCORE_PREFETCH 1
#endif
constexpr int kPrefetchBatches = NRB_SCORE_PREFETCH;

__device__ __forceinline__ void prefetch_row_l2(const char* row, int bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(row), "r"(bytes) : "memory");
}

template <typename T, int NV>
__device__ __forceinline__ void load_row(const char* base, int lane, uint4 (&v)[NV]) {
#pragma unroll
  for (int i = 0; i < NV; ++i) v[i] = ldg_stream_128(base + (size_t)(lane + 32 * i) * 16);
}

template <typename T, int NV, int MODE>
__global__ void __launch_bounds__(kScoreWarps * 32, 16 / kScoreWarps)
score_rank_kernel(const ScoreRankParams p) {
  constexpr int EPV = Vec16<T>::EPV;
  constexpr int EPL = NV * EPV;  // elements owned by one lane
  __shared__ float s_scores[kScoreWarps][kRankCap];
  __shared__ int32_t s_ranks[kScoreWarps][kRankCap];

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * kScoreWarps;

  for (int64_t imp = (int64_t)blockIdx.x * kScoreWarps + warp; imp < p.n_imp; imp += stride) {
    const int64_t h0 = p.hist_off[imp], h1 = p.hist_off[imp + 1];
    const int64_t c0 = p.cand_off[imp], c1 = p.cand_off[imp + 1];

    float num[EPL];
    float den[MODE == NRB_POOL_FINAL_ATTENTION ? EPL : 1];
#pragma unroll
    for (int i = 0; i < EPL; ++i) num[i] = 0.f;
    if (MODE == NRB_POOL_FINAL_ATTENTION) {
#pragma unroll
      for (int i = 0; i < EPL; ++i) den[i] = 0.f;
    }

    // ---- history: gather rows, accumulate in registers -------------------------------
    // HR rows (x MODE-0's two tables) are requested back to back and only then consumed: the
    // __syncwarp() between the loads and their first use keeps ptxas from interleaving
    // load -> use -> load (which leaves 1-2 requests in flight per lane and is latency bound).
    constexpr int kTables = MODE == NRB_POOL_FINAL_ATTENTION ? 2 : 1;
    constexpr int HR = (16 / (NV * kTables)) > 0 ? (16 / (NV * kTables)) : 1;  // ~16 requests of 16 B per lane
    for (int64_t base = h0; base < h1; base += 32) {
      const int cnt = (int)min((int64_t)32, h1 - base);
      int my = 0;
      if (lane < cnt) {
        my = p.hist_idx[base + lane];
        if ((uint32_t)my >= (uint64_t)p.n_rows) {
          atomicOr(p.err_flag, 1);
          my = 0;
        }
      }
      for (int s = 0; s < cnt; s += HR) {
        // rows of the next kPrefetchBatches batches of this chunk -> L2 (see prefetch_row_l2)
        if (lane >= s + HR && lane < min(s + HR * (kPrefetchBatches + 1), cnt) &&
            (s == 0 || lane >= s + HR * kPrefetchBatches)) {
          prefetch_row_l2(p.hist_x + (int64_t)my * p.hist_stride_bytes, NV * 512);
          if (MODE == NRB_POOL_FINAL_ATTENTION) prefetch_row_l2(p.hist_e + (int64_t)my * p.hist_stride_bytes, NV * 512);
        }
        uint4 x[HR][NV];
        uint4 e[MODE == NRB_POOL_FINAL_ATTENTION ? HR : 1][NV];
#pragma unroll
        for (int q = 0; q < HR; ++q) {
          // past the end: re-request the last valid row (an L2 hit, ignored below) so that the loads
          // stay unconditional
          const int r = __shfl_sync(kFullMask, my, min(s + q, cnt - 1));
          load_row<T, NV>(p.hist_x + (int64_t)r * p.hist_stride_bytes, lane, x[q]);
          if (MODE == NRB_POOL_FINAL_ATTENTION)
            load_row<T, NV>(p.hist_e + (int64_t)r * p.hist_stride_bytes, lane, e[q]);
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < HR; ++q) {
          if (s + q < cnt) {
#pragma unroll
            for (int i = 0; i < NV; ++i) {
              float xf[EPV];
              Vec16<T>::unpack(x[q][i], xf);
              if (MODE == NRB_POOL_FINAL_ATTENTION) {
                float ef[EPV];
                Vec16<T>::unpack(e[q][i], ef);
#pragma unroll
                for (int k = 0; k < EPV; ++k) {
                  num[i * EPV + k] = fmaf(xf[k], ef[k], num[i * EPV + k]);
                  den[i * EPV + k] += ef[k];
                }
              } else {
#pragma unroll
                for (int k = 0; k < EPV; ++k) num[i * EPV + k] += xf[k];
              }
            }
          }
        }
      }
    }

    // ---- user vector ---------------------------------------------------------------------
    float ss = 0.f;
    if (MODE == NRB_POOL_FINAL_ATTENTION) {
#pragma unroll
      for (int i = 0; i < EPL; ++i) {
        num[i] = num[i] / (den[i] + 1e-10f);  // modeling_utils.py:225
        ss = fmaf(num[i], num[i], ss);
      }
    } else {
      // warp-uniform divisors are applied as one reciprocal + multiplies (<= 1 ulp from the division; an IEEE
      // divide is ~12 instructions and there are 3 x 32 of them per impression here)
      const float inv_cnt = 1.0f / (float)(h1 - h0);  // empty history: 0 * inf = NaN like the reference's 0/0 (:168)
#pragma unroll
      for (int i = 0; i < EPL; ++i) {
        num[i] = num[i] * inv_cnt;
        ss = fmaf(num[i], num[i], ss);
      }
      const float inv_nrm = 1.0f / fmaxf(sqrtf(warp_sum(ss)), 1e-12f);  // F.normalize eps
      ss = 0.f;
#pragma unroll
      for (int i = 0; i < EPL; ++i) {
        num[i] = num[i] * inv_nrm;
        ss = fmaf(num[i], num[i], ss);
      }
    }
    if (p.user_out != nullptr) {
      float* dst = p.user_out + imp * (int64_t)p.dim;
#pragma unroll
      for (int i = 0; i < NV; ++i) {
#pragma unroll
        for (int q = 0; q < EPV / 4; ++q) {
          float4 o = make_float4(num[i * EPV + 4 * q], num[i * EPV + 4 * q + 1], num[i * EPV + 4 * q + 2],
                                 num[i * EPV + 4 * q + 3]);
          *reinterpret_cast<float4*>(dst + (size_t)(lane + 32 * i) * EPV + 4 * q) = o;
        }
      }
    }
    // F.cosine_similarity: x / max(|x|, 1e-8) first (data_model_helper.py:224-227)
    const float inv_unorm = 1.0f / fmaxf(sqrtf(warp_sum(ss)), 1e-8f);
#pragma unroll
    for (int i = 0; i < EPL; ++i) num[i] = num[i] * inv_unorm;

    // ---- candidates: dot + norm per row, warp-shuffle reduction -------------------------
    const int n_cand = (int)(c1 - c0);
    for (int64_t base = c0; base < c1; base += 32) {
      const int cnt = (int)min((int64_t)32, c1 - base);
      int my = 0;
      if (lane < cnt) {
        my = p.cand_idx[base + lane];
        if ((uint32_t)my >= (uint64_t)p.n_rows) {
          atomicOr(p.err_flag, 1);
          my = 0;
        }
      }
      // lane l keeps the (dot, |c|^2) sums of candidate base + l; the sqrt / divide / blend then run once per lane
      // after the block instead of once per candidate on all 32 lanes
      float my_dot = 0.f, my_sq = 0.f;
      constexpr int CR = (16 / NV) > 0 ? (16 / NV) : 1;  // candidate rows in flight per iteration
      for (int s = 0; s < cnt; s += CR) {
        if (lane >= s + CR && lane < min(s + CR * (kPrefetchBatches + 1), cnt) &&
            (s == 0 || lane >= s + CR * kPrefetchBatches))
          prefetch_row_l2(p.cand + (int64_t)my * p.cand_stride_bytes, NV * 512);
        uint4 a[CR][NV];
#pragma unroll
        for (int q = 0; q < CR; ++q) {
          const int r = __shfl_sync(kFullMask, my, min(s + q, cnt - 1));
          load_row<T, NV>(p.cand + (int64_t)r * p.cand_stride_bytes, lane, a[q]);
        }
        __syncwarp();  // all loads issued before the first use (see the history loop)
        float dot[CR], sq[CR];
#pragma unroll
        for (int q = 0; q < CR; ++q) {
          dot[q] = 0.f;
          sq[q] = 0.f;
#pragma unroll
          for (int i = 0; i < NV; ++i) {
            float f[EPV];
            Vec16<T>::unpack(a[q][i], f);
#pragma unroll
            for (int k = 0; k < EPV; ++k) {
              dot[q] = fmaf(f[k], num[i * EPV + k], dot[q]);
              sq[q] = fmaf(f[k], f[k], sq[q]);
            }
          }
        }
        if constexpr ((CR & (CR - 1)) == 0) {
          // candidate q's totals land in lanes [q*32/CR, (q+1)*32/CR); lane s+q fetches them from there
          // (14 shuffles per 4 candidates instead of 40; the compute phase between two load batches is what the
          // kernel's bandwidth is sensitive to: +0.7 % FinalAttention pooling, +2..5 % mean pooling, same box)
          const float d = warp_sum_transposed<CR>(dot, lane), n2 = warp_sum_transposed<CR>(sq, lane);
          const int src = (lane & (CR - 1)) * (32 / CR);
          const float gd = __shfl_sync(kFullMask, d, src), gn = __shfl_sync(kFullMask, n2, src);
          if (lane >= s && lane < s + CR) {
            my_dot = gd;
            my_sq = gn;
          }
        } else {
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
            for (int q = 0; q < CR; ++q) {
              dot[q] += __shfl_xor_sync(kFullMask, dot[q], o);
              sq[q] += __shfl_xor_sync(kFullMask, sq[q], o);
            }
          }
#pragma unroll
          for (int q = 0; q < CR; ++q) {
            if (lane == s + q) {
              my_dot = dot[q];
              my_sq = sq[q];
            }
          }
        }
      }
      float my_score = my_dot / fmaxf(sqrtf(my_sq), 1e-8f);
      if (p.cand_base != nullptr && lane < cnt) {
        // WeightedSumModel (modeling_utils.py:158-165) fused behind the cosine; rows without history keep
        // the classification baseline alone (data_model_helper.py:284-299)
        const float cb = p.cand_base[my];
        my_score = (h1 > h0) ? my_score * p.alpha + cb * (1.0f - p.alpha) : cb;
      }
      if (lane < cnt) {
        p.scores[base + lane] = my_score;
        const int pos = (int)(base - c0) + lane;
        if (pos < kRankCap) s_scores[warp][pos] = my_score;
      }
    }

    // ---- dense rank -----------------------------------------------------------------------
    if (p.ranks != nullptr) {
      __syncwarp();
      if (n_cand <= kRankCap) {
        warp_dense_rank(s_scores[warp], s_ranks[warp], n_cand, lane);
        __syncwarp();
        for (int k = lane; k < n_cand; k += 32) p.ranks[c0 + k] = s_ranks[warp][k];
      } else {
        __threadfence_block();
        warp_dense_rank(p.scores + c0, p.ranks + c0, n_cand, lane);
      }
    }
    __syncwarp();
  }
}

template <typename T, int MODE>
static int launch_score_rank_nv(int nv, const ScoreRankParams& p, int grid, cudaStream_t st) {
  const dim3 block(kScoreWarps * 32);
  switch (nv) {
#define NRB_CASE(N)                                                  \
  case N:                                                            \
    score_rank_kernel<T, N, MODE><<<grid, block, 0, st>>>(p); note_launch();        \
    break;
    NRB_CASE(1)
    NRB_CASE(2)
    NRB_CASE(3)
    NRB_CASE(4)
    NRB_CASE(5)
    NRB_CASE(6)
    NRB_CASE(7)
    NRB_CASE(8)
#undef NRB_CASE
    default:
      set_error("nrb_score_rank: dim*elemsize must be a multiple of 512 bytes and <= 4096 (got %d vectors/lane)", nv);
      return NRB_E_INVALID;
  }
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

// ---- standalone dense rank (rank_group_preds drop-in) ---------------------------------------
// V = float (the hot path's score dtype) or double (rank_group_preds on float64 scores: scipy ranks the
// array in its own dtype, so values that differ only below fp32 resolution must not become ties).
template <typename V, int WARPS>
__global__ void __launch_bounds__(WARPS * 32)
dense_rank_kernel(const V* scores, const int64_t* offsets, int64_t n_groups, int32_t* ranks) {
  __shared__ V s_scores[WARPS][kRankCap];
  __shared__ int32_t s_ranks[WARPS][kRankCap];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * WARPS;
  for (int64_t g = (int64_t)blockIdx.x * WARPS + warp; g < n_groups; g += stride) {
    const int64_t c0 = offsets[g], c1 = offsets[g + 1];
    const int64_t n64 = c1 - c0;
    if (n64 <= kRankCap) {
      const int n = (int)n64;
      for (int k = lane; k < n; k += 32) s_scores[warp][k] = scores[c0 + k];
      __syncwarp();
      warp_dense_rank(s_scores[warp], s_ranks[warp], n, lane);
      __syncwarp();
      for (int k = lane; k < n; k += 32) ranks[c0 + k] = s_ranks[warp][k];
    } else {
      warp_dense_rank(scores + c0, ranks + c0, (int)n64, lane);
    }
    __syncwarp();
  }
}

// ---- warp-level top-k ordering ---------------------------------------------------------------------
// out[g, p] = position (within the group) of the candidate at place p of the descending order, p < k;
// equal scores keep their original order (== np.argsort(-scores, kind="stable")[:k]); -1 pads groups
// shorter than k.  NaN scores sort last.  One warp per group; place(j) = #{s_i > s_j} + #{i < j : s_i == s_j}.
__global__ void __launch_bounds__(kWarpsPerCta * 32)
topk_order_kernel(const float* scores, const int64_t* offsets, int64_t n_groups, int k, int32_t* out) {
  __shared__ float s_scores[kWarpsPerCta][kRankCap];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t stride = (int64_t)gridDim.x * kWarpsPerCta;
  for (int64_t g = (int64_t)blockIdx.x * kWarpsPerCta + warp; g < n_groups; g += stride) {
    const int64_t c0 = offsets[g];
    const int n = (int)(offsets[g + 1] - c0);
    const bool in_smem = n <= kRankCap;
    if (in_smem) {
      for (int i = lane; i < n; i += 32) s_scores[warp][i] = scores[c0 + i];
      __syncwarp();
    }
    const float* s = in_smem ? s_scores[warp] : scores + c0;
    for (int p = lane; p < k; p += 32) out[g * k + p] = -1;
    __syncwarp();
    for (int j = lane; j < n; j += 32) {
      const float v = s[j];
      const bool vnan = v != v;
      int place = 0;
      for (int i = 0; i < n; ++i) {
        const float u = s[i];
        const bool unan = u != u;
        // u sorts before v: larger, or equal and earlier; NaNs after every number, among themselves by position
        const bool before = vnan ? (!unan || i < j) : (!unan && (u > v || (u == v && i < j)));
        place += before;
      }
      if (place < k) out[g * k + place] = j;
    }
    __syncwarp();
  }
}

// ---- padded gather (final_attention_eval_collate_fn drop-in) -----------------------------------
// one warp per (group, slot): copies one table row (or zeros) with 128-bit accesses.
__global__ void __launch_bounds__(256)
gather_collate_kernel(const char* table, int64_t n_rows, int row_bytes, int64_t table_stride_bytes,
                      const int32_t* idx, const int64_t* offsets, int64_t n_groups, int max_len,
                      char* emb_out, int32_t* mask_out, int32_t* err_flag) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t total = n_groups * (int64_t)max_len;
  const int nvec = row_bytes / 16;
  for (int64_t slot = warp_id; slot < total; slot += n_warps) {
    const int64_t g = slot / max_len;
    const int s = (int)(slot - g * max_len);
    const int64_t o0 = offsets[g];
    const int len = (int)(offsets[g + 1] - o0);
    const bool valid = s < len;
    uint4* dst = reinterpret_cast<uint4*>(emb_out + slot * (int64_t)row_bytes);
    if (valid) {
      int r = idx[o0 + s];
      if ((uint32_t)r >= (uint64_t)n_rows) {
        if (lane == 0) atomicOr(err_flag, 1);
        r = 0;
      }
      const char* src = table + (int64_t)r * table_stride_bytes;
      for (int v = lane; v < nvec; v += 32) dst[v] = ldg_stream_128(src + (size_t)v * 16);
    } else {
      for (int v = lane; v < nvec; v += 32) dst[v] = make_uint4(0, 0, 0, 0);
    }
    if (lane == 0) mask_out[slot] = valid ? 1 : 0;
  }
}

// int32 dense ranks -> int16 (halves the device->host bytes of the ranks; a rank never exceeds the candidate count
// of its impression).  Values that do not fit set bit 1 of *err_flag and saturate.
__global__ void __launch_bounds__(256)
narrow_ranks_kernel(const int32_t* src, int16_t* dst, int64_t n, int32_t* err_flag) {
  const int64_t n8 = n / 8;
  bool bad = false;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n8; i += (int64_t)gridDim.x * blockDim.x) {
    const int4 a = *reinterpret_cast<const int4*>(src + i * 8), b = *reinterpret_cast<const int4*>(src + i * 8 + 4);
    const int v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      bad |= v[2 * k] > 32767 || v[2 * k + 1] > 32767;
      o[k] = (uint32_t)min(v[2 * k], 32767) | ((uint32_t)min(v[2 * k + 1], 32767) << 16);
    }
    *reinterpret_cast<uint4*>(dst + i * 8) = make_uint4(o[0], o[1], o[2], o[3]);
  }
  for (int64_t i = n8 * 8 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    bad |= src[i] > 32767;
    dst[i] = (int16_t)min(src[i], 32767);
  }
  if (bad) atomicOr(err_flag, 2);
}

}  // namespace nrb

using namespace nrb;

extern "C" int nrb_narrow_ranks(const int32_t* ranks, int16_t* ranks16, int64_t n, int32_t* err_flag,
                                nrb_stream_t stream) {
  NRB_REQUIRE(n >= 0, "nrb_narrow_ranks: n < 0");
  if (n == 0) return NRB_OK;
  NRB_REQUIRE(ranks && ranks16 && err_flag, "nrb_narrow_ranks: null pointer");
  NRB_REQUIRE((reinterpret_cast<uintptr_t>(ranks) & 15) == 0 && (reinterpret_cast<uintptr_t>(ranks16) & 15) == 0,
              "nrb_narrow_ranks: buffers must be 16-byte aligned");
  const int64_t want = (n / 8 + 255) / 256 + 1;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count_cached() * 16);
  narrow_ranks_kernel<<<grid, 256, 0, as_stream(stream)>>>(ranks, ranks16, n, err_flag);
  note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

template <typename V, int WARPS>
static int launch_dense_rank(const V* scores, const int64_t* offsets, int64_t n_groups, int32_t* ranks,
                             nrb_stream_t stream, const char* what) {
  NRB_REQUIRE(n_groups >= 0, "%s: n_groups < 0", what);
  if (n_groups == 0) return NRB_OK;
  NRB_REQUIRE(scores && offsets && ranks, "%s: null pointer", what);
  const int64_t want = (n_groups + WARPS - 1) / WARPS;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count_cached() * 32);
  dense_rank_kernel<V, WARPS><<<grid, WARPS * 32, 0, as_stream(stream)>>>(scores, offsets, n_groups, ranks);
  note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

extern "C" int nrb_dense_rank(const float* scores, const int64_t* offsets, int64_t n_groups, int32_t* ranks,
                              nrb_stream_t stream) {
  return launch_dense_rank<float, kWarpsPerCta>(scores, offsets, n_groups, ranks, stream, "nrb_dense_rank");
}

extern "C" int nrb_dense_rank_f64(const double* scores, const int64_t* offsets, int64_t n_groups, int32_t* ranks,
                                  nrb_stream_t stream) {
  return launch_dense_rank<double, 4>(scores, offsets, n_groups, ranks, stream, "nrb_dense_rank_f64");
}

extern "C" int nrb_topk_order(const float* scores, const int64_t* offsets, int64_t n_groups, int k, int32_t* out_idx,
                              nrb_stream_t stream) {
  NRB_REQUIRE(n_groups >= 0 && k >= 1, "nrb_topk_order: bad sizes");
  if (n_groups == 0) return NRB_OK;
  NRB_REQUIRE(scores && offsets && out_idx, "nrb_topk_order: null pointer");
  const int64_t want = (n_groups + kWarpsPerCta - 1) / kWarpsPerCta;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count_cached() * 32);
  topk_order_kernel<<<grid, kWarpsPerCta * 32, 0, as_stream(stream)>>>(scores, offsets, n_groups, k, out_idx);
  note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

extern "C" int nrb_gather_collate(const void* table, int dtype, int64_t n_rows, int dim, int64_t table_stride,
                                  const int32_t* idx, const int64_t* offsets, int64_t n_groups, int max_len,
                                  void* emb_out, int32_t* mask_out, int32_t* err_flag, nrb_stream_t stream) {
  NRB_REQUIRE(dtype == NRB_F32 || dtype == NRB_BF16, "nrb_gather_collate: bad dtype %d", dtype);
  const int es = dtype == NRB_F32 ? 4 : 2;
  NRB_REQUIRE(dim > 0 && (dim * es) % 16 == 0, "nrb_gather_collate: dim*elemsize must be a multiple of 16 bytes");
  NRB_REQUIRE((table_stride * es) % 16 == 0, "nrb_gather_collate: table stride must keep rows 16-byte aligned");
  NRB_REQUIRE(n_groups >= 0 && max_len >= 0, "nrb_gather_collate: negative size");
  if (n_groups == 0 || max_len == 0) return NRB_OK;
  NRB_REQUIRE(table && idx && offsets && emb_out && mask_out && err_flag, "nrb_gather_collate: null pointer");
  const int64_t total = n_groups * (int64_t)max_len;
  const int64_t want = (total + 7) / 8;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count_cached() * 32);
  gather_collate_kernel<<<grid, 256, 0, as_stream(stream)>>>(
      (const char*)table, n_rows, dim * es, table_stride * es, idx, offsets, n_groups, max_len, (char*)emb_out,
      mask_out, err_flag); note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

extern "C" int nrb_score_rank(int pool_mode, int dtype, int dim, int64_t n_rows, const void* hist_x,
                              const void* hist_e, int64_t hist_stride, const void* cand, int64_t cand_stride,
                              const float* cand_base, float blend_alpha, const int32_t* hist_idx, const int64_t* hist_off, const int32_t* cand_idx,
                              const int64_t* cand_off, int64_t n_imp, float* user_out, float* scores,
                              int32_t* ranks, int32_t* err_flag, nrb_stream_t stream) {
  NRB_REQUIRE(dtype == NRB_F32 || dtype == NRB_BF16, "nrb_score_rank: bad dtype %d", dtype);
  NRB_REQUIRE(pool_mode == NRB_POOL_FINAL_ATTENTION || pool_mode == NRB_POOL_MEAN_L2,
              "nrb_score_rank: bad pool_mode %d", pool_mode);
  const int es = dtype == NRB_F32 ? 4 : 2;
  NRB_REQUIRE(dim > 0 && (dim * es) % 512 == 0 && dim * es <= 4096,
              "nrb_score_rank: dim*elemsize must be a multiple of 512 bytes and <= 4096 (dim=%d)", dim);
  NRB_REQUIRE((hist_stride * es) % 16 == 0 && (cand_stride * es) % 16 == 0,
              "nrb_score_rank: row strides must keep rows 16-byte aligned");
  NRB_REQUIRE(n_imp >= 0 && n_rows > 0, "nrb_score_rank: bad sizes");
  if (n_imp == 0) return NRB_OK;
  NRB_REQUIRE(hist_x && cand && hist_idx && hist_off && cand_idx && cand_off && scores && err_flag,
              "nrb_score_rank: null pointer");
  NRB_REQUIRE(pool_mode != NRB_POOL_FINAL_ATTENTION || hist_e, "nrb_score_rank: hist_e required");
  ScoreRankParams p;
  p.hist_x = (const char*)hist_x;
  p.hist_e = (const char*)hist_e;
  p.cand = (const char*)cand;
  p.cand_base = cand_base;
  p.alpha = blend_alpha;
  p.hist_stride_bytes = hist_stride * es;
  p.cand_stride_bytes = cand_stride * es;
  p.hist_idx = hist_idx;
  p.hist_off = hist_off;
  p.cand_idx = cand_idx;
  p.cand_off = cand_off;
  p.n_imp = n_imp;
  p.n_rows = n_rows;
  p.dim = dim;
  p.user_out = user_out;
  p.scores = scores;
  p.ranks = ranks;
  p.err_flag = err_flag;
  const int nv = dim * es / 512;
  const int64_t want = (n_imp + kScoreWarps - 1) / kScoreWarps;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count_cached() * (16 / kScoreWarps) * NRB_SCORE_GRID_MULT * 8);
  cudaStream_t st = as_stream(stream);
  if (dtype == NRB_F32) {
    return pool_mode == NRB_POOL_FINAL_ATTENTION
               ? launch_score_rank_nv<float, NRB_POOL_FINAL_ATTENTION>(nv, p, grid, st)
               : launch_score_rank_nv<float, NRB_POOL_MEAN_L2>(nv, p, grid, st);
  }
  return pool_mode == NRB_POOL_FINAL_ATTENTION
             ? launch_score_rank_nv<__nv_bfloat16, NRB_POOL_FINAL_ATTENTION>(nv, p, grid, st)
             : launch_score_rank_nv<__nv_bfloat16, NRB_POOL_MEAN_L2>(nv, p, grid, st);
}
