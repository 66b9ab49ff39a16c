// Retrieval: the k best rows of the resident table, or of a pool of its rows, for each user (nrb_recommend,
// nrb_recommend_pool_blend).
//
//   cos(u, r)   = (u / max(|u|, 1e-8)) . c_r / max(|c_r|, 1e-8)      -- the cosine nrb_score_rank computes
//   score(u, r) = cos(u, r); with a baseline: cos * alpha + base[r] * (1 - alpha), or base[r] alone for a user with
//                 an empty history (a select: a NaN user vector cannot reach the list)
//
// One tcgen05 GEMM of the normalised users against the table (or the pool's rows of it) with a top-k epilogue
// (gemm_tc.cu, NRB_EPI_TOPK, or NRB_EPI_TOPK_BLEND with a baseline): the scores never leave TMEM.  Around it:
//   pool_gather_kernel   the pool's rows of the GEMM operand -> workspace [n_pool, K'], ids validated (pool only)
//   user_operand_kernel  u / max(|u|, 1e-8) -> bf16, or -> [hi|hi|lo] split-bf16 (fp32 tables, K' = 3d); the
//                        empty-history flags of the users (baseline only)
//   row_scale_kernel     1 / max(|c_r|, 1e-8) of the stored table and base[r], in column order (pool order with a
//                        pool), NaN past the last column: never scores
//   sort_excl_kernel     each user's excluded rows as columns, sorted ascending (any length), range-checked
//   merge_kernel         one warp per user merges its partial lists into the final [U, k], columns -> table rows
// Order: score descending, equal scores by ascending row id; NaN never returned; (-1, NaN) once rows run out.
#include "dense.cuh"

#include <algorithm>

namespace nrb {

constexpr int kRecMaxK = 32;
constexpr int kSortChunk = 2048;  // excluded ids sorted per shared-memory pass

// One warp per pool entry: copies table_op row pool[i] (16-byte vectors) and checks that the ids are strictly
// ascending and in [0, n_rows); a bad id sets bit 0 of *err_flag and its row is zero-filled.
__global__ void __launch_bounds__(256)
pool_gather_kernel(const __nv_bfloat16* op, int64_t ld, int kdim, const int32_t* pool, int64_t n_pool, int64_t n_rows,
                   __nv_bfloat16* out, int32_t* err_flag) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int nv = kdim / 8;
  for (int64_t i = warp_id; i < n_pool; i += n_warps) {
    const int32_t id = pool[i];
    const bool ok = id >= 0 && (int64_t)id < n_rows && (i == 0 || pool[i - 1] < id);
    if (!ok && lane == 0) atomicOr(err_flag, 1);
    const uint4* src = reinterpret_cast<const uint4*>(op + (int64_t)(ok ? id : 0) * ld);
    uint4* dst = reinterpret_cast<uint4*>(out + i * kdim);
    for (int j = lane; j < nv; j += 32) dst[j] = ok ? src[j] : make_uint4(0u, 0u, 0u, 0u);
  }
}

__global__ void __launch_bounds__(256)
user_operand_kernel(const float* users, int64_t ldu, int64_t n_users, int dim, int split, __nv_bfloat16* out,
                    int64_t ldo, const int64_t* hist_off, uint8_t* cold) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = warp_id; r < n_users; r += n_warps) {
    const float* u = users + r * ldu;
    float ss = 0.f;
    for (int i = lane; i < dim; i += 32) ss = fmaf(u[i], u[i], ss);
    const float inv = 1.0f / fmaxf(sqrtf(warp_sum(ss)), 1e-8f);  // NaN users stay NaN
    __nv_bfloat16* o = out + r * ldo;
    for (int i = lane; i < dim; i += 32) {
      const float v = u[i] * inv;
      const __nv_bfloat16 hi = __float2bfloat16_rn(v);
      o[i] = hi;
      if (split) {  // nrb_split_rows role 0: [hi | hi | lo]
        o[dim + i] = hi;
        o[2 * dim + i] = __float2bfloat16_rn(v - __bfloat162float(hi));
      }
    }
    if (cold != nullptr && lane == 0) cold[r] = hist_off != nullptr && hist_off[r + 1] <= hist_off[r];
  }
}

// Column c of the GEMM is table row pool[c] (pool != NULL) or row c; an id outside [0, n_rows) (pool_gather_kernel
// flags it) gets NaN and never scores.  base_out (when base != NULL): base of the column's row, NaN past the last one.
__global__ void __launch_bounds__(256)
row_scale_kernel(const void* table, int dtype, int64_t ld, int64_t n_rows, int dim, const int32_t* pool,
                 int64_t n_cols, int64_t n_pad, float* scale, const float* base, float* base_out) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t c = warp_id; c < n_pad; c += n_warps) {
    float ss = 0.f;
    const int64_t r = c >= n_cols ? -1 : pool != nullptr ? (int64_t)pool[c] : c;
    const bool ok = r >= 0 && r < n_rows;
    if (ok) {
      if (dtype == NRB_F32) {
        const float* c = reinterpret_cast<const float*>(table) + r * ld;
        for (int i = lane; i < dim; i += 32) ss = fmaf(c[i], c[i], ss);
      } else {
        const __nv_bfloat16* c = reinterpret_cast<const __nv_bfloat16*>(table) + r * ld;
        for (int i = lane; i < dim; i += 32) {
          const float x = __bfloat162float(c[i]);
          ss = fmaf(x, x, ss);
        }
      }
    }
    ss = warp_sum(ss);
    if (lane == 0) {
      scale[c] = ok ? 1.0f / fmaxf(sqrtf(ss), 1e-8f) : __int_as_float(0x7fc00000);
      if (base != nullptr) base_out[c] = ok ? base[r] : __int_as_float(0x7fc00000);
    }
  }
}

// ascending bitonic sort of n_pow2 ints in shared memory (the whole block takes part)
__device__ void block_bitonic_sort(int32_t* s, int n_pow2) {
  for (int size = 2; size <= n_pow2; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      __syncthreads();
      for (int i = threadIdx.x; i < n_pow2 / 2; i += blockDim.x) {
        const int lo = 2 * i - (i & (stride - 1));
        const int hi = lo + stride;
        const bool up = (lo & size) == 0;
        const int32_t a = s[lo], b = s[hi];
        if ((a > b) == up) {
          s[lo] = b;
          s[hi] = a;
        }
      }
    }
  }
  __syncthreads();
}

// Column of table row `id` in the ascending pool: its position, or n_pool when the row is not in the pool (the
// epilogue's cursor never reaches a column >= n_pool, so such an id excludes nothing).
__device__ __forceinline__ int32_t pool_column(const int32_t* pool, int64_t n_pool, int32_t id) {
  int64_t lo = 0, hi = n_pool;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if (pool[mid] < id) lo = mid + 1; else hi = mid;
  }
  return (int32_t)(lo < n_pool && pool[lo] == id ? lo : n_pool);
}

// One block per user.  Histories up to kSortChunk ids are sorted in shared memory; longer ones are sorted in chunks
// into `tmp`, then every id goes straight to its final place: its position in its own chunk plus, in every other
// chunk, the number of ids that precede it (ids of earlier chunks first among equals).  With a pool the ids are
// range-checked as table rows, then sorted as GEMM columns (pool_column).
__global__ void __launch_bounds__(256)
sort_excl_kernel(const int32_t* idx, const int64_t* off, int64_t n_rows, const int32_t* pool, int64_t n_pool,
                 int32_t* tmp, int32_t* out, int32_t* err_flag) {
  __shared__ int32_t s[kSortChunk];
  const int64_t g = blockIdx.x;
  const int64_t o0 = off[g], n = off[g + 1] - o0;
  if (n <= 0) return;
  bool bad = false;
  for (int64_t c0 = 0; c0 < n; c0 += kSortChunk) {
    const int m = (int)(n - c0 < kSortChunk ? n - c0 : kSortChunk);
    int p2 = 32;
    while (p2 < m) p2 <<= 1;
    __syncthreads();
    for (int i = threadIdx.x; i < p2; i += blockDim.x) {
      int32_t v = 0x7fffffff;
      if (i < m) {
        v = idx[o0 + c0 + i];
        bad |= v < 0 || (int64_t)v >= n_rows;
        if (pool != nullptr) v = pool_column(pool, n_pool, v);
      }
      s[i] = v;
    }
    block_bitonic_sort(s, p2);
    int32_t* dst = (n <= kSortChunk ? out : tmp) + o0 + c0;
    for (int i = threadIdx.x; i < m; i += blockDim.x) dst[i] = s[i];
  }
  if (bad) atomicOr(err_flag, 1);
  if (n <= kSortChunk) return;
  __threadfence_block();
  __syncthreads();
  const int64_t n_chunks = (n + kSortChunk - 1) / kSortChunk;
  for (int64_t i = threadIdx.x; i < n; i += blockDim.x) {
    const int64_t own = i / kSortChunk;
    const int32_t x = tmp[o0 + i];
    int64_t rank = i - own * kSortChunk;
    for (int64_t c = 0; c < n_chunks; ++c) {
      if (c == own) continue;
      const int32_t* a = tmp + o0 + c * kSortChunk;
      int64_t lo = 0, hi = n - c * kSortChunk < kSortChunk ? n - c * kSortChunk : kSortChunk;
      while (lo < hi) {  // c < own: ids <= x precede it; c > own: ids < x
        const int64_t mid = (lo + hi) >> 1;
        if (c < own ? a[mid] <= x : a[mid] < x) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    out[o0 + rank] = x;
  }
}

// total order key: larger = better (score descending, then row ascending); 0 = empty entry
__device__ __forceinline__ unsigned long long topk_key(uint2 e) {
  if ((int32_t)e.y < 0) return 0ull;
  const uint32_t b = __float_as_uint(__uint_as_float(e.x) + 0.f);
  const uint32_t ord = (b & 0x80000000u) ? ~b : (b | 0x80000000u);
  return ((unsigned long long)ord << 32) | (uint32_t)(~e.y);
}

// One warp per user: k rounds of "best head among the user's sorted partial lists".  Lane l owns lists l, l+32, ...
// (their heads in shared memory) and keeps the best of them; the winning lane advances its head and rescans.
// Entries hold GEMM columns; with a pool, column c is table row pool[c] (ascending, so the column order is the row order).
__global__ void __launch_bounds__(256)
merge_kernel(const uint2* parts, TopkPlan plan, int64_t n_users, int k, const int32_t* pool, int32_t* out_rows,
             float* out_scores) {
  extern __shared__ int32_t heads_all[];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int64_t u = (int64_t)blockIdx.x * (blockDim.x >> 5) + w;
  if (u >= n_users) return;
  const int64_t S = plan.slots;
  int32_t* heads = heads_all + (int64_t)w * 2 * S;
  const int64_t m_u = u / (128 * plan.cg);
  const int64_t c_first = plan.first_owner(m_u);
  const int n_used = (int)(plan.last_owner(m_u) - c_first + 1);
  const int n_lists = 2 * n_used;
  auto list_base = [&](int i) {  // list i = (half i / n_used, slot i % n_used)
    return parts + ((u * 2 + i / n_used) * S + (i % n_used)) * k;
  };
  for (int i = lane; i < n_lists; i += 32) heads[i] = 0;
  __syncwarp();
  auto rescan = [&](unsigned long long& best, int& best_i) {
    best = 0ull;
    best_i = -1;
    for (int i = lane; i < n_lists; i += 32) {
      const int h = heads[i];
      if (h >= k) continue;
      const unsigned long long key = topk_key(list_base(i)[h]);
      if (key > best) {
        best = key;
        best_i = i;
      }
    }
  };
  unsigned long long best;
  int best_i;
  rescan(best, best_i);
  for (int j = 0; j < k; ++j) {
    unsigned long long m = best;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(kFullMask, m, o));
    if (lane == 0) {
      const int32_t col = (int32_t)(~(uint32_t)m);
      out_rows[u * k + j] = m == 0ull ? -1 : pool != nullptr ? pool[col] : col;
      const uint32_t ord = (uint32_t)(m >> 32);
      const uint32_t b = (ord & 0x80000000u) ? (ord & 0x7fffffffu) : ~ord;
      out_scores[u * k + j] = m == 0ull ? __int_as_float(0x7fc00000) : __uint_as_float(b);
    }
    if (m == 0ull) continue;  // lists exhausted: the rest is padding
    if (best == m) {          // row ids are unique across lists: exactly one lane wins
      heads[best_i] += 1;
      rescan(best, best_i);
    }
    __syncwarp();
  }
}

struct RecLayout {
  void* user_op;
  void* pool_op;  // the pool's rows of table_op (pool only)
  float* scale;
  float* base;    // base in column order (baseline only)
  uint8_t* cold;  // per user: empty history (baseline only)
  int32_t* excl_sorted;
  int32_t* excl_tmp;
  uint2* parts;
  size_t bytes;
};

// n_pool < 0: the whole table.  The plan is the GEMM's over max(columns, 1): an empty pool launches no GEMM.
static RecLayout rec_layout(void* base, int precision, int dim, int64_t n_users, int64_t n_excl, int k, int64_t n_pool,
                            const TopkPlan& plan) {
  Workspace ws(base, (size_t)-1);
  RecLayout L;
  const int kdim = precision == NRB_BF16 ? dim : 3 * dim;
  L.user_op = ws.take((size_t)n_users * kdim * 2);
  L.pool_op = n_pool > 0 ? ws.take((size_t)n_pool * kdim * 2) : nullptr;
  L.scale = (float*)ws.take((size_t)plan.n_per_row * 256 * 4);
  L.base = (float*)ws.take((size_t)plan.n_per_row * 256 * 4);
  L.cold = (uint8_t*)ws.take((size_t)n_users);
  L.excl_sorted = (int32_t*)ws.take((size_t)std::max<int64_t>(n_excl, 1) * 4);
  L.excl_tmp = (int32_t*)ws.take((size_t)std::max<int64_t>(n_excl, 1) * 4);
  L.parts = (uint2*)ws.take((size_t)plan.m_blocks * 128 * plan.cg * 2 * plan.slots * k * 8);
  L.bytes = ws.used + 256;
  return L;
}

static int check_recommend_args(int precision, int dim, int64_t n_rows, int64_t n_users, int64_t n_excl, int k,
                                int64_t n_pool) {
  NRB_REQUIRE(precision == NRB_BF16 || precision == NRB_F32, "nrb_recommend: precision must be NRB_BF16 or NRB_F32");
  NRB_REQUIRE(k >= 1 && k <= kRecMaxK,
              "nrb_recommend: k must be in [1, %d] (got %d): each epilogue thread keeps its list in %d shared-memory "
              "entries",
              kRecMaxK, k, kRecMaxK);
  NRB_REQUIRE(dim > 0 && dim % 64 == 0, "nrb_recommend: dim must be a positive multiple of 64 (got %d)", dim);
  NRB_REQUIRE(n_rows >= 1 && n_rows <= 0x7fffffff - 256, "nrb_recommend: n_rows must be in [1, 2^31 - 257]");
  NRB_REQUIRE(n_users >= 1, "nrb_recommend: n_users must be >= 1");
  NRB_REQUIRE(n_excl >= 0, "nrb_recommend: n_excl must be >= 0");
  NRB_REQUIRE(n_pool <= n_rows, "nrb_recommend: a pool of strictly ascending row ids has at most n_rows entries");
  return NRB_OK;
}

static TopkPlan rec_plan(int64_t n_users, int64_t n_rows, int64_t n_pool) {
  return topk_plan(n_users, n_pool < 0 ? n_rows : std::max<int64_t>(n_pool, 1));
}

}  // namespace nrb

using namespace nrb;

extern "C" size_t nrb_recommend_pool_blend_workspace_bytes(int precision, int dim, int64_t n_rows, int64_t n_users,
                                                           int64_t n_excl, int k, int64_t n_pool) {
  if (check_recommend_args(precision, dim, n_rows, n_users, n_excl, k, n_pool) != NRB_OK) return 0;
  return rec_layout(nullptr, precision, dim, n_users, n_excl, k, n_pool, rec_plan(n_users, n_rows, n_pool)).bytes;
}

extern "C" size_t nrb_recommend_workspace_bytes(int precision, int dim, int64_t n_rows, int64_t n_users,
                                                int64_t n_excl, int k) {
  return nrb_recommend_pool_blend_workspace_bytes(precision, dim, n_rows, n_users, n_excl, k, -1);
}

extern "C" int nrb_recommend_pool_blend(int precision, int dim, int64_t n_rows, const void* table,
                                        int64_t table_stride, const void* table_op, int64_t op_stride,
                                        const float* users, int64_t users_stride, int64_t n_users,
                                        const int32_t* excl_idx, const int64_t* excl_off, int64_t n_excl, int k,
                                        const int32_t* pool, int64_t n_pool, const float* cand_base,
                                        float blend_alpha, const int64_t* hist_off, int32_t* out_rows,
                                        float* out_scores, int32_t* err_flag, void* workspace,
                                        size_t workspace_bytes, nrb_stream_t stream) {
  int rc = check_recommend_args(precision, dim, n_rows, n_users, n_excl, k, n_pool);
  if (rc != NRB_OK) return rc;
  NRB_REQUIRE(table && table_op && users && out_rows && out_scores && err_flag && workspace,
              "nrb_recommend: null pointer");
  NRB_REQUIRE((excl_idx == nullptr) == (excl_off == nullptr), "nrb_recommend: excl_idx and excl_off go together");
  NRB_REQUIRE(n_pool <= 0 || pool != nullptr, "nrb_recommend: a pool of n_pool > 0 ids needs `pool`");
  NRB_REQUIRE(table_stride >= dim && users_stride >= dim && op_stride >= (precision == NRB_BF16 ? dim : 3 * dim),
              "nrb_recommend: row strides must cover the row");
  NRB_REQUIRE(n_pool < 0 || (op_stride % 8 == 0 && (reinterpret_cast<uintptr_t>(table_op) & 15) == 0),
              "nrb_recommend: with a pool, table_op must be 16-byte aligned with a 16-byte multiple row pitch");
  const bool has_pool = n_pool >= 0;
  const int64_t n_cols = has_pool ? n_pool : n_rows;
  const TopkPlan plan = rec_plan(n_users, n_rows, n_pool);
  const RecLayout L = rec_layout(workspace, precision, dim, n_users, n_excl, k, n_pool, plan);
  if (workspace_bytes < L.bytes) {
    set_error("nrb_recommend: workspace too small (%zu < %zu bytes)", workspace_bytes, L.bytes);
    return NRB_E_WORKSPACE;
  }
  cudaStream_t st = as_stream(stream);
  const int sms = sm_count_cached();
  const int kdim = precision == NRB_BF16 ? dim : 3 * dim;
  auto warps_grid = [&](int64_t n) { return (int)std::max<int64_t>(1, std::min<int64_t>((n + 7) / 8, (int64_t)sms * 16)); };
  auto sort_excl = [&]() -> int {
    sort_excl_kernel<<<(unsigned)n_users, 256, 0, st>>>(excl_idx, excl_off, n_rows, has_pool ? pool : nullptr,
                                                        n_pool, L.excl_tmp, L.excl_sorted, err_flag);
    note_launch();
    NRB_CUDA_CHECK(cudaGetLastError());
    return NRB_OK;
  };

  if (n_cols == 0) {  // empty pool: nothing is eligible; excluded ids are still range-checked
    NRB_CUDA_CHECK(cudaMemsetAsync(out_rows, 0xff, (size_t)n_users * k * sizeof(int32_t), st));  // -1
    NRB_CUDA_CHECK(cudaMemsetAsync(out_scores, 0xff, (size_t)n_users * k * sizeof(float), st));  // NaN
    return excl_idx != nullptr ? sort_excl() : NRB_OK;
  }
  const void* gemm_op = table_op;
  int64_t gemm_ld = op_stride;
  if (has_pool) {
    pool_gather_kernel<<<warps_grid(n_pool), 256, 0, st>>>((const __nv_bfloat16*)table_op, op_stride, kdim, pool,
                                                            n_pool, n_rows, (__nv_bfloat16*)L.pool_op, err_flag);
    note_launch();
    NRB_CUDA_CHECK(cudaGetLastError());
    gemm_op = L.pool_op;
    gemm_ld = kdim;
  }
  user_operand_kernel<<<warps_grid(n_users), 256, 0, st>>>(users, users_stride, n_users, dim, precision != NRB_BF16,
                                                           (__nv_bfloat16*)L.user_op, kdim, hist_off,
                                                           cand_base != nullptr ? L.cold : nullptr);
  note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  const int64_t n_pad = plan.n_per_row * 256;
  row_scale_kernel<<<warps_grid(n_pad), 256, 0, st>>>(table, precision, table_stride, n_rows, dim,
                                                      has_pool ? pool : nullptr, n_cols, n_pad, L.scale, cand_base,
                                                      L.base);
  note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  if (excl_idx != nullptr) {
    rc = sort_excl();
    if (rc != NRB_OK) return rc;
  }
  rc = gemm_topk_tc(L.user_op, kdim, gemm_op, gemm_ld, L.scale, excl_off, excl_idx ? L.excl_sorted : nullptr,
                    n_users, (int)n_cols, kdim, k, plan, L.parts, cand_base != nullptr ? L.base : nullptr, L.cold,
                    blend_alpha, st);
  if (rc != NRB_OK) return rc;
  const size_t merge_smem = (size_t)8 * 2 * plan.slots * sizeof(int32_t);
  if (merge_smem > 48 * 1024) NRB_CUDA_CHECK(cudaFuncSetAttribute(merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)merge_smem));
  merge_kernel<<<(unsigned)((n_users + 7) / 8), 256, merge_smem, st>>>(L.parts, plan, n_users, k,
                                                                       has_pool ? pool : nullptr, out_rows,
                                                                       out_scores);
  note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

extern "C" int nrb_recommend(int precision, int dim, int64_t n_rows, const void* table, int64_t table_stride,
                             const void* table_op, int64_t op_stride, const float* users, int64_t users_stride,
                             int64_t n_users, const int32_t* excl_idx, const int64_t* excl_off, int64_t n_excl, int k,
                             int32_t* out_rows, float* out_scores, int32_t* err_flag, void* workspace,
                             size_t workspace_bytes, nrb_stream_t stream) {
  return nrb_recommend_pool_blend(precision, dim, n_rows, table, table_stride, table_op, op_stride, users,
                                  users_stride, n_users, excl_idx, excl_off, n_excl, k, nullptr, -1, nullptr, 1.0f,
                                  nullptr, out_rows, out_scores, err_flag, workspace, workspace_bytes, stream);
}
