// Row-wise helper kernels around the dense contractions + the FinalAttention per-row transform.
//
//   layer_norm_rows  : torch.nn.LayerNorm (eps 1e-5, biased variance) -- latent_attention.py:10-19
//   softmax_groups   : softmax over the latents of one head           -- latent_attention.py:69-72
//   nrb_final_attention_rows : modeling_utils.py:218-224 hoisted from per-history-slot to per-table-row
#include "dense.cuh"

#include <algorithm>

namespace nrb {

__device__ __forceinline__ float load_elem(const void* p, int dt, int64_t i) {
  return dt == NRB_F32 ? reinterpret_cast<const float*>(p)[i]
                       : __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(p)[i]);
}
__device__ __forceinline__ void store_elem(void* p, int dt, int64_t i, float v) {
  if (dt == NRB_F32)
    reinterpret_cast<float*>(p)[i] = v;
  else
    reinterpret_cast<__nv_bfloat16*>(p)[i] = __float2bfloat16_rn(v);
}

// One warp per row.  Two-pass mean / variance in fp32 of x - x0 (x0 = the row's first element, see
// layer_norm_vec_kernel); the row is re-read from L1 rather than cached so that any `dim` works.
// Optionally gathers the source row through `row_map` (varlen token packing) and emits an fp32 copy
// of the raw row (the residual operand).
__global__ void __launch_bounds__(256)
layer_norm_kernel(const void* x, int x_dtype, int64_t ldx, const int32_t* row_map, const float* gamma,
                  const float* beta, void* y, int y_dtype, int64_t ldy, float* copy_f32, int64_t ldcopy,
                  int64_t rows, const int* rows_dev, int dim, float eps) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t n = rows_dev != nullptr ? min(rows, (int64_t)*rows_dev) : rows;
  for (int64_t r = warp_id; r < n; r += n_warps) {
    const int64_t src = row_map != nullptr ? (int64_t)row_map[r] : r;
    const int64_t xo = src * ldx;
    const float x0 = load_elem(x, x_dtype, xo);  // shift of the statistics (see layer_norm_vec_kernel)
    float s = 0.f;
    for (int i = lane; i < dim; i += 32) s += load_elem(x, x_dtype, xo + i) - x0;
    const float mean = warp_sum(s) / (float)dim;  // of x - x0
    float q = 0.f;
    for (int i = lane; i < dim; i += 32) {
      const float d = (load_elem(x, x_dtype, xo + i) - x0) - mean;
      q = fmaf(d, d, q);
    }
    const float rstd = rsqrtf(warp_sum(q) / (float)dim + eps);
    for (int i = lane; i < dim; i += 32) {
      const float v = load_elem(x, x_dtype, xo + i);
      store_elem(y, y_dtype, r * ldy + i, ((v - x0) - mean) * rstd * gamma[i] + beta[i]);
      if (copy_f32 != nullptr) copy_f32[r * ldcopy + i] = v;
    }
  }
}

// Vectorised single-pass variant: the row lives in registers (NV 16-byte vectors per lane), so x is read
// once; used whenever dim*elemsize is a multiple of 512 bytes (768 / 1024-wide rows in both dtypes).
template <typename TIN, int NV>
__global__ void __launch_bounds__(256, NV <= 3 ? 3 : 2)
layer_norm_vec_kernel(const void* x, int64_t ldx, const int32_t* row_map, const float* gamma, const float* beta,
                      void* y, int y_dtype, int64_t ldy, float* copy_f32, int64_t ldcopy, int64_t rows,
                      const int* rows_dev, int dim, float eps) {
  constexpr int EPV = Vec16<TIN>::EPV;
  const int lane = threadIdx.x & 31;
  const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t n = rows_dev != nullptr ? min(rows, (int64_t)*rows_dev) : rows;
  const TIN* xin = reinterpret_cast<const TIN*>(x);
  // the row-map entry of the NEXT row is requested one row ahead: the gather costs no dependent-load latency
  int64_t src_next = warp_id < n ? (row_map != nullptr ? (int64_t)row_map[warp_id] : warp_id) : 0;
  for (int64_t r = warp_id; r < n; r += n_warps) {
    const int64_t src = src_next;
    if (r + n_warps < n) src_next = row_map != nullptr ? (int64_t)row_map[r + n_warps] : r + n_warps;
    const char* base = reinterpret_cast<const char*>(xin + src * ldx);
    float v[NV][EPV];
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const uint4 u = *reinterpret_cast<const uint4*>(base + (size_t)(lane + 32 * i) * 16);
      Vec16<TIN>::unpack(u, v[i]);
    }
    // Statistics of x - x0, x0 = the row's first element: sum(x) / dim rounds the mean by up to an ulp of x, and
    // (x - mean) * rsqrt(var + eps) turns that into O(1) when the spread is far below the magnitude -- a constant
    // row with eps 1e-12 came out as beta +- 0.4 gamma.  x - x0 is exact there, so the mean and every deviation are.
    const float x0 = __shfl_sync(kFullMask, v[0][0], 0);
    float s = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
      for (int k = 0; k < EPV; ++k) s += v[i][k] - x0;
    const float mean = warp_sum(s) / (float)dim;  // of x - x0
    float q = 0.f;
#pragma unroll
    for (int i = 0; i < NV; ++i)
#pragma unroll
      for (int k = 0; k < EPV; ++k) {
        const float d = (v[i][k] - x0) - mean;
        q = fmaf(d, d, q);
      }
    const float rstd = rsqrtf(warp_sum(q) / (float)dim + eps);
#pragma unroll
    for (int i = 0; i < NV; ++i) {
      const int e0 = (lane + 32 * i) * EPV;
      float o[EPV];
#pragma unroll
      for (int k = 0; k < EPV; k += 4) {
        const float4 g4 = *reinterpret_cast<const float4*>(gamma + e0 + k);
        const float4 b4 = *reinterpret_cast<const float4*>(beta + e0 + k);
        o[k] = ((v[i][k] - x0) - mean) * rstd * g4.x + b4.x;
        o[k + 1] = ((v[i][k + 1] - x0) - mean) * rstd * g4.y + b4.y;
        o[k + 2] = ((v[i][k + 2] - x0) - mean) * rstd * g4.z + b4.z;
        o[k + 3] = ((v[i][k + 3] - x0) - mean) * rstd * g4.w + b4.w;
      }
      if (y_dtype == NRB_BF16) {
        __nv_bfloat16* yo = reinterpret_cast<__nv_bfloat16*>(y) + r * ldy + e0;
#pragma unroll
        for (int k = 0; k < EPV; k += 4)
          *reinterpret_cast<uint2*>(yo + k) = make_uint2(pack_bf16x2(o[k], o[k + 1]), pack_bf16x2(o[k + 2], o[k + 3]));
      } else {
        float* yo = reinterpret_cast<float*>(y) + r * ldy + e0;
#pragma unroll
        for (int k = 0; k < EPV; k += 4) *reinterpret_cast<float4*>(yo + k) = make_float4(o[k], o[k + 1], o[k + 2], o[k + 3]);
      }
      if (copy_f32 != nullptr) {
        float* co = copy_f32 + r * ldcopy + e0;
#pragma unroll
        for (int k = 0; k < EPV; k += 4)
          *reinterpret_cast<float4*>(co + k) = make_float4(v[i][k], v[i][k + 1], v[i][k + 2], v[i][k + 3]);
      }
    }
  }
}

int layer_norm_rows(const void* x, int x_dtype, int64_t ldx, const int32_t* row_map, const float* gamma,
                    const float* beta, void* y, int y_dtype, int64_t ldy, float* copy_f32, int64_t ldcopy,
                    int64_t rows, const int* rows_dev, int dim, cudaStream_t st, float eps) {
  if (rows <= 0) return NRB_OK;
  const int64_t want = (rows + 7) / 8;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count_cached() * 16);
  const int es = x_dtype == NRB_F32 ? 4 : 2;
  const int yes = y_dtype == NRB_F32 ? 4 : 2;
  const bool aligned = (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (ldx * es) % 16 == 0 &&
                       (reinterpret_cast<uintptr_t>(y) & 15) == 0 && (ldy * yes) % 16 == 0 &&
                       (reinterpret_cast<uintptr_t>(gamma) & 15) == 0 && (reinterpret_cast<uintptr_t>(beta) & 15) == 0 &&
                       (copy_f32 == nullptr || ((reinterpret_cast<uintptr_t>(copy_f32) & 15) == 0 && ldcopy % 4 == 0));
  const int nv = (dim * es) % 512 == 0 ? dim * es / 512 : 0;
  bool done = false;
  if (aligned && nv >= 1 && nv <= 8) {
    done = true;
#define NRB_LN_CASE(T, N)                                                                                          \
  case N:                                                                                                          \
    layer_norm_vec_kernel<T, N><<<grid, 256, 0, st>>>(x, ldx, row_map, gamma, beta, y, y_dtype, ldy, copy_f32,      \
                                                      ldcopy, rows, rows_dev, dim, eps);                           \
    break;
    if (x_dtype == NRB_F32) {
      switch (nv) {
        NRB_LN_CASE(float, 1) NRB_LN_CASE(float, 2) NRB_LN_CASE(float, 3) NRB_LN_CASE(float, 4)
        NRB_LN_CASE(float, 6) NRB_LN_CASE(float, 8)
        default: done = false;
      }
    } else {
      switch (nv) {
        NRB_LN_CASE(__nv_bfloat16, 1) NRB_LN_CASE(__nv_bfloat16, 2) NRB_LN_CASE(__nv_bfloat16, 3)
        NRB_LN_CASE(__nv_bfloat16, 4)
        default: done = false;
      }
    }
#undef NRB_LN_CASE
  }
  if (!done)
    layer_norm_kernel<<<grid, 256, 0, st>>>(x, x_dtype, ldx, row_map, gamma, beta, y, y_dtype, ldy, copy_f32, ldcopy,
                                            rows, rows_dev, dim, eps);
  note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

// One warp per (row, group): p = softmax(logits[group]) over the first `valid` columns of the group,
// zeros in the padded columns.
__global__ void __launch_bounds__(256)
softmax_groups_kernel(const float* logits, int64_t ldl, void* p, int p_dtype, int64_t ldp, int64_t rows,
                      const int* rows_dev, int n_groups, int group, int valid) {
  const int lane = threadIdx.x & 31;
  const int64_t warp_id = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t n = rows_dev != nullptr ? min(rows, (int64_t)*rows_dev) : rows;
  const int64_t total = n * n_groups;
  for (int64_t w = warp_id; w < total; w += n_warps) {
    const int64_t r = w / n_groups;
    const int g = (int)(w - r * n_groups);
    const float* src = logits + r * ldl + (int64_t)g * group;
    float m = -INFINITY;
    for (int i = lane; i < valid; i += 32) m = fmaxf(m, src[i]);
    m = warp_max(m);
    float s = 0.f;
    for (int i = lane; i < valid; i += 32) s += expf(src[i] - m);
    s = warp_sum(s);
    const float inv = 1.0f / s;
    for (int i = lane; i < group; i += 32) {
      const float v = i < valid ? expf(src[i] - m) * inv : 0.f;
      store_elem(p, p_dtype, r * ldp + (int64_t)g * group + i, v);
    }
  }
}

int softmax_groups(const float* logits, int64_t ldl, void* p, int p_dtype, int64_t ldp, int64_t rows,
                   const int* rows_dev, int n_groups, int group, int valid, cudaStream_t st) {
  if (rows <= 0) return NRB_OK;
  const int64_t want = (rows * n_groups + 7) / 8;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count_cached() * 16);
  softmax_groups_kernel<<<grid, 256, 0, st>>>(logits, ldl, p, p_dtype, ldp, rows, rows_dev, n_groups, group, valid); note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

__global__ void __launch_bounds__(256)
convert_rows_kernel(const void* src, int src_dtype, int64_t lds, void* dst, int dst_dtype, int64_t ldd,
                    int64_t rows, int cols) {
  const int64_t total = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols;
    const int c = (int)(i - r * cols);
    store_elem(dst, dst_dtype, r * ldd + c, load_elem(src, src_dtype, r * lds + c));
  }
}

// fp32 -> bf16, 8 elements per thread: two 128-bit loads, one 128-bit store (the host-table upload path)
__global__ void __launch_bounds__(256)
convert_f32_bf16_vec_kernel(const float* src, int64_t lds, __nv_bfloat16* dst, int64_t ldd, int64_t rows, int cols8) {
  const int64_t total = rows * cols8;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols8;
    const int c = (int)(i - r * cols8) * 8;
    const uint4 a = ldg_stream_128(src + r * lds + c), b = ldg_stream_128(src + r * lds + c + 4);
    uint4 o;
    o.x = pack_bf16x2(__uint_as_float(a.x), __uint_as_float(a.y));
    o.y = pack_bf16x2(__uint_as_float(a.z), __uint_as_float(a.w));
    o.z = pack_bf16x2(__uint_as_float(b.x), __uint_as_float(b.y));
    o.w = pack_bf16x2(__uint_as_float(b.z), __uint_as_float(b.w));
    *reinterpret_cast<uint4*>(dst + r * ldd + c) = o;
  }
}

// fp32 -> three bf16 column blocks for the split-bf16 tensor-core path: with hi = bf16(v), lo = bf16(v - hi)
//   role 0 (activation rows):  [ hi | hi | lo ]        role 1 (weight rows):  [ hi | lo | hi ]
// so that ONE bf16 GEMM over K' = 3K accumulates a_hi w_hi + a_hi w_lo + a_lo w_hi in fp32 (the dropped a_lo w_lo
// term and the 16-bit truncation of each operand are ~2^-17 relative).
__global__ void __launch_bounds__(256)
split_rows_kernel(const float* src, int64_t lds, __nv_bfloat16* dst, int64_t ldd, int64_t rows, int k4, int role) {
  const int64_t total = rows * k4;
  const int K = k4 * 4;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / k4;
    const int c = (int)(i - r * k4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(src + r * lds + c);
    const float f[4] = {v.x, v.y, v.z, v.w};
    float hi[4], lo[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      hi[q] = __bfloat162float(__float2bfloat16_rn(f[q]));
      lo[q] = f[q] - hi[q];  // exact in fp32
    }
    const uint2 H = make_uint2(pack_bf16x2(hi[0], hi[1]), pack_bf16x2(hi[2], hi[3]));
    const uint2 L = make_uint2(pack_bf16x2(lo[0], lo[1]), pack_bf16x2(lo[2], lo[3]));
    __nv_bfloat16* d = dst + r * ldd + c;
    *reinterpret_cast<uint2*>(d) = H;
    *reinterpret_cast<uint2*>(d + K) = role == 0 ? H : L;
    *reinterpret_cast<uint2*>(d + 2 * K) = role == 0 ? L : H;
  }
}

int split_rows(const float* src, int64_t lds, void* dst, int64_t ldd, int64_t rows, int K, int role, cudaStream_t st) {
  if (rows <= 0) return NRB_OK;
  const int64_t want = (rows * (K / 4) + 255) / 256;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count_cached() * 16);
  split_rows_kernel<<<grid, 256, 0, st>>>(src, lds, (__nv_bfloat16*)dst, ldd, rows, K / 4, role);
  note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

int convert_rows(const void* src, int src_dtype, int64_t lds, void* dst, int dst_dtype, int64_t ldd, int64_t rows,
                 int cols, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return NRB_OK;
  if (src_dtype == NRB_F32 && dst_dtype == NRB_BF16 && cols % 8 == 0 && lds % 4 == 0 && ldd % 8 == 0 &&
      (reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 15) == 0) {
    const int64_t want8 = (rows * (cols / 8) + 255) / 256;
    const int grid8 = (int)std::min<int64_t>(want8, (int64_t)sm_count_cached() * 16);
    convert_f32_bf16_vec_kernel<<<grid8, 256, 0, st>>>((const float*)src, lds, (__nv_bfloat16*)dst, ldd, rows,
                                                       cols / 8);
    note_launch();
    NRB_CUDA_CHECK(cudaGetLastError());
    return NRB_OK;
  }
  const int64_t want = (rows * cols + 255) / 256;
  const int grid = (int)std::min<int64_t>(want, (int64_t)sm_count_cached() * 32);
  convert_rows_kernel<<<grid, 256, 0, st>>>(src, src_dtype, lds, dst, dst_dtype, ldd, rows, cols); note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

__global__ void transpose_f32_kernel(const float* src, int rows, int cols, float* dst) {
  __shared__ float tile[32][33];
  const int c0 = blockIdx.x * 32, r0 = blockIdx.y * 32;
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int r = r0 + j, c = c0 + threadIdx.x;
    if (r < rows && c < cols) tile[j][threadIdx.x] = src[(int64_t)r * cols + c];
  }
  __syncthreads();
  for (int j = threadIdx.y; j < 32; j += blockDim.y) {
    const int c = c0 + j, r = r0 + threadIdx.x;
    if (r < rows && c < cols) dst[(int64_t)c * rows + r] = tile[threadIdx.x][j];
  }
}

int transpose_f32(const float* src, int rows, int cols, float* dst, cudaStream_t st) {
  dim3 grid((cols + 31) / 32, (rows + 31) / 32), block(32, 8);
  transpose_f32_kernel<<<grid, block, 0, st>>>(src, rows, cols, dst); note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

__global__ void scale_cols_kernel(float* x, int64_t ld, int64_t rows, int cols, float s) {
  const int64_t total = rows * cols;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = i / cols;
    x[r * ld + (i - r * cols)] *= s;
  }
}

int scale_cols_f32(float* x, int64_t ld, int64_t rows, int cols, float s, cudaStream_t st) {
  const int64_t want = (rows * cols + 255) / 256;
  const int grid = (int)std::min<int64_t>(std::max<int64_t>(want, 1), (int64_t)sm_count_cached() * 8);
  scale_cols_kernel<<<grid, 256, 0, st>>>(x, ld, rows, cols, s); note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

int linear(int precision, int epi, int out_dtype, const void* a, int64_t lda, const void* w, int64_t ldw,
           const float* bias, const void* res, int64_t ldres, void* y, int64_t ldy, int64_t M, const int* m_dev,
           int N, int K, cudaStream_t st, int group, int group_valid, int res_dtype, const int32_t* res_map) {
  if (precision == NRB_BF16)
    return gemm_bf16_tc(epi, out_dtype, a, lda, w, ldw, bias, res, ldres, y, ldy, M, m_dev, N, K, group,
                        group_valid, st, res_dtype, res_map);
  if (precision == NRB_F32 && epi == NRB_EPI_SOFTMAX) {
    set_error("nrb_linear(fp32): the fused softmax epilogue exists only on the tensor-core path");
    return NRB_E_INVALID;
  }
  if (precision == NRB_F32)
    return gemm_f32_simt(epi, out_dtype, a, lda, w, ldw, bias, res, ldres, y, ldy, M, m_dev, N, K, st, res_dtype,
                         res_map);
  set_error("nrb_linear: bad precision %d", precision);
  return NRB_E_INVALID;
}

constexpr int64_t kFaChunkRows = 16384;

}  // namespace nrb

using namespace nrb;

extern "C" int nrb_convert_rows(const void* src, int src_dtype, int64_t src_stride, void* dst, int dst_dtype,
                                int64_t dst_stride, int64_t n_rows, int dim, nrb_stream_t stream) {
  NRB_REQUIRE((src_dtype == NRB_F32 || src_dtype == NRB_BF16) && (dst_dtype == NRB_F32 || dst_dtype == NRB_BF16),
              "nrb_convert_rows: bad dtype");
  NRB_REQUIRE(n_rows >= 0 && dim > 0, "nrb_convert_rows: bad sizes");
  if (n_rows == 0) return NRB_OK;
  NRB_REQUIRE(src && dst, "nrb_convert_rows: null pointer");
  return convert_rows(src, src_dtype, src_stride, dst, dst_dtype, dst_stride, n_rows, dim, as_stream(stream));
}

extern "C" int nrb_layer_norm(const void* x, int x_dtype, int64_t ldx, const float* gamma, const float* beta, float eps,
                              void* y, int y_dtype, int64_t ldy, int64_t rows, int dim, nrb_stream_t stream) {
  NRB_REQUIRE(x && gamma && beta && y, "nrb_layer_norm: null pointer");
  NRB_REQUIRE((x_dtype == NRB_F32 || x_dtype == NRB_BF16) && (y_dtype == NRB_F32 || y_dtype == NRB_BF16),
              "nrb_layer_norm: bad dtype");
  NRB_REQUIRE(rows >= 0 && dim > 0 && eps >= 0.f, "nrb_layer_norm: bad sizes");
  return layer_norm_rows(x, x_dtype, ldx, nullptr, gamma, beta, y, y_dtype, ldy, nullptr, 0, rows, nullptr, dim,
                         as_stream(stream), eps);
}

extern "C" int nrb_linear(int precision, int epilogue, int out_dtype, const void* a, int64_t lda, const void* w,
                          int64_t ldw, const float* bias, const float* res, int64_t ldres, void* y, int64_t ldy,
                          int64_t M, int N, int K, int group, int group_valid, nrb_stream_t stream) {
  NRB_REQUIRE(a && w && y, "nrb_linear: null pointer");
  return linear(precision, epilogue, out_dtype, a, lda, w, ldw, bias, res, ldres, y, ldy, M, nullptr, N, K,
                as_stream(stream), group, group_valid);
}

extern "C" int nrb_split_rows(const float* src, int64_t src_stride, void* dst, int64_t dst_stride, int64_t n_rows,
                              int dim, int role, nrb_stream_t stream) {
  NRB_REQUIRE(n_rows >= 0 && dim > 0 && dim % 4 == 0, "nrb_split_rows: dim must be a positive multiple of 4");
  NRB_REQUIRE(role == 0 || role == 1, "nrb_split_rows: role must be 0 (activations) or 1 (weights)");
  if (n_rows == 0) return NRB_OK;
  NRB_REQUIRE(src && dst, "nrb_split_rows: null pointer");
  NRB_REQUIRE(src_stride % 4 == 0 && dst_stride % 4 == 0 && dst_stride >= 3 * (int64_t)dim &&
                  (reinterpret_cast<uintptr_t>(src) & 15) == 0 && (reinterpret_cast<uintptr_t>(dst) & 7) == 0,
              "nrb_split_rows: alignment / stride");
  return split_rows(src, src_stride, dst, dst_stride, n_rows, dim, role, as_stream(stream));
}

// split-bf16 variant of the FinalAttention row transform: fp32 table in, fp32 x / exp(logit) out, every Linear as ONE
// tcgen05 GEMM over K' = 3K on [hi|hi|lo] x [hi|lo|hi] operands (weights pre-split by nrb_split_rows, role 1)
static size_t fa_split_ws(int64_t n_rows, int dim, int hidden, float** act, void** sp, void* base) {
  const int64_t chunk = std::min<int64_t>(n_rows, kFaChunkRows);
  const int wide = std::max(dim, hidden);
  Workspace ws(base, (size_t)-1);
  float* a = (float*)ws.take((size_t)chunk * wide * 4);
  void* s3 = ws.take((size_t)chunk * 3 * wide * 2);
  if (act) *act = a;
  if (sp) *sp = s3;
  return ws.used + 256;
}

extern "C" size_t nrb_final_attention_rows_split_workspace_bytes(int64_t n_rows, int dim, int hidden) {
  return fa_split_ws(n_rows, dim, hidden, nullptr, nullptr, nullptr);
}

extern "C" int nrb_final_attention_rows_split(const float* table, int64_t table_stride, int64_t n_rows, int dim,
                                              int hidden, const void* w1s, const float* b1, const void* w2s,
                                              const float* b2, const void* w3s, const float* b3, const void* w4s,
                                              const float* b4, const void* w5s, float* x_out, float* e_out,
                                              int64_t out_stride, void* workspace, size_t workspace_bytes,
                                              nrb_stream_t stream) {
  NRB_REQUIRE(n_rows > 0 && dim > 0 && hidden > 0 && dim % 64 == 0 && hidden % 64 == 0,
              "nrb_final_attention_rows_split: dim and hidden must be multiples of 64");
  NRB_REQUIRE(table && w1s && b1 && w2s && b2 && w3s && b3 && w4s && b4 && w5s && x_out && e_out && workspace,
              "nrb_final_attention_rows_split: null pointer");
  float* act;
  void* sp;
  if (workspace_bytes < fa_split_ws(n_rows, dim, hidden, &act, &sp, workspace)) {
    set_error("nrb_final_attention_rows_split: workspace too small");
    return NRB_E_WORKSPACE;
  }
  cudaStream_t st = as_stream(stream);
  const int64_t chunk = std::min<int64_t>(n_rows, kFaChunkRows);
  const int d3 = 3 * dim, h3 = 3 * hidden;
  for (int64_t r0 = 0; r0 < n_rows; r0 += chunk) {
    const int64_t m = std::min<int64_t>(chunk, n_rows - r0);
    float* xo = x_out + r0 * out_stride;
    float* eo = e_out + r0 * out_stride;
    int rc;
#define NRB_SPLIT_LINEAR(SRC, LDS, KIN, W, BIAS, EPI, DST, LDD, NOUT)                                                  \
  if ((rc = split_rows(SRC, LDS, sp, 3 * (KIN), m, KIN, 0, st)) != NRB_OK) return rc;                                  \
  if ((rc = gemm_bf16_tc(EPI, NRB_F32, sp, 3 * (KIN), W, 3 * (KIN), BIAS, nullptr, 0, DST, LDD, m, nullptr, NOUT,      \
                         3 * (KIN), 0, 0, st)) != NRB_OK)                                                              \
    return rc;
    // x = W3 relu(W2 relu(W1 e + b1) + b2) + b3          (modeling_utils.py:218-220)
    NRB_SPLIT_LINEAR(table + r0 * table_stride, table_stride, dim, w1s, b1, NRB_EPI_RELU, act, hidden, hidden)
    NRB_SPLIT_LINEAR(act, hidden, hidden, w2s, b2, NRB_EPI_RELU, act, hidden, hidden)
    NRB_SPLIT_LINEAR(act, hidden, hidden, w3s, b3, NRB_EPI_NONE, xo, out_stride, dim)
    // elog = exp(W5 relu(W4 x + b4))                        (modeling_utils.py:221-224)
    NRB_SPLIT_LINEAR(xo, out_stride, dim, w4s, b4, NRB_EPI_RELU, act, hidden, hidden)
    NRB_SPLIT_LINEAR(act, hidden, hidden, w5s, nullptr, NRB_EPI_EXP, eo, out_stride, dim)
#undef NRB_SPLIT_LINEAR
    (void)d3;
    (void)h3;
  }
  return NRB_OK;
}

extern "C" size_t nrb_final_attention_rows_workspace_bytes(int precision, int64_t n_rows, int dim, int hidden) {
  const int64_t chunk = std::min<int64_t>(n_rows, kFaChunkRows);
  Workspace ws(nullptr, 0);
  ws.take((size_t)chunk * hidden * dtype_size(precision));  // h1
  ws.take((size_t)chunk * hidden * dtype_size(precision));  // h2
  ws.take((size_t)chunk * dim * dtype_size(precision));     // x in compute dtype
  return ws.used + 256;
}

extern "C" int nrb_final_attention_rows(int precision, int out_dtype, const void* table, int64_t table_stride,
                                        int64_t n_rows, int dim, int hidden, const void* w1, const float* b1,
                                        const void* w2, const float* b2, const void* w3, const float* b3,
                                        const void* w4, const float* b4, const void* w5, void* x_out, void* e_out,
                                        int64_t out_stride, void* workspace, size_t workspace_bytes,
                                        nrb_stream_t stream) {
  NRB_REQUIRE(precision == NRB_F32 || precision == NRB_BF16, "nrb_final_attention_rows: bad precision");
  NRB_REQUIRE(out_dtype == NRB_F32 || out_dtype == NRB_BF16, "nrb_final_attention_rows: bad out_dtype");
  NRB_REQUIRE(n_rows > 0 && dim > 0 && hidden > 0, "nrb_final_attention_rows: bad sizes");
  NRB_REQUIRE(table && w1 && b1 && w2 && b2 && w3 && b3 && w4 && b4 && w5 && x_out && e_out && workspace,
              "nrb_final_attention_rows: null pointer");
  if (workspace_bytes < nrb_final_attention_rows_workspace_bytes(precision, n_rows, dim, hidden)) {
    set_error("nrb_final_attention_rows: workspace too small");
    return NRB_E_WORKSPACE;
  }
  cudaStream_t st = as_stream(stream);
  const size_t es = dtype_size(precision), os = dtype_size(out_dtype);
  const int64_t chunk = std::min<int64_t>(n_rows, kFaChunkRows);
  Workspace ws(workspace, workspace_bytes);
  void* h1 = ws.take((size_t)chunk * hidden * es);
  void* h2 = ws.take((size_t)chunk * hidden * es);
  void* xc = ws.take((size_t)chunk * dim * es);
  for (int64_t r0 = 0; r0 < n_rows; r0 += chunk) {
    const int64_t m = std::min<int64_t>(chunk, n_rows - r0);
    const void* e = (const char*)table + (size_t)r0 * table_stride * es;
    void* xo = (char*)x_out + (size_t)r0 * out_stride * os;
    void* eo = (char*)e_out + (size_t)r0 * out_stride * os;
    int rc;
    // x = W3 relu(W2 relu(W1 e + b1) + b2) + b3          (modeling_utils.py:218-220)
    if ((rc = linear(precision, NRB_EPI_RELU, precision, e, table_stride, w1, dim, b1, nullptr, 0, h1, hidden, m,
                     nullptr, hidden, dim, st)) != NRB_OK)
      return rc;
    if ((rc = linear(precision, NRB_EPI_RELU, precision, h1, hidden, w2, hidden, b2, nullptr, 0, h2, hidden, m,
                     nullptr, hidden, hidden, st)) != NRB_OK)
      return rc;
    if ((rc = linear(precision, NRB_EPI_NONE, out_dtype, h2, hidden, w3, hidden, b3, nullptr, 0, xo, out_stride, m,
                     nullptr, dim, hidden, st)) != NRB_OK)
      return rc;
    const void* xin = xo;
    int64_t ldxin = out_stride;
    if (out_dtype != precision) {
      if ((rc = convert_rows(xo, out_dtype, out_stride, xc, precision, dim, m, dim, st)) != NRB_OK) return rc;
      xin = xc;
      ldxin = dim;
    }
    // elog = exp(W5 relu(W4 x + b4))                        (modeling_utils.py:221-224)
    if ((rc = linear(precision, NRB_EPI_RELU, precision, xin, ldxin, w4, dim, b4, nullptr, 0, h1, hidden, m,
                     nullptr, hidden, dim, st)) != NRB_OK)
      return rc;
    if ((rc = linear(precision, NRB_EPI_EXP, out_dtype, h1, hidden, w5, hidden, nullptr, nullptr, 0, eo,
                     out_stride, m, nullptr, dim, hidden, st)) != NRB_OK)
      return rc;
  }
  return NRB_OK;
}
