// Internal interfaces shared by the dense-path translation units.
#pragma once

#include "common.cuh"

namespace nrb {

// gemm_tc.cu -- tcgen05 / TMA / TMEM (bf16 operands)
int gemm_bf16_tc(int epi, int out_dtype, const void* a, int64_t lda, const void* w, int64_t ldw, const float* bias,
                 const void* res, int64_t ldres, void* y, int64_t ldy, int64_t M, const int* m_dev, int N, int K,
                 int group, int group_valid, cudaStream_t st, int res_dtype = NRB_F32,
                 const int32_t* res_map = nullptr);
// gemm_tc.cu -- tcgen05 GEMM with the fused top-k epilogue (NRB_EPI_TOPK, or NRB_EPI_TOPK_BLEND when base != NULL)
struct TopkPlan {
  int cg;              // 1: single CTA (M <= 128), 2: CTA pairs
  int rows_per_block;  // 128 * cg
  int64_t m_tiles, n_per_row, units, n_units, slots;
};
// CTA (pair) whose contiguous unit range holds unit u: the largest c with floor(c * units / n_units) <= u
__host__ __device__ inline int64_t topk_owner(const TopkPlan& t, int64_t u) {
  return ((u + 1) * t.n_units - 1) / t.units;
}
TopkPlan topk_plan(int64_t M, int64_t N);
int gemm_topk_tc(const void* a, int64_t lda, const void* w, int64_t ldw, const float* scale, const int64_t* excl_off,
                 const int32_t* excl_sorted, int64_t M, int N, int K, int k, const TopkPlan& plan, void* parts,
                 const float* base, const uint8_t* cold, float alpha, cudaStream_t st);
// gemm_simt.cu -- FFMA (fp32 operands)
int gemm_f32_simt(int epi, int out_dtype, const void* a, int64_t lda, const void* w, int64_t ldw,
                  const float* bias, const void* res, int64_t ldres, void* y, int64_t ldy, int64_t M,
                  const int* m_dev, int N, int K, cudaStream_t st, int res_dtype = NRB_F32,
                  const int32_t* res_map = nullptr);

// precision-dispatching linear
int linear(int precision, int epi, int out_dtype, const void* a, int64_t lda, const void* w, int64_t ldw,
           const float* bias, const void* res, int64_t ldres, void* y, int64_t ldy, int64_t M, const int* m_dev,
           int N, int K, cudaStream_t st, int group = 0, int group_valid = 0, int res_dtype = NRB_F32,
           const int32_t* res_map = nullptr);

// dense.cu -- row-wise helpers (all take an optional device-side row count)
int layer_norm_rows(const void* x, int x_dtype, int64_t ldx, const int32_t* row_map, const float* gamma,
                    const float* beta, void* y, int y_dtype, int64_t ldy, float* copy_f32, int64_t ldcopy,
                    int64_t rows, const int* rows_dev, int dim, cudaStream_t st, float eps = 1e-5f);
int softmax_groups(const float* logits, int64_t ldl, void* p, int p_dtype, int64_t ldp, int64_t rows,
                   const int* rows_dev, int n_groups, int group, int valid, cudaStream_t st);
int convert_rows(const void* src, int src_dtype, int64_t lds, void* dst, int dst_dtype, int64_t ldd, int64_t rows,
                 int cols, cudaStream_t st);
int transpose_f32(const float* src, int rows, int cols, float* dst, cudaStream_t st);
int scale_cols_f32(float* x, int64_t ld, int64_t rows, int cols, float s, cudaStream_t st);

static inline size_t dtype_size(int dt) { return dt == NRB_F32 ? 4 : 2; }
static inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

// bump allocator over a caller-provided workspace
struct Workspace {
  char* base;
  size_t size;
  size_t used = 0;
  bool ok = true;
  Workspace(void* b, size_t s) : base((char*)b), size(s) {}
  void* take(size_t bytes) {
    const size_t off = align_up(used, 256);
    if (base != nullptr && off + bytes > size) ok = false;
    used = off + bytes;
    return base ? base + off : nullptr;
  }
};

}  // namespace nrb
