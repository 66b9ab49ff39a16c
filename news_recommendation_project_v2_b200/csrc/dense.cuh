// Internal interfaces shared by the dense-path translation units.
#pragma once

#include "common.cuh"

namespace nrb {

// gemm_tc.cu -- tcgen05 / TMA / TMEM (bf16 operands)
int gemm_bf16_tc(int epi, int out_dtype, const void* a, int64_t lda, const void* w, int64_t ldw, const float* bias,
                 const void* res, int64_t ldres, void* y, int64_t ldy, int64_t M, const int* m_dev, int N, int K,
                 int group, int group_valid, cudaStream_t st, int res_dtype = NRB_F32,
                 const int32_t* res_map = nullptr);
// Persistent tile schedule of the tcgen05 GEMM (gemm_tc.cu).  A scheduling unit is one row block of 128 * cg rows
// (cg = 2: a CTA pair) by cs neighbouring bn-column tiles (cs > 1: a softmax cluster); units are numbered row block
// by row block, N tiles ascending.  The n_ctas CTAs (pairs, clusters) of the grid take them strided
// (u = c, c + n_ctas, ...), or, for the top-k epilogue, in contiguous ranges, so that the tiles a CTA does for one row
// block are consecutive (a "segment").
struct TileSchedule {
  int cg, cs;
  int n_per_row;     // units per row block
  int64_t m_blocks;  // row blocks
  int64_t units;     // m_blocks * n_per_row
  uint32_t n_ctas;

  // The N tiles of a row are a multiple of cs; n_ctas = min(units, max_ctas).
  __host__ __device__ TileSchedule(int64_t M, int N, int bn, int cg_, int cs_, uint32_t max_ctas)
      : cg(cg_), cs(cs_), n_per_row((N + bn - 1) / bn / cs_), m_blocks((M + 128 * cg_ - 1) / (128 * cg_)),
        units(m_blocks * n_per_row), n_ctas(units < max_ctas ? (uint32_t)units : max_ctas) {}

  // units of CTA c: first, first + step, ... below end
  __host__ __device__ int64_t first(int64_t c, bool contiguous) const { return contiguous ? c * units / n_ctas : c; }
  __host__ __device__ int64_t end(int64_t c, bool contiguous) const {
    return contiguous ? (c + 1) * units / n_ctas : units;
  }
  __host__ __device__ int64_t step(bool contiguous) const { return contiguous ? 1 : n_ctas; }
  // 128-row block and bn-column tile of CTA `rank` of the pair / cluster that does unit u
  __host__ __device__ int m_blk(int64_t u, int rank) const { return (int)(u / n_per_row) * cg + (cg == 2 ? rank : 0); }
  __host__ __device__ int n_blk(int64_t u, int rank) const { return (int)(u % n_per_row) * cs + (cg == 2 ? 0 : rank); }
  // contiguous ranges: unit u starts / ends the segment of its row block in a range [first, end)
  __host__ __device__ bool starts_segment(int64_t u, int64_t first) const { return u == first || u % n_per_row == 0; }
  __host__ __device__ bool ends_segment(int64_t u, int64_t end) const {
    return u + 1 == end || (u + 1) % n_per_row == 0;
  }
  // contiguous ranges: the CTA whose range holds unit u (the largest c with first(c) <= u), and the first and last
  // CTA whose range touches row block m
  __host__ __device__ int64_t owner(int64_t u) const { return ((u + 1) * n_ctas - 1) / units; }
  __host__ __device__ int64_t first_owner(int64_t m) const { return owner(m * n_per_row); }
  __host__ __device__ int64_t last_owner(int64_t m) const { return owner((m + 1) * n_per_row - 1); }
};

// gemm_tc.cu -- tcgen05 GEMM with the fused top-k epilogue (NRB_EPI_TOPK, or NRB_EPI_TOPK_BLEND when base != NULL).
// cg = 1 when M <= 128, else CTA pairs; 256-column tiles; slots = the most CTAs whose range touches one row block,
// i.e. the partial lists each (row, half) may get.
struct TopkPlan : TileSchedule {
  int64_t slots;
};
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
