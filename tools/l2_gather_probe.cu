// L2 gather-rate probe: how fast can the SMs gather random 128-byte lines that sit in L2?
//
// The score/rank kernel reads 2*sum(H) + sum(C) random table rows per step.  Every step of its arithmetic except
// the final cosine scalars works column by column, so it could instead run as passes over 128-byte column slices
// of the rows: one slice of the three tables (X, E, T) is 3 * n_rows * 128 B, which fits the 126 MB L2 at the
// MIND-large shape (161,013 rows).  Whether that pays depends on one number nobody had measured: the rate at
// which warps gather random 128-byte lines from L2.  This program measures it for the kernel's access pattern:
//
//   * uniformly random row ids over N rows, streamed from DRAM (evict_first cache hint), one per lane;
//   * one 128-byte line per row at base + r*2048 + s*128, rotating over 3 tables;
//   * a warp issues 4 B per lane, so one load instruction is one line, DEPTH lines in flight per warp;
//   * 1- or 2-warp CTAs, one wave of as many as fit (32 resident warps per SM, or what registers allow).
//
// It sweeps the slice working set (3 * N * 128 B) over 15 / 31 / 62 / 124 MB and, as the baseline, times the
// current pattern: whole 2 KB rows from three 0.99 GB tables.  No torch; prints one JSON document.
//
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o l2_gather_probe tools/l2_gather_probe.cu
//   ./l2_gather_probe > result.json
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>

#include <algorithm>
#include <string>
#include <vector>

#define CHECK(x)                                                                                  \
  do {                                                                                            \
    cudaError_t e_ = (x);                                                                         \
    if (e_ != cudaSuccess) {                                                                      \
      fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_));          \
      exit(1);                                                                                    \
    }                                                                                             \
  } while (0)

constexpr int kRowBytes = 2048;  // bf16 d=1024 / fp32 d=512: the bench's row width
constexpr unsigned kFull = 0xffffffffu;

// Scalar loads take their L2 eviction priority from a createpolicy operand (.L2::cache_hint).
__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ uint64_t policy_evict_last() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
  return p;
}
__device__ __forceinline__ int32_t ld_hint_i32(const int32_t* p, uint64_t pol) {
  int32_t v;
  asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
// HINT 0: no L2 hint (evict_normal), 1: L2::evict_last
template <int HINT>
__device__ __forceinline__ uint32_t ld_line_u32(const char* p, uint64_t pol) {
  uint32_t v;
  if (HINT == 1)
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.b32 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  else
    asm volatile("ld.global.nc.L1::no_allocate.b32 %0, [%1];" : "=r"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ uint4 ld_row_128(const char* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

__global__ void fill_idx(int32_t* idx, int64_t n, uint32_t n_rows, uint64_t seed) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    uint64_t z = seed + (uint64_t)i * 0x9E3779B97F4A7C15ull;  // splitmix64
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    z ^= z >> 31;
    idx[i] = (int32_t)((z >> 32) % n_rows);
  }
}

__global__ void fill_bytes(uint32_t* p, int64_t n_words) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (int64_t)gridDim.x * blockDim.x)
    p[i] = (uint32_t)(i * 2654435761u);
}

struct Tables {
  const char* t[3];
};

// Slice pattern: index k -> line (table k % 3, row idx[k], slice s).  Each warp takes 32 indices at a time (one
// coalesced 128-byte index load) and gathers their lines DEPTH at a time, all loads issued before any use.
template <int DEPTH, int HINT>
__global__ void gather_slices(Tables tb, const int32_t* idx, int64_t n_idx, int slice, uint32_t* sink) {
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const size_t off = (size_t)slice * 128 + (size_t)lane * 4;
  const uint64_t first = policy_evict_first(), last = policy_evict_last();
  uint32_t acc = 0;
  for (int64_t base = warp * 32; base < n_idx; base += n_warps * 32) {
    const int my = ld_hint_i32(idx + base + lane, first);  // n_idx is a multiple of 32
#pragma unroll
    for (int j = 0; j < 32; j += DEPTH) {
      uint32_t v[DEPTH];
#pragma unroll
      for (int q = 0; q < DEPTH; ++q) {
        const int r = __shfl_sync(kFull, my, j + q);
        v[q] = ld_line_u32<HINT>(tb.t[(j + q) % 3] + (size_t)r * kRowBytes + off, last);
      }
#pragma unroll
      for (int q = 0; q < DEPTH; ++q) acc ^= v[q];
    }
  }
  if (acc == 0x9E3779B9u) sink[0] = acc;  // keeps the loads; practically never true
}

// Baseline: index k -> the whole 2 KB row idx[k] of table k % 3, 16 B per lane per load, 4 rows in flight per warp
// (16 loads per lane, as score_rank_kernel keeps for d*es = 2048).
__global__ void gather_rows(Tables tb, const int32_t* idx, int64_t n_idx, uint32_t* sink) {
  constexpr int NV = kRowBytes / 512, ROWS = 16 / NV;
  const int lane = threadIdx.x & 31;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t n_warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const uint64_t first = policy_evict_first();
  uint32_t acc = 0;
  for (int64_t base = warp * 32; base < n_idx; base += n_warps * 32) {
    const int my = ld_hint_i32(idx + base + lane, first);
#pragma unroll
    for (int j = 0; j < 32; j += ROWS) {
      uint4 v[ROWS][NV];
#pragma unroll
      for (int q = 0; q < ROWS; ++q) {
        const int r = __shfl_sync(kFull, my, j + q);
        const char* row = tb.t[(j + q) % 3] + (size_t)r * kRowBytes;
#pragma unroll
        for (int i = 0; i < NV; ++i) v[q][i] = ld_row_128(row + (size_t)(lane + 32 * i) * 16);
      }
#pragma unroll
      for (int q = 0; q < ROWS; ++q)
#pragma unroll
        for (int i = 0; i < NV; ++i) acc ^= v[q][i].x ^ v[q][i].y ^ v[q][i].z ^ v[q][i].w;
    }
  }
  if (acc == 0x9E3779B9u) sink[0] = acc;
}

static std::string shell_line(const char* cmd) {
  std::string out;
  if (FILE* f = popen(cmd, "r")) {
    char buf[512];
    while (fgets(buf, sizeof buf, f)) out += buf;
    pclose(f);
  }
  while (!out.empty() && (out.back() == '\n' || out.back() == ' ')) out.pop_back();
  for (char& c : out)
    if (c == '"' || c == '\\' || c == '\n') c = ' ';
  return out.empty() ? "unknown" : out;
}

// CTAs of `threads` threads that fit on one SM
template <typename K>
static int ctas_per_sm(K kernel, int threads) {
  int n = 0;
  CHECK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, kernel, threads, 0));
  return n;
}

// median over `reps` timed launches (after one untimed launch that fills L2 with the working set)
template <typename F>
static double time_ms(F&& launch, int reps) {
  cudaEvent_t a, b;
  CHECK(cudaEventCreate(&a));
  CHECK(cudaEventCreate(&b));
  launch();
  CHECK(cudaGetLastError());
  std::vector<float> t;
  for (int i = 0; i < reps; ++i) {
    CHECK(cudaEventRecord(a));
    launch();
    CHECK(cudaEventRecord(b));
    CHECK(cudaEventSynchronize(b));
    float ms;
    CHECK(cudaEventElapsedTime(&ms, a, b));
    t.push_back(ms);
  }
  CHECK(cudaGetLastError());
  std::sort(t.begin(), t.end());
  CHECK(cudaEventDestroy(a));
  CHECK(cudaEventDestroy(b));
  return t[t.size() / 2];
}

int main() {
  int dev = 0, sms = 0, l2 = 0;
  CHECK(cudaSetDevice(dev));
  cudaDeviceProp prop;
  CHECK(cudaGetDeviceProperties(&prop, dev));
  CHECK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  CHECK(cudaDeviceGetAttribute(&l2, cudaDevAttrL2CacheSize, dev));
  const std::string smi =
      shell_line("nvidia-smi -i 0 --query-gpu=name,power.limit,clocks.max.sm,clocks.max.mem --format=csv,noheader");

  const int64_t kMindRows = 161013;                  // MIND-large news table: slice of 3 tables = 61.8 MB
  const int64_t kMaxRows = 2600000;                  // 1 GB of slices: the DRAM reference point
  const int64_t n_idx = (int64_t)256 << 20;          // 1 GiB of indices: streamed from DRAM, not L2-resident
  const int64_t n_idx_rows = (int64_t)64 << 20;      // baseline: 64 Mi whole rows = 137 GB per launch
  const int reps = 9;

  char* tab;
  int32_t* idx;
  uint32_t* sink;
  const size_t tab_bytes = (size_t)kMaxRows * kRowBytes;
  CHECK(cudaMalloc(&tab, 3 * tab_bytes));
  CHECK(cudaMalloc(&idx, (size_t)n_idx * 4));
  CHECK(cudaMalloc(&sink, 4));
  fill_bytes<<<sms * 8, 256>>>((uint32_t*)tab, (int64_t)(3 * tab_bytes / 4));
  CHECK(cudaGetLastError());
  Tables tb{{tab, tab + tab_bytes, tab + 2 * tab_bytes}};

  printf("{\n  \"what\": \"random 128-byte line gathers from L2 (slice pattern) vs whole 2 KB rows from HBM\",\n");
  printf("  \"device\": \"%s\",\n  \"nvidia_smi\": \"%s\",\n", prop.name, smi.c_str());
  printf("  \"sms\": %d,\n  \"l2_bytes\": %d,\n  \"n_idx\": %lld,\n  \"reps\": %d,\n", sms, l2, (long long)n_idx, reps);
  printf("  \"slices\": [\n");

  const double mb_sizes[4] = {15.5, 31, 62, 124};
  bool first = true;
  double rate_62 = 0;
  for (double mb : mb_sizes) {
    const int64_t n_rows = std::min<int64_t>(kMaxRows, (int64_t)(mb * 1e6 / (3 * 128)));
    fill_idx<<<sms * 8, 256>>>(idx, n_idx, (uint32_t)n_rows, 0x1234567ull + n_rows);
    CHECK(cudaGetLastError());
    for (int wpc : {1, 2}) {
      for (int depth : {16, 32}) {
        for (int hint : {0, 1}) {
          // one wave of as many CTAs as fit (32 per SM at most): 32 resident warps, or what registers allow
          const int per_sm = depth == 16 ? (hint ? ctas_per_sm(gather_slices<16, 1>, 32 * wpc)
                                                 : ctas_per_sm(gather_slices<16, 0>, 32 * wpc))
                                         : (hint ? ctas_per_sm(gather_slices<32, 1>, 32 * wpc)
                                                 : ctas_per_sm(gather_slices<32, 0>, 32 * wpc));
          const int grid = sms * per_sm;
          auto run = [&] {
            const int s = 5;
            if (depth == 16)
              hint ? gather_slices<16, 1><<<grid, 32 * wpc>>>(tb, idx, n_idx, s, sink)
                   : gather_slices<16, 0><<<grid, 32 * wpc>>>(tb, idx, n_idx, s, sink);
            else
              hint ? gather_slices<32, 1><<<grid, 32 * wpc>>>(tb, idx, n_idx, s, sink)
                   : gather_slices<32, 0><<<grid, 32 * wpc>>>(tb, idx, n_idx, s, sink);
          };
          const double ms = time_ms(run, reps);
          const double line_gbs = (double)n_idx * 128 / (ms * 1e6);
          const double idx_gbs = (double)n_idx * 4 / (ms * 1e6);
          if (mb == 62) rate_62 = std::max(rate_62, line_gbs);
          printf("%s    {\"slice_mb\": %.1f, \"n_rows\": %lld, \"warps_per_sm\": %d, \"lines_in_flight_per_warp\": %d, "
                 "\"l2_hint\": \"%s\", \"ms\": %.4f, \"line_gbs\": %.1f, \"index_gbs\": %.1f}",
                 first ? "" : ",\n", 3 * n_rows * 128 / 1e6, (long long)n_rows, per_sm * wpc, depth,
                 hint ? "evict_last" : "none", ms, line_gbs, idx_gbs);
          first = false;
          fflush(stdout);
        }
      }
    }
  }
  printf("\n  ],\n");

  // finer curve at the best configuration above, up to a slice set 8x the L2 (served from DRAM)
  printf("  \"curve_32_warps_16_in_flight\": [\n");
  first = true;
  for (double mb : {15.5, 20.0, 25.0, 31.0, 40.0, 50.0, 62.0, 80.0, 124.0, 250.0, 998.0}) {
    const int64_t n_rows = std::min<int64_t>(kMaxRows, (int64_t)(mb * 1e6 / (3 * 128)));
    fill_idx<<<sms * 8, 256>>>(idx, n_idx, (uint32_t)n_rows, 0x2345678ull + n_rows);
    CHECK(cudaGetLastError());
    const int grid = sms * ctas_per_sm(gather_slices<16, 0>, 32);
    const double ms = time_ms([&] { gather_slices<16, 0><<<grid, 32>>>(tb, idx, n_idx, 5, sink); }, reps);
    printf("%s    {\"slice_mb\": %.1f, \"n_rows\": %lld, \"ms\": %.4f, \"line_gbs\": %.1f}", first ? "" : ",\n",
           3 * n_rows * 128 / 1e6, (long long)n_rows, ms, (double)n_idx * 128 / (ms * 1e6));
    first = false;
    fflush(stdout);
  }
  printf("\n  ],\n");

  // baseline: today's pattern, whole rows of the three 0.99 GB tables
  fill_idx<<<sms * 8, 256>>>(idx, n_idx_rows, (uint32_t)kMindRows, 0x7654321ull);
  CHECK(cudaGetLastError());
  Tables tb_rows{{tab, tab + (size_t)kMindRows * kRowBytes, tab + 2 * (size_t)kMindRows * kRowBytes}};
  printf("  \"whole_rows\": [\n");
  first = true;
  for (int wpc : {1, 2}) {
    const int per_sm = ctas_per_sm(gather_rows, 32 * wpc);
    const int grid = sms * per_sm;
    const double ms = time_ms([&] { gather_rows<<<grid, 32 * wpc>>>(tb_rows, idx, n_idx_rows, sink); }, reps);
    printf("%s    {\"tables_gb\": %.3f, \"warps_per_sm\": %d, \"ms\": %.4f, \"row_gbs\": %.1f}", first ? "" : ",\n",
           3.0 * kMindRows * kRowBytes / 1e9, per_sm * wpc, ms, (double)n_idx_rows * kRowBytes / (ms * 1e6));
    first = false;
  }
  printf("\n  ],\n");
  // score/rank bytes of one bench step (2*sum(H) + sum(C) rows of 2 KB): 438.6 GB
  printf("  \"best_line_gbs_at_62mb\": %.1f,\n  \"predicted_score_kernel_ms\": %.1f\n}\n", rate_62,
         438.6e9 / (rate_62 * 1e6));
  CHECK(cudaFree(tab));
  CHECK(cudaFree(idx));
  CHECK(cudaFree(sink));
  return 0;
}
