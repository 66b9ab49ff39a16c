// Dense row kernel on the 5th-gen tensor cores:  y = epilogue(a[M,K] @ w[N,K]^T + bias).
//
// This is the torch.nn.Linear contraction of the reference (latent_attention.py:65-74,33-37;
// modeling_utils.py:218-222), bf16 operands, fp32 accumulation, with the op that FOLLOWS the Linear in
// the reference fused into the epilogue: ReLU / exp (FinalAttention), residual add, GEGLU with erf-GELU
// (FeedForward), and the per-head softmax over the latents (SDPA, latent_attention.py:69-72).
//
// B200 design (one CTA per SM, persistent over output tiles, warp specialised, 384 threads):
//   warp 0    : TMA producer -- cp.async.bulk.tensor 2-D tiles of A (128x64) and W (BNx64) into a
//               ring of 128B-swizzled shared-memory stages, mbarrier complete_tx.
//   warp 1    : MMA issuer   -- one thread issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16)
//               on UMMA smem descriptors; fp32 accumulators live in TMEM, double buffered (2 x BN columns)
//               so the epilogue of tile i overlaps the mainloop of tile i+1; tcgen05.commit frees smem
//               stages and publishes accumulators.
//   warp 2    : TMEM allocator.
//   warp 3    : all-gather carrier -- when a push job is attached (row-sharded table build) it streams finished
//               rows of the PREVIOUS chunk to every rank's table with NVLink multicast stores (multimem.st),
//               so the collective overlaps the tensor-core work inside the same kernel.
//   warps 4-11: epilogue     -- two warps per TMEM lane quadrant, 128 accumulator columns each:
//               tcgen05.ld (32 lanes x 32 columns) -> registers -> fused math -> either
//                 * bf16 outputs: 128B-swizzled staging tile in smem -> TMA store (coalesced, async), or
//                 * fp32 outputs: 128-bit global stores.
//   softmax   : a softmax row (one head, Lp latents) spans Lp/256 N-tiles.  Those tiles are computed at the
//               same time by the CTAs of one thread-block CLUSTER; the per-row (max, sum) statistics are
//               exchanged through distributed shared memory (st.shared::cluster + remote mbarrier arrive),
//               so probabilities are normalised with the exact row statistics before their single bf16
//               rounding and P never exists in fp32 in HBM.
#include "common.cuh"
#include "dense.cuh"
#include "ptx.cuh"

#include <algorithm>
#include <mutex>

namespace nrb {

constexpr int kBM = 128;
constexpr int kBK = 64;  // 64 bf16 = 128 bytes = one swizzle-128B row
constexpr int kUmmaK = 16;
constexpr int kCtrlWarps = 4;  // TMA, MMA, TMEM-alloc, spare
constexpr int kEpiWarps = 8;
constexpr int kGemmThreads = (kCtrlWarps + kEpiWarps) * 32;
constexpr int kGroupBytes = kBM * 128;  // one 128-row x 64-column bf16 staging group (swizzle-128B)
constexpr int kMaxCluster = 4;  // softmax groups up to 4 x 256 = 1024 columns
constexpr int kSmemLimit = 232448;  // 227 KB opt-in limit per CTA
constexpr int kTopkMaxK = 32;       // NRB_EPI_TOPK: longest list an epilogue thread keeps (8-byte entries in smem)

template <int BN, int EPI, bool OUT_BF16, int CG = 1>
struct GemmCfg {
  static_assert(CG == 1 || (CG == 2 && BN == 256 && EPI != NRB_EPI_SOFTMAX), "CTA pairs: 256-wide tiles, no softmax");
  static constexpr bool kStaged = OUT_BF16;
  static constexpr bool kSoftmax = EPI == NRB_EPI_SOFTMAX;
  static constexpr bool kTopk = EPI == NRB_EPI_TOPK || EPI == NRB_EPI_TOPK_BLEND;
  static constexpr bool kBlend = EPI == NRB_EPI_TOPK_BLEND;
  // fp32 outputs: every epilogue warp transposes its 32x32 accumulator chunk through a private 4 KB smem patch so
  // that the residual loads and the output stores touch 4 rows x 128 contiguous bytes per instruction instead of
  // 32 rows x 16 bytes (GEGLU with fp32 output -- unused on the hot path -- keeps the direct row-per-lane stores)
  static constexpr bool kXpose = !OUT_BF16 && EPI != NRB_EPI_GEGLU && !kTopk;
  static constexpr int kXposeBytes = kXpose ? kEpiWarps * 4096 : 0;
  static constexpr int kHalves = BN / 128;  // epilogue column halves (128 accumulator columns each)
  static constexpr int kABytes = kBM * kBK * 2;
  static constexpr int kBBytes = (BN / CG) * kBK * 2;  // a CTA pair splits the N rows of W between its two CTAs
  static constexpr int kStageBytes = kABytes + kBBytes;
  static constexpr int kStagingBytes = kStaged ? kHalves * 2 * kGroupBytes : 0;  // double buffered per half
  static constexpr int kXchgBytes = kSoftmax ? 2 * 2 * (2 * kMaxCluster) * 128 * 4 : 0;  // [parity][m|s][participant][row]
  // top-k: one list of kTopkMaxK (score, row) entries per epilogue thread, entry j of thread t at [j][t]
  static constexpr int kListBytes = kTopk ? kTopkMaxK * kEpiWarps * 32 * 8 : 0;
  static constexpr int kFixedBytes =
      1024 /*align*/ + 512 /*barriers*/ + kStagingBytes + kXposeBytes + kXchgBytes + kListBytes;
  static constexpr int kStagesRaw = (kSmemLimit - kFixedBytes) / kStageBytes;
#ifndef NRB_MAX_STAGES
#define NRB_MAX_STAGES 6
#endif
  static constexpr int kStages = kStagesRaw > NRB_MAX_STAGES ? NRB_MAX_STAGES : kStagesRaw;
  static constexpr int kTmemCols = 2 * BN;
  static constexpr int kSmemBytes = kStages * kStageBytes + kFixedBytes;
  static_assert(kStages >= 2, "pipeline too shallow");
  static_assert(!kSoftmax || OUT_BF16, "softmax epilogue writes bf16 probabilities");
  static_assert(!kTopk || (!OUT_BF16 && BN == 256), "top-k epilogue: 256-wide tiles, no output tile");
};

struct GemmParams {
  int64_t M;         // row capacity (TMA extent); effective rows = min(M, *m_dev) when m_dev != NULL
  const int* m_dev;  // optional device-side row count (varlen token packing, no host sync)
  int N, K;
  const float* bias;
  const void* res;          // residual operand: fp32 or bf16 rows ...
  int res_dtype;            // NRB_F32 | NRB_BF16
  const int32_t* res_map;   // ... optionally gathered through a row map (varlen token packing: res = the raw input)
  int64_t ldres;
  void* y;  // direct-store epilogues only
  int64_t ldy;
  int group;        // softmax: padded group width Lp (power of two >= 32)
  int group_valid;  // softmax: valid columns per group (L <= Lp)
  int cluster;      // softmax: CTAs per cluster = max(1, Lp / 256)
  PushJob push;     // rows of an earlier result that the spare warp multicasts to every rank while the GEMM runs
  // NRB_EPI_TOPK / NRB_EPI_TOPK_BLEND, which read no other field but the shape (placed last, so that the parameter
  // offsets of every other epilogue stay as they are)
  struct TopkArgs {
    const float* scale;          // per-column 1 / max(|w_n|, 1e-8), NaN from column N up to the next multiple of 256
    const int64_t* excl_off;     // CSR offsets [M + 1] of the excluded columns of each row (NULL: nothing excluded)
    const int32_t* excl_sorted;  // the excluded columns, sorted ascending within each row
    uint2* parts;                // partial lists, 8-byte (score, column) entries [rows][2 halves][slots][k]
    int64_t slots;               // per (row, half): CTAs (pairs) whose contiguous unit range touches one row block
    int k;
    const float* base;           // blend: per-column baseline, NaN from column N up to the next multiple of 256
    const uint8_t* cold;         // blend: per row, 1 = empty history, the score is base alone
    float alpha;                 // blend: score = acc * scale * alpha + base * (1 - alpha) for the other rows
  } topk;
};

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float rcp_approx(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
constexpr float kLog2e = 1.4426950408889634f;

// ---- packed fp32 pairs (Blackwell FFMA2 / FMUL2 / FADD2: two IEEE fp32 operations per lane per instruction) ----
// The fused epilogues are bound by the FMA pipe (a 3-register FFMA issues every other cycle per SM sub-partition);
// the packed forms halve the instruction count of the polynomial / scaling work.  A pair lives in one 64-bit
// register; tcgen05.ld hands out consecutive registers, so neighbouring accumulator columns pack for free.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pack2(float lo, float hi) {
  f32x2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(f32x2 v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ f32x2 splat2(float v) { return pack2(v, v); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) {
  f32x2 d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
  return d;
}
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) {
  f32x2 d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
  return d;
}

// erf-GELU (F.gelu default, latent_attention.py:27): g * Phi(g) with Phi from the Abramowitz-Stegun 7.1.26
// erfc approximation (|abs err| <= 1.5e-7, far below the bf16 rounding of the output); the negative branch
// uses erfc directly so that there is no cancellation.
__device__ __forceinline__ float gelu_erf_fast(float g) {
  const float z = fabsf(g) * 0.70710678118654752440f;
  const float t = rcp_approx(fmaf(0.3275911f, z, 1.0f));
  float p = fmaf(t, 0.5f * 1.061405429f, 0.5f * -1.453152027f);
  p = fmaf(p, t, 0.5f * 1.421413741f);
  p = fmaf(p, t, 0.5f * -0.284496736f);
  p = fmaf(p, t, 0.5f * 0.254829592f);
  const float half_erfc = p * t * ex2_approx(z * (z * -kLog2e));  // 0.5 * erfc(|z|)
  // g * Phi(g) = relu(g) - |g| * half_erfc  (g >= 0: g(1-h); g < 0: g*h) -- no select, no cancellation
  return fmaf(-fabsf(g), half_erfc, fmaxf(g, 0.f));
}
// the same for two gates at once: a2 * gelu(g2), 12 packed FMA-pipe instructions + 4 MUFU per pair of outputs
__device__ __forceinline__ f32x2 geglu2(f32x2 a2, f32x2 g2) {
  float g0, g1;
  unpack2(g2, g0, g1);
  const f32x2 ag = pack2(fabsf(g0), fabsf(g1));
  const f32x2 z = mul2(ag, splat2(0.70710678118654752440f));
  float d0, d1;
  unpack2(fma2(splat2(0.3275911f), z, splat2(1.0f)), d0, d1);
  const f32x2 t = pack2(rcp_approx(d0), rcp_approx(d1));
  // coefficients carry -0.5: p = -0.5 * poly(t), so that the last step is one fused multiply-add
  f32x2 p = fma2(t, splat2(-0.5f * 1.061405429f), splat2(-0.5f * -1.453152027f));
  p = fma2(p, t, splat2(-0.5f * 1.421413741f));
  p = fma2(p, t, splat2(-0.5f * -0.284496736f));
  p = fma2(p, t, splat2(-0.5f * 0.254829592f));
  float e0, e1;
  unpack2(mul2(z, mul2(z, splat2(-kLog2e))), e0, e1);
  const f32x2 ex = pack2(ex2_approx(e0), ex2_approx(e1));
  const f32x2 neg_half_erfc = mul2(mul2(p, t), ex);  // -0.5 * erfc(|z|)
  const f32x2 gelu = fma2(ag, neg_half_erfc, pack2(fmaxf(g0, 0.f), fmaxf(g1, 0.f)));
  return mul2(a2, gelu);
}

// ---- shared epilogue math: 32 accumulator columns of one row -> post-activation fp32 values -------------
template <int EPI>
__device__ __forceinline__ void activate_chunk(const uint32_t (&acc)[32], const GemmParams& p, int64_t row,
                                               int col0, bool row_ok, float (&v)[32]) {
  if (p.bias != nullptr) {
#pragma unroll
    for (int j = 0; j < 32; j += 4) {
      const float4 b = *reinterpret_cast<const float4*>(p.bias + col0 + j);
      unpack2(add2(pack2(__uint_as_float(acc[j]), __uint_as_float(acc[j + 1])), pack2(b.x, b.y)), v[j], v[j + 1]);
      unpack2(add2(pack2(__uint_as_float(acc[j + 2]), __uint_as_float(acc[j + 3])), pack2(b.z, b.w)), v[j + 2],
              v[j + 3]);
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(acc[j]);
  }
  if (EPI == NRB_EPI_RELU) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = fmaxf(v[j], 0.f);
  } else if (EPI == NRB_EPI_EXP) {
#pragma unroll
    for (int j = 0; j < 32; ++j) v[j] = ex2_approx(v[j] * kLog2e);
  } else if (EPI == NRB_EPI_RESIDUAL) {
    if (row_ok) {
      const int64_t rrow = p.res_map != nullptr ? (int64_t)p.res_map[row] : row;
      if (p.res_dtype == NRB_F32) {
        const float* r = reinterpret_cast<const float*>(p.res) + rrow * p.ldres + col0;
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const float4 b = *reinterpret_cast<const float4*>(r + j);
          v[j] += b.x;
          v[j + 1] += b.y;
          v[j + 2] += b.z;
          v[j + 3] += b.w;
        }
      } else {
        const __nv_bfloat16* r = reinterpret_cast<const __nv_bfloat16*>(p.res) + rrow * p.ldres + col0;
#pragma unroll
        for (int j = 0; j < 32; j += 8) {
          const uint4 b = *reinterpret_cast<const uint4*>(r + j);
          float f[8];
          Vec16<__nv_bfloat16>::unpack(b, f);
#pragma unroll
          for (int k = 0; k < 8; ++k) v[j + k] += f[k];
        }
      }
    }
  } else if (EPI == NRB_EPI_GEGLU) {
    // W rows interleaved in pairs (a0,a1,g0,g1,a2,a3,g2,g3,...): neighbouring accumulator columns hold two values
    // or two gates, i.e. one packed operand each; 32 accumulator columns -> 16 outputs in v[0..15]
#pragma unroll
    for (int q = 0; q < 8; ++q)
      unpack2(geglu2(pack2(v[4 * q], v[4 * q + 1]), pack2(v[4 * q + 2], v[4 * q + 3])), v[2 * q], v[2 * q + 1]);
  }
}

// 16-byte chunk j (0..7) of row r inside a 128-row x 128-byte swizzle-128B staging group
__device__ __forceinline__ uint32_t stage_addr(uint32_t base, int r, int j) {
  return base + (uint32_t)r * 128u + (uint32_t)((j ^ (r & 7)) << 4);
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
// NOUT consecutive bf16 outputs of row r, starting at 16-byte chunk j0 of the staging group
template <int NOUT>
__device__ __forceinline__ void stage_values(uint32_t base, int r, int j0, const float* v) {
#pragma unroll
  for (int q = 0; q < NOUT / 8; ++q)
    st_shared_v4(stage_addr(base, r, j0 + q), pack_bf16x2(v[8 * q], v[8 * q + 1]),
                 pack_bf16x2(v[8 * q + 2], v[8 * q + 3]), pack_bf16x2(v[8 * q + 4], v[8 * q + 5]),
                 pack_bf16x2(v[8 * q + 6], v[8 * q + 7]));
}

// Position in a ring of N mbarrier-guarded buffers, and the parity of the pass over the ring it is in
template <int N>
struct Ring {
  int i = 0;
  uint32_t phase = 0;
  __device__ __forceinline__ void advance() {
    if (++i == N) {
      i = 0;
      phase ^= 1;
    }
  }
};

// The 4 x 32-column accumulator chunks of this warp's half (TMEM address taddr), each loaded while the one before it
// is worked on:
//   TmemChunks ch(taddr);
//   #pragma unroll
//   for (int c = 0; c < 4; ++c) { const uint32_t(&r)[32] = ch.wait(c, release); ... }
// wait(c) returns chunk c and starts the load of chunk c + 1.  release() runs once the last load has completed, before
// the last chunk's math: with it the epilogue hands the accumulator back to the MMA warp as early as it can.  (The
// loop body stays in the caller: as a lambda, the top-k body compiled to more registers and a longer insertion path.)
struct TmemChunks {
  uint32_t taddr;
  uint32_t rbuf[2][32];
  __device__ __forceinline__ explicit TmemChunks(uint32_t a) : taddr(a) { ptx::tmem_ld_32x32(taddr, rbuf[0]); }
  template <typename Release>
  __device__ __forceinline__ const uint32_t (&wait(int c, Release release))[32] {
    ptx::tmem_ld_wait();
    if (c + 1 < 4) ptx::tmem_ld_32x32(taddr + (uint32_t)((c + 1) * 32), rbuf[(c + 1) & 1]);  // prefetch
    if (c == 3) release();
    return rbuf[c & 1];
  }
};

// One epilogue half's two 128-row x 64-column bf16 staging buffers, filled in turn ("groups") by the half's 4 warps
// and written out by TMA stores of the half's first thread.
struct StoreGroups {
  uint8_t* base;
  int bar_id;  // named barrier of the half (128 threads)
  bool issuer;
  uint32_t gsel = 0;  // buffer of the current group
  __device__ __forceinline__ uint8_t* buf() const { return base + gsel * kGroupBytes; }
  __device__ __forceinline__ void begin() {  // the buffer used two groups ago must be drained
    if (issuer) ptx::tma_store_wait_read1();
    ptx::named_bar_sync(bar_id, 128);
  }
  __device__ __forceinline__ void end(const CUtensorMap* map, bool store, int col, int row) {
    ptx::fence_proxy_async();
    ptx::named_bar_sync(bar_id, 128);
    if (issuer) {
      if (store) ptx::tma_store_2d(map, buf(), col, row);
      ptx::tma_store_commit();  // committed even when empty: keeps the group count in step with gsel
    }
    gsel ^= 1;
  }
};

template <int BN, int EPI, bool OUT_BF16, int CG>
__global__ void __launch_bounds__(kGemmThreads, 1)
gemm_tc_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_w,
               const __grid_constant__ CUtensorMap map_y, const GemmParams p) {
  using Cfg = GemmCfg<BN, EPI, OUT_BF16, CG>;
  constexpr int kStages = Cfg::kStages;
  constexpr int kHalves = Cfg::kHalves;
  constexpr bool kGeglu = EPI == NRB_EPI_GEGLU;
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment required by the 128B swizzle atom
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  uint8_t* smem_a = smem;
  uint8_t* smem_b = smem + kStages * Cfg::kABytes;
  uint8_t* staging = smem + kStages * Cfg::kStageBytes;  // [kHalves][2][16 KB], 1024-aligned
  uint8_t* xpose = staging + Cfg::kStagingBytes;                         // [kEpiWarps][4 KB]
  float* xbuf = reinterpret_cast<float*>(xpose + Cfg::kXposeBytes);      // [2][2*kMaxCluster][128]
  uint2* topk_list = reinterpret_cast<uint2*>(xpose + Cfg::kXposeBytes + Cfg::kXchgBytes);  // [kTopkMaxK][256]
  uint64_t* bars = reinterpret_cast<uint64_t*>(xpose + Cfg::kXposeBytes + Cfg::kXchgBytes + Cfg::kListBytes);
  uint64_t* full_bar = bars;                      // [kStages] TMA -> MMA
  uint64_t* empty_bar = bars + kStages;           // [kStages] MMA -> TMA
  uint64_t* tmem_full = bars + 2 * kStages;       // [2] MMA -> epilogue
  uint64_t* tmem_empty = bars + 2 * kStages + 2;  // [2] epilogue -> MMA
  uint64_t* xbar = bars + 2 * kStages + 4;        // [2] softmax statistics exchange (max, sum)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStages + 6);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  // CS: CTAs of a cluster share one 128-row block and take neighbouring N tiles (softmax statistics exchange)
  // CG: CTA pair (cta_group::2): two neighbouring 128-row blocks, ONE N tile; tcgen05.mma spans both SMs
  const int CS = Cfg::kSoftmax ? p.cluster : 1;
  const bool clustered = CS > 1 || CG == 2;
  const uint32_t cta_rank = clustered ? ptx::cluster_ctarank() : 0;
  const uint32_t unit = clustered ? ptx::cluster_id_x() : blockIdx.x;  // scheduling unit = cluster

  const int64_t M = p.m_dev != nullptr ? min(p.M, (int64_t)*p.m_dev) : p.M;
  const TileSchedule sched(M, p.N, BN, CG, CS, clustered ? ptx::num_clusters_x() : gridDim.x);
  const int k_blocks = p.K / kBK;
  // top-k: each CTA (pair) takes one contiguous range, so that a thread's list lives across all the tiles its CTA
  // does for one row block and is written out once per (row block, CTA)
  const int64_t u_first = sched.first(unit, Cfg::kTopk), u_last = sched.end(unit, Cfg::kTopk);
  const int64_t u_step = sched.step(Cfg::kTopk);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_a);
    ptx::prefetch_tensormap(&map_w);
    if (Cfg::kStaged) ptx::prefetch_tensormap(&map_y);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < kStages; ++s) {
      ptx::mbar_init(&full_bar[s], 1);  // pair: only the leader arrives (expect_tx covers both CTAs' bytes)
      ptx::mbar_init(&empty_bar[s], 1);
    }
    for (int s = 0; s < 2; ++s) {
      ptx::mbar_init(&tmem_full[s], 1);
      ptx::mbar_init(&tmem_empty[s], 4 * kHalves * CG);  // one arrive per active epilogue warp (of both CTAs)
      ptx::mbar_init(&xbar[s], 1);  // one local expect_tx arrive per tile; the statistics arrive as st.async bytes
    }
    ptx::fence_barrier_init();
  }
  if (warp == 2) {
    ptx::tmem_alloc<CG>(tmem_slot, Cfg::kTmemCols);
    ptx::tmem_relinquish<CG>();
  }
  ptx::tc_fence_before();
  __syncthreads();
  if (clustered) ptx::cluster_sync_all();  // peers' barriers are initialised before any remote arrive
  ptx::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      Ring<kStages> s;
      for (int64_t u = u_first; u < u_last; u += u_step) {
        const int m_blk = sched.m_blk(u, cta_rank), n_blk = sched.n_blk(u, cta_rank);
        for (int kb = 0; kb < k_blocks; ++kb) {
          ptx::mbar_wait(&empty_bar[s.i], s.phase ^ 1);
          // a pair counts both CTAs' bytes on the LEADER's barrier (the peer's bytes can only be issued after the
          // stage's previous phase completed, so they are always accounted to the right phase even if they land
          // before the leader's expect_tx); each CTA loads its A tile and its 1 / CG of the W tile
          if (CG == 1 || cta_rank == 0) ptx::mbar_expect_tx(&full_bar[s.i], CG * Cfg::kStageBytes);
          ptx::tma_load_2d<CG>(smem_a + s.i * Cfg::kABytes, &map_a, &full_bar[s.i], kb * kBK, m_blk * kBM);
          ptx::tma_load_2d<CG>(smem_b + s.i * Cfg::kBBytes, &map_w, &full_bar[s.i], kb * kBK,
                               n_blk * BN + (CG == 2 ? (int)cta_rank * (BN / 2) : 0));
          s.advance();
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (lane == 0 && (CG == 1 || cta_rank == 0)) {  // pair: only the leader CTA issues
      constexpr uint32_t idesc = ptx::make_idesc_bf16(kBM * CG, BN);
      Ring<kStages> s;
      Ring<2> acc;
      for (int64_t u = u_first; u < u_last; u += u_step) {
        ptx::mbar_wait(&tmem_empty[acc.i], acc.phase ^ 1);
        ptx::tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc.i * BN);
        for (int kb = 0; kb < k_blocks; ++kb) {
          ptx::mbar_wait(&full_bar[s.i], s.phase);
          ptx::tc_fence_after();
          const uint32_t a_addr = ptx::smem_u32(smem_a + s.i * Cfg::kABytes);
          const uint32_t b_addr = ptx::smem_u32(smem_b + s.i * Cfg::kBBytes);
#pragma unroll
          for (int k = 0; k < kBK / kUmmaK; ++k) {
            const uint64_t da = ptx::make_smem_desc_sw128(a_addr + k * kUmmaK * 2);
            const uint64_t db = ptx::make_smem_desc_sw128(b_addr + k * kUmmaK * 2);
            ptx::mma_bf16_ss<CG>(tmem_d, da, db, idesc, (kb | k) != 0 ? 1u : 0u);
          }
          ptx::mma_commit<CG>(&empty_bar[s.i]);  // smem stage reusable once these MMAs retire (pair: in both CTAs)
          s.advance();
        }
        ptx::mma_commit<CG>(&tmem_full[acc.i]);  // accumulator complete (pair: both CTAs' epilogues)
        acc.advance();
      }
    }
  } else if (warp == 3) {
    // ===================== all-gather carrier (NVLS multicast stores) =====================
    if (p.push.n_seg > 0) push_job_warp(p.push, blockIdx.x, gridDim.x, lane);
  } else if (warp >= kCtrlWarps && (warp - kCtrlWarps) < 4 * kHalves) {
    // ===================== epilogue =====================
    const int e = warp - kCtrlWarps;
    const int quad = e & 3;  // == warp & 3: the TMEM lane quadrant this warp may access
    const int hf = e >> 2;   // which 128-column half of the accumulator tile
    const int r_tile = quad * 32 + lane;
    const bool issuer = (quad == 0 && lane == 0);
    StoreGroups out{staging + hf * 2 * kGroupBytes, 1 + hf, issuer};
    Ring<2> acc;
    uint32_t it = 0;
    int topk_cnt = 0;            // top-k: entries in this thread's list
    float topk_thr = -INFINITY;  // top-k: score a column must beat (the k-th best once the list is full)
    int64_t hcur = 0, hend = 0;  // top-k: cursor into this row's sorted excluded columns
    bool topk_cold = false;      // top-k blend: this row scores by the baseline alone
    // accumulator hand-back: the (leader's) MMA warp waits for every epilogue warp of the pair
    // (TMEM reads are ordered by tcgen05.fence::before_thread_sync; no memory release is needed, which spares the
    //  peer CTA a cluster-scope MEMBAR per tile)
    auto release_tmem = [&] {
      ptx::tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (CG == 2 && cta_rank != 0)
          ptx::mbar_arrive_cluster_relaxed(ptx::leader_addr(ptx::smem_u32(&tmem_empty[acc.i])));
        else
          ptx::mbar_arrive(&tmem_empty[acc.i]);
      }
    };
    for (int64_t u = u_first; u < u_last; u += u_step, ++it) {
      const int m_blk = sched.m_blk(u, cta_rank), n_blk = sched.n_blk(u, cta_rank);
      ptx::mbar_wait(&tmem_full[acc.i], acc.phase);
      ptx::tc_fence_after();
      const int64_t row = (int64_t)m_blk * kBM + r_tile;
      const bool row_ok = row < M;
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc.i * BN + hf * 128);
      const int colh = n_blk * BN + hf * 128;  // first accumulator column of this half

      if constexpr (Cfg::kSoftmax) {
        // ---------- per-head softmax over Lp columns: two TMEM passes + ONE statistics exchange ----------
        // pass A: per 32-column chunk (m_c, s_c = sum exp(x - m_c)); chunks merged to the group in registers;
        //         groups wider than this warp's 128 columns merge the (m, s) pairs of all participants
        //         (the other half of this CTA and the other CTAs of the cluster) through DSMEM.
        //         exp(x - m_c) is written back to TMEM in place of the logit (tcgen05.st).
        // pass B: p = TMEM value * 2^((m_c - M) log2e) / S: one ex2 per element, one bf16 rounding.
        const int lp = p.group, lv = p.group_valid;
        const bool masked = lv < lp;
        const bool half_ok = colh < p.N;
        float mx[4], sm[4], mcb[4];  // group max / sum, chunk-local max * log2e
        TmemChunks pass_a(taddr);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t(&r)[32] = pass_a.wait(c, [] {});
          float xv[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const bool ok = !masked || (((colh + c * 32 + j) & (lp - 1)) < lv);
            xv[j] = ok ? __uint_as_float(r[j]) : -INFINITY;
          }
          float m4[4] = {xv[0], xv[1], xv[2], xv[3]};  // 4 independent chains instead of one of length 32
#pragma unroll
          for (int j = 4; j < 32; ++j) m4[j & 3] = fmaxf(m4[j & 3], xv[j]);
          const float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
          // A chunk with no valid column (only when lp >= 64) exponentiates from 0 here, which gives exp(-inf) = 0,
          // and keeps -inf as its pass-B scale: 2^(0 - M log2e) would overflow to +inf once the group max M is below
          // about -88.7, and 0 * inf is NaN.
          const float mb = (m == -INFINITY ? 0.f : m) * kLog2e;
          f32x2 s2[2] = {splat2(0.f), splat2(0.f)};  // 4 independent chains, two per packed register
          const f32x2 l2e = splat2(kLog2e), nmb = splat2(-mb);
          uint32_t ev[32];
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            float a0, a1;
            unpack2(fma2(pack2(xv[j], xv[j + 1]), l2e, nmb), a0, a1);
            const float e0 = ex2_approx(a0), e1 = ex2_approx(a1);
            s2[(j >> 1) & 1] = add2(s2[(j >> 1) & 1], pack2(e0, e1));
            ev[j] = __float_as_uint(e0);
            ev[j + 1] = __float_as_uint(e1);
          }
          float s4[4];
          unpack2(s2[0], s4[0], s4[1]);
          unpack2(s2[1], s4[2], s4[3]);
          // exp(x - m_c) replaces the logit IN TMEM: pass B only rescales, so each element costs one ex2
          ptx::tmem_st_32x32(taddr + (uint32_t)(c * 32), ev);
          mx[c] = m;
          mcb[c] = m == -INFINITY ? -INFINITY : mb;
          sm[c] = (s4[0] + s4[1]) + (s4[2] + s4[3]);
        }
        ptx::tmem_st_wait();
        // merge (m, s) pairs: s_total = sum_c s_c * 2^((m_c - m) log2e)
        auto merge2 = [](float& ma, float& sa, float mb_, float sb_) {
          const float m = fmaxf(ma, mb_);
          const float ms = (m == -INFINITY ? 0.f : m);
          sa = sa * ex2_approx((ma - ms) * kLog2e) + sb_ * ex2_approx((mb_ - ms) * kLog2e);
          ma = m;
        };
        if (lp >= 64) {
          merge2(mx[0], sm[0], mx[1], sm[1]);
          merge2(mx[2], sm[2], mx[3], sm[3]);
          mx[1] = mx[0];
          sm[1] = sm[0];
          mx[3] = mx[2];
          sm[3] = sm[2];
        }
        if (lp >= 128) {
          merge2(mx[0], sm[0], mx[2], sm[2]);
          mx[1] = mx[2] = mx[3] = mx[0];
          sm[1] = sm[2] = sm[3] = sm[0];
        }
        if (lp >= 256) {
          const int n_part = kHalves * CS;
          const uint32_t parity = it & 1;
          const int me = (int)cta_rank * kHalves + hf;
          // (m, s) pairs travel as st.async (DSMEM) whose completion bytes are counted on the DESTINATION's
          // mbarrier: no release fence on the producer side.  Slots and barriers alternate with the tile
          // parity: a peer can reach tile it+2 (same parity) only after this thread contributed to it+1,
          // i.e. after it has read the slots of tile `it`.
          float2* xb2 = reinterpret_cast<float2*>(xbuf) + parity * (2 * kMaxCluster * 128);
          if (e == 0 && lane == 0) ptx::mbar_expect_tx(&xbar[parity], (uint32_t)(n_part * 128 * 8));
          const uint32_t slot = ptx::smem_u32(xb2 + me * 128 + r_tile);
          const uint32_t bar = ptx::smem_u32(&xbar[parity]);
          for (int c = 0; c < CS; ++c)
            ptx::st_async_v2_f32(ptx::map_to_cta(slot, c), mx[0], sm[0], ptx::map_to_cta(bar, c));
          ptx::mbar_wait(&xbar[parity], (it >> 1) & 1);
          float m = -INFINITY;
          for (int q = 0; q < n_part; ++q) m = fmaxf(m, xb2[q * 128 + r_tile].x);
          float st = 0.f;
          for (int q = 0; q < n_part; ++q) {
            const float2 ms = xb2[q * 128 + r_tile];
            st += ms.y * ex2_approx((ms.x - m) * kLog2e);
          }
          mx[0] = mx[1] = mx[2] = mx[3] = m;
          sm[0] = sm[1] = sm[2] = sm[3] = st;
        }
        TmemChunks pass_b(taddr);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t(&r)[32] = pass_b.wait(c, release_tmem);
          // p = exp(x - m_c) * 2^((m_c - M) log2e) / S   (masked columns already hold exp(-inf) = 0; a chunk with
          // no valid column has m_c = -inf, so its factor is 2^-inf = 0)
          const float f = ex2_approx(mcb[c] - mx[c] * kLog2e) / sm[c];
          float v[32];
          const f32x2 f2 = splat2(f);
#pragma unroll
          for (int j = 0; j < 32; j += 2)
            unpack2(mul2(pack2(__uint_as_float(r[j]), __uint_as_float(r[j + 1])), f2), v[j], v[j + 1]);
          if ((c & 1) == 0) out.begin();
          stage_values<32>(ptx::smem_u32(out.buf()), r_tile, (c & 1) * 4, v);
          if ((c & 1) == 1) out.end(&map_y, half_ok, colh + (c >> 1) * 64, m_blk * kBM);
        }
      } else if constexpr (Cfg::kTopk) {
        // ---------- top-k: score = acc * scale[col]; columns that beat the k-th best enter a smem list ----------
        // (blend: score = cold ? base[col] : acc * scale[col] * alpha + base[col] * (1 - alpha), a select so that a
        //  NaN user vector of an empty history cannot reach the list)
        const int k = p.topk.k;
        uint2* const list = topk_list + (e * 32 + lane);
        constexpr int kLs = kEpiWarps * 32;  // stride between a thread's entries (conflict-free: lane-contiguous)
        const int32_t* const hist = p.topk.excl_sorted;
        if (sched.starts_segment(u, u_first)) {  // a row-block segment starts: empty list, cursor to colh
          topk_cnt = 0;
          topk_thr = -INFINITY;
          hcur = hend = 0;
          if constexpr (Cfg::kBlend) topk_cold = row_ok && p.topk.cold[row] != 0;
          if (p.topk.excl_off != nullptr && row_ok) {
            int64_t lo = p.topk.excl_off[row], hi = p.topk.excl_off[row + 1];
            hend = hi;
            while (lo < hi) {
              const int64_t mid = (lo + hi) >> 1;
              if (hist[mid] < colh) lo = mid + 1; else hi = mid;
            }
            hcur = lo;
          }
        }
        // Columns reach a thread in ascending order within a segment, so a column that ties the k-th best comes
        // after it in the (score desc, column asc) order and is rejected by the strict compare; NaN never passes.
        auto consider = [&](float v, int col) {
          if (!(v > topk_thr)) return;
          if (hcur < hend) {  // the cursor only moves forward: one L2 load per excluded column crossed
            while (hcur < hend && hist[hcur] < col) ++hcur;
            if (hcur < hend && hist[hcur] == col) return;
          }
          v += 0.f;  // -0.0 -> +0.0
          int pos = topk_cnt < k ? topk_cnt : k - 1;
          while (pos > 0) {
            const uint2 prev = list[(pos - 1) * kLs];
            if (__uint_as_float(prev.x) >= v) break;
            list[pos * kLs] = prev;
            --pos;
          }
          list[pos * kLs] = make_uint2(__float_as_uint(v), (uint32_t)col);
          if (topk_cnt < k) ++topk_cnt;
          if (topk_cnt == k) topk_thr = __uint_as_float(list[(k - 1) * kLs].x);
        };
        TmemChunks ch(taddr);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t(&r)[32] = ch.wait(c, release_tmem);
          const int col0 = colh + c * 32;
          if (!row_ok || col0 >= p.N) continue;
          float v[32];
          bool any = false;
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            // scale is NaN past column N: the TMA's zero fill there never scores
            const float4 sc = *reinterpret_cast<const float4*>(p.topk.scale + col0 + j);
            v[j] = __uint_as_float(r[j]) * sc.x;
            v[j + 1] = __uint_as_float(r[j + 1]) * sc.y;
            v[j + 2] = __uint_as_float(r[j + 2]) * sc.z;
            v[j + 3] = __uint_as_float(r[j + 3]) * sc.w;
            if constexpr (Cfg::kBlend) {  // base is NaN past column N as well: cold rows never score the zero fill
              // The fused products are spelled out, and on purpose not alike: x fuses acc * alpha, y, z and w fuse
              // base * (1 - alpha).  That is the rounding this epilogue has always produced (the compiler used to
              // pick it, and its pick changes with the code around it); one form for all four lanes would change
              // scores in the last bit.
              const float4 b = *reinterpret_cast<const float4*>(p.topk.base + col0 + j);
              const float a = p.topk.alpha, oma = 1.0f - p.topk.alpha;
              v[j] = topk_cold ? b.x : __fmaf_rn(v[j], a, __fmul_rn(b.x, oma));
              v[j + 1] = topk_cold ? b.y : __fmaf_rn(b.y, oma, __fmul_rn(v[j + 1], a));
              v[j + 2] = topk_cold ? b.z : __fmaf_rn(b.z, oma, __fmul_rn(v[j + 2], a));
              v[j + 3] = topk_cold ? b.w : __fmaf_rn(b.w, oma, __fmul_rn(v[j + 3], a));
            }
            any |= (v[j] > topk_thr) | (v[j + 1] > topk_thr) | (v[j + 2] > topk_thr) | (v[j + 3] > topk_thr);
          }
          if (any) {  // rare once the list is full
#pragma unroll
            for (int j = 0; j < 32; ++j) consider(v[j], col0 + j);
          }
        }
        // segment ends (row block changes or the range ends): write the list out, padded with (NaN, -1)
        if (sched.ends_segment(u, u_last) && row_ok) {
          const int64_t slot = (int64_t)unit - sched.first_owner(u / sched.n_per_row);
          uint2* dst = p.topk.parts + ((row * 2 + hf) * p.topk.slots + slot) * k;
          for (int j = 0; j < k; ++j)
            dst[j] = j < topk_cnt ? list[j * kLs] : make_uint2(0x7fc00000u, 0xffffffffu);
        }
      } else if constexpr (Cfg::kStaged) {
        // ---------- element-wise epilogue, bf16 output through smem + TMA store ----------
        TmemChunks ch(taddr);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t(&r)[32] = ch.wait(c, release_tmem);
          const int col0 = colh + c * 32;
          const bool active = col0 < p.N;  // uniform across the half
          float v[32];
          if (active) activate_chunk<EPI>(r, p, row, col0, row_ok, v);
          constexpr int kChunksPerGroup = kGeglu ? 4 : 2;  // accumulator chunks that fill one 64-column group
          const int cg = c % kChunksPerGroup;
          if (cg == 0) out.begin();
          if (active) {
            if (kGeglu)
              stage_values<16>(ptx::smem_u32(out.buf()), r_tile, cg * 2, v);
            else
              stage_values<32>(ptx::smem_u32(out.buf()), r_tile, cg * 4, v);
          }
          if (cg == kChunksPerGroup - 1) {
            const int out_col = kGeglu ? (colh >> 1) : (colh + (c / 2) * 64);
            out.end(&map_y, out_col < (kGeglu ? (p.N >> 1) : p.N), out_col, m_blk * kBM);
          }
        }
      } else if constexpr (Cfg::kXpose) {
        // ---------- element-wise epilogue, fp32 output, coalesced through a per-warp smem transpose ----------
        // phase 1: lane = accumulator row; (acc + bias, activation) -> 8 x 16 B into row `lane` of the warp's patch
        //          (16-byte chunk j of row r sits at j ^ (r & 7): conflict-free for both phases)
        // phase 2: lane = (row 4i + lane/8, chunk lane%8): LDS.128 + residual LDG.128 + add + STG.128, i = 0..7
        //          -> a warp instruction covers 4 rows x 128 contiguous bytes
        const uint32_t patch = ptx::smem_u32(xpose + e * 4096);
        const int sub_row = lane >> 3, chunk16 = lane & 7;
        const int64_t row0 = (int64_t)m_blk * kBM + quad * 32;
        TmemChunks ch(taddr);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t(&r)[32] = ch.wait(c, release_tmem);
          const int col0 = colh + c * 32;
          if (col0 >= p.N) continue;  // warp-uniform
          // residual rows of phase 2 are requested first: their latency hides behind phase 1
          uint4 rres[8];
          if (EPI == NRB_EPI_RESIDUAL) {
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int64_t rr = row0 + 4 * i + sub_row;
              rres[i] = make_uint4(0, 0, 0, 0);
              if (rr < M) {
                const int64_t rrow = p.res_map != nullptr ? (int64_t)p.res_map[rr] : rr;
                if (p.res_dtype == NRB_F32) {
                  rres[i] = ldg_stream_128(reinterpret_cast<const float*>(p.res) + rrow * p.ldres + col0 + chunk16 * 4);
                } else {
                  const uint2 h = *reinterpret_cast<const uint2*>(reinterpret_cast<const __nv_bfloat16*>(p.res) +
                                                                  rrow * p.ldres + col0 + chunk16 * 4);
                  rres[i] = make_uint4(h.x << 16, h.x & 0xffff0000u, h.y << 16, h.y & 0xffff0000u);
                }
              }
            }
          }
          float v[32];
          activate_chunk<EPI == NRB_EPI_RESIDUAL ? NRB_EPI_NONE : EPI>(r, p, row, col0, row_ok, v);
          __syncwarp();  // the previous chunk's phase-2 reads of the patch are complete
#pragma unroll
          for (int j = 0; j < 8; ++j)
            st_shared_v4(patch + (uint32_t)lane * 128u + (uint32_t)((j ^ (lane & 7)) << 4), __float_as_uint(v[4 * j]),
                         __float_as_uint(v[4 * j + 1]), __float_as_uint(v[4 * j + 2]), __float_as_uint(v[4 * j + 3]));
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rl = 4 * i + sub_row;
            const int64_t rr = row0 + rl;
            uint4 a;
            asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];"
                         : "=r"(a.x), "=r"(a.y), "=r"(a.z), "=r"(a.w)
                         : "r"(patch + (uint32_t)rl * 128u + (uint32_t)((chunk16 ^ (rl & 7)) << 4)));
            float4 o = make_float4(__uint_as_float(a.x), __uint_as_float(a.y), __uint_as_float(a.z), __uint_as_float(a.w));
            if (EPI == NRB_EPI_RESIDUAL) {
              o.x += __uint_as_float(rres[i].x);
              o.y += __uint_as_float(rres[i].y);
              o.z += __uint_as_float(rres[i].z);
              o.w += __uint_as_float(rres[i].w);
            }
            if (rr < M) *reinterpret_cast<float4*>(reinterpret_cast<float*>(p.y) + rr * p.ldy + col0 + chunk16 * 4) = o;
          }
        }
      } else {
        // ---------- element-wise epilogue, fp32 output with 128-bit global stores (GEGLU + fp32 only) ----------
        TmemChunks ch(taddr);
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const uint32_t(&r)[32] = ch.wait(c, release_tmem);
          const int col0 = colh + c * 32;
          if (col0 >= p.N || !row_ok) continue;  // col0 >= p.N: warp-uniform
          float v[32];
          activate_chunk<EPI>(r, p, row, col0, row_ok, v);
          float* y = reinterpret_cast<float*>(p.y) + row * p.ldy + (col0 >> 1);
#pragma unroll
          for (int j = 0; j < 16; j += 4)
            *reinterpret_cast<float4*>(y + j) = make_float4(v[j], v[j + 1], v[j + 2], v[j + 3]);
        }
      }
      acc.advance();
    }
    if (Cfg::kStaged && issuer) ptx::tma_store_wait_all();
  }

  ptx::tc_fence_before();
  __syncthreads();
  if (clustered) ptx::cluster_sync_all();  // no CTA may exit while a peer can still touch its smem / TMEM
  if (warp == 2) {
    ptx::tc_fence_after();
    ptx::tmem_dealloc<CG>(tmem_base, Cfg::kTmemCols);
  }
}

// ---- host side ---------------------------------------------------------------------------

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(sym);
  });
  return fn;
}

// 2-D bf16 row-major [rows, cols] with leading dimension ld (elements); box = [box_rows, 64 cols], 128B swizzle.
int make_tmap_bf16(CUtensorMap* map, const void* ptr, int64_t rows, int64_t cols, int64_t ld, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled unavailable (no CUDA driver?)");
    return NRB_E_CUDA;
  }
  NRB_REQUIRE((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "TMA operand must be 16-byte aligned");
  NRB_REQUIRE((ld * 2) % 16 == 0, "TMA operand leading dimension must be a multiple of 8 elements");
  cuuint64_t gdim[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t gstr[1] = {(cuuint64_t)(ld * 2)};
  cuuint32_t box[2] = {(cuuint32_t)kBK, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(ptr), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows=%lld cols=%lld ld=%lld)", (int)r,
              (long long)rows, (long long)cols, (long long)ld);
    return NRB_E_CUDA;
  }
  return NRB_OK;
}

template <int BN, int EPI, bool OUT_BF16, int CG = 1>
static int launch_gemm(const CUtensorMap& ma, const CUtensorMap& mw, const CUtensorMap& my, const GemmParams& p,
                       cudaStream_t st) {
  using Cfg = GemmCfg<BN, EPI, OUT_BF16, CG>;
  auto kern = gemm_tc_kernel<BN, EPI, OUT_BF16, CG>;
  // function attributes are per device: one flag per (kernel instantiation, device)
  static bool attr_set[64] = {};
  int dev = 0;
  NRB_CUDA_CHECK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64 || !attr_set[dev]) {
    NRB_CUDA_CHECK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    if (dev >= 0 && dev < 64) attr_set[dev] = true;
  }
  const int n_split = Cfg::kSoftmax ? p.cluster : 1;  // CTAs of a softmax cluster split the N tiles of a unit
  const int cs = CG * n_split;                         // CTAs per scheduling unit
  int max_units = sm_count_cached() / cs;
  if (cs > 1 || Cfg::kSoftmax) {  // softmax always launches as a cluster (st.async / mapa need one, even of size 1)
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(kGemmThreads);
    cfg.dynamicSmemBytes = Cfg::kSmemBytes;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = cs;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    // A persistent kernel must not ask for more clusters than can be co-resident: the GPCs hold 16 / 18 / 20 SMs, so
    // clusters of 4 fit 33 times (132 SMs), not 148 / 4 = 37 -- the 4 surplus clusters would run as a second wave
    // after the first one has finished all of its tiles (cluster-of-4 softmax: 517 -> ~1000 TFLOP/s).
    static int max_clusters[64][9] = {};
    if (cs > 2 && dev >= 0 && dev < 64 && cs <= 8) {
      if (max_clusters[dev][cs] == 0) {
        cfg.gridDim = dim3(max_units * cs);
        int n = 0;
        if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) != cudaSuccess || n <= 0) {
          (void)cudaGetLastError();
          n = max_units;
        }
        max_clusters[dev][cs] = n;
      }
      max_units = std::min(max_units, max_clusters[dev][cs]);
    }
    cfg.gridDim = dim3((int)TileSchedule(p.M, p.N, BN, CG, n_split, max_units).n_ctas * cs);
    NRB_CUDA_CHECK(cudaLaunchKernelEx(&cfg, kern, ma, mw, my, p));
  } else {
    const int grid = (int)TileSchedule(p.M, p.N, BN, CG, 1, max_units).n_ctas;
    kern<<<grid, kGemmThreads, Cfg::kSmemBytes, st>>>(ma, mw, my, p);
  }
  note_launch();
  NRB_CUDA_CHECK(cudaGetLastError());
  return NRB_OK;
}

template <int BN, bool OUT_BF16, int CG = 1>
static int dispatch_epi(int epi, const CUtensorMap& ma, const CUtensorMap& mw, const CUtensorMap& my,
                        const GemmParams& p, cudaStream_t st) {
  switch (epi) {
    case NRB_EPI_NONE:
      return launch_gemm<BN, NRB_EPI_NONE, OUT_BF16, CG>(ma, mw, my, p, st);
    case NRB_EPI_RELU:
      return launch_gemm<BN, NRB_EPI_RELU, OUT_BF16, CG>(ma, mw, my, p, st);
    case NRB_EPI_EXP:
      return launch_gemm<BN, NRB_EPI_EXP, OUT_BF16, CG>(ma, mw, my, p, st);
    case NRB_EPI_RESIDUAL:
      return launch_gemm<BN, NRB_EPI_RESIDUAL, OUT_BF16, CG>(ma, mw, my, p, st);
    case NRB_EPI_GEGLU:
      return launch_gemm<BN, NRB_EPI_GEGLU, OUT_BF16, CG>(ma, mw, my, p, st);
    default:
      set_error("nrb_linear(bf16): unsupported epilogue %d", epi);
      return NRB_E_INVALID;
  }
}

// y = epi(a @ w^T + bias); a [M,K] bf16, w [N,K] bf16.
int gemm_bf16_tc(int epi, int out_dtype, const void* a, int64_t lda, const void* w, int64_t ldw, const float* bias,
                 const void* res, int64_t ldres, void* y, int64_t ldy, int64_t M, const int* m_dev, int N, int K,
                 int group, int group_valid, cudaStream_t st, int res_dtype, const int32_t* res_map) {
  NRB_REQUIRE(M > 0 && N > 0 && K > 0, "nrb_linear: empty problem");
  NRB_REQUIRE(K % kBK == 0, "nrb_linear(bf16): K must be a multiple of 64 (got %d)", K);
  NRB_REQUIRE(N % 32 == 0, "nrb_linear(bf16): N must be a multiple of 32 (got %d)", N);
  NRB_REQUIRE(out_dtype == NRB_F32 || out_dtype == NRB_BF16, "nrb_linear: bad out_dtype");
  NRB_REQUIRE(epi != NRB_EPI_RESIDUAL || res != nullptr, "nrb_linear: residual epilogue needs res");
  const int64_t ycols_align = out_dtype == NRB_BF16 ? 8 : 4;
  NRB_REQUIRE(ldy % ycols_align == 0 && (reinterpret_cast<uintptr_t>(y) & 15) == 0,
              "nrb_linear: y must be 16-byte aligned with a 16-byte multiple row pitch");
  NRB_REQUIRE(res == nullptr || (ldres % (res_dtype == NRB_BF16 ? 8 : 4) == 0 &&
                                 (reinterpret_cast<uintptr_t>(res) & 15) == 0),
              "nrb_linear: res must be 16-byte aligned");
  NRB_REQUIRE(bias == nullptr || (reinterpret_cast<uintptr_t>(bias) & 15) == 0, "nrb_linear: bias alignment");
  const bool softmax = epi == NRB_EPI_SOFTMAX;
  int cluster = 1;
  if (softmax) {
    NRB_REQUIRE(out_dtype == NRB_BF16, "nrb_linear: the softmax epilogue writes bf16");
    NRB_REQUIRE(group >= 32 && (group & (group - 1)) == 0 && group <= 256 * kMaxCluster,
                "nrb_linear: softmax group must be a power of two in [32, %d] (got %d)", 256 * kMaxCluster, group);
    NRB_REQUIRE(group_valid >= 1 && group_valid <= group, "nrb_linear: bad softmax group_valid %d", group_valid);
    NRB_REQUIRE(N % group == 0 && N % 256 == 0, "nrb_linear: softmax needs N %% group == 0 and N %% 256 == 0");
    NRB_REQUIRE(bias == nullptr, "nrb_linear: softmax epilogue takes no bias");
    cluster = group > 256 ? group / 256 : 1;
  }
  const bool small_n = N <= 128 && !softmax;
  // CTA pairs (tcgen05 cta_group::2): each SM stages only half of the W tile -> 1/3 less shared-memory
  // operand traffic per MMA
  const bool pair = !small_n && !softmax && M > kBM;
  CUtensorMap ma, mw, my;
  int rc = make_tmap_bf16(&ma, a, M, K, lda, kBM);
  if (rc != NRB_OK) return rc;
  rc = make_tmap_bf16(&mw, w, N, K, ldw, (small_n || pair) ? 128 : 256);
  if (rc != NRB_OK) return rc;
  const int n_out = epi == NRB_EPI_GEGLU ? N / 2 : N;
  if (out_dtype == NRB_BF16) {
    rc = make_tmap_bf16(&my, y, M, n_out, ldy, kBM);
    if (rc != NRB_OK) return rc;
  } else {
    my = ma;  // unused by the direct-store epilogue
  }
  GemmParams p;
  p.M = M;
  p.m_dev = m_dev;
  p.N = N;
  p.K = K;
  p.bias = bias;
  p.res = res;
  p.res_dtype = res_dtype;
  p.res_map = res_map;
  p.ldres = ldres;
  p.y = y;
  p.ldy = ldy;
  p.group = group;
  p.group_valid = group_valid;
  p.cluster = cluster;
  take_push_share(&p.push);  // a share of the pending all-gather segments rides along (nrb_push_attach)
  if (softmax) return launch_gemm<256, NRB_EPI_SOFTMAX, true>(ma, mw, my, p, st);
  if (small_n) {
    return out_dtype == NRB_BF16 ? dispatch_epi<128, true>(epi, ma, mw, my, p, st)
                                 : dispatch_epi<128, false>(epi, ma, mw, my, p, st);
  }
  if (pair) {
    return out_dtype == NRB_BF16 ? dispatch_epi<256, true, 2>(epi, ma, mw, my, p, st)
                                 : dispatch_epi<256, false, 2>(epi, ma, mw, my, p, st);
  }
  return out_dtype == NRB_BF16 ? dispatch_epi<256, true>(epi, ma, mw, my, p, st)
                               : dispatch_epi<256, false>(epi, ma, mw, my, p, st);
}

// The schedule launch_gemm gives the top-k GEMM
TopkPlan topk_plan(int64_t M, int64_t N) {
  const int cg = M > kBM ? 2 : 1;
  TopkPlan t{TileSchedule(M, (int)N, 256, cg, 1, sm_count_cached() / cg), 1};
  for (int64_t m = 0; m < t.m_blocks; ++m) t.slots = std::max(t.slots, t.last_owner(m) - t.first_owner(m) + 1);
  return t;
}

// Partial top-k lists of (a[M,K] . w[N,K]^T) * scale[N] per row, blended with base[N] when base != NULL: see
// GemmParams::TopkArgs.
int gemm_topk_tc(const void* a, int64_t lda, const void* w, int64_t ldw, const float* scale, const int64_t* excl_off,
                 const int32_t* excl_sorted, int64_t M, int N, int K, int k, const TopkPlan& plan, void* parts,
                 const float* base, const uint8_t* cold, float alpha, cudaStream_t st) {
  NRB_REQUIRE(M > 0 && N > 0 && K > 0 && K % kBK == 0, "nrb_recommend: bad GEMM shape");
  NRB_REQUIRE(k >= 1 && k <= kTopkMaxK, "nrb_recommend: k must be in [1, %d]", kTopkMaxK);
  CUtensorMap ma, mw;
  int rc = make_tmap_bf16(&ma, a, M, K, lda, kBM);
  if (rc != NRB_OK) return rc;
  rc = make_tmap_bf16(&mw, w, N, K, ldw, plan.cg == 2 ? 128 : 256);
  if (rc != NRB_OK) return rc;
  GemmParams p = {};  // no all-gather rides along: it rides on the dense row kernels only
  p.M = M;
  p.N = N;
  p.K = K;
  p.topk = {scale, excl_off, excl_sorted, static_cast<uint2*>(parts), plan.slots, k, base, cold, alpha};
  if (base != nullptr) {
    if (plan.cg == 2) return launch_gemm<256, NRB_EPI_TOPK_BLEND, false, 2>(ma, mw, ma, p, st);
    return launch_gemm<256, NRB_EPI_TOPK_BLEND, false, 1>(ma, mw, ma, p, st);
  }
  if (plan.cg == 2) return launch_gemm<256, NRB_EPI_TOPK, false, 2>(ma, mw, ma, p, st);
  return launch_gemm<256, NRB_EPI_TOPK, false, 1>(ma, mw, ma, p, st);
}

}  // namespace nrb
