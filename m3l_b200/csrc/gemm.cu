// m3l_b200 — persistent warp-specialised bf16 GEMM on tcgen05 / TMEM / TMA (sm_100a).
//
//   C[M,N] = epilogue( sum_k A[m,k] * B[n,k] )
//
// This one kernel serves every dense contraction of the VTMAE step that the reference hands to
// cuBLAS through nn.Linear (vit_pytorch Attention.to_qkv / to_out / FeedForward.net, the patch
// embedding Linear and the to_pixels / to_tactiles heads: /root/reference/models/
// pretrain_models.py:113-116,766-779,784) and their autograd dgrad / wgrad products:
//   * forward and dgrad: both operands K-major (activations [M,K]; weights [N,K], or the bf16
//     transposed shadow copy of the weight for dgrad);
//   * wgrad dW[n,k] = sum_m dY[m,n] X[m,k]: both operands MN-major (the contraction runs over
//     the token rows), split-K over the token dimension, fp32 TMA reduce-add into the grad arena.
//
// Structure (one CTA per SM, persistent over a static tile schedule):
//   warp 0      TMA producer   cp.async.bulk.tensor -> 128B-swizzled smem ring (mbarrier tx)
//   warp 1      MMA issuer     one lane issues tcgen05.mma (128 x BN x 16), fp32 accum in TMEM,
//                              tcgen05.commit frees smem stages / publishes the accumulator
//   warps 2..9  epilogue       tcgen05.ld TMEM -> registers (thread = tile row) -> math -> the
//                              thread's row of a 128B-swizzled [32 x 128 B] smem tile -> ONE TMA
//                              store (or fp32 reduce-add) per 32 x 64 sub-tile.  Residual / GELU'
//                              operands come in the same way (TMA load, prefetched one round
//                              ahead) and the result is written in place over them.
// TMEM holds two accumulators (2 x BN columns) so the epilogue of tile i overlaps the MMAs of
// tile i+1 (K is only 256 for most of these GEMMs: SURVEY.md §7.3 hard part 2).
//
// Why the epilogue looks like this (measured, profiles/r01_gemm_epilogue.md): with K = 256 a tile
// is 16 MMAs = 2048 clk of tensor work, and the previous epilogue (registers -> smem transpose ->
// ld.shared -> per-thread 16-byte global stores, residual through per-thread global loads) took
// ~3900 clk per tile per warp as one long dependent chain (LDTM -> F2FP -> STS -> LDS -> address
// math -> STG; 24 % issue utilisation), i.e. the GEMMs ran at < 50 % of the MMA rate with every
// memory pipe below 40 %.  TMA does the address generation, coalescing and bounds handling.
#include <stdlib.h>

#include "common.cuh"
#include "dropout.cuh"
#include "m3l_internal.h"

namespace m3l {

namespace {

constexpr int BM = 128;
constexpr int BK = 64;
constexpr int kNumEpiWarps = 8;
constexpr int kNumThreads = 32 * (2 + kNumEpiWarps);
constexpr int kStgTileBytes = 32 * 128;   // one staging tile: 32 rows x 128 B

// WS ("weight stationary", K <= 256): the whole [BN x K] slice of the B operand (the weight) stays
// resident in shared memory for the life of the CTA and only A tiles stream through the ring,
// which removes 2/3 of the operand traffic through the L2 -> SM path for the K = 256 GEMMs.
constexpr int kWsMaxKb = 4;
template <int BN, bool WS>
struct GemmCfg {
  static constexpr int kABytes = BM * BK * 2;
  static constexpr int kBBytes = BN * BK * 2;
  static constexpr int kStgBufs = WS ? 1 : 2;                     // staging tiles per epilogue warp
  static constexpr int kStages = WS ? (BN == 256 ? 4 : 8) : ((BN == 256) ? 3 : (BN == 128 ? 4 : 6));
  static constexpr int kStageBytes = WS ? kABytes : kABytes + kBBytes;
  static constexpr int kResidentBytes = WS ? kWsMaxKb * kBBytes : 0;
  static constexpr int kStagingBytes = kNumEpiWarps * kStgBufs * kStgTileBytes;
  static constexpr int kTmemCols = 2 * BN;
  static constexpr int kScratchBytes = WS ? 0 : 4096;             // EPI_LN_BWD: row-sum exchange between column halves
  static constexpr int kSmemBytes =
      1024 /*align slack*/ + kStages * kStageBytes + kResidentBytes + kStagingBytes + 512 + kScratchBytes;
};

struct alignas(8) GemmBarriers {
  uint64_t full[8];
  uint64_t empty[8];
  uint64_t tmem_full[2];
  uint64_t tmem_empty[2];
  uint64_t b_full;                      // WS: resident weight slice landed
  uint64_t side_full[kNumEpiWarps][2];  // per epilogue warp: residual / aux tile landed
  uint32_t tmem_base;
};
static_assert(sizeof(GemmBarriers) <= 512, "barrier block");

// Epilogue flavours (compile time, so the inner loops carry no mode branches):
enum : int {
  EPI_BF16 = 0,      // out bf16 = acc (+ bias) (+ residual)
  EPI_GELU_FWD = 1,  // out bf16 = GELU(acc + bias) ; aux_out bf16 = GELU'(acc + bias)
  EPI_GELU_BWD = 2,  // out bf16 = acc * aux_in   (aux_in = the stored GELU')
  EPI_F32 = 3,       // out fp32 = acc (+ bias)
  EPI_F32_RED = 4,   // out fp32 += acc  (TMA reduce-add, split-K)
  EPI_LN_BWD = 5,    // out bf16 = LayerNorm backward of acc (+ skip); dgamma / dbeta / dx column sums (N == BN == 256)
  // dropout (training; mask Z of dropout.cuh, row / column of the output, plane 0, site drop_site):
  EPI_GELU_DROP = 6, // out bf16 = Z o GELU(acc + bias) ; aux_out bf16 = Z o GELU'(acc + bias)
  EPI_BF16_DROP = 7, // out bf16 = residual + Z o (acc + bias) (out2: the same values)
};

// column sums over the 32 lanes of a warp: v[c] of lane l is element (row l, column c); returns, in lane l, the sum over
// the rows of column l (reduce-scatter butterfly, 31 shuffles; destroys v)
M3L_DEVINL float warp_colsum32(float (&v)[32], int lane) {
#pragma unroll
  for (int off = 16; off >= 1; off >>= 1) {
    const bool hi = (lane & off) != 0;
#pragma unroll
    for (int i = 0; i < off; ++i) {
      const float send = hi ? v[i] : v[i + off];
      const float keep = hi ? v[i + off] : v[i];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  return v[0];
}

// ---- staging tile: 32 rows x 128 B, 16-byte chunks XOR-swizzled by (row & 7) == SWIZZLE_128B ------
// thread `lane` owns row `lane` (this is how tcgen05.ld hands out the accumulator); bank-conflict free.
M3L_DEVINL void stg_store_row(uint32_t stg, int lane, const uint32_t* w) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t addr = stg + lane * 128 + ((j ^ (lane & 7)) << 4);
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(w[4 * j]), "r"(w[4 * j + 1]),
                 "r"(w[4 * j + 2]), "r"(w[4 * j + 3])
                 : "memory");
  }
}
M3L_DEVINL void stg_load_row(uint32_t stg, int lane, uint32_t* w) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const uint32_t addr = stg + lane * 128 + ((j ^ (lane & 7)) << 4);
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(w[4 * j]), "=r"(w[4 * j + 1]), "=r"(w[4 * j + 2]), "=r"(w[4 * j + 3])
                 : "r"(addr)
                 : "memory");
  }
}
// 32-bit word `lane` (= bf16 columns 2*lane, 2*lane+1) of row r: one conflict-free column read
M3L_DEVINL uint32_t stg_load_word(uint32_t stg, int lane, int r) {
  const uint32_t addr = stg + r * 128 + ((((lane >> 2) ^ (r & 7))) << 4) + ((lane & 3) << 2);
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
  return v;
}

// Static tile schedule of one CTA (identical in the producer, MMA and epilogue roles).
//   streaming : items blockIdx.x, +gridDim.x, ... over (m tile, n tile, split), n fastest
//   WS        : the CTA owns n tile (blockIdx.x % tiles_n) and walks m tiles q, q + G, ...
struct TileSched {
  int tiles_n, splits, count, first, step, n_fixed;
  bool ws;
  M3L_DEVINL void get(int i, int BN_, int* m0, int* n0, int* split) const {
    const int item = first + i * step;
    if (ws) {
      *m0 = item * BM; *n0 = n_fixed * BN_; *split = 0;
    } else {
      *split = item % splits;
      const int t = item / splits;
      *n0 = (t % tiles_n) * BN_;
      *m0 = (t / tiles_n) * BM;
    }
  }
};

template <int BN, bool A_MN, bool B_MN, int EPI, bool WS>
__global__ void __launch_bounds__(kNumThreads, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                 const __grid_constant__ CUtensorMap map_out, const __grid_constant__ CUtensorMap map_aux,
                 const __grid_constant__ CUtensorMap map_side, const GemmArgs p) {
  static_assert(!WS || (!A_MN && !B_MN), "weight-stationary mode is for K-major operands");
  using Cfg = GemmCfg<BN, WS>;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* resident = smem + Cfg::kStages * Cfg::kStageBytes;      // WS: [kb][BN x 64] weight slice
  uint8_t* staging = resident + Cfg::kResidentBytes;
  GemmBarriers* bars = reinterpret_cast<GemmBarriers*>(staging + Cfg::kStagingBytes);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  const int tiles_n = (p.N + BN - 1) / BN;
  const int tiles_m = (p.M + BM - 1) / BM;
  const int kb_total = (p.K + BK - 1) / BK;
  const int kb_per_split = (kb_total + p.splits - 1) / p.splits;
  TileSched sched;
  sched.tiles_n = tiles_n; sched.splits = p.splits; sched.ws = WS;
  if (WS) {
    const int n_idx = blockIdx.x % tiles_n, q = blockIdx.x / tiles_n;
    const int group = ((int)gridDim.x - n_idx + tiles_n - 1) / tiles_n;   // CTAs that own this n tile
    sched.n_fixed = n_idx; sched.first = q; sched.step = group;
    sched.count = q < tiles_m ? (tiles_m - q + group - 1) / group : 0;
  } else {
    const int num_items = tiles_m * tiles_n * p.splits;
    sched.n_fixed = 0; sched.first = blockIdx.x; sched.step = gridDim.x;
    sched.count = (int)blockIdx.x < num_items
                      ? (num_items - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  }

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_a);
    tma_prefetch_desc(&map_b);
    tma_prefetch_desc(&map_out);
    constexpr bool kPlain = EPI == EPI_BF16 || EPI == EPI_BF16_DROP;
    if (EPI == EPI_GELU_FWD || EPI == EPI_GELU_DROP || (kPlain && p.out2 != nullptr)) tma_prefetch_desc(&map_aux);
    if (EPI == EPI_GELU_BWD || kPlain || EPI == EPI_LN_BWD) tma_prefetch_desc(&map_side);
    if (EPI == EPI_LN_BWD) tma_prefetch_desc(&map_aux);
    for (int s = 0; s < Cfg::kStages; ++s) {
      mbar_init(&bars->full[s], 1);
      mbar_init(&bars->empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&bars->tmem_full[b], 1);
      mbar_init(&bars->tmem_empty[b], kNumEpiWarps);
    }
    mbar_init(&bars->b_full, 1);
    for (int w = 0; w < kNumEpiWarps; ++w) {
      mbar_init(&bars->side_full[w][0], 1);
      mbar_init(&bars->side_full[w][1], 1);
    }
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&bars->tmem_base, Cfg::kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_base;
  pdl_wait();      // prologue above overlapped the predecessor kernel; global memory from here on
  pdl_trigger();

  if (warp == 0) {
    // ------------------------------- TMA producer ---------------------------------------
    if (elect_one()) {      // single issuing thread; elect (not lane == 0) keeps TMA / MMA operands in uniform registers
      int stage = 0;
      uint32_t phase = 0;
      if (WS && sched.count > 0) {
        mbar_arrive_expect_tx(&bars->b_full, kb_total * Cfg::kBBytes);
        for (int kb = 0; kb < kb_total; ++kb)
          tma_load_2d(resident + kb * Cfg::kBBytes, &map_b, &bars->b_full, kb * BK, sched.n_fixed * BN);
      }
      for (int i = 0; i < sched.count; ++i) {
        int m0, n0, split;
        sched.get(i, BN, &m0, &n0, &split);
        const int kb0 = split * kb_per_split;
        const int kb1 = min(kb0 + kb_per_split, kb_total);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&bars->empty[stage], phase ^ 1);
          uint8_t* sa = smem + stage * Cfg::kStageBytes;
          uint8_t* sb = sa + Cfg::kABytes;
          mbar_arrive_expect_tx(&bars->full[stage], Cfg::kStageBytes);
          if (!A_MN) {
            tma_load_2d(sa, &map_a, &bars->full[stage], kb * BK, m0);
          } else {
#pragma unroll
            for (int j = 0; j < BM / 64; ++j)
              tma_load_2d(sa + j * 8192, &map_a, &bars->full[stage], m0 + 64 * j, kb * BK);
          }
          if (WS) {
            // weight slice already resident
          } else if (!B_MN) {
            tma_load_2d(sb, &map_b, &bars->full[stage], kb * BK, n0);
          } else {
#pragma unroll
            for (int j = 0; j < BN / 64; ++j)
              tma_load_2d(sb + j * 8192, &map_b, &bars->full[stage], n0 + 64 * j, kb * BK);
          }
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer -----------------------------------------
    if (elect_one()) {      // single issuing thread; elect (not lane == 0) keeps TMA / MMA operands in uniform registers
      constexpr uint32_t idesc = umma_idesc_bf16(BM, BN, A_MN ? 1 : 0, B_MN ? 1 : 0);
      int stage = 0;
      uint32_t phase = 0;
      if (WS && sched.count > 0) mbar_wait(&bars->b_full, 0);
      for (int it = 0; it < sched.count; ++it) {
        int m0, n0, split;
        sched.get(it, BN, &m0, &n0, &split);
        const int kb0 = split * kb_per_split;
        const int kb1 = min(kb0 + kb_per_split, kb_total);
        const int buf = it & 1;
        const uint32_t acc_phase = (it >> 1) & 1;
        mbar_wait(&bars->tmem_empty[buf], acc_phase ^ 1);
        tc_fence_after_sync();
        const uint32_t tmem_d = tmem_base + buf * BN;
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&bars->full[stage], phase);
          tc_fence_after_sync();
          const uint32_t a_addr = smem_u32(smem + stage * Cfg::kStageBytes);
          const uint32_t b_addr = WS ? smem_u32(resident + kb * Cfg::kBBytes) : a_addr + Cfg::kABytes;
#pragma unroll
          for (int k = 0; k < BK / 16; ++k) {
            const uint64_t adesc = A_MN ? umma_smem_desc(a_addr + k * 2048, 8192, 1024)
                                        : umma_smem_desc(a_addr + k * 32, 16, 1024);
            const uint64_t bdesc = B_MN ? umma_smem_desc(b_addr + k * 2048, 8192, 1024)
                                        : umma_smem_desc(b_addr + k * 32, 16, 1024);
            umma_bf16(tmem_d, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          umma_commit(&bars->empty[stage]);
          if (++stage == Cfg::kStages) { stage = 0; phase ^= 1; }
        }
        umma_commit(&bars->tmem_full[buf]);
      }
    }
  } else if constexpr (EPI == EPI_LN_BWD) {
    // ------------------------------- epilogue: fused LayerNorm backward ------------------
    // The accumulator tile holds dy = grad w.r.t. LayerNorm's output for 128 FULL rows (BN == N == 256).  Per row
    //   g = dy * gamma,  xhat = (x - mean) * rstd,  dx = rstd * (g - mean_j(g) - xhat * mean_j(g * xhat)) + skip
    // thread = row; a warp owns 32 rows x one 128-column half, in two rounds of 64 columns.  Pass 1 forms the two row
    // sums (the halves meet through 8 bytes of shared memory per row), pass 2 re-reads the accumulator from tensor memory
    // and x through TMA, writes dx in place over the skip tile and stores it with TMA; dgamma / dbeta / column sums of dx
    // come from register butterflies (no staging).  With K = 768 / 1024 the products of a tile take 6 - 8 k clk, the
    // epilogue is hidden behind them: the separate LayerNorm-backward kernel (29 us, six per step) and the dy round
    // trip through HBM disappear.
    const int ew = warp - 2;
    const int quad = warp & 3;
    const int col_half = ew >> 2;
    const int span0 = col_half * 128;
    const uint32_t stg = smem_u32(staging + ew * 2 * kStgTileBytes);
    float2* scratch = reinterpret_cast<float2*>(reinterpret_cast<uint8_t*>(bars) + 512);     // [2][4 quads][2 halves][32]
    const bool has_skip = p.ln_skip != nullptr;
    uint32_t uses0 = 0, uses1 = 0;                       // completed phases of side_full[ew][0 / 1]
    auto load_side = [&](int b, const CUtensorMap* map, int col, int row) {      // elected lane
      mbar_arrive_expect_tx(&bars->side_full[ew][b], kStgTileBytes);
      tma_load_2d_u32(stg + b * kStgTileBytes, map, &bars->side_full[ew][b], col, row);
    };
    float acc_g[4] = {0.f, 0.f, 0.f, 0.f}, acc_b[4] = {0.f, 0.f, 0.f, 0.f}, acc_c[4] = {0.f, 0.f, 0.f, 0.f};
    for (int it = 0; it < sched.count; ++it) {
      int m0, n0, split;
      sched.get(it, BN, &m0, &n0, &split);
      const int row0 = m0 + quad * 32;
      const int my_row = row0 + lane;
      const bool in = my_row < p.M;
      float mean = 0.f, rstd = 0.f;
      if (in) {
        const float2 ms = __ldg(reinterpret_cast<const float2*>(p.ln_stats) + my_row);
        mean = ms.x; rstd = ms.y;
      }
      // x tiles of both rounds (buffer 1 may still be read by the previous tile's last dx store)
      if (elect_one()) {
        load_side(0, &map_side, span0, row0);
        tma_wait_group_read<0>();
        fence_proxy_async_smem();
        load_side(1, &map_side, span0 + 64, row0);
      }
      __syncwarp();
      const int buf = it & 1;
      mbar_wait(&bars->tmem_full[buf], (it >> 1) & 1);
      tc_fence_after_sync();
      const uint32_t t_acc = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * BN + span0;
      // ---------------- pass 1: row sums
      float s1 = 0.f, s2 = 0.f;
#pragma unroll 1
      for (int r = 0; r < 2; ++r) {
        uint32_t v[64], w[32];
        tmem_ld_32x32(t_acc + r * 64, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
        tmem_ld_32x32(t_acc + r * 64 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
        if (r == 0) { mbar_wait(&bars->side_full[ew][0], uses0 & 1); ++uses0; }
        else { mbar_wait(&bars->side_full[ew][1], uses1 & 1); ++uses1; }
        stg_load_row(stg + r * kStgTileBytes, lane, w);
        __syncwarp();                                  // every lane has its x row of this buffer in registers
        if (elect_one()) {                             // pass 2, round 0: x again into buffer 0, skip into buffer 1
          fence_proxy_async_smem();
          if (r == 0) load_side(0, &map_side, span0, row0);
          else if (has_skip) load_side(1, &map_aux, span0, row0);
        }
        tmem_ld_wait();
#pragma unroll
        for (int j = 0; j < 64; j += 4) {
          const float4 gm = __ldg(reinterpret_cast<const float4*>(p.ln_gamma + span0 + r * 64 + j));
          const float2 x01 = unpack_bf16x2(w[j >> 1]), x23 = unpack_bf16x2(w[(j >> 1) + 1]);
          const float g0 = __uint_as_float(v[j]) * gm.x, g1 = __uint_as_float(v[j + 1]) * gm.y;
          const float g2 = __uint_as_float(v[j + 2]) * gm.z, g3 = __uint_as_float(v[j + 3]) * gm.w;
          s1 += (g0 + g1) + (g2 + g3);
          s2 = fmaf(g0, (x01.x - mean) * rstd, s2);
          s2 = fmaf(g1, (x01.y - mean) * rstd, s2);
          s2 = fmaf(g2, (x23.x - mean) * rstd, s2);
          s2 = fmaf(g3, (x23.y - mean) * rstd, s2);
        }
      }
      // the two column halves of a row meet (parity-double-buffered scratch: one barrier per tile suffices)
      float2* my_slot = scratch + (((it & 1) * 4 + quad) * 2 + col_half) * 32 + lane;
      *my_slot = make_float2(s1, s2);
      named_bar_sync(1 + quad, 64);
      const float2 other = scratch[(((it & 1) * 4 + quad) * 2 + (col_half ^ 1)) * 32 + lane];
      const float c1 = (s1 + other.x) * (1.0f / 256.0f), c2 = (s2 + other.y) * (1.0f / 256.0f);
      // ---------------- pass 2: dx, parameter-gradient column sums (32 columns at a time: register budget)
#pragma unroll 1
      for (int r = 0; r < 2; ++r) {
        mbar_wait(&bars->side_full[ew][0], uses0 & 1); ++uses0;
        if (has_skip) { mbar_wait(&bars->side_full[ew][1], uses1 & 1); ++uses1; }
        else if (r == 1) tma_wait_group_read<0>();       // round 0's store has left buffer 1
#pragma unroll 1
        for (int grp = 0; grp < 2; ++grp) {
          uint32_t v[32], wx[16], ws[16];
          tmem_ld_32x32(t_acc + r * 64 + grp * 32, v);
#pragma unroll
          for (int k = 0; k < 4; ++k) {                  // chunks grp*4 .. grp*4+3 of this thread's 128-byte rows
            const uint32_t off = lane * 128 + (((grp * 4 + k) ^ (lane & 7)) << 4);
            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                         : "=r"(wx[4 * k]), "=r"(wx[4 * k + 1]), "=r"(wx[4 * k + 2]), "=r"(wx[4 * k + 3]) : "r"(stg + off) : "memory");
            if (has_skip) {
              asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                           : "=r"(ws[4 * k]), "=r"(ws[4 * k + 1]), "=r"(ws[4 * k + 2]), "=r"(ws[4 * k + 3])
                           : "r"(stg + kStgTileBytes + off) : "memory");
            } else {
              ws[4 * k] = ws[4 * k + 1] = ws[4 * k + 2] = ws[4 * k + 3] = 0u;
            }
          }
          tmem_ld_wait();
          if (r == 1 && grp == 1) {                      // last read of this accumulator
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->tmem_empty[buf]);
          }
          float a_g[32], a_c[32];
          uint32_t outw[16];
#pragma unroll
          for (int j = 0; j < 32; j += 2) {
            const float2 gm = __ldg(reinterpret_cast<const float2*>(p.ln_gamma + span0 + r * 64 + grp * 32 + j));
            const float2 xv = unpack_bf16x2(wx[j >> 1]), kv = unpack_bf16x2(ws[j >> 1]);
            const float dy0 = in ? __uint_as_float(v[j]) : 0.f, dy1 = in ? __uint_as_float(v[j + 1]) : 0.f;
            const float xh0 = (xv.x - mean) * rstd, xh1 = (xv.y - mean) * rstd;
            const float dx0 = in ? fmaf(rstd, dy0 * gm.x - c1 - xh0 * c2, kv.x) : 0.f;
            const float dx1 = in ? fmaf(rstd, dy1 * gm.y - c1 - xh1 * c2, kv.y) : 0.f;
            a_g[j] = dy0 * xh0; a_g[j + 1] = dy1 * xh1;
            a_c[j] = dx0; a_c[j + 1] = dx1;
            v[j] = __float_as_uint(dy0); v[j + 1] = __float_as_uint(dy1);
            outw[j >> 1] = pack_bf16x2(dx0, dx1);
          }
          // dx in place over the skip tile (buffer 1)
          __syncwarp();
#pragma unroll
          for (int k = 0; k < 4; ++k) {
            const uint32_t off = lane * 128 + (((grp * 4 + k) ^ (lane & 7)) << 4);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(stg + kStgTileBytes + off), "r"(outw[4 * k]),
                         "r"(outw[4 * k + 1]), "r"(outw[4 * k + 2]), "r"(outw[4 * k + 3]) : "memory");
          }
          float a_b[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) a_b[j] = __uint_as_float(v[j]);
          const float tg = warp_colsum32(a_g, lane), tb = warp_colsum32(a_b, lane), tc = warp_colsum32(a_c, lane);
#pragma unroll
          for (int q = 0; q < 4; ++q)            // static register indexing
            if (q == r * 2 + grp) { acc_g[q] += tg; acc_b[q] += tb; acc_c[q] += tc; }
        }
        __syncwarp();                                   // every lane is done with the x tile of buffer 0
        fence_proxy_async_smem();
        if (r == 0 && elect_one()) load_side(0, &map_side, span0 + 64, row0);       // x of round 1
        __syncwarp();
        if (elect_one()) {
          tma_store_2d(&map_out, stg + kStgTileBytes, span0 + r * 64, row0);
          tma_commit_group();
          if (r == 0 && has_skip) {                    // skip of round 1 into the same buffer, once the store has read it
            tma_wait_group_read<0>();
            fence_proxy_async_smem();
            load_side(1, &map_aux, span0 + 64, row0);
          }
        }
        __syncwarp();
      }
    }
    // parameter gradients: lane l holds columns span0 + q * 32 + l of this warp's rows
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int c = span0 + q * 32 + lane;
      atomicAdd(p.ln_dgamma + c, acc_g[q]);
      atomicAdd(p.ln_dbeta + c, acc_b[q]);
      if (p.ln_dxcol != nullptr) atomicAdd(p.ln_dxcol + c, acc_c[q]);
    }
    tma_wait_group_read<0>();
  } else {
    // ------------------------------- epilogue -------------------------------------------
    const int ew = warp - 2;
    const int quad = warp & 3;                 // TMEM lane quadrant this warp may access
    const int col_half = ew >> 2;
    // columns of the tile this warp drains: BN >= 128 -> its half; BN == 64 -> half 0 takes all
    constexpr int kSpan = BN >= 128 ? BN / 2 : 64;
    const bool active = BN >= 128 || col_half == 0;
    const int span0 = BN >= 128 ? col_half * kSpan : 0;
    constexpr bool kF32 = (EPI == EPI_F32 || EPI == EPI_F32_RED);
    constexpr int kRoundCols = kF32 ? 32 : 64;   // one staging tile (128 B per row) per round
    constexpr int kRounds = kSpan / kRoundCols;
    constexpr int kBufs = Cfg::kStgBufs;
    const uint32_t stg = smem_u32(staging + ew * kBufs * kStgTileBytes);
    const bool has_bias = (EPI != EPI_GELU_BWD && EPI != EPI_F32_RED) && p.bias != nullptr;
    // side operand (TMA-loaded, result written in place): residual (EPI_BF16) or aux_in (GELU')
    const bool has_dot = EPI == EPI_BF16 && p.dot_out != nullptr;    // side = dot operand, output = acc
    const bool has_side = kBufs == 2 && ((EPI == EPI_BF16 && (p.residual != nullptr || has_dot)) || EPI == EPI_GELU_BWD ||
                                         EPI == EPI_BF16_DROP);
    constexpr bool kDrop = EPI == EPI_GELU_DROP || EPI == EPI_BF16_DROP;
    uint64_t dkey = 0;
    if constexpr (kDrop) dkey = drop_key_load(p.drop_key);
    const bool want_colsum = !kF32 && p.colsum_out != nullptr;
    // fused column sums of the bf16 output (bias gradient): lane accumulates 8 columns (16-byte chunk
    // lane & 7) over the rows = (lane >> 3) mod 4 of every staged tile, in registers while this CTA
    // stays on the same n tile (the host sizes the grid as a multiple of tiles_n so that it always does)
    float csum[kRounds][8];
    int csum_n0 = -1;
    const int cs_row = lane >> 3, cs_chunk = lane & 7;
    auto flush_colsum = [&]() {
      if (csum_n0 < 0) return;
#pragma unroll
      for (int r = 0; r < kRounds; ++r) {
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          float t = csum[r][e];
          t += __shfl_xor_sync(0xffffffffu, t, 8);
          t += __shfl_xor_sync(0xffffffffu, t, 16);
          const int gc = csum_n0 + span0 + r * kRoundCols + cs_chunk * 8 + e;
          if (cs_row == 0 && gc < p.N) atomicAdd(p.colsum_out + gc, t);
        }
      }
    };
    // column sums of the tile just staged at `sb` (bf16), rows beyond M excluded
    auto add_colsum = [&](uint32_t sb, int row0, int r) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int rr = 4 * i + cs_row;
        const uint32_t addr = sb + rr * 128 + ((cs_chunk ^ (rr & 7)) << 4);
        uint4 u;
        asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];"
                     : "=r"(u.x), "=r"(u.y), "=r"(u.z), "=r"(u.w) : "r"(addr) : "memory");
        if (row0 + rr < p.M) {
          const float2 a = unpack_bf16x2(u.x), b = unpack_bf16x2(u.y), c = unpack_bf16x2(u.z), d = unpack_bf16x2(u.w);
#pragma unroll
          for (int q = 0; q < kRounds; ++q)      // static register indexing
            if (q == r) {
              csum[q][0] += a.x; csum[q][1] += a.y; csum[q][2] += b.x; csum[q][3] += b.y;
              csum[q][4] += c.x; csum[q][5] += c.y; csum[q][6] += d.x; csum[q][7] += d.y;
            }
        }
      }
    };
    const int total_rounds = active ? sched.count * kRounds : 0;
    auto issue_side = [&](int gi) {   // lane 0: prefetch the side tile of global round gi
      int m0, n0, split;
      sched.get(gi / kRounds, BN, &m0, &n0, &split);
      const int b = gi & 1;
      mbar_arrive_expect_tx(&bars->side_full[ew][b], kStgTileBytes);
      tma_load_2d_u32(stg + b * kStgTileBytes, &map_side, &bars->side_full[ew][b],
                      n0 + span0 + (gi % kRounds) * kRoundCols, m0 + quad * 32);
    };
    if (has_side && total_rounds > 0 && elect_one()) issue_side(0);
    int g = 0;      // global round counter of this warp
    int ob = 0;     // staging buffer of the next output tile (modes without a side operand)
    // stage one 32 x 128 B tile (row-mapped registers) and hand it to TMA; returns the smem tile
    auto stage_and_store = [&](const CUtensorMap* map, const uint32_t* w, int col, int row, bool reduce) {
      const uint32_t dst = stg + ob * kStgTileBytes;
      tma_wait_group_read<kBufs - 1>();   // (issuing lane) the tile last stored from this buffer was read
      __syncwarp();
      stg_store_row(dst, lane, w);
      fence_proxy_async_smem();
      __syncwarp();
      if (elect_one()) {
        if (reduce) tma_reduce_add_2d(map, dst, col, row); else tma_store_2d(map, dst, col, row);
        tma_commit_group();
      }
      ob = (ob + 1 == kBufs) ? 0 : ob + 1;
      return dst;
    };
    for (int it = 0; it < sched.count; ++it) {
      int m0, n0, split;
      sched.get(it, BN, &m0, &n0, &split);
      if (want_colsum && active && n0 != csum_n0) {
        flush_colsum();
        csum_n0 = n0;
#pragma unroll
        for (int r = 0; r < kRounds; ++r)
#pragma unroll
          for (int e = 0; e < 8; ++e) csum[r][e] = 0.f;
      }
      const int buf = it & 1;
      const uint32_t acc_phase = (it >> 1) & 1;
      mbar_wait(&bars->tmem_full[buf], acc_phase);
      tc_fence_after_sync();
      const int row0 = m0 + quad * 32;
      const uint32_t t_acc = tmem_base + (static_cast<uint32_t>(quad * 32) << 16) + buf * BN;
      if (!active) {
        tc_fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bars->tmem_empty[buf]);
        continue;
      }
#pragma unroll 1
      for (int r = 0; r < kRounds; ++r, ++g) {
        const int c0 = span0 + r * kRoundCols;        // first tile column of this round
        const int gcol = n0 + c0;
        if constexpr (!kF32) {
          // ---------------- bf16 outputs: 64 columns per round ----------------
          uint32_t v[64];
          tmem_ld_32x32(t_acc + c0, *reinterpret_cast<uint32_t(*)[32]>(&v[0]));
          tmem_ld_32x32(t_acc + c0 + 32, *reinterpret_cast<uint32_t(*)[32]>(&v[32]));
          if (has_side && g + 1 < total_rounds) {
            __syncwarp();    // every lane is done with buffer (g+1)&1 (round g-1: row + column-sum reads)
            if (elect_one()) {
              tma_wait_group_read<0>();     // ... and so is the TMA store that was issued from it
              fence_proxy_async_smem();
              issue_side(g + 1);
            }
          }
          tmem_ld_wait();
          if (r == kRounds - 1) {
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->tmem_empty[buf]);
          }
          if (has_bias) {
#pragma unroll
            for (int j = 0; j < 64; j += 4) {
              const int c = gcol + j;
              float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
              if (c < p.N) b = __ldg(reinterpret_cast<const float4*>(p.bias + c));
              v[j] = __float_as_uint(__uint_as_float(v[j]) + b.x);
              v[j + 1] = __float_as_uint(__uint_as_float(v[j + 1]) + b.y);
              v[j + 2] = __float_as_uint(__uint_as_float(v[j + 2]) + b.z);
              v[j + 3] = __float_as_uint(__uint_as_float(v[j + 3]) + b.w);
            }
          }
          if (EPI == EPI_BF16 && p.act == 3) {            // ReLU (EarlyCNN conv stem)
#pragma unroll
            for (int j = 0; j < 64; ++j) v[j] = __float_as_uint(fmaxf(__uint_as_float(v[j]), 0.f));
          }
          uint32_t keep[2];                               // dropout: keep bits of this row's 64 columns
          if constexpr (kDrop) {
            keep[0] = drop_keep32(dkey, gcol, row0 + lane, 0, p.drop_site, p.drop_thr);
            keep[1] = drop_keep32(dkey, gcol + 32, row0 + lane, 0, p.drop_site, p.drop_thr);
          }
          if constexpr (EPI == EPI_BF16_DROP) {
#pragma unroll
            for (int j = 0; j < 64; ++j)
              v[j] = __float_as_uint((keep[j >> 5] >> (j & 31)) & 1u ? __uint_as_float(v[j]) * p.drop_scale : 0.f);
          }
          uint32_t w[32];
          if constexpr (EPI == EPI_GELU_FWD || EPI == EPI_GELU_DROP) {
            // out = GELU(v); aux_out = GELU'(v) (bf16) so that the backward pass is a plain multiply
            // and never evaluates erf again (the exp(-v^2/2) is shared between the two here)
            if (p.aux_out != nullptr) {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                f32x2 hh, gg;
                gelu_pair(v[2 * j], v[2 * j + 1], hh, gg);
                if constexpr (EPI == EPI_GELU_DROP) {
                  const int c = 2 * j;
                  const f32x2 z = f2_pack((keep[c >> 5] >> (c & 31)) & 1u ? p.drop_scale : 0.f,
                                          (keep[c >> 5] >> ((c + 1) & 31)) & 1u ? p.drop_scale : 0.f);
                  hh = f2_mul(hh, z);
                  gg = f2_mul(gg, z);
                }
                float g0, g1;
                f2_unpack(gg, g0, g1);
                w[j] = pack_bf16x2(g0, g1);
                f2_unpacku(hh, v[2 * j], v[2 * j + 1]);
              }
              stage_and_store(&map_aux, w, gcol, row0, false);
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {      // same packed evaluation as above: eval and training agree bitwise
                f32x2 hh, gg;
                gelu_pair(v[2 * j], v[2 * j + 1], hh, gg);
                if constexpr (EPI == EPI_GELU_DROP) {
                  const int c = 2 * j;
                  hh = f2_mul(hh, f2_pack((keep[c >> 5] >> (c & 31)) & 1u ? p.drop_scale : 0.f,
                                          (keep[c >> 5] >> ((c + 1) & 31)) & 1u ? p.drop_scale : 0.f));
                }
                f2_unpacku(hh, v[2 * j], v[2 * j + 1]);
              }
            }
          }
          if (has_side) {
            const uint32_t sb = stg + (g & 1) * kStgTileBytes;
            mbar_wait(&bars->side_full[ew][g & 1], (g >> 1) & 1);
            stg_load_row(sb, lane, w);
            if (has_dot) {
              // out = acc (rounded to bf16 first: the consumer sees exactly these values); dot over this
              // round's 64 columns with the side operand (dO . O per head = FlashAttention's delta)
              float dot = 0.f;
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const float2 s2 = unpack_bf16x2(w[j]);
                w[j] = pack_bf16x2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
                const float2 o2 = unpack_bf16x2(w[j]);
                dot = fmaf(o2.x, s2.x, dot);
                dot = fmaf(o2.y, s2.y, dot);
              }
              if (row0 + lane < p.M && gcol < p.N) p.dot_out[(size_t)(row0 + lane) * (p.N >> 6) + (gcol >> 6)] = dot;
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const float2 s2 = unpack_bf16x2(w[j]);
                if constexpr (EPI == EPI_GELU_BWD) {   // aux_in holds GELU'(pre-activation)
                  w[j] = pack_bf16x2(__uint_as_float(v[2 * j]) * s2.x, __uint_as_float(v[2 * j + 1]) * s2.y);
                } else {
                  w[j] = pack_bf16x2(__uint_as_float(v[2 * j]) + s2.x, __uint_as_float(v[2 * j + 1]) + s2.y);
                }
              }
            }
            stg_store_row(sb, lane, w);      // in place: every thread only touches its own row
            fence_proxy_async_smem();
            __syncwarp();
            if (elect_one()) {
              tma_store_2d(&map_out, sb, gcol, row0);
              if ((EPI == EPI_BF16 || EPI == EPI_BF16_DROP) && p.out2 != nullptr)
                tma_store_2d(&map_aux, sb, gcol, row0);   // second copy of the output
              tma_commit_group();
            }
            if (want_colsum) add_colsum(sb, row0, r);
          } else {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              w[j] = pack_bf16x2(__uint_as_float(v[2 * j]), __uint_as_float(v[2 * j + 1]));
            const uint32_t sb = stage_and_store(&map_out, w, gcol, row0, false);
            if (want_colsum) add_colsum(sb, row0, r);
          }
        } else {
          // ---------------- fp32 outputs: 32 columns per round ----------------
          uint32_t v[32];
          tmem_ld_32x32(t_acc + c0, v);
          tmem_ld_wait();
          if (r == kRounds - 1) {
            tc_fence_before_sync();
            __syncwarp();
            if (lane == 0) mbar_arrive(&bars->tmem_empty[buf]);
          }
          if (has_bias) {
#pragma unroll
            for (int j = 0; j < 32; j += 4) {
              const int c = gcol + j;
              float4 b = make_float4(0.f, 0.f, 0.f, 0.f);
              if (c < p.N) b = __ldg(reinterpret_cast<const float4*>(p.bias + c));
              v[j] = __float_as_uint(__uint_as_float(v[j]) + b.x);
              v[j + 1] = __float_as_uint(__uint_as_float(v[j + 1]) + b.y);
              v[j + 2] = __float_as_uint(__uint_as_float(v[j + 2]) + b.z);
              v[j + 3] = __float_as_uint(__uint_as_float(v[j + 3]) + b.w);
            }
          }
          stage_and_store(&map_out, v, gcol, row0, EPI == EPI_F32_RED);
        }
      }
    }
    if (want_colsum && active) flush_colsum();
    // (issuing lane) every store / reduce of this warp has READ its staging tile; the writes themselves are complete
    // at grid completion, which is what dependents wait for (griddepcontrol.wait / stream order)
    tma_wait_group_read<0>();
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, Cfg::kTmemCols);
  }
}

template <int BN, bool A_MN, bool B_MN, int EPI, bool WS = false>
int launch_variant(const GemmPlan& plan, cudaStream_t stream) {
  using Cfg = GemmCfg<BN, WS>;
  static_assert(Cfg::kSmemBytes <= 227 * 1024, "shared memory budget");
  auto kern = gemm_bf16_kernel<BN, A_MN, B_MN, EPI, WS>;
  static bool configured = false;
  if (!configured) {
    M3L_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::kSmemBytes));
    configured = true;
  }
  M3L_CUDA(launch_kernel(kern, dim3(plan.grid), dim3(kNumThreads), Cfg::kSmemBytes, stream, plan.map_a,
                         plan.map_b, plan.map_out, plan.map_aux, plan.map_side, plan.args));
  M3L_CUDA(cudaGetLastError());
  return M3L_OK;
}

template <int BN>
int launch_bn(const GemmPlan& plan, cudaStream_t stream) {
  const GemmArgs& p = plan.args;
  if (p.a_mn_major) return launch_variant<BN, true, true, EPI_F32_RED>(plan, stream);
  if (p.drop_key != nullptr)
    return p.act == 1 ? launch_variant<BN, false, false, EPI_GELU_DROP>(plan, stream)
                      : launch_variant<BN, false, false, EPI_BF16_DROP>(plan, stream);
  if constexpr (BN >= 128) {
    if (plan.ws) {
      if (p.out_mode == 1) return launch_variant<BN, false, false, EPI_F32, true>(plan, stream);
      if (p.act == 1) return launch_variant<BN, false, false, EPI_GELU_FWD, true>(plan, stream);
      return launch_variant<BN, false, false, EPI_BF16, true>(plan, stream);
    }
  }
  if constexpr (BN == 256) {
    if (p.ln_x != nullptr) return launch_variant<BN, false, false, EPI_LN_BWD>(plan, stream);
  }
  if (p.out_mode == 1) return launch_variant<BN, false, false, EPI_F32>(plan, stream);
  if (p.act == 1) return launch_variant<BN, false, false, EPI_GELU_FWD>(plan, stream);
  if (p.act == 2) return launch_variant<BN, false, false, EPI_GELU_BWD>(plan, stream);
  return launch_variant<BN, false, false, EPI_BF16>(plan, stream);
}

}  // namespace

int gemm_pick_bn(int M, int N) {
  const int sms = device_sm_count();
  const int tiles_m = (M + BM - 1) / BM;
  if (N % 256 == 0 && tiles_m * (N / 256) >= sms) return 256;
  if (N >= 128 && tiles_m * ((N + 127) / 128) >= sms / 2) return 128;
  if (N % 128 == 0 && N >= 512) return 128;
  return N >= 128 && (N % 128 == 0) ? 128 : 64;
}

int gemm_make_plan(GemmPlan* plan, const GemmArgs& args, int bn) {
  GemmArgs p = args;
  M3L_REQUIRE(p.M > 0 && p.N > 0 && p.K > 0, "gemm: bad shape M=%d N=%d K=%d", p.M, p.N, p.K);
  M3L_REQUIRE(p.N % 8 == 0, "gemm: N=%d must be a multiple of 8", p.N);
  M3L_REQUIRE(p.a_mn_major == p.b_mn_major,
              "gemm: mixed operand majors are not instantiated (a=%d b=%d)", p.a_mn_major,
              p.b_mn_major);
  M3L_REQUIRE(p.out != nullptr && p.a != nullptr && p.b != nullptr, "gemm: null pointer");
  if (p.splits < 1) p.splits = 1;
  const int kb_total = (p.K + BK - 1) / BK;
  if (p.splits > kb_total) p.splits = kb_total;
  // every split must own at least one k-block
  while (p.splits > 1 && ((kb_total + p.splits - 1) / p.splits) * (p.splits - 1) >= kb_total)
    --p.splits;
  M3L_REQUIRE(p.splits == 1 || p.out_mode == 2, "gemm: split-K requires the atomic output mode");
  M3L_REQUIRE(p.alpha == 1.0f, "gemm: alpha != 1 is not supported");
  M3L_REQUIRE((p.out_mode == 2) == (p.a_mn_major != 0),
              "gemm: the accumulate output mode goes with MN-major operands (wgrad) and vice versa");
  M3L_REQUIRE(p.a_mn_major == 0 || (p.bias == nullptr && p.residual == nullptr && p.act == 0),
              "gemm: wgrad mode takes no bias / residual / activation");
  M3L_REQUIRE(p.out_mode != 1 || (p.act == 0 && p.residual == nullptr),
              "gemm: fp32 store mode supports bias only");
  M3L_REQUIRE(p.act == 0 || p.residual == nullptr, "gemm: activation and residual cannot be combined");
  M3L_REQUIRE(p.act != 2 || (p.aux_in != nullptr && p.bias == nullptr), "gemm: GELU' needs aux_in and no bias");
  M3L_REQUIRE(p.ldo % 8 == 0 && (p.residual == nullptr || p.ldr % 8 == 0) &&
                  ((p.aux_in == nullptr && p.aux_out == nullptr) || p.ld_aux % 8 == 0),
              "gemm: output / residual / aux leading dimensions must be multiples of 8");
  M3L_REQUIRE((p.dot_out == nullptr) == (p.dot_side == nullptr), "gemm: dot_side and dot_out go together");
  M3L_REQUIRE(p.out2 == nullptr || (p.out_mode == 0 && p.act == 0 && p.residual != nullptr && p.aux_out == nullptr),
              "gemm: out2 needs the bf16 output mode with a residual and no activation");
  M3L_REQUIRE(p.act >= 0 && p.act <= 3 && (p.act != 3 || p.out_mode == 0), "gemm: act=%d unsupported here", p.act);
  M3L_REQUIRE(p.dot_out == nullptr || (p.out_mode == 0 && p.act == 0 && p.residual == nullptr && p.N % 64 == 0 &&
                                       p.ld_dot % 8 == 0 && !p.a_mn_major),
              "gemm: the fused row-dot needs a plain bf16 output with N %% 64 == 0");
  M3L_REQUIRE(p.drop_key != nullptr || p.drop_p == 0.f, "gemm: null dropout key with p > 0");
  if (p.drop_key != nullptr) {
    M3L_REQUIRE(drop_threshold(p.drop_p, &p.drop_thr, &p.drop_scale), "gemm: dropout probability %g outside [0, 1)",
                (double)p.drop_p);
    const bool plain = p.out_mode == 0 && !p.a_mn_major && p.ln_x == nullptr && p.dot_out == nullptr && p.splits == 1;
    M3L_REQUIRE(plain && ((p.act == 1 && p.residual == nullptr && p.out2 == nullptr) ||
                          (p.act == 0 && p.residual != nullptr && p.aux_out == nullptr)),
                "gemm: dropout goes with the GELU epilogue or with bias + residual only");
  }
  if (p.ln_x != nullptr) {
    M3L_REQUIRE(p.N == 256 && p.out_mode == 0 && !p.a_mn_major && p.splits == 1, "gemm: the LayerNorm-backward epilogue needs n == 256, bf16 output, K-major operands");
    M3L_REQUIRE(p.bias == nullptr && p.residual == nullptr && p.act == 0 && p.colsum_out == nullptr && p.dot_out == nullptr &&
                    p.out2 == nullptr && p.aux_out == nullptr,
                "gemm: the LayerNorm-backward epilogue excludes the other epilogue options");
    M3L_REQUIRE(p.ln_stats && p.ln_gamma && p.ln_dgamma && p.ln_dbeta, "gemm: LayerNorm-backward epilogue: null pointer");
    M3L_REQUIRE(p.ldo == 256, "gemm: LayerNorm-backward epilogue writes a contiguous [m, 256] output");
    bn = 256;
  }
  if (bn == 0) bn = gemm_pick_bn(p.M, p.N);
  M3L_REQUIRE(bn == 64 || bn == 128 || bn == 256, "gemm: BN=%d unsupported", bn);
  plan->bn = bn;
  plan->args = p;
  int s;
  if (!p.a_mn_major) {
    if ((s = make_tmap_2d_bf16(&plan->map_a, p.a, p.M, p.K, p.lda, BM))) return s;
    if ((s = make_tmap_2d_bf16(&plan->map_b, p.b, p.N, p.K, p.ldb, bn))) return s;
  } else {
    // operands stored [K rows, M or N columns]
    if ((s = make_tmap_2d_bf16(&plan->map_a, p.a, p.K, p.M, p.lda, BK))) return s;
    if ((s = make_tmap_2d_bf16(&plan->map_b, p.b, p.K, p.N, p.ldb, BK))) return s;
  }
  // epilogue tiles: 32 rows x 128 B (64 bf16 / 32 fp32 columns)
  if (p.out_mode == 0) {
    if ((s = make_tmap_2d_bf16(&plan->map_out, p.out, p.M, p.N, p.ldo, 32))) return s;
  } else {
    if ((s = make_tmap_2d_f32(&plan->map_out, p.out, p.M, p.N, p.ldo, 32))) return s;
  }
  plan->map_aux = plan->map_out;
  plan->map_side = plan->map_out;
  if (p.ln_x != nullptr) {
    if ((s = make_tmap_2d_bf16(&plan->map_side, p.ln_x, p.M, p.N, p.N, 32))) return s;
    if (p.ln_skip != nullptr && (s = make_tmap_2d_bf16(&plan->map_aux, p.ln_skip, p.M, p.N, p.N, 32))) return s;
  }
  if (p.aux_out != nullptr && (s = make_tmap_2d_bf16(&plan->map_aux, p.aux_out, p.M, p.N, p.ld_aux, 32))) return s;
  if (p.out2 != nullptr && (s = make_tmap_2d_bf16(&plan->map_aux, p.out2, p.M, p.N, p.ldo, 32))) return s;
  if (p.act == 2) {
    if ((s = make_tmap_2d_bf16(&plan->map_side, p.aux_in, p.M, p.N, p.ld_aux, 32))) return s;
  } else if (p.residual != nullptr) {
    if ((s = make_tmap_2d_bf16(&plan->map_side, p.residual, p.M, p.N, p.ldr, 32))) return s;
  } else if (p.dot_out != nullptr) {
    if ((s = make_tmap_2d_bf16(&plan->map_side, p.dot_side, p.M, p.N, p.ld_dot, 32))) return s;
  }
  const int tiles_n = (p.N + bn - 1) / bn;
  const int tiles = ((p.M + BM - 1) / BM) * tiles_n * p.splits;
  plan->grid = tiles < device_sm_count() ? tiles : device_sm_count();
  // weight-stationary mode: K fits the resident slice, no side operand (its staging is single
  // buffered) and every CTA gets several m tiles to amortise the one-off weight load over
  // (M3L_GEMM_WS=0 disables it, for A/B measurements)
  static const bool ws_allowed = [] { const char* e = getenv("M3L_GEMM_WS"); return !(e && e[0] == '0'); }();
  plan->ws = ws_allowed && !p.a_mn_major && p.drop_key == nullptr && kb_total <= kWsMaxKb && p.splits == 1 && bn >= 128 &&
             p.residual == nullptr && p.dot_out == nullptr && p.act != 2 && p.ln_x == nullptr &&
             tiles >= 2 * device_sm_count() && tiles_n <= plan->grid;
  // decoder feed-forward forward shape (GELU + GELU' outputs, K <= 256, N % 256 == 0): dedicated kernel
  // with 16 epilogue warps (M3L_GELU16=0 falls back to the generic epilogue, for A/B measurements)
  static const bool g16_allowed = [] { const char* e = getenv("M3L_GELU16"); return !(e && e[0] == '0'); }();
  plan->gelu16 = g16_allowed && plan->ws && bn == 256 && p.act == 1 && p.out_mode == 0 && p.N % 256 == 0 &&
                 p.colsum_out == nullptr;
  if (plan->gelu16) {
    if ((s = make_tmap_2d_bf16_sw64(&plan->map_out32, p.out, p.M, p.N, p.ldo, 32))) return s;
    plan->map_aux32 = plan->map_out32;
    if (p.aux_out != nullptr &&
        (s = make_tmap_2d_bf16_sw64(&plan->map_aux32, p.aux_out, p.M, p.N, p.ld_aux, 32))) return s;
  }
  if (p.colsum_out != nullptr) {
    M3L_REQUIRE(p.out_mode == 0, "gemm: colsum_out needs the bf16 output mode");
    // keep every CTA on one N tile so the column sums stay in registers across its tiles
    if (plan->grid > tiles_n) plan->grid = (plan->grid / tiles_n) * tiles_n;
  }
  return M3L_OK;
}

int gemm_run(const GemmPlan& plan, cudaStream_t stream) {
  if (plan.gelu16) return gemm_gelu16_run(plan, stream);
  switch (plan.bn) {
    case 64: return launch_bn<64>(plan, stream);
    case 128: return launch_bn<128>(plan, stream);
    case 256: return launch_bn<256>(plan, stream);
  }
  set_last_error("gemm: BN=%d unsupported", plan.bn);
  return M3L_ERR_INVALID;
}

}  // namespace m3l

// ---------------------------------------------------------------------------------------
// C-ABI (include/m3l_b200.h)
// ---------------------------------------------------------------------------------------
extern "C" int m3l_gemm_bf16(const m3l_gemm_args* a, void* stream) {
  if (a == nullptr) return m3l::M3L_ERR_INVALID;
  m3l::GemmArgs g;
  g.a = a->a; g.b = a->b; g.lda = a->lda; g.ldb = a->ldb;
  g.a_mn_major = a->a_mn_major; g.b_mn_major = a->b_mn_major;
  g.M = a->m; g.N = a->n; g.K = a->k; g.splits = a->splits;
  g.out = a->out; g.ldo = a->ldo; g.out_mode = a->out_mode;
  g.bias = a->bias; g.residual = (const m3l::bf16*)a->residual; g.ldr = a->ldr;
  g.act = a->act; g.aux_out = (m3l::bf16*)a->aux_out; g.aux_in = (const m3l::bf16*)a->aux_in;
  g.ld_aux = a->ld_aux; g.alpha = a->alpha; g.colsum_out = a->colsum_out; g.out2 = (m3l::bf16*)a->out2;
  g.dot_side = (const m3l::bf16*)a->dot_side; g.ld_dot = a->ld_dot; g.dot_out = a->dot_out;
  g.ln_x = (const m3l::bf16*)a->ln_x; g.ln_stats = a->ln_stats; g.ln_gamma = a->ln_gamma;
  g.ln_skip = (const m3l::bf16*)a->ln_skip; g.ln_dgamma = a->ln_dgamma; g.ln_dbeta = a->ln_dbeta; g.ln_dxcol = a->ln_dxcol;
  g.drop_key = a->drop_key; g.drop_site = (uint32_t)a->drop_site; g.drop_p = a->drop_p;
  m3l::GemmPlan plan;
  int s = m3l::gemm_make_plan(&plan, g, a->bn);
  if (s) return s;
  return m3l::gemm_run(plan, (cudaStream_t)stream);
}
