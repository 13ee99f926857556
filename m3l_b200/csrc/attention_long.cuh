// m3l_b200 — fused multi-head attention for sequences of any length on tcgen05 / TMEM / TMA (sm_100a), forward and
// backward, as a template on the head width kDh in {32, 64, 128}.  attention_long.cu instantiates kDh = 64,
// attention_dh.cu kDh = 32 and 128.
//
// attention.cu holds a sample's whole key sequence in one CTA and is limited to n <= 256 (DinoV2 at 224 x 224 has
// 261 tokens, at its default 518 x 518 1374).  The kernels here loop over 128-key tiles instead:
//
//   forward, persistent CTA over (sample, head, 128-query tile) items, FlashAttention-style online softmax:
//     warp 0     TMA loader: Q tile (double-buffered across items), K / V tiles through a kFwdStages-deep ring
//     warp 1     MMA issuer: S_j = Q K_j^T into one of two TMEM S slots, issued BEFORE O += P_{j-1} V_{j-1}, so the
//                tensor core computes the next scores while the softmax warps work on the current ones
//     warps 2..5 softmax, one TMEM lane (= query row) per thread; running max / sum in registers, P_j (bf16) ->
//                swizzled smem.  O (TMEM) is rescaled only when a row's max grows by more than kRescaleLog2: the
//                reference max may then lag the true one by up to that much (P <= 2^kRescaleLog2, harmless in
//                bf16 / fp32), and the result is exact because the final division and the LSE use the same max.
//     out bf16 [B*n, heads*dh] and lse fp32 [B, heads, n] (natural log of the scaled scores): the contract of
//     m3l_attention_fwd, so either backward reads either forward's output.
//
//   backward, two deterministic kernels (no atomics; every gradient element is summed in one fixed order), both
//   recomputing P = exp(S * scale - LSE) and dS = P (dP - delta) scale from the saved LSE:
//     KV-stationary  CTA = (sample, head, 128-key tile): loops over the query tiles, dV += P^T dO, dK += dS^T Q
//     Q-stationary   CTA = (sample, head, 128-query tile): loops over the key tiles, dQ += dS K
//   warp 0 TMA loader (stationary pair once, streamed pair through a ring of LongCfg::bwd_stages), warp 1 MMA issuer
//   (S / dP of step s+1 issued before the accumulating products of step s when the ring has more than one stage),
//   warps 2..9 two groups of 128 threads, thread = (query row, 64-key half), as in attention.cu's backward.
//
// What depends on the head width (LongCfg):
//   operand tiles  [128 rows x kN] bf16 with kN = max(dh, 64), stored as kN / 64 panels of [128 x 64] 128B-swizzled
//                  (one TMA box each).  dh = 32 loads a 64-wide box, so the upper 32 columns hold the next head's
//                  (or, past the tensor, TMA's zero-filled) values: Q K^T and dO V^T contract over the first 32
//                  columns only (K = 32), and the N = dh products (P V, dS K, P^T dO, dS^T Q) run at N = 64 with
//                  the upper half of their accumulators never read.  dh = 128: K-major k-steps 4..7 are in the
//                  second panel; MN-major operands with N = 128 take LBO = the panel stride.
//   shared memory  (227 KB a block)  forward 2 Q + 2 * kFwdStages K|V tiles + the 32 KB P slab:
//                    dh <= 64: 3 stages, 161 KB;  dh = 128: 2 stages, 225 KB (3 would need 289 KB).
//                  backward stationary pair + stages * streamed pair + P and dS slabs (32 KB each):
//                    dh <= 64: 3 stages, 193 KB in both kernels;
//                    dh = 128 KV-stationary: 1 stage, 193 KB.  Two stages need 257 KB; with one the next step's
//                      S / dP cannot be issued ahead (its Q|dO would overwrite the current one), so that look-ahead
//                      is given up at this width;
//                    dh = 128 Q-stationary: 2 stages, 225 KB, with no P slab (this kernel only multiplies dS).
//   tensor memory  (512 columns)  forward S 2 x 128 + O kN;  backward S 128 + dP 128 + dV|dQ kN + dK kN (= 512 at
//                  dh = 128).
#pragma once
#include "common.cuh"
#include "dropout.cuh"
#include "m3l_internal.h"

namespace m3l {
namespace {

constexpr int kTile = 128;                    // query / key rows per tile
constexpr int kPanelBytes = kTile * 64 * 2;   // [128 x 64] bf16 panel, 128B-swizzled: one TMA box
constexpr int kPBytes = 2 * kPanelBytes;      // P / dS slab: [2 panels of 64 keys][128 q x 64], for every dh
constexpr float kLog2e = 1.4426950408889634f;
constexpr float kLn2 = 0.6931471805599453f;
constexpr float kRescaleLog2 = 8.0f;

template <int kDh>
struct LongCfg {
  static_assert(kDh == 32 || kDh == 64 || kDh == 128, "head widths 32, 64 and 128 only");
  static constexpr int kN = kDh < 64 ? 64 : kDh;            // loaded tile width = N of the N = dh products
  static constexpr int kPanels = kN / 64;
  static constexpr int kTileBytes = kPanels * kPanelBytes;  // one [128 x kN] operand tile
  // LBO of an MN-major operand = stride between its 64-wide MN blocks (ignored with one block)
  static constexpr uint32_t kMnLbo = kPanels == 1 ? 8192u : (uint32_t)kPanelBytes;
  static constexpr int kFwdStages = kDh == 128 ? 2 : 3;
  static constexpr int bwd_stages(bool kv) { return kDh == 128 ? (kv ? 1 : 2) : 3; }
  static constexpr bool bwd_has_p(bool kv) { return kv || kDh != 128; }
  static constexpr int kFwdSmem = 1024 + 2 * kTileBytes + kFwdStages * 2 * kTileBytes + kPBytes + 256;
  static constexpr int bwd_smem(bool kv) {
    return 1024 + 2 * kTileBytes + bwd_stages(kv) * 2 * kTileBytes + (bwd_has_p(kv) ? 2 : 1) * kPBytes + 256;
  }
  static_assert(kFwdSmem <= 232448 && bwd_smem(true) <= 232448 && bwd_smem(false) <= 232448, "shared memory");
};

// byte offset of K-major k-step k (16 bf16 columns) inside a panelled tile
M3L_DEVINL constexpr uint32_t kmajor_off(int k) { return (k >> 2) * kPanelBytes + (k & 3) * 32; }

// one [128 x kPanels*64] operand tile at columns [col, col + kPanels*64) of rows [row, row + 128) of sample b
template <int kPanels>
M3L_DEVINL void tma_load_tile(uint8_t* dst, const CUtensorMap* map, uint64_t* bar, int col, int row, int b) {
#pragma unroll
  for (int pn = 0; pn < kPanels; ++pn) tma_load_3d(dst + pn * kPanelBytes, map, bar, col + pn * 64, row, b);
}

M3L_DEVINL void st_swz_chunk(uint32_t slab_u32, int row, int chunk, uint4 v) {
  const uint32_t addr = slab_u32 + row * 128 + ((chunk ^ (row & 7)) << 4);
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

M3L_DEVINL void tmem_st_32x32(uint32_t taddr, const uint32_t (&v)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0],"
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16,"
      " %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};" ::"r"(taddr),
      "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]), "r"(v[9]),
      "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]), "r"(v[16]), "r"(v[17]), "r"(v[18]),
      "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]), "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]),
      "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
      : "memory");
}
M3L_DEVINL void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// first kCols (8 .. 32, multiple of 8) fp32 of one 32-column TMEM chunk * s -> bf16 at dst (16-byte stores)
template <int kCols>
M3L_DEVINL void store_row_chunk_scaled(bf16* dst, const uint32_t (&a)[32], float s) {
#pragma unroll
  for (int g = 0; g < kCols / 8; ++g) {
    uint4 u;
    u.x = pack_bf16x2(__uint_as_float(a[g * 8 + 0]) * s, __uint_as_float(a[g * 8 + 1]) * s);
    u.y = pack_bf16x2(__uint_as_float(a[g * 8 + 2]) * s, __uint_as_float(a[g * 8 + 3]) * s);
    u.z = pack_bf16x2(__uint_as_float(a[g * 8 + 4]) * s, __uint_as_float(a[g * 8 + 5]) * s);
    u.w = pack_bf16x2(__uint_as_float(a[g * 8 + 6]) * s, __uint_as_float(a[g * 8 + 7]) * s);
    *reinterpret_cast<uint4*>(dst + g * 8) = u;
  }
}

// 64 fp32 (two 32-column TMEM chunks) * s -> 64 bf16 at dst (16-byte stores)
M3L_DEVINL void store_row64_scaled(bf16* dst, const uint32_t (&a0)[32], const uint32_t (&a1)[32], float s) {
#pragma unroll
  for (int g = 0; g < 8; ++g) {
    const uint32_t(&a)[32] = g < 4 ? a0 : a1;
    const int o = (g & 3) * 8;
    uint4 u;
    u.x = pack_bf16x2(__uint_as_float(a[o + 0]) * s, __uint_as_float(a[o + 1]) * s);
    u.y = pack_bf16x2(__uint_as_float(a[o + 2]) * s, __uint_as_float(a[o + 3]) * s);
    u.z = pack_bf16x2(__uint_as_float(a[o + 4]) * s, __uint_as_float(a[o + 5]) * s);
    u.w = pack_bf16x2(__uint_as_float(a[o + 6]) * s, __uint_as_float(a[o + 7]) * s);
    *reinterpret_cast<uint4*>(dst + g * 8) = u;
  }
}

// kCols fp32 columns of this thread's TMEM lane from taddr, * s -> kCols bf16 at dst when `valid`.  64 columns at a
// time (two 32-column loads in flight), or one chunk for kCols <= 32.  tcgen05.ld is warp-collective, so every lane
// loads and `valid` only gates the stores.
template <int kCols>
M3L_DEVINL void tmem_row_to_bf16(bf16* dst, uint32_t taddr, float s, bool valid) {
  if constexpr (kCols <= 32) {
    uint32_t a0[32];
    tmem_ld_32x32(taddr, a0);
    tmem_ld_wait();
    if (valid) store_row_chunk_scaled<kCols>(dst, a0, s);
  } else {
#pragma unroll
    for (int c0 = 0; c0 < kCols; c0 += 64) {
      uint32_t a0[32], a1[32];
      tmem_ld_32x32(taddr + c0, a0);
      tmem_ld_32x32(taddr + c0 + 32, a1);
      tmem_ld_wait();
      if (valid) store_row64_scaled(dst + c0, a0, a1, s);
    }
  }
}

// ------------------------------------------------------------------------------------------
// forward
// TMEM columns: [0,128) S slot 0, [128,256) S slot 1, [256,256+kN) O
// ------------------------------------------------------------------------------------------
template <int kStages>
struct LongFwdBars {
  uint64_t q_full[2], q_empty[2], kv_full[kStages], kv_empty[kStages], s_full[2], s_free[2], p_full, o_done;
  uint32_t tmem_base;
};

struct LongFwdParams {
  bf16* out;
  float* lse;
  int n, heads, inner, tiles, num_items;
  float scale;
};

// kDrop: dropout on the probabilities that multiply V (attention_dropout.cu).  The row sums and the LSE use the
// undropped P, so lse equals the lse without dropout.
template <int kDh, bool kDrop>
__device__ __forceinline__ void attn_long_fwd_body(const CUtensorMap& map_qkv, const LongFwdParams& p,
                                                   const DropParams& dp) {
  using Cfg = LongCfg<kDh>;
  constexpr int kTileBytes = Cfg::kTileBytes, kFwdStages = Cfg::kFwdStages, kN = Cfg::kN;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sQ = smem;                                   // [2][128 x kN]
  uint8_t* sKV = sQ + 2 * kTileBytes;                   // [kFwdStages][K | V]
  uint8_t* sP = sKV + kFwdStages * 2 * kTileBytes;      // [2 slabs of 64 keys][128 q x 64]
  LongFwdBars<kFwdStages>* bars = reinterpret_cast<LongFwdBars<kFwdStages>*>(sP + kPBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr uint32_t kTmemCols = 512, kColO = 256;
  const int n = p.n;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_qkv);
    for (int i = 0; i < 2; ++i) {
      mbar_init(&bars->q_full[i], 1);
      mbar_init(&bars->q_empty[i], 1);
      mbar_init(&bars->s_full[i], 1);
      mbar_init(&bars->s_free[i], 128);
    }
    for (int i = 0; i < kFwdStages; ++i) {
      mbar_init(&bars->kv_full[i], 1);
      mbar_init(&bars->kv_empty[i], 1);
    }
    mbar_init(&bars->p_full, 128);
    mbar_init(&bars->o_done, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&bars->tmem_base, kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_base;
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ------------------------------- TMA loader -----------------------------------------
    if (elect_one()) {
      int it = 0, g = 0;
      for (int item = blockIdx.x; item < p.num_items; item += gridDim.x, ++it) {
        const int t = item % p.tiles, bh = item / p.tiles;
        const int h = bh % p.heads, b = bh / p.heads;
        const int qb = it & 1;
        mbar_wait(&bars->q_empty[qb], ((it >> 1) & 1) ^ 1);
        mbar_arrive_expect_tx(&bars->q_full[qb], kTileBytes);
        tma_load_tile<Cfg::kPanels>(sQ + qb * kTileBytes, &map_qkv, &bars->q_full[qb], h * kDh, t * kTile, b);
        for (int j = 0; j < p.tiles; ++j, ++g) {
          const int st = g % kFwdStages;
          mbar_wait(&bars->kv_empty[st], ((g / kFwdStages) & 1) ^ 1);
          uint8_t* dst = sKV + st * 2 * kTileBytes;
          mbar_arrive_expect_tx(&bars->kv_full[st], 2 * kTileBytes);
          tma_load_tile<Cfg::kPanels>(dst, &map_qkv, &bars->kv_full[st], p.inner + h * kDh, j * kTile, b);
          tma_load_tile<Cfg::kPanels>(dst + kTileBytes, &map_qkv, &bars->kv_full[st], 2 * p.inner + h * kDh,
                                      j * kTile, b);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer -----------------------------------------
    if (elect_one()) {
      const uint32_t idesc_s = umma_idesc_bf16(128, kTile, 0, 0);
      const uint32_t idesc_o = umma_idesc_bf16(128, kN, 0, 1);   // A = P K-major, B = V MN-major
      const uint32_t p_addr = smem_u32(sP);
      // O (+)= P_g V_g once the softmax warps have written P_g
      auto issue_pv = [&](int gp, bool first) {
        mbar_wait(&bars->p_full, gp & 1);
        tc_fence_after_sync();
        const int st = gp % kFwdStages;
        uint64_t d_v = umma_smem_desc(smem_u32(sKV + st * 2 * kTileBytes + kTileBytes), Cfg::kMnLbo, 1024);
#pragma unroll
        for (int kp = 0; kp < 2; ++kp) {
          const uint64_t d_p = umma_smem_desc(p_addr + kp * kPanelBytes, 16, 1024);
#pragma unroll
          for (int k4 = 0; k4 < 4; ++k4) {
            umma_bf16(tmem_base + kColO, d_p + k4 * (32 >> 4), d_v, idesc_o, (!first || kp > 0 || k4 > 0) ? 1u : 0u);
            d_v += 2048 >> 4;
          }
        }
        umma_commit(&bars->o_done);
        umma_commit(&bars->kv_empty[st]);
      };
      int it = 0, g = 0, pend = -1;
      bool pend_first = false;
      for (int item = blockIdx.x; item < p.num_items; item += gridDim.x, ++it) {
        const int qb = it & 1;
        mbar_wait(&bars->q_full[qb], (it >> 1) & 1);
        const uint32_t q_addr = smem_u32(sQ + qb * kTileBytes);
        for (int j = 0; j < p.tiles; ++j, ++g) {
          const int st = g % kFwdStages, slot = g & 1;
          mbar_wait(&bars->kv_full[st], (g / kFwdStages) & 1);
          mbar_wait(&bars->s_free[slot], ((g >> 1) & 1) ^ 1);
          tc_fence_after_sync();
          const uint32_t k_addr = smem_u32(sKV + st * 2 * kTileBytes);
#pragma unroll
          for (int k = 0; k < kDh / 16; ++k)
            umma_bf16(tmem_base + slot * kTile, umma_smem_desc(q_addr + kmajor_off(k), 16, 1024),
                      umma_smem_desc(k_addr + kmajor_off(k), 16, 1024), idesc_s, k > 0 ? 1u : 0u);
          umma_commit(&bars->s_full[slot]);
          if (j == p.tiles - 1) umma_commit(&bars->q_empty[qb]);
          if (pend >= 0) issue_pv(pend, pend_first);
          pend = g;
          pend_first = j == 0;
        }
      }
      if (pend >= 0) issue_pv(pend, pend_first);
    }
  } else {
    // ------------------------------- softmax + epilogue ---------------------------------
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t t_lane = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const uint32_t p_u32 = smem_u32(sP);
    const float sl2 = p.scale * kLog2e;
    const f32x2 sl2_2 = f2_splat(sl2);
    uint64_t dkey = 0;
    if constexpr (kDrop) dkey = drop_key_load(dp.key);
    int g = 0;
    for (int item = blockIdx.x; item < p.num_items; item += gridDim.x) {
      const int t = item % p.tiles, bh = item / p.tiles;
      const int h = bh % p.heads, b = bh / p.heads;
      float m_ref = -INFINITY;       // reference max of this row, log2 domain (raw score * scale * log2 e)
      float sum = 0.f;               // sum of exp2(s * sl2 - m_ref) over the keys seen so far
      for (int j = 0; j < p.tiles; ++j, ++g) {
        const int slot = g & 1;
        const int kvalid = min(kTile, n - j * kTile);   // keys of this tile inside the sequence (>= 1)
        const uint32_t ts = t_lane + slot * kTile;
        uint32_t keep[4];                               // kDrop: keep bits of the tile's 128 keys, while S is computed
        if constexpr (kDrop) {
#pragma unroll
          for (int q = 0; q < 4; ++q) keep[q] = drop_keep32(dkey, j * kTile + q * 32, t * kTile + row, bh, dp.site, dp.thr);
        }
        mbar_wait(&bars->s_full[slot], (g >> 1) & 1);
        tc_fence_after_sync();
        // ---- pass 1: tile max, four independent chains
        float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
        {
          uint32_t va[32], vb[32];
#pragma unroll
          for (int c = 0; c < 4; c += 2) {
            tmem_ld_32x32(ts + c * 32, va);
            tmem_ld_32x32(ts + (c + 1) * 32, vb);
            tmem_ld_wait();
            if ((c + 2) * 32 <= kvalid) {
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                mx4[e & 3] = fmaxf(mx4[e & 3], __uint_as_float(va[e]));
                mx4[e & 3] = fmaxf(mx4[e & 3], __uint_as_float(vb[e]));
              }
            } else {
#pragma unroll
              for (int e = 0; e < 32; ++e) {
                if (c * 32 + e < kvalid) mx4[e & 3] = fmaxf(mx4[e & 3], __uint_as_float(va[e]));
                if ((c + 1) * 32 + e < kvalid) mx4[e & 3] = fmaxf(mx4[e & 3], __uint_as_float(vb[e]));
              }
            }
          }
        }
        const float m_tile = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3])) * sl2;
        float corr = 1.f;
        if (m_tile > m_ref + kRescaleLog2) {            // always true for the first tile (m_ref = -inf)
          corr = exp2f(m_ref - m_tile);                 // 0 for the first tile
          m_ref = m_tile;
        }
        // ---- pass 2: P = exp2(s * sl2 - m_ref) -> packed bf16 registers; two partial sums
        uint32_t pw[64];
        float sum0 = 0.f, sum1 = 0.f;
        {
          const f32x2 nm2 = f2_splat(-m_ref);
          uint32_t va[32], vb[32];
#pragma unroll
          for (int c = 0; c < 4; c += 2) {
            tmem_ld_32x32(ts + c * 32, va);
            tmem_ld_32x32(ts + (c + 1) * 32, vb);
            tmem_ld_wait();
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2) {
              const uint32_t(&v)[32] = h2 == 0 ? va : vb;
              const int col0 = (c + h2) * 32;
              const bool full = col0 + 32 <= kvalid;
#pragma unroll
              for (int e = 0; e < 32; e += 2) {
                float a0, a1;
                f2_unpack(f2_fma(f2_packu(v[e], v[e + 1]), sl2_2, nm2), a0, a1);
                float p0 = exp2f(a0), p1 = exp2f(a1);
                if (!full) {
                  p0 = col0 + e < kvalid ? p0 : 0.f;
                  p1 = col0 + e + 1 < kvalid ? p1 : 0.f;
                }
                if (e & 2) sum1 += p0 + p1; else sum0 += p0 + p1;
                if constexpr (kDrop) {
                  p0 = (keep[(c + h2)] >> e) & 1u ? p0 * dp.scale : 0.f;
                  p1 = (keep[(c + h2)] >> (e + 1)) & 1u ? p1 * dp.scale : 0.f;
                }
                pw[(col0 + e) >> 1] = pack_bf16x2(p0, p1);
              }
            }
          }
        }
        tc_fence_before_sync();
        mbar_arrive(&bars->s_free[slot]);               // S slot may take the scores after next
        // ---- O of the previous tile complete: P buffer free, O may be rescaled
        if (g > 0) mbar_wait(&bars->o_done, (g - 1) & 1);
        tc_fence_after_sync();
        if (j > 0 && __any_sync(0xffffffffu, corr != 1.f)) {
          // 64 of the kN accumulator columns at a time (dh = 32 rescales its unread upper half too)
#pragma unroll
          for (int c0 = 0; c0 < kN; c0 += 64) {
            uint32_t o0[32], o1[32];
            tmem_ld_32x32(t_lane + kColO + c0, o0);
            tmem_ld_32x32(t_lane + kColO + c0 + 32, o1);
            tmem_ld_wait();
#pragma unroll
            for (int e = 0; e < 32; ++e) {
              o0[e] = __float_as_uint(__uint_as_float(o0[e]) * corr);
              o1[e] = __float_as_uint(__uint_as_float(o1[e]) * corr);
            }
            tmem_st_32x32(t_lane + kColO + c0, o0);
            tmem_st_32x32(t_lane + kColO + c0 + 32, o1);
            tmem_st_wait();
          }
        }
        sum = sum * corr + (sum0 + sum1);
#pragma unroll
        for (int ch = 0; ch < 16; ++ch)
          st_swz_chunk(p_u32 + (ch >> 3) * 16384, row, ch & 7,
                       make_uint4(pw[4 * ch], pw[4 * ch + 1], pw[4 * ch + 2], pw[4 * ch + 3]));
        fence_proxy_async_smem();
        tc_fence_before_sync();
        mbar_arrive(&bars->p_full);
      }
      // ---- epilogue: O / sum -> bf16, LSE
      mbar_wait(&bars->o_done, (g - 1) & 1);
      tc_fence_after_sync();
      if constexpr (kDh == 64) {
        uint32_t o0[32], o1[32];
        tmem_ld_32x32(t_lane + kColO, o0);
        tmem_ld_32x32(t_lane + kColO + 32, o1);
        tmem_ld_wait();
        const int grow = t * kTile + row;
        if (grow < n) {
          store_row64_scaled(p.out + ((size_t)b * n + grow) * p.inner + h * kDh, o0, o1, 1.0f / sum);
          if (p.lse) p.lse[((size_t)b * p.heads + h) * n + grow] = m_ref * kLn2 + __logf(sum);
        }
      } else {
        // the same through tmem_row_to_bf16 (kept apart so that the dh = 64 code is as it was before the other
        // widths were added)
        const int grow = t * kTile + row;
        tmem_row_to_bf16<kDh>(p.out + ((size_t)b * n + grow) * p.inner + h * kDh, t_lane + kColO, 1.0f / sum,
                              grow < n);
        if (grow < n && p.lse) p.lse[((size_t)b * p.heads + h) * n + grow] = m_ref * kLn2 + __logf(sum);
      }
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

template <int kDh>
__global__ void __launch_bounds__(192, 1)
attn_long_fwd_kernel(const __grid_constant__ CUtensorMap map_qkv, const LongFwdParams p) {
  attn_long_fwd_body<kDh, false>(map_qkv, p, DropParams{});
}

template <int kDh>
__global__ void __launch_bounds__(192, 1)
attn_long_drop_fwd_kernel(const __grid_constant__ CUtensorMap map_qkv, const LongFwdParams p, const DropParams dp) {
  attn_long_fwd_body<kDh, true>(map_qkv, p, dp);
}

// ------------------------------------------------------------------------------------------
// backward.  kKV = true: KV-stationary (dK, dV); false: Q-stationary (dQ).
// TMEM columns: [0,128) S  [128,256) dP  [256,256+kN) dV | dQ  [256+kN,256+2kN) dK
// ------------------------------------------------------------------------------------------
template <int kStages>
struct LongBwdBars {
  uint64_t stat_full, st_full[kStages], st_empty[kStages], sdp_full, sdp_free, pds_full, pds_free, acc_full;
  uint32_t tmem_base;
};

struct LongBwdParams {
  const bf16* o;
  const bf16* dout;
  const float* lse;
  const float* delta;   // [batch*n, heads] rowsum(dO * O), or nullptr (computed here from o / dout)
  bf16* dqkv;
  int n, heads, inner, tiles;
  float scale;
};

// delta = rowsum(dO * O) of one (token, head) row of kDh elements, from global memory
template <int kDh>
M3L_DEVINL float row_delta(const bf16* po, const bf16* pd) {
  float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
  for (int q = 0; q < kDh / 8; ++q) {
    const uint4 a = __ldg(reinterpret_cast<const uint4*>(po) + q);
    const uint4 d = __ldg(reinterpret_cast<const uint4*>(pd) + q);
    const float2 a0 = unpack_bf16x2(a.x), a1 = unpack_bf16x2(a.y), a2 = unpack_bf16x2(a.z), a3 = unpack_bf16x2(a.w);
    const float2 d0 = unpack_bf16x2(d.x), d1 = unpack_bf16x2(d.y), d2 = unpack_bf16x2(d.z), d3 = unpack_bf16x2(d.w);
    acc0 += a0.x * d0.x + a0.y * d0.y + a1.x * d1.x + a1.y * d1.y;
    acc1 += a2.x * d2.x + a2.y * d2.y + a3.x * d3.x + a3.y * d3.y;
  }
  return acc0 + acc1;
}

// kDrop: with the dropout mask Z (scale folded in) the P slab is P o Z and dS = P o (Z o dP - delta) scale; delta =
// rowsum(dO o O) is the same expression as without dropout.
template <int kDh, bool kKV, bool kDrop>
__device__ __forceinline__ void attn_long_bwd_body(const CUtensorMap& map_qkv, const CUtensorMap& map_do,
                                                   const LongBwdParams& p, const DropParams& dp) {
  using Cfg = LongCfg<kDh>;
  constexpr int kTileBytes = Cfg::kTileBytes, kN = Cfg::kN;
  constexpr int kBwdStages = Cfg::bwd_stages(kKV);
  constexpr bool kHasP = Cfg::bwd_has_p(kKV);
  constexpr bool kAhead = kBwdStages > 1;     // S / dP of step s+1 issued before the products of step s
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~static_cast<uintptr_t>(1023));
  uint8_t* sA = smem;                                   // stationary pair: [K | V] (kKV) or [Q | dO]
  uint8_t* sS = sA + 2 * kTileBytes;                    // streamed pairs:  [kBwdStages][Q | dO] (kKV) or [K | V]
  uint8_t* sP = sS + kBwdStages * 2 * kTileBytes;       // [2 slabs of 64 keys][128 q x 64] (kHasP)
  uint8_t* sDS = sP + (kHasP ? kPBytes : 0);            // same layout
  LongBwdBars<kBwdStages>* bars = reinterpret_cast<LongBwdBars<kBwdStages>*>(sDS + kPBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr uint32_t kTmemCols = 512, kColS = 0, kColDP = 128, kColA = 256, kColB = 256 + kN;
  const int n = p.n, tile = blockIdx.x, h = blockIdx.y, b = blockIdx.z;
  const int steps = p.tiles;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&map_qkv);
    tma_prefetch_desc(&map_do);
    mbar_init(&bars->stat_full, 1);
    for (int i = 0; i < kBwdStages; ++i) {
      mbar_init(&bars->st_full[i], 1);
      mbar_init(&bars->st_empty[i], 1);
    }
    mbar_init(&bars->sdp_full, 1);
    mbar_init(&bars->sdp_free, 256);
    mbar_init(&bars->pds_full, 256);
    mbar_init(&bars->pds_free, 1);
    mbar_init(&bars->acc_full, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(&bars->tmem_base, kTmemCols);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem_base = bars->tmem_base;
  pdl_wait();
  pdl_trigger();

  if (warp == 0) {
    // ------------------------------- TMA loader -----------------------------------------
    if (elect_one()) {
      constexpr int kPn = Cfg::kPanels;
      mbar_arrive_expect_tx(&bars->stat_full, 2 * kTileBytes);
      if (kKV) {
        tma_load_tile<kPn>(sA, &map_qkv, &bars->stat_full, p.inner + h * kDh, tile * kTile, b);
        tma_load_tile<kPn>(sA + kTileBytes, &map_qkv, &bars->stat_full, 2 * p.inner + h * kDh, tile * kTile, b);
      } else {
        tma_load_tile<kPn>(sA, &map_qkv, &bars->stat_full, h * kDh, tile * kTile, b);
        tma_load_tile<kPn>(sA + kTileBytes, &map_do, &bars->stat_full, h * kDh, tile * kTile, b);
      }
      for (int s = 0; s < steps; ++s) {
        const int st = s % kBwdStages;
        mbar_wait(&bars->st_empty[st], ((s / kBwdStages) & 1) ^ 1);
        uint8_t* dst = sS + st * 2 * kTileBytes;
        mbar_arrive_expect_tx(&bars->st_full[st], 2 * kTileBytes);
        if (kKV) {
          tma_load_tile<kPn>(dst, &map_qkv, &bars->st_full[st], h * kDh, s * kTile, b);
          tma_load_tile<kPn>(dst + kTileBytes, &map_do, &bars->st_full[st], h * kDh, s * kTile, b);
        } else {
          tma_load_tile<kPn>(dst, &map_qkv, &bars->st_full[st], p.inner + h * kDh, s * kTile, b);
          tma_load_tile<kPn>(dst + kTileBytes, &map_qkv, &bars->st_full[st], 2 * p.inner + h * kDh, s * kTile, b);
        }
      }
    }
  } else if (warp == 1) {
    // ------------------------------- MMA issuer -----------------------------------------
    if (elect_one()) {
      const uint32_t idesc_s = umma_idesc_bf16(128, kTile, 0, 0);
      const uint32_t idesc_dq = umma_idesc_bf16(128, kN, 0, 1);    // A K-major (dS), B MN-major (K)
      const uint32_t idesc_dkv = umma_idesc_bf16(128, kN, 1, 1);   // both MN-major
      const uint32_t a_addr = smem_u32(sA), p_addr = smem_u32(sP), ds_addr = smem_u32(sDS);
      auto s_addr = [&](int s) { return smem_u32(sS + (s % kBwdStages) * 2 * kTileBytes); };
      // S = Q K^T, dP = dO V^T of step s
      auto issue_sdp = [&](int s) {
        mbar_wait(&bars->st_full[s % kBwdStages], (s / kBwdStages) & 1);
        if (s > 0) mbar_wait(&bars->sdp_free, (s - 1) & 1);
        tc_fence_after_sync();
        const uint32_t q = kKV ? s_addr(s) : a_addr, dO = q + kTileBytes;
        const uint32_t k = kKV ? a_addr : s_addr(s), v = k + kTileBytes;
#pragma unroll
        for (int kk = 0; kk < kDh / 16; ++kk)
          umma_bf16(tmem_base + kColS, umma_smem_desc(q + kmajor_off(kk), 16, 1024),
                    umma_smem_desc(k + kmajor_off(kk), 16, 1024), idesc_s, kk > 0 ? 1u : 0u);
#pragma unroll
        for (int kk = 0; kk < kDh / 16; ++kk)
          umma_bf16(tmem_base + kColDP, umma_smem_desc(dO + kmajor_off(kk), 16, 1024),
                    umma_smem_desc(v + kmajor_off(kk), 16, 1024), idesc_s, kk > 0 ? 1u : 0u);
        umma_commit(&bars->sdp_full);
      };
      mbar_wait(&bars->stat_full, 0);
      if constexpr (kAhead) issue_sdp(0);
      for (int s = 0; s < steps; ++s) {
        if constexpr (kAhead) {
          if (s + 1 < steps) issue_sdp(s + 1);
        } else {
          issue_sdp(s);
        }
        mbar_wait(&bars->pds_full, s & 1);
        tc_fence_after_sync();
        if (kKV) {
          // dV += P^T dO, dK += dS^T Q: contraction over the 128 query rows of this step
          const uint32_t q = s_addr(s), dO = q + kTileBytes;
          uint64_t d_p = umma_smem_desc(p_addr, 16384, 1024), d_do = umma_smem_desc(dO, Cfg::kMnLbo, 1024);
          uint64_t d_ds = umma_smem_desc(ds_addr, 16384, 1024), d_q = umma_smem_desc(q, Cfg::kMnLbo, 1024);
#pragma unroll
          for (int kk = 0; kk < kTile / 16; ++kk) {
            const uint32_t acc = (s > 0 || kk > 0) ? 1u : 0u;
            umma_bf16(tmem_base + kColA, d_p, d_do, idesc_dkv, acc);
            umma_bf16(tmem_base + kColB, d_ds, d_q, idesc_dkv, acc);
            d_p += 2048 >> 4; d_do += 2048 >> 4; d_ds += 2048 >> 4; d_q += 2048 >> 4;
          }
        } else {
          // dQ += dS K: contraction over the 128 keys of this step, two 64-key panels
          uint64_t d_k = umma_smem_desc(s_addr(s), Cfg::kMnLbo, 1024);
#pragma unroll
          for (int kp = 0; kp < 2; ++kp) {
            const uint64_t d_a = umma_smem_desc(ds_addr + kp * 16384, 16, 1024);
#pragma unroll
            for (int k4 = 0; k4 < 4; ++k4) {
              umma_bf16(tmem_base + kColA, d_a + k4 * (32 >> 4), d_k, idesc_dq, (s > 0 || kp > 0 || k4 > 0) ? 1u : 0u);
              d_k += 2048 >> 4;
            }
          }
        }
        umma_commit(&bars->pds_free);
        umma_commit(&bars->st_empty[s % kBwdStages]);
      }
      umma_commit(&bars->acc_full);
    }
  } else {
    // ------------------------------- P / dS producers + epilogue ------------------------
    const int wg = (warp - 2) >> 2;
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    const uint32_t t_row = tmem_base + (static_cast<uint32_t>(quad * 32) << 16);
    const uint32_t p_slab = smem_u32(sP + wg * 16384), ds_slab = smem_u32(sDS + wg * 16384);
    const float sl2 = p.scale * kLog2e;
    const float* lse_bh = p.lse + ((size_t)b * p.heads + h) * n;
    // row statistics (log2-domain LSE, delta) of query row `grow`
    auto stats = [&](int grow, float& lg, float& dl) {
      lg = 0.f; dl = 0.f;
      if (grow < n) {
        lg = __ldg(lse_bh + grow) * kLog2e;
        if (p.delta != nullptr) {
          dl = __ldg(p.delta + ((size_t)b * n + grow) * p.heads + h);
        } else {
          const size_t off = ((size_t)b * n + grow) * p.inner + h * kDh;
          dl = row_delta<kDh>(p.o + off, p.dout + off);
        }
      }
    };
    float lg = 0.f, dl = 0.f;
    if (!kKV) stats(tile * kTile + row, lg, dl);
    uint64_t dkey = 0;
    if constexpr (kDrop) dkey = drop_key_load(dp.key);
    const uint32_t plane = (uint32_t)b * p.heads + h;
    for (int s = 0; s < steps; ++s) {
      const int qi = kKV ? s : tile, kj = kKV ? tile : s;
      const int grow = qi * kTile + row;
      const bool valid = grow < n;
      if (kKV) stats(grow, lg, dl);
      const int key0 = kj * kTile + wg * 64;
      const bool interior = (qi * kTile + quad * 32 + 32 <= n) && (key0 + 64 <= n);   // warp-uniform
      uint32_t keep[2];                                 // kDrop: keep bits of this thread's 64 keys, while S / dP are computed
      if constexpr (kDrop) {
        keep[0] = drop_keep32(dkey, key0, grow, plane, dp.site, dp.thr);
        keep[1] = drop_keep32(dkey, key0 + 32, grow, plane, dp.site, dp.thr);
      }
      mbar_wait(&bars->sdp_full, s & 1);
      tc_fence_after_sync();
      uint32_t pw[32], dw[32];
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        uint32_t sv[32], dv[32];
        tmem_ld_32x32(t_row + kColS + wg * 64 + c * 32, sv);
        tmem_ld_32x32(t_row + kColDP + wg * 64 + c * 32, dv);
        tmem_ld_wait();
        if (c == 1) {
          tc_fence_before_sync();
          mbar_arrive(&bars->sdp_free);
        }
        if (interior) {
          const f32x2 sl2_2 = f2_splat(sl2), nlg2 = f2_splat(-lg), ndl2 = f2_splat(-dl), sc2 = f2_splat(p.scale);
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            float t0, t1;
            f2_unpack(f2_fma(f2_packu(sv[e], sv[e + 1]), sl2_2, nlg2), t0, t1);
            const float p0 = exp2f(t0), p1 = exp2f(t1);
            f32x2 dpv = f2_packu(dv[e], dv[e + 1]);
            float z0 = 1.f, z1 = 1.f;
            if constexpr (kDrop) {
              z0 = (keep[c] >> e) & 1u ? dp.scale : 0.f;
              z1 = (keep[c] >> (e + 1)) & 1u ? dp.scale : 0.f;
              dpv = f2_mul(dpv, f2_pack(z0, z1));
            }
            const f32x2 ds = f2_mul(f2_mul(f2_pack(p0, p1), f2_add(dpv, ndl2)), sc2);
            float d0, d1;
            f2_unpack(ds, d0, d1);
            if constexpr (kDrop) pw[c * 16 + (e >> 1)] = pack_bf16x2(p0 * z0, p1 * z1);
            else pw[c * 16 + (e >> 1)] = pack_bf16x2(p0, p1);
            dw[c * 16 + (e >> 1)] = pack_bf16x2(d0, d1);
          }
        } else {
#pragma unroll
          for (int e = 0; e < 32; e += 2) {
            const int key = key0 + c * 32 + e;
            const float p0 = exp2f(fmaf(__uint_as_float(sv[e]), sl2, -lg));
            const float p1 = exp2f(fmaf(__uint_as_float(sv[e + 1]), sl2, -lg));
            const float q0 = (valid && key < n) ? p0 : 0.f, q1 = (valid && key + 1 < n) ? p1 : 0.f;
            float dp0 = __uint_as_float(dv[e]), dp1 = __uint_as_float(dv[e + 1]);
            if constexpr (kDrop) {
              const float z0 = (keep[c] >> e) & 1u ? dp.scale : 0.f, z1 = (keep[c] >> (e + 1)) & 1u ? dp.scale : 0.f;
              dp0 *= z0;
              dp1 *= z1;
              pw[c * 16 + (e >> 1)] = pack_bf16x2(q0 * z0, q1 * z1);
            } else {
              pw[c * 16 + (e >> 1)] = pack_bf16x2(q0, q1);
            }
            dw[c * 16 + (e >> 1)] = pack_bf16x2(q0 * (dp0 - dl) * p.scale, q1 * (dp1 - dl) * p.scale);
          }
        }
      }
      // the slabs are still read by the previous step's accumulating products
      if (s > 0) mbar_wait(&bars->pds_free, (s - 1) & 1);
#pragma unroll
      for (int ch = 0; ch < 8; ++ch) {
        if (kHasP)
          st_swz_chunk(p_slab, row, ch, make_uint4(pw[4 * ch], pw[4 * ch + 1], pw[4 * ch + 2], pw[4 * ch + 3]));
        st_swz_chunk(ds_slab, row, ch, make_uint4(dw[4 * ch], dw[4 * ch + 1], dw[4 * ch + 2], dw[4 * ch + 3]));
      }
      fence_proxy_async_smem();
      tc_fence_before_sync();
      mbar_arrive(&bars->pds_full);
    }
    // ---- epilogue
    mbar_wait(&bars->acc_full, 0);
    tc_fence_after_sync();
    if constexpr (kDh == 64) {
      // the general form below, as written before the other widths were added
      if (kKV) {
        // group 0: dV, group 1: dK of key row `row` of this tile
        uint32_t a0[32], a1[32];
        const uint32_t col = wg == 0 ? kColA : kColB;
        tmem_ld_32x32(t_row + col, a0);
        tmem_ld_32x32(t_row + col + 32, a1);
        tmem_ld_wait();
        const int key = tile * kTile + row;
        if (key < n)
          store_row64_scaled(p.dqkv + ((size_t)b * n + key) * 3 * p.inner + (wg == 0 ? 2 : 1) * p.inner + h * kDh, a0,
                             a1, 1.f);
      } else {
        // group w: dQ columns [32 w, 32 w + 32) of query row `row`
        uint32_t a0[32];
        tmem_ld_32x32(t_row + kColA + wg * 32, a0);
        tmem_ld_wait();
        const int grow = tile * kTile + row;
        if (grow < n) {
          bf16* dst = p.dqkv + ((size_t)b * n + grow) * 3 * p.inner + h * kDh + wg * 32;
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            uint4 u;
            u.x = pack_bf16x2(__uint_as_float(a0[g * 8 + 0]), __uint_as_float(a0[g * 8 + 1]));
            u.y = pack_bf16x2(__uint_as_float(a0[g * 8 + 2]), __uint_as_float(a0[g * 8 + 3]));
            u.z = pack_bf16x2(__uint_as_float(a0[g * 8 + 4]), __uint_as_float(a0[g * 8 + 5]));
            u.w = pack_bf16x2(__uint_as_float(a0[g * 8 + 6]), __uint_as_float(a0[g * 8 + 7]));
            *reinterpret_cast<uint4*>(dst + g * 8) = u;
          }
        }
      }
    } else if (kKV) {
      // group 0: dV, group 1: dK of key row `row` of this tile
      const uint32_t col = wg == 0 ? kColA : kColB;
      const int key = tile * kTile + row;
      tmem_row_to_bf16<kDh>(p.dqkv + ((size_t)b * n + key) * 3 * p.inner + (wg == 0 ? 2 : 1) * p.inner + h * kDh,
                            t_row + col, 1.f, key < n);
    } else {
      // group w: dQ columns [w dh/2, (w + 1) dh/2) of query row `row`
      constexpr int kHalf = kDh / 2;
      const int grow = tile * kTile + row;
      tmem_row_to_bf16<kHalf>(p.dqkv + ((size_t)b * n + grow) * 3 * p.inner + h * kDh + wg * kHalf,
                              t_row + kColA + wg * kHalf, 1.f, grow < n);
    }
  }
  tc_fence_before_sync();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after_sync();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

template <int kDh, bool kKV>
__global__ void __launch_bounds__(320, 1)
attn_long_bwd_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_do,
                     const LongBwdParams p) {
  attn_long_bwd_body<kDh, kKV, false>(map_qkv, map_do, p, DropParams{});
}

template <int kDh, bool kKV>
__global__ void __launch_bounds__(320, 1)
attn_long_drop_bwd_kernel(const __grid_constant__ CUtensorMap map_qkv, const __grid_constant__ CUtensorMap map_do,
                          const LongBwdParams p, const DropParams dp) {
  attn_long_bwd_body<kDh, kKV, true>(map_qkv, map_do, p, dp);
}

// ------------------------------------------------------------------------------------------
// host launchers (arguments already checked by the entry points)
// ------------------------------------------------------------------------------------------
// kDrop: the dropout kernels (attention_dropout.cu), with the mask of `dp`
template <int kDh, bool kDrop = false>
int long_fwd_launch(const char* who, const void* qkv_bf16, int batch, int n, int heads, float scale, void* out_bf16,
                    float* lse, void* stream, const DropParams& dp = DropParams{}) {
  using Cfg = LongCfg<kDh>;
  const int inner = heads * kDh;
  CUtensorMap map_qkv;
  int s = make_tmap_3d_bf16(&map_qkv, qkv_bf16, 3 * inner, n, batch, 3 * inner, (uint64_t)n * 3 * inner, kTile);
  if (s) return s;
  LongFwdParams p;
  p.out = (bf16*)out_bf16; p.lse = lse; p.n = n; p.heads = heads; p.inner = inner; p.scale = scale;
  p.tiles = (n + kTile - 1) / kTile;
  const long long items = (long long)batch * heads * p.tiles;
  M3L_REQUIRE(items < (1ll << 31), "%s: too many (sample, head, tile) items", who);
  p.num_items = (int)items;
  static bool configured = false;
  const int grid = std::min(p.num_items, device_sm_count());
  if constexpr (kDrop) {
    if (!configured) {
      M3L_CUDA(cudaFuncSetAttribute(attn_long_drop_fwd_kernel<kDh>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    Cfg::kFwdSmem));
      configured = true;
    }
    M3L_CUDA(launch_kernel(attn_long_drop_fwd_kernel<kDh>, dim3(grid), dim3(192), Cfg::kFwdSmem, (cudaStream_t)stream,
                           map_qkv, p, dp));
  } else {
    if (!configured) {
      M3L_CUDA(cudaFuncSetAttribute(attn_long_fwd_kernel<kDh>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    Cfg::kFwdSmem));
      configured = true;
    }
    M3L_CUDA(launch_kernel(attn_long_fwd_kernel<kDh>, dim3(grid), dim3(192), Cfg::kFwdSmem, (cudaStream_t)stream,
                           map_qkv, p));
  }
  M3L_CUDA(cudaGetLastError());
  return M3L_OK;
}

template <int kDh, bool kDrop = false>
int long_bwd_launch(const char* who, const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                    const float* lse, const float* delta, int batch, int n, int heads, float scale, void* dqkv_bf16,
                    void* stream, const DropParams& dp = DropParams{}) {
  using Cfg = LongCfg<kDh>;
  M3L_REQUIRE(batch <= 65535, "%s: batch %d > 65535", who, batch);
  const int inner = heads * kDh;
  CUtensorMap map_qkv, map_do;
  int s = make_tmap_3d_bf16(&map_qkv, qkv_bf16, 3 * inner, n, batch, 3 * inner, (uint64_t)n * 3 * inner, kTile);
  if (s) return s;
  s = make_tmap_3d_bf16(&map_do, dout_bf16, inner, n, batch, inner, (uint64_t)n * inner, kTile);
  if (s) return s;
  LongBwdParams p;
  p.o = (const bf16*)out_bf16; p.dout = (const bf16*)dout_bf16; p.lse = lse; p.delta = delta;
  p.dqkv = (bf16*)dqkv_bf16;
  p.n = n; p.heads = heads; p.inner = inner; p.scale = scale;
  p.tiles = (n + kTile - 1) / kTile;
  constexpr int kSmemQ = Cfg::bwd_smem(false), kSmemKV = Cfg::bwd_smem(true);
  static bool configured = false;
  const dim3 grid(p.tiles, heads, batch);
  if constexpr (kDrop) {
    if (!configured) {
      M3L_CUDA(cudaFuncSetAttribute(attn_long_drop_bwd_kernel<kDh, false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    kSmemQ));
      M3L_CUDA(cudaFuncSetAttribute(attn_long_drop_bwd_kernel<kDh, true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    kSmemKV));
      configured = true;
    }
    M3L_CUDA(launch_kernel(attn_long_drop_bwd_kernel<kDh, false>, grid, dim3(320), kSmemQ, (cudaStream_t)stream,
                           map_qkv, map_do, p, dp));
    M3L_CUDA(cudaGetLastError());
    M3L_CUDA(launch_kernel(attn_long_drop_bwd_kernel<kDh, true>, grid, dim3(320), kSmemKV, (cudaStream_t)stream,
                           map_qkv, map_do, p, dp));
  } else {
    if (!configured) {
      M3L_CUDA(cudaFuncSetAttribute(attn_long_bwd_kernel<kDh, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemQ));
      M3L_CUDA(cudaFuncSetAttribute(attn_long_bwd_kernel<kDh, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemKV));
      configured = true;
    }
    M3L_CUDA(launch_kernel(attn_long_bwd_kernel<kDh, false>, grid, dim3(320), kSmemQ, (cudaStream_t)stream, map_qkv,
                           map_do, p));
    M3L_CUDA(cudaGetLastError());
    M3L_CUDA(launch_kernel(attn_long_bwd_kernel<kDh, true>, grid, dim3(320), kSmemKV, (cudaStream_t)stream, map_qkv,
                           map_do, p));
  }
  M3L_CUDA(cudaGetLastError());
  return M3L_OK;
}

}  // namespace
}  // namespace m3l
