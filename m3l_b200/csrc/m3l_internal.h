// m3l_b200 — internal (C++) declarations shared by the kernels and the step engine.
#pragma once

#include "../../include/m3l_b200.h"
#include "common.cuh"

namespace m3l {

// ----------------------------------------------------------------------------- GEMM (gemm.cu)
struct GemmArgs {
  const void* a = nullptr;  // bf16; K-major: [M, K] (lda); MN-major: [K, M] (lda)
  const void* b = nullptr;  // bf16; K-major: [N, K] (ldb); MN-major: [K, N] (ldb)
  int lda = 0, ldb = 0;
  int a_mn_major = 0, b_mn_major = 0;
  int M = 0, N = 0, K = 0;
  int splits = 1;           // split-K (requires out_mode 2)
  void* out = nullptr;      // [M, ldo]
  int ldo = 0;
  int out_mode = 0;         // 0 bf16 store, 1 fp32 store, 2 fp32 red.add
  const float* bias = nullptr;      // [N] fp32
  const bf16* residual = nullptr;   // [M, ldr] bf16, added after activation
  int ldr = 0;
  int act = 0;              // 0 none; 1 GELU (aux_out <- GELU'(pre-activation)); 2 multiply by aux_in; 3 ReLU
  bf16* aux_out = nullptr;
  const bf16* aux_in = nullptr;
  int ld_aux = 0;
  float alpha = 1.0f;
  float* colsum_out = nullptr;  // [N] fp32: += column sums of the (bf16) output, e.g. the bias gradient
  bf16* out2 = nullptr;             // [M, ldo] bf16: second copy of the output (EPI_BF16 with a residual)
  const bf16* dot_side = nullptr;   // [M, ld_dot] bf16: dot_out[row, c] = sum_{j<64} out[row, 64c+j] * dot_side[row, 64c+j]
  int ld_dot = 0;
  float* dot_out = nullptr;         // [M, N/64] fp32
  // fused LayerNorm backward epilogue (EPI_LN_BWD; see m3l_gemm_args in include/m3l_b200.h)
  const bf16* ln_x = nullptr;
  const float* ln_stats = nullptr;
  const float* ln_gamma = nullptr;
  const bf16* ln_skip = nullptr;
  float* ln_dgamma = nullptr;
  float* ln_dbeta = nullptr;
  float* ln_dxcol = nullptr;
  // dropout epilogues (EPI_GELU_DROP / EPI_BF16_DROP; mask of dropout.cuh): key on the device, threshold / scale
  // derived from drop_p by gemm_make_plan
  const int64_t* drop_key = nullptr;
  uint32_t drop_site = 0;
  float drop_p = 0.f;
  uint32_t drop_thr = 0;
  float drop_scale = 1.f;
};

struct GemmPlan {
  CUtensorMap map_a, map_b;
  CUtensorMap map_out, map_aux, map_side;   // epilogue tiles: output, second output (GELU' / out2), side operand
  GemmArgs args;
  int bn = 0;
  int grid = 0;
  bool ws = false;          // weight-stationary schedule (gemm.cu)
  bool gelu16 = false;      // FF1 forward shape: the 16-epilogue-warp GELU kernel (gemm_gelu.cu)
  CUtensorMap map_out32, map_aux32;   // its 32-column (64 B, SWIZZLE_64B) output tiles
};

int gemm_pick_bn(int M, int N);
int gemm_make_plan(GemmPlan* plan, const GemmArgs& args, int bn /*0 = auto*/);
int gemm_run(const GemmPlan& plan, cudaStream_t stream);
int gemm_gelu16_run(const GemmPlan& plan, cudaStream_t stream);   // gemm_gelu.cu

}  // namespace m3l
