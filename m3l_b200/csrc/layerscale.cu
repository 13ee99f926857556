// m3l_b200 — LayerScale fold / unfold for fine-tuning DINOv2 (m3l_b200/dinov2.py).
//
// The forward folds a block's LayerScale gamma into the Linear before it: W' = gamma o W (row i scaled by gamma_i),
// b' = gamma o b, so the projection / FF2 GEMMs need no extra epilogue.  Training keeps the fold:
//   fold:   bf16 W' in the plain [rows, cols] and the transposed [cols, rows] layouts (the dgrad GEMMs read W'^T),
//           fp32 b'.  The product is one fp32 multiply rounded to nearest, then rounded to bf16 (nearest even), which
//           is what torch's (gamma[:, None] * W).to(torch.bfloat16) computes, so the operands are bit-identical to the
//           frozen path's.  gamma == nullptr casts W unscaled (the qkv / FF1 weights).
//   unfold: from the fp32 gradients dW', db' of the folded Linear:
//           dW = gamma o dW',  db = gamma o db',  dgamma_i = sum_j W_ij dW'_ij + b_i db'_i.
#include "common.cuh"
#include "m3l_internal.h"

namespace m3l {
namespace {

__global__ void layerscale_fold_kernel(const float* __restrict__ w, const float* __restrict__ b,
                                       const float* __restrict__ gamma, int rows, int cols, bf16* __restrict__ wf,
                                       bf16* __restrict__ wf_t, float* __restrict__ bf) {
  pdl_wait();
  pdl_trigger();
  __shared__ bf16 tile[32][34];
  const int tiles_c = (cols + 31) / 32, tiles_r = (rows + 31) / 32;
  for (int t = blockIdx.x; t < tiles_r * tiles_c; t += gridDim.x) {
    const int tr = t / tiles_c, tc = t - tr * tiles_c;
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {
      const int r = tr * 32 + i, c = tc * 32 + threadIdx.x;
      if (r < rows && c < cols) {
        const float v = gamma ? __fmul_rn(gamma[r], w[(size_t)r * cols + c]) : w[(size_t)r * cols + c];
        const bf16 h = __float2bfloat16_rn(v);
        wf[(size_t)r * cols + c] = h;
        tile[i][threadIdx.x] = h;
      }
      if (bf && tc == 0 && threadIdx.x == 0 && r < rows) bf[r] = gamma ? __fmul_rn(gamma[r], b[r]) : b[r];
    }
    __syncthreads();
    if (wf_t) {
      for (int i = threadIdx.y; i < 32; i += blockDim.y) {
        const int c = tc * 32 + i, r = tr * 32 + threadIdx.x;
        if (r < rows && c < cols) wf_t[(size_t)c * rows + r] = tile[threadIdx.x][i];
      }
    }
    __syncthreads();
  }
}

// one block per row
__global__ void layerscale_unfold_kernel(const float* __restrict__ dwf, const float* __restrict__ dbf,
                                         const float* __restrict__ w, const float* __restrict__ b,
                                         const float* __restrict__ gamma, int cols, float* __restrict__ dw,
                                         float* __restrict__ db, float* __restrict__ dgamma) {
  pdl_wait();
  pdl_trigger();
  __shared__ float red[32];
  const int r = blockIdx.x;
  const float g = gamma[r];
  const float* dwr = dwf + (size_t)r * cols;
  const float* wr = w + (size_t)r * cols;
  float* dwo = dw + (size_t)r * cols;
  float acc = 0.f;
  for (int c = threadIdx.x; c < cols; c += blockDim.x) {
    const float d = dwr[c];
    dwo[c] = g * d;
    acc = fmaf(wr[c], d, acc);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) red[warp] = acc;
  __syncthreads();
  if (warp == 0) {
    float t = lane < (int)(blockDim.x >> 5) ? red[lane] : 0.f;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    if (lane == 0) {
      db[r] = g * dbf[r];
      dgamma[r] = fmaf(b[r], dbf[r], t);
    }
  }
}

}  // namespace
}  // namespace m3l

using namespace m3l;

extern "C" int m3l_layerscale_fold(const float* w, const float* b, const float* gamma, int rows, int cols,
                                   void* wf_bf16, void* wf_t_bf16, float* bf, void* stream) {
  M3L_REQUIRE(w && wf_bf16, "layerscale_fold: null pointer");
  M3L_REQUIRE(bf == nullptr || b != nullptr, "layerscale_fold: bf needs b");
  M3L_REQUIRE(rows > 0 && cols > 0, "layerscale_fold: empty matrix %d x %d", rows, cols);
  const int tiles = ((rows + 31) / 32) * ((cols + 31) / 32);
  const int grid = std::min(tiles, device_sm_count() * 8);
  M3L_CUDA(launch_kernel(layerscale_fold_kernel, dim3(grid), dim3(32, 8), 0, (cudaStream_t)stream, w, b, gamma, rows,
                         cols, (bf16*)wf_bf16, (bf16*)wf_t_bf16, bf));
  M3L_CUDA(cudaGetLastError());
  return M3L_OK;
}

extern "C" int m3l_layerscale_unfold(const float* dwf, const float* dbf, const float* w, const float* b,
                                     const float* gamma, int rows, int cols, float* dw, float* db, float* dgamma,
                                     void* stream) {
  M3L_REQUIRE(dwf && dbf && w && b && gamma && dw && db && dgamma, "layerscale_unfold: null pointer");
  M3L_REQUIRE(rows > 0 && cols > 0, "layerscale_unfold: empty matrix %d x %d", rows, cols);
  M3L_CUDA(launch_kernel(layerscale_unfold_kernel, dim3(rows), dim3(256), 0, (cudaStream_t)stream, dwf, dbf, w, b,
                         gamma, cols, dw, db, dgamma));
  M3L_CUDA(cudaGetLastError());
  return M3L_OK;
}
