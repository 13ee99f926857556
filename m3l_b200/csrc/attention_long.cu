// m3l_b200 — fused multi-head attention for sequences of any length, dim_head = 64, on tcgen05 / TMEM / TMA
// (sm_100a), forward and backward.  The kernels are the kDh = 64 instantiation of attention_long.cuh (algorithm and
// layouts described there); attention_dh.cu instantiates the 32- and 128-wide heads.
#include "attention_long.cuh"

namespace m3l {
namespace {

int long_check(int n, int heads, int dim_head, int batch) {
  if (dim_head != 64) {
    set_last_error("attention_long: dim_head=%d unsupported (only 64)", dim_head);
    return M3L_ERR_UNSUPPORTED;
  }
  M3L_REQUIRE(n >= 1 && heads >= 1 && batch >= 0, "attention_long: bad n/heads/batch (%d, %d, %d)", n, heads, batch);
  return M3L_OK;
}

}  // namespace
}  // namespace m3l

using namespace m3l;

extern "C" int m3l_attention_long_fwd(const void* qkv_bf16, int batch, int n, int heads, int dim_head, float scale,
                                      void* out_bf16, float* lse, void* stream) {
  M3L_REQUIRE(qkv_bf16 && out_bf16, "attention_long_fwd: null pointer");
  int s = long_check(n, heads, dim_head, batch);
  if (s) return s;
  if (batch == 0) return M3L_OK;
  return long_fwd_launch<64>("attention_long_fwd", qkv_bf16, batch, n, heads, scale, out_bf16, lse, stream);
}

extern "C" int m3l_attention_long_bwd(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                                      const float* lse, const float* delta, int batch, int n, int heads, int dim_head,
                                      float scale, void* dqkv_bf16, void* stream) {
  M3L_REQUIRE(qkv_bf16 && out_bf16 && dout_bf16 && lse && dqkv_bf16, "attention_long_bwd: null pointer");
  int s = long_check(n, heads, dim_head, batch);
  if (s) return s;
  if (batch == 0) return M3L_OK;
  return long_bwd_launch<64>("attention_long_bwd", qkv_bf16, out_bf16, dout_bf16, lse, delta, batch, n, heads, scale,
                             dqkv_bf16, stream);
}
