// m3l_b200 — fused multi-head attention for 32- and 128-wide heads, any sequence length, on tcgen05 / TMEM / TMA
// (sm_100a), forward and backward: the kDh = 32 and 128 instantiations of attention_long.cuh (algorithm, layouts and
// the shared / tensor memory budget of each width are described there).  64-wide heads have their own entry points
// (m3l_attention_fwd/bwd for n <= 256, m3l_attention_long_fwd/bwd for any n).
#include "attention_long.cuh"

namespace m3l {
namespace {

int dh_check(int n, int heads, int dim_head, int batch) {
  if (dim_head != 32 && dim_head != 128) {
    set_last_error("attention_dh: dim_head=%d unsupported (32 or 128; 64 has its own kernels)", dim_head);
    return M3L_ERR_UNSUPPORTED;
  }
  M3L_REQUIRE(n >= 1 && heads >= 1 && batch >= 0, "attention_dh: bad n/heads/batch (%d, %d, %d)", n, heads, batch);
  return M3L_OK;
}

}  // namespace
}  // namespace m3l

using namespace m3l;

extern "C" int m3l_attention_dh_fwd(const void* qkv_bf16, int batch, int n, int heads, int dim_head, float scale,
                                    void* out_bf16, float* lse, void* stream) {
  M3L_REQUIRE(qkv_bf16 && out_bf16, "attention_dh_fwd: null pointer");
  int s = dh_check(n, heads, dim_head, batch);
  if (s) return s;
  if (batch == 0) return M3L_OK;
  return dim_head == 32
             ? long_fwd_launch<32>("attention_dh_fwd", qkv_bf16, batch, n, heads, scale, out_bf16, lse, stream)
             : long_fwd_launch<128>("attention_dh_fwd", qkv_bf16, batch, n, heads, scale, out_bf16, lse, stream);
}

extern "C" int m3l_attention_dh_bwd(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                                    const float* lse, const float* delta, int batch, int n, int heads, int dim_head,
                                    float scale, void* dqkv_bf16, void* stream) {
  M3L_REQUIRE(qkv_bf16 && out_bf16 && dout_bf16 && lse && dqkv_bf16, "attention_dh_bwd: null pointer");
  int s = dh_check(n, heads, dim_head, batch);
  if (s) return s;
  if (batch == 0) return M3L_OK;
  return dim_head == 32 ? long_bwd_launch<32>("attention_dh_bwd", qkv_bf16, out_bf16, dout_bf16, lse, delta, batch, n,
                                              heads, scale, dqkv_bf16, stream)
                        : long_bwd_launch<128>("attention_dh_bwd", qkv_bf16, out_bf16, dout_bf16, lse, delta, batch,
                                               n, heads, scale, dqkv_bf16, stream);
}
