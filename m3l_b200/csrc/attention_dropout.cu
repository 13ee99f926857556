// m3l_b200 — multi-head attention with dropout on the attention probabilities (vit_pytorch Attention's
// `attn = self.dropout(attn)` before `attn @ v`, training mode), forward and backward, for 32-, 64- and 128-wide heads
// and any sequence length: the kDrop instantiations of attention_long.cuh.  The mask is dropout.cuh's, with
// row = query index, col = key index, plane = sample * heads + head.
//   forward:  the row sums and the LSE use the undropped P (lse is the lse without dropout); O = (P o Z) V / sum.
//   backward: dV = (P o Z)^T dO, dS = P o (Z o dP - delta) scale, delta = rowsum(dO o O) as without dropout.
// Z holds 0 or 65536 / (65536 - thr).  At p = 0 every result is bit-identical to the kernels without dropout.
#include "attention_long.cuh"

namespace m3l {
namespace {

int drop_attn_check(const char* who, int n, int heads, int dim_head, int batch, const int64_t* key, float p,
                    DropParams* dp) {
  if (dim_head != 32 && dim_head != 64 && dim_head != 128) {
    set_last_error("%s: dim_head=%d unsupported (32, 64 or 128)", who, dim_head);
    return M3L_ERR_UNSUPPORTED;
  }
  M3L_REQUIRE(n >= 1 && heads >= 1 && batch >= 0, "%s: bad n/heads/batch (%d, %d, %d)", who, n, heads, batch);
  M3L_REQUIRE(drop_threshold(p, &dp->thr, &dp->scale), "%s: dropout probability %g outside [0, 1)", who, (double)p);
  M3L_REQUIRE(key != nullptr || dp->thr == 0, "%s: null dropout key with p > 0", who);
  dp->key = key;
  return M3L_OK;
}

}  // namespace
}  // namespace m3l

using namespace m3l;

extern "C" int m3l_attention_dropout_fwd(const void* qkv_bf16, int batch, int n, int heads, int dim_head, float scale,
                                         const int64_t* drop_key, int drop_site, float drop_p, void* out_bf16,
                                         float* lse, void* stream) {
  const char* who = "attention_dropout_fwd";
  M3L_REQUIRE(qkv_bf16 && out_bf16, "%s: null pointer", who);
  DropParams dp;
  int s = drop_attn_check(who, n, heads, dim_head, batch, drop_key, drop_p, &dp);
  if (s) return s;
  dp.site = (uint32_t)drop_site;
  if (batch == 0) return M3L_OK;
  switch (dim_head) {
    case 32: return long_fwd_launch<32, true>(who, qkv_bf16, batch, n, heads, scale, out_bf16, lse, stream, dp);
    case 64: return long_fwd_launch<64, true>(who, qkv_bf16, batch, n, heads, scale, out_bf16, lse, stream, dp);
    default: return long_fwd_launch<128, true>(who, qkv_bf16, batch, n, heads, scale, out_bf16, lse, stream, dp);
  }
}

extern "C" int m3l_attention_dropout_bwd(const void* qkv_bf16, const void* out_bf16, const void* dout_bf16,
                                         const float* lse, const float* delta, int batch, int n, int heads,
                                         int dim_head, float scale, const int64_t* drop_key, int drop_site,
                                         float drop_p, void* dqkv_bf16, void* stream) {
  const char* who = "attention_dropout_bwd";
  M3L_REQUIRE(qkv_bf16 && out_bf16 && dout_bf16 && lse && dqkv_bf16, "%s: null pointer", who);
  DropParams dp;
  int s = drop_attn_check(who, n, heads, dim_head, batch, drop_key, drop_p, &dp);
  if (s) return s;
  dp.site = (uint32_t)drop_site;
  if (batch == 0) return M3L_OK;
  switch (dim_head) {
    case 32:
      return long_bwd_launch<32, true>(who, qkv_bf16, out_bf16, dout_bf16, lse, delta, batch, n, heads, scale,
                                       dqkv_bf16, stream, dp);
    case 64:
      return long_bwd_launch<64, true>(who, qkv_bf16, out_bf16, dout_bf16, lse, delta, batch, n, heads, scale,
                                       dqkv_bf16, stream, dp);
    default:
      return long_bwd_launch<128, true>(who, qkv_bf16, out_bf16, dout_bf16, lse, delta, batch, n, heads, scale,
                                        dqkv_bf16, stream, dp);
  }
}
