// m3l_b200 — the dropout mask: one definition for every kernel that applies dropout (attention_dropout.cu, the
// GEMM epilogues of gemm.cu, m3l_dropout_bwd in elementwise.cu) and for the numpy reference of the tests.
//
// The mask is a pure function of logical coordinates, never of tiling, grid or stream, so the forward and the
// backward kernels agree by construction and a host-side generator can regenerate it:
//   Philox4x32-10 (Random123 / cuRAND), key = the 64-bit dropout key (read from device memory by the kernels),
//   counter = (col >> 3, row, plane, site)
//     attention:   row = query index, col = key index, plane = sample * heads + head
//     activations: row / col of the [rows, features] matrix, plane = 0
//     site = (layer << 2) | s, s = 0 attention probabilities, 1 attention output, 2 after GELU, 3 FF output.
// The four output words are eight 16-bit uniforms, low half first; element `col & 7` keeps when its uniform is
// >= thr = floor(p * 65536 + 0.5) and is then multiplied by 65536 / (65536 - thr), so the expectation is exact.
#pragma once
#include <cmath>
#include <cstdint>

namespace m3l {

struct DropParams {
  const int64_t* key = nullptr;   // device; NULL only with thr == 0 (nothing dropped)
  uint32_t site = 0;
  uint32_t thr = 0;               // keep iff u16 >= thr
  float scale = 1.f;              // 65536 / (65536 - thr)
};

__host__ __device__ __forceinline__ void philox_mulhilo(uint32_t a, uint32_t b, uint32_t& hi, uint32_t& lo) {
#ifdef __CUDA_ARCH__
  lo = a * b;
  hi = __umulhi(a, b);
#else
  const uint64_t p = (uint64_t)a * b;
  lo = (uint32_t)p;
  hi = (uint32_t)(p >> 32);
#endif
}

// Philox4x32-10 of counter c under key (k0, k1); c is overwritten with the output
__host__ __device__ __forceinline__ void philox4x32_10(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
#ifdef __CUDA_ARCH__
  // opaque to the optimiser: the ten round keys are formed here, not hoisted out of the caller's loops, where they
  // would hold 18 registers for the whole kernel
  asm volatile("" : "+r"(k0), "+r"(k1));
#endif
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    if (r > 0) {
      k0 += 0x9E3779B9u;
      k1 += 0xBB67AE85u;
    }
    uint32_t hi0, lo0, hi1, lo1;
    philox_mulhilo(0xD2511F53u, c[0], hi0, lo0);
    philox_mulhilo(0xCD9E8D57u, c[2], hi1, lo1);
    const uint32_t x0 = hi1 ^ c[1] ^ k0, x2 = hi0 ^ c[3] ^ k1;
    c[0] = x0; c[1] = lo1; c[2] = x2; c[3] = lo0;
  }
}

// the four Philox words serving columns [col0, col0 + 8) of `row` (col0 a multiple of 8)
__host__ __device__ __forceinline__ void drop_words(uint32_t (&w)[4], uint64_t key, uint32_t col0, uint32_t row,
                                                    uint32_t plane, uint32_t site) {
  w[0] = col0 >> 3; w[1] = row; w[2] = plane; w[3] = site;
  philox4x32_10(w, (uint32_t)key, (uint32_t)(key >> 32));
}

// multiplier of element e (0..7) of the group the words serve: `scale` if kept, else 0
__host__ __device__ __forceinline__ float drop_factor(const uint32_t (&w)[4], int e, uint32_t thr, float scale) {
  const uint32_t u = (w[e >> 1] >> (16 * (e & 1))) & 0xffffu;
  return u >= thr ? scale : 0.f;
}

// thr / scale of probability p; false for p outside [0, 1) (or so close to 1 that nothing is kept), and NaN
inline bool drop_threshold(float p, uint32_t* thr, float* scale) {
  if (!(p >= 0.f && p < 1.f)) return false;
  const double t = std::floor((double)p * 65536.0 + 0.5);
  if (t >= 65536.0) return false;
  *thr = (uint32_t)t;
  *scale = (float)(65536.0 / (65536.0 - t));
  return true;
}

#ifdef __CUDACC__
__device__ __forceinline__ uint64_t drop_key_load(const int64_t* key) {
  return key != nullptr ? (uint64_t)__ldg(reinterpret_cast<const long long*>(key)) : 0ull;
}

// keep bits of columns [col0, col0 + 32) of `row` (col0 a multiple of 8): bit i set = column col0 + i kept
__device__ __forceinline__ uint32_t drop_keep32(uint64_t key, uint32_t col0, uint32_t row, uint32_t plane,
                                                uint32_t site, uint32_t thr) {
  uint32_t bits = 0;
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    uint32_t w[4];
    drop_words(w, key, col0 + 8 * g, row, plane, site);
#pragma unroll
    for (int e = 0; e < 8; ++e) bits |= (((w[e >> 1] >> (16 * (e & 1))) & 0xffffu) >= thr ? 1u : 0u) << (8 * g + e);
  }
  return bits;
}
#endif

}  // namespace m3l
