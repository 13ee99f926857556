"""Shows that the GEMM tests can tell a subtly wrong kernel from a right one: builds variants of the library in which
csrc/gemm.cu, csrc/common.cuh (GELU of gemm.cu and gemm_gelu.cu) or csrc/rowblock.cu differs in ONE arithmetic value or
comparison constant, runs pytest selections against each and prints which selection kills which variant.

    python tools/gemm_mutants.py --build-only     # compile the variants (no GPU needed)
    python tools/gemm_mutants.py                  # compile if needed, then run (GPU)

"new" is tests/test_gemm_bounds_gpu.py; "old" the GEMM, ln_mlp and LayerNorm-backward-epilogue tests of
tests/test_ops_gpu.py and test_gemm_dropout_epilogues (see tools/_mutants.py for how the variants are built)."""
from __future__ import annotations

import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from tools import _mutants  # noqa: E402

F32_BIAS = ("for (int j = 0; j < 32; j += 4) {\n              const int c = gcol + j;\n"
            "              float4 b = make_float4(0.f, 0.f, 0.f, 0.f);\n"
            "              if (c < p.N) b = __ldg(reinterpret_cast<const float4*>(p.bias + c));")
# name -> (source under csrc, what is wrong, [(exact text, replacement), ...]); every text occurs once in its source
MUTANTS = {
    "colsum_row_M": ("gemm.cu", "column sums admit row M (row0 + rr < p.M + 1)",
                     [("if (row0 + rr < p.M) {", "if (row0 + rr < p.M + 1) {")]),
    "residual_scaled": ("gemm.cu", "residual add off by 0.4 %",
                        [("w[j] = pack_bf16x2(__uint_as_float(v[2 * j]) + s2.x, __uint_as_float(v[2 * j + 1]) + s2.y);",
                          "w[j] = pack_bf16x2(__uint_as_float(v[2 * j]) + s2.x * 1.004f, "
                          "__uint_as_float(v[2 * j + 1]) + s2.y * 1.004f);")]),
    "f32_bias": ("gemm.cu", "fp32-output bias off by a relative 2^-14",
                 [(F32_BIAS, F32_BIAS.replace("p.bias + c));", "p.bias + c)); b.x *= 1.00006103515625f; "
                                              "b.y *= 1.00006103515625f; b.z *= 1.00006103515625f; "
                                              "b.w *= 1.00006103515625f;"))]),
    "rowdot_unrounded": ("gemm.cu", "row-dot of the unrounded accumulator instead of the bf16 output",
                         [("dot = fmaf(o2.x, s2.x, dot);\n                dot = fmaf(o2.y, s2.y, dot);",
                           "dot = fmaf(__uint_as_float(v[2 * j]), s2.x, dot);\n"
                           "                dot = fmaf(__uint_as_float(v[2 * j + 1]), s2.y, dot);")]),
    "ln_c2_255": ("gemm.cu", "LayerNorm backward: c2 divided by 255",
                  [("c2 = (s2 + other.y) * (1.0f / 256.0f)", "c2 = (s2 + other.y) * (1.0f / 255.0f)")]),
    "relu_clamp": ("gemm.cu", "ReLU clamps at -2^-10",
                   [("fmaxf(__uint_as_float(v[j]), 0.f)", "fmaxf(__uint_as_float(v[j]), -0.0009765625f)")]),
    "drop_scale": ("gemm.cu", "dropout scale off by 0.2 % (bias + residual epilogue)",
                   [("__uint_as_float(v[j]) * p.drop_scale : 0.f", "__uint_as_float(v[j]) * (p.drop_scale * 1.002f) : 0.f")]),
    "as_coef": ("common.cuh", "GELU: A&S coefficient 1.061405429 -> 1.061415429 (also gelu16)",
                [("f2_splat(-0.5f * 1.061405429f)", "f2_splat(-0.5f * 1.061415429f)")]),
    "gelu_pdf": ("common.cuh", "GELU': pdf constant 0.39894228 -> 0.39895228 (also gelu16)",
                 [("f2_splat(0.39894228040143268f), cdf)", "f2_splat(0.39895228040143268f), cdf)")]),
    "ln_mlp_eps": ("rowblock.cu", "ln_mlp: rstd with 1.5 x eps",
                   [("rsqrtf(var + p.eps)", "rsqrtf(var + 1.5f * p.eps)")]),
}
SELECTIONS = {
    "new": ["tests/test_gemm_bounds_gpu.py"],
    "old": ["tests/test_ops_gpu.py", "tests/test_dropout_gpu.py::test_gemm_dropout_epilogues", "-k", "gemm or ln_mlp"],
}

if __name__ == "__main__":
    _mutants.main(__doc__, MUTANTS, SELECTIONS)
