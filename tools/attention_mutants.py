"""Shows that the attention tests can tell a subtly wrong kernel from a right one: builds variants of the library
whose csrc/attention.cu differs in ONE arithmetic value or comparison constant (never an address, an index, a trip
count or a barrier, so no variant can fault), runs pytest selections against each through M3L_B200_LIB, and prints
which selection kills which variant.

    python tools/attention_mutants.py --build-only     # compile the variants (no GPU needed)
    python tools/attention_mutants.py                  # compile if needed, then run (GPU)

The mutated sources go to a temporary copy; m3l_b200/csrc is not touched.  The libraries are written to
m3l_b200/build/mutants/ (ignored by git) and link the shipped library's other objects."""
from __future__ import annotations

import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from tools import _mutants  # noqa: E402

SRC = "attention.cu"
# name -> (what is wrong, [(exact text, replacement), ...]); every text must occur exactly once in attention.cu
MUTANTS = {
    "fwd_exp_scaled": (
        "forward exponent off by 0.2 %: exp2f(a) -> exp2f(a * 1.002f)",
        [("pv[j] = exp2f(a0);\n                  pv[j + 1] = exp2f(a1);",
          "pv[j] = exp2f(a0 * 1.002f);\n                  pv[j + 1] = exp2f(a1 * 1.002f);")]),
    "fwd_pad_leak": (
        "forward: a padded key enters the softmax at weight 1/256 instead of 0",
        [("pv[j] = (col0 + g * 8 + j < n) ? pv[j] : 0.f;", "pv[j] = (col0 + g * 8 + j < n) ? pv[j] : 0.00390625f;")]),
    "lse_offset": (
        "forward LSE off by 1e-3",
        [("= mx * p.scale + __logf(sum);", "= mx * p.scale + __logf(sum) + 1e-3f;")]),
    "bwd_delta_scaled": (
        "tcgen05 backward: delta off by 0.4 %",
        [("const float dl = delta[i], lg", "const float dl = delta[i] * 1.004f, lg")]),
    "small_mask_finite": (
        "n <= 16 forward masks padded keys with -20 instead of -inf",
        [("sc[nt][e] = ok ? sc[nt][e] * scale : -INFINITY;", "sc[nt][e] = ok ? sc[nt][e] * scale : -20.f;"),
         ("sc[nt][2 + e] = ok ? sc[nt][2 + e] * scale : -INFINITY;", "sc[nt][2 + e] = ok ? sc[nt][2 + e] * scale : -20.f;")]),
    "bwd_exp_shift": (
        "tcgen05 backward exponent subtracts lg + 0.003 (interior and edge paths)",
        [("nlg2 = f2_splat(-lg)", "nlg2 = f2_splat(-(lg + 0.003f))"),
         ("exp2f(fmaf(__uint_as_float(sv[e]), sl2, -lg))", "exp2f(fmaf(__uint_as_float(sv[e]), sl2, -(lg + 0.003f)))"),
         ("exp2f(fmaf(__uint_as_float(sv[e + 1]), sl2, -lg))",
          "exp2f(fmaf(__uint_as_float(sv[e + 1]), sl2, -(lg + 0.003f)))")]),
}
SELECTIONS = {
    "new": ["tests/test_attention_bounds_gpu.py"],
    "old": ["tests/test_ops_gpu.py::test_attention_fwd_bwd"],
}
if __name__ == "__main__":
    _mutants.main(__doc__, {name: (SRC, what, subs) for name, (what, subs) in MUTANTS.items()}, SELECTIONS)
