"""Shows that the attention tests can tell a subtly wrong kernel from a right one: builds variants of the library
whose csrc/attention.cu differs in ONE arithmetic value or comparison constant (never an address, an index, a trip
count or a barrier, so no variant can fault), runs pytest selections against each through M3L_B200_LIB, and prints
which selection kills which variant.

    python tools/attention_mutants.py --build-only     # compile the variants (no GPU needed)
    python tools/attention_mutants.py                  # compile if needed, then run (GPU)

The mutated sources go to a temporary copy; m3l_b200/csrc is not touched.  The libraries are written to
m3l_b200/build/mutants/ (ignored by git) and link the shipped library's other objects."""
from __future__ import annotations

import argparse
import os
import shutil
import subprocess
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from m3l_b200 import build as B  # noqa: E402

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
OUT = B.OBJ / "mutants"


def mutate(text: str, subs) -> str:
    for old, new in subs:
        count = text.count(old)
        if count != 1:
            raise SystemExit(f"substitution text found {count} times (expected once): {old!r}")
        text = text.replace(old, new)
    return text


def build_mutant(name: str) -> Path:
    """attention.cu with the mutant's substitutions, linked with the shipped library's other objects."""
    subs = MUTANTS[name][1]
    lib = OUT / f"{name}.so"
    with tempfile.TemporaryDirectory() as tmp:
        csrc = Path(tmp) / "m3l_b200" / "csrc"
        shutil.copytree(B.CSRC, csrc)
        shutil.copytree(ROOT / "include", Path(tmp) / "include")
        src = csrc / SRC
        src.write_text(mutate(src.read_text(), subs))
        obj = Path(tmp) / "attention.o"
        cmd = [B.NVCC, *B.ARCH_FLAGS, *B.flags_for(src), "-c", str(src), "-o", str(obj)]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode:
            raise SystemExit(f"{name}: nvcc failed\n{r.stderr}")
        others = [str(B.OBJ / (s.stem + ".o")) for s in B._sources() if s.name != SRC]
        subprocess.run([B.NVCC, *B.ARCH_FLAGS, "-shared", "-o", str(lib), str(obj), *others, "-lcudart"], check=True)
    return lib


def run(lib: Path, selection: list[str], timeout: int) -> tuple[str, float]:
    env = dict(os.environ, M3L_B200_LIB=str(lib))
    t0 = time.time()
    try:
        r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-p", "no:cacheprovider", *selection], cwd=ROOT,
                           env=env, capture_output=True, text=True, timeout=timeout)
    except subprocess.TimeoutExpired:
        return "timeout", time.time() - t0
    # pytest: 0 all passed, 1 some test failed; anything else (collection error, crash) is not a verdict
    verdict = {0: "survived", 1: "killed"}.get(r.returncode, f"error {r.returncode}")
    if verdict == "killed":
        failed = [l for l in r.stdout.splitlines() if l.startswith("FAILED")]
        verdict += f" ({failed[0].split()[1].split('::')[-1]})" if failed else ""
    return verdict, time.time() - t0


def main() -> None:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--build-only", action="store_true")
    ap.add_argument("--mutants", nargs="*", default=list(MUTANTS))
    ap.add_argument("--selections", nargs="*", default=list(SELECTIONS))
    ap.add_argument("--timeout", type=int, default=900, help="seconds per pytest run")
    args = ap.parse_args()
    B.build(verbose=False)
    OUT.mkdir(parents=True, exist_ok=True)
    for name in args.mutants:
        mutate((B.CSRC / SRC).read_text(), MUTANTS[name][1])      # every substitution matches exactly once
    stale = [m for m in args.mutants
             if not (OUT / f"{m}.so").exists() or (OUT / f"{m}.so").stat().st_mtime < (B.CSRC / SRC).stat().st_mtime]
    with ThreadPoolExecutor(max_workers=len(stale) or 1) as ex:
        for lib in ex.map(build_mutant, stale):
            print(f"built {lib.relative_to(ROOT)}", flush=True)
    if args.build_only:
        return
    rows = []
    for name in args.mutants:
        lib = OUT / f"{name}.so"
        row = [name, MUTANTS[name][0]]
        for sel in args.selections:
            verdict, secs = run(lib, SELECTIONS[sel], args.timeout)
            row.append(f"{verdict}, {secs:.0f} s")
            print(f"{name} / {sel}: {verdict} ({secs:.0f} s)", flush=True)
        rows.append(row)
    head = ["mutant", "what is wrong", *(" ".join(SELECTIONS[s]) for s in args.selections)]
    print("\n| " + " | ".join(head) + " |\n|" + "---|" * len(head))
    for row in rows:
        print("| " + " | ".join(row) + " |")


if __name__ == "__main__":
    main()
