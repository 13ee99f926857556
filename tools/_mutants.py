"""Mutant builds shared by tools/attention_mutants.py and tools/gemm_mutants.py: a mutant changes ONE arithmetic value or
comparison constant in one source file (never an address, an index, a trip count or a barrier, so no variant can
fault).  A mutant of a .cu file rebuilds that object; a mutant of a header names the objects that include it and
rebuilds those.  The mutated sources go to a temporary copy (m3l_b200/csrc is not touched); the libraries are written
to m3l_b200/build/mutants/ (ignored by git) and link the shipped library's other objects.  Each is run against pytest
selections through M3L_B200_LIB."""
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

OUT = B.OBJ / "mutants"
# header -> the .cu files whose objects a mutant of it rebuilds
HEADER_USERS = {"common.cuh": ("gemm.cu", "gemm_gelu.cu")}


def mutate(text: str, subs) -> str:
    for old, new in subs:
        count = text.count(old)
        if count != 1:
            raise SystemExit(f"substitution text found {count} times (expected once): {old!r}")
        text = text.replace(old, new)
    return text


def objects_of(src: str) -> tuple[str, ...]:
    return HEADER_USERS[src] if src.endswith((".cuh", ".h")) else (src,)


def build_mutant(name: str, src: str, subs) -> Path:
    """The library with `src` mutated: the objects that depend on it recompiled, the others as shipped."""
    lib = OUT / f"{name}.so"
    rebuilt = objects_of(src)
    with tempfile.TemporaryDirectory() as tmp:
        csrc = Path(tmp) / "m3l_b200" / "csrc"
        shutil.copytree(B.CSRC, csrc)
        shutil.copytree(ROOT / "include", Path(tmp) / "include")
        (csrc / src).write_text(mutate((csrc / src).read_text(), subs))
        objs = []
        for cu in rebuilt:
            obj = Path(tmp) / (Path(cu).stem + ".o")
            cmd = [B.NVCC, *B.ARCH_FLAGS, *B.flags_for(csrc / cu), "-c", str(csrc / cu), "-o", str(obj)]
            r = subprocess.run(cmd, capture_output=True, text=True)
            if r.returncode:
                raise SystemExit(f"{name}: nvcc failed\n{r.stderr}")
            objs.append(str(obj))
        others = [str(B.OBJ / (s.stem + ".o")) for s in B._sources() if s.name not in rebuilt]
        subprocess.run([B.NVCC, *B.ARCH_FLAGS, "-shared", "-o", str(lib), *objs, *others, "-lcudart"], check=True)
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


def main(doc: str, mutants: dict, selections: dict) -> None:
    """mutants: name -> (source file under csrc, what is wrong, [(exact text, replacement), ...]);
    selections: name -> pytest arguments."""
    ap = argparse.ArgumentParser(description=doc, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--build-only", action="store_true")
    ap.add_argument("--mutants", nargs="*", default=list(mutants))
    ap.add_argument("--selections", nargs="*", default=list(selections))
    ap.add_argument("--timeout", type=int, default=900, help="seconds per pytest run")
    args = ap.parse_args()
    B.build(verbose=False)
    OUT.mkdir(parents=True, exist_ok=True)
    for name in args.mutants:
        src, _, subs = mutants[name]
        mutate((B.CSRC / src).read_text(), subs)      # every substitution matches exactly once
    newest = max(p.stat().st_mtime for p in list(B.CSRC.glob("*.cu*")) + list(B.CSRC.glob("*.h")))
    stale = [m for m in args.mutants if not (OUT / f"{m}.so").exists() or (OUT / f"{m}.so").stat().st_mtime < newest]
    with ThreadPoolExecutor(max_workers=min(8, len(stale)) or 1) as ex:
        for lib in ex.map(lambda m: build_mutant(m, mutants[m][0], mutants[m][2]), stale):
            print(f"built {lib.relative_to(ROOT)}", flush=True)
    if args.build_only:
        return
    rows = []
    for name in args.mutants:
        lib = OUT / f"{name}.so"
        row = [name, mutants[name][1]]
        for sel in args.selections:
            verdict, secs = run(lib, selections[sel], args.timeout)
            row.append(f"{verdict}, {secs:.0f} s")
            print(f"{name} / {sel}: {verdict} ({secs:.0f} s)", flush=True)
        rows.append(row)
    head = ["mutant", "what is wrong", *(" ".join(selections[s]) for s in args.selections)]
    print("\n| " + " | ".join(head) + " |\n|" + "---|" * len(head))
    for row in rows:
        print("| " + " | ".join(row) + " |")
