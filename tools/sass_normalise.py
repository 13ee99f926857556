"""Print the SASS of a CUDA object with kernel names, addresses and encodings normalised away, one kernel after the
other in a fixed order, so that two builds of the same kernels can be compared instruction for instruction.

    python tools/sass_normalise.py m3l_b200/build/attention_long.o > a.sass
    python tools/sass_normalise.py --digest m3l_b200/build/attention_long.o

Kernels are identified by the base name before the template arguments (`attn_long_fwd_kernel`, ...) and their
boolean template argument, if any; everything else in a mangled name (namespaces, the anonymous-namespace hash,
the head-width argument) is dropped."""
from __future__ import annotations

import argparse
import hashlib
import re
import shutil
import subprocess
import sys
from pathlib import Path

_ADDR = re.compile(r"/\*[0-9a-f]{4,}\*/")
_ENC = re.compile(r"/\* 0x[0-9a-f]+ \*/")


def _kernel_key(mangled: str) -> str:
    """`_ZN<len><name>...<len><kernel>I<args>E...` -> `kernel` or `kernel<flag>` (the bool template argument)."""
    if not mangled.startswith("_ZN"):
        return mangled
    i, names = 3, []
    while i < len(mangled) and mangled[i].isdigit():
        j = i
        while mangled[j].isdigit():
            j += 1
        length = int(mangled[i:j])
        names.append(mangled[j:j + length])
        i = j + length
    flag = re.match(r"I(?:Li\d+E)*Lb([01])E", mangled[i:])
    return names[-1] + (f"<{flag.group(1)}>" if flag else "")


def normalised_sass(obj: Path) -> dict[str, list[str]]:
    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    out = subprocess.run([cuobjdump, "-sass", str(obj)], capture_output=True, text=True, check=True).stdout
    kernels: dict[str, list[str]] = {}
    cur = None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = kernels.setdefault(_kernel_key(m.group(1)), [])
            continue
        if cur is None:
            continue
        text = _ENC.sub("", _ADDR.sub("", line)).strip()
        if text and not text.startswith(".") and text not in ("}", "{"):
            cur.append(text)
    return kernels


def digest(obj: Path) -> str:
    k = normalised_sass(obj)
    return hashlib.sha256("\n".join(f"== {name}\n" + "\n".join(k[name]) for name in sorted(k)).encode()).hexdigest()


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("obj", type=Path)
    ap.add_argument("--digest", action="store_true", help="print only the SHA-256 of the normalised listing")
    a = ap.parse_args()
    if a.digest:
        print(digest(a.obj))
        return 0
    k = normalised_sass(a.obj)
    for name in sorted(k):
        print(f"== {name} ({len(k[name])} instructions)")
        print("\n".join(k[name]))
    return 0


if __name__ == "__main__":
    sys.exit(main())
