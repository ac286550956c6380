"""Check that a change left existing kernels' machine code alone: dump the SASS of two builds of libcerb_post.so with
``cuobjdump -sass``, split it by function and compare every function of the OLD build with its namesake in the new one
(instructions and their encodings).  Functions only the new build has are listed, not compared.  Runs on any machine
with the CUDA toolkit; no GPU needed.

    python tools/sass_identity.py OLD.so NEW.so [--out report.txt]

Exit status 0 when every old function is present and identical, 1 otherwise.  A function whose mangled name carries the
hash nvcc derives from a file's contents (anonymous namespaces) is matched by its name with that hash removed.
"""
from __future__ import annotations

import argparse
import os
import re
import shutil
import subprocess
import sys
from typing import Dict, List, Tuple

_FUNC = re.compile(r"^\s*Function\s*:\s*(\S+)\s*$")
_INSN = re.compile(r"^\s*/\*([0-9a-f]{4,})\*/\s*(.*?)\s*;?\s*/\*\s*(0x[0-9a-f]+)\s*\*/\s*$")
_ENC2 = re.compile(r"^\s*/\*\s*(0x[0-9a-f]+)\s*\*/\s*$")
_ANON = re.compile(r"_GLOBAL__N__[0-9a-f]+_\d+_[A-Za-z0-9_]+?_[0-9a-f]{8}")


def parse_sass(text: str) -> Dict[str, List[Tuple[str, str]]]:
    """``{function name: [(instruction text, encoding), ...]}`` from ``cuobjdump -sass`` output.  The instruction text
    drops the address; the encoding joins the two 64-bit halves cuobjdump prints on consecutive lines."""
    funcs: Dict[str, List[Tuple[str, str]]] = {}
    cur = None
    for line in text.splitlines():
        m = _FUNC.match(line)
        if m:
            cur = funcs.setdefault(normalise_name(m.group(1)), [])
            continue
        if cur is None:
            continue
        m = _INSN.match(line)
        if m:
            cur.append((re.sub(r"\s+", " ", m.group(2)).rstrip(" ;"), m.group(3)))
            continue
        m = _ENC2.match(line)
        if m and cur:
            text_, enc = cur[-1]
            cur[-1] = (text_, enc + ":" + m.group(1))
    return funcs


def normalise_name(name: str) -> str:
    return _ANON.sub("_GLOBAL__N__<anon>", name)


def compare(old: Dict[str, list], new: Dict[str, list]) -> Tuple[List[str], List[str], List[str], List[str]]:
    """``(identical, differing, missing, added)`` function names."""
    same, diff, missing = [], [], []
    for name in sorted(old):
        if name not in new:
            missing.append(name)
        elif old[name] == new[name]:
            same.append(name)
        else:
            diff.append(name)
    added = sorted(n for n in new if n not in old)
    return same, diff, missing, added


def cuobjdump(lib: str) -> str:
    exe = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    return subprocess.run([exe, "-sass", lib], check=True, capture_output=True, text=True).stdout


def report(same, diff, missing, added) -> str:
    lines = [f"identical: {len(same)}  differing: {len(diff)}  missing: {len(missing)}  new: {len(added)}"]
    lines += [f"DIFF     {n}" for n in diff] + [f"MISSING  {n}" for n in missing]
    lines += [f"same     {n}" for n in same] + [f"new      {n}" for n in added]
    return "\n".join(lines) + "\n"


def main(argv=None) -> int:
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("old")
    ap.add_argument("new")
    ap.add_argument("--out", help="also write the report here")
    a = ap.parse_args(argv)
    same, diff, missing, added = compare(parse_sass(cuobjdump(a.old)), parse_sass(cuobjdump(a.new)))
    text = report(same, diff, missing, added)
    sys.stdout.write(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text)
    return 1 if diff or missing else 0


if __name__ == "__main__":
    sys.exit(main())
