#!/usr/bin/env python3
"""Check that every kernel of a base build has the same SASS in the current build.

    python tools/sass_compare.py [--rev HEAD~1] [--base-lib PATH] [--out FILE]

Builds libnka_b200.so from git revision --rev in a temporary directory (or takes --base-lib), builds the
working tree's library in place, dumps both with `cuobjdump -sass`, and compares the instructions of each
kernel the base library holds, function by function.  Kernels only the current build has (new features)
are listed but not compared.  Exit status 1 if any base kernel is missing or differs.  Needs nvcc and
cuobjdump, no GPU.
"""
from __future__ import annotations

import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def build_rev(rev: str, tmp: str) -> str:
    src = os.path.join(tmp, "base")
    os.makedirs(src)
    archive = subprocess.run(["git", "-C", ROOT, "archive", rev], check=True, capture_output=True).stdout
    subprocess.run(["tar", "-x", "-C", src], input=archive, check=True)
    code = "import sys; sys.path.insert(0, %r); from nka_b200 import build; print(build.build_library(force=True))" % src
    out = subprocess.run([sys.executable, "-c", code], check=True, capture_output=True, text=True, cwd=src)
    return out.stdout.strip().splitlines()[-1]


def sass_by_function(lib: str) -> dict[str, str]:
    text = subprocess.run(["cuobjdump", "-sass", lib], check=True, capture_output=True, text=True).stdout
    funcs: dict[str, list[str]] = {}
    cur = None
    for line in text.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
            continue
        if cur is not None and re.match(r"\s*/\*[0-9a-f]{4,}\*/", line):
            funcs[cur].append(line.strip())
    return {k: "\n".join(v) for k, v in funcs.items()}


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--rev", default="HEAD~1", help="git revision of the base build (default HEAD~1)")
    ap.add_argument("--base-lib", help="an already built base libnka_b200.so instead of --rev")
    ap.add_argument("--out", help="write the report here as well")
    args = ap.parse_args()
    sys.path.insert(0, ROOT)
    from nka_b200 import build
    cur_lib = build.build_library()
    with tempfile.TemporaryDirectory() as tmp:
        base_lib = args.base_lib or build_rev(args.rev, tmp)
        base = sass_by_function(base_lib)
    cur = sass_by_function(cur_lib)
    same = sorted(k for k in base if cur.get(k) == base[k])
    differ = sorted(k for k in base if k in cur and cur[k] != base[k])
    missing = sorted(k for k in base if k not in cur)
    new = sorted(k for k in cur if k not in base)
    lines = ["base kernels: %d, identical SASS: %d, differing: %d, missing: %d; kernels only in this build: %d"
             % (len(base), len(same), len(differ), len(missing), len(new))]
    lines += ["DIFFERS %s" % k for k in differ] + ["MISSING %s" % k for k in missing]
    lines += ["new %s" % k for k in new]
    report = "\n".join(lines)
    print(report)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(report + "\n")
    return 1 if (differ or missing) else 0


if __name__ == "__main__":
    sys.exit(main())
