"""Compare the SASS of two builds of libwsocean.so kernel by kernel.

    python tools/sass_identity.py --base-rev HEAD~1            # build that revision in a temporary directory
    python tools/sass_identity.py --base-lib OLD.so [--head-lib NEW.so]

Every kernel that exists in both builds must compile to the same instruction stream.  Kernel names are demangled
(cu++filt) and normalised before they are matched: a trailing `float4` template argument - the default texel type of the
map kernels (RGBA32F) - is dropped, so `wso_pass2_kernel<..., LaunchArgsT<64>, float4>` of a build that has a texel
parameter matches `wso_pass2_kernel<..., LaunchArgsT<64>>` of one that has not.  Instructions are compared as text plus
their encoding words, addresses stripped.  Exit status 0: identical; 1: a kernel differs or is missing from the head build.
Needs cuobjdump and cu++filt (CUDA toolkit); no GPU.
"""
from __future__ import annotations

import argparse
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUDA_BIN = "/usr/local/cuda/bin"


def _tool(name):
    p = os.path.join(CUDA_BIN, name)
    return p if os.path.exists(p) else name


def sass_by_kernel(lib: str) -> dict[str, list[str]]:
    out = subprocess.run([_tool("cuobjdump"), "-sass", lib], capture_output=True, text=True, check=True).stdout
    kernels: dict[str, list[str]] = {}
    cur = None
    for line in out.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            cur = m.group(1)
            kernels[cur] = []
            continue
        if cur is None:
            continue
        s = line.strip()
        m = re.match(r"/\*[0-9a-f]{4,}\*/\s*(.*)$", s)
        if m:
            kernels[cur].append(m.group(1).strip())
        elif s.startswith("/* 0x"):
            kernels[cur].append(s)  # second encoding word
    return kernels


def normalise(mangled: list[str]) -> dict[str, str]:
    dem = subprocess.run([_tool("cu++filt")], input="\n".join(mangled), capture_output=True, text=True,
                         check=True).stdout.splitlines()
    return {m: re.sub(r",\s*float4>", ">", d) for m, d in zip(mangled, dem)}


def build_rev(rev: str, tmp: str) -> str:
    subprocess.run(f"git -C {ROOT} archive {rev} | tar -x -C {tmp}", shell=True, check=True)
    code = "import sys; sys.path.insert(0, sys.argv[1]); from watersurfacerendering_b200 import build as b; print(b.build(force=True))"
    return subprocess.run([sys.executable, "-c", code, tmp], capture_output=True, text=True,
                          check=True).stdout.strip().splitlines()[-1]


def main() -> int:
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    g = ap.add_mutually_exclusive_group(required=True)
    g.add_argument("--base-rev", help="git revision to build and compare against")
    g.add_argument("--base-lib", help="an already built base libwsocean.so")
    ap.add_argument("--head-lib", default=None, help="default: the in-tree build (built if needed)")
    a = ap.parse_args()
    head = a.head_lib
    if head is None:
        sys.path.insert(0, ROOT)
        from watersurfacerendering_b200 import build as B
        head = B.build()
    with tempfile.TemporaryDirectory() as tmp:
        base = a.base_lib or build_rev(a.base_rev, tmp)
        kb, kh = sass_by_kernel(base), sass_by_kernel(head)
    nb, nh = normalise(list(kb)), normalise(list(kh))
    head_by_name = {}
    for m, d in nh.items():
        head_by_name.setdefault(d, []).append(m)
    same, differ, missing = 0, [], []
    for m, d in sorted(nb.items(), key=lambda x: x[1]):
        cands = head_by_name.get(d, [])
        if len(cands) != 1:
            missing.append(d)
            continue
        if kb[m] == kh[cands[0]]:
            same += 1
        else:
            differ.append(d)
    matched = {c for d in nb.values() for c in head_by_name.get(d, [])}
    only_head = sorted(nh[m] for m in kh if m not in matched)
    print(f"base {len(kb)} kernels, head {len(kh)} kernels")
    print(f"identical instruction streams: {same}; different: {len(differ)}; base kernels without a head match: {len(missing)}")
    for d in differ:
        print("  DIFFERENT:", d)
    for d in missing:
        print("  MISSING:", d)
    print(f"head-only kernels: {len(only_head)}")
    for d in only_head:
        print("  new:", d)
    return 0 if not differ and not missing else 1


if __name__ == "__main__":
    sys.exit(main())
