#!/usr/bin/env python3
"""One line per kernel of a built libb200rt.so: a hash of its SASS, its instruction count and its demangled name.

usage: sass_digest.py [lib.so]   (default: ensem3a_openclraytracer_b200/lib/libb200rt.so)

Two builds compile a kernel to the same code iff their lines for it agree.  Addresses and encodings are dropped, and
parameter-bank offsets (c[0x0][0x...]) are masked, so a kernel whose code is unchanged keeps its digest when a field is
added to or removed from its parameter struct."""
import hashlib
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CUOBJDUMP = os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")


def kernels(lib):
    txt = subprocess.run([CUOBJDUMP, "-sass", lib], capture_output=True, text=True, check=True).stdout
    out, name = {}, None
    for line in txt.splitlines():
        m = re.match(r"\s*Function : (\S+)", line)
        if m:
            name = m.group(1)
            out[name] = []
            continue
        m = re.match(r"\s*/\*[0-9a-f]{4,}\*/\s+(.*?)\s*;", line)
        if name is not None and m:
            out[name].append(re.sub(r"c\[0x0\]\[0x[0-9a-f]+\]", "c[0x0][P]", m.group(1)))
    return out


def main():
    lib = sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "ensem3a_openclraytracer_b200", "lib", "libb200rt.so")
    ks = kernels(lib)
    names = sorted(ks)
    dem = subprocess.run(["c++filt"], input="\n".join(names), capture_output=True, text=True, check=True).stdout.split("\n")
    for d, n in sorted((re.sub(r"^void b200rt::", "", d), n) for n, d in zip(names, dem)):
        print(f"{hashlib.sha256(chr(10).join(ks[n]).encode()).hexdigest()[:16]} {len(ks[n]):6d} {d}")
    print(f"{len(ks)} kernels", file=sys.stderr)


if __name__ == "__main__":
    main()
