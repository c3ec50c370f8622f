#!/usr/bin/env python3
"""Writes tests/golden/cr_hard_cases.npz and its C table ensem3a_openclraytracer_b200/csrc/cr_hard_cases.inc: every
binary32 input, on the domains the kernels reach, whose binary64 function value lies within WINDOW binary64 ulps of
a binary32 rounding boundary, with its correctly rounded result.

Domains (every float in each):
  sin, cos      |a| <= 8         (cr_sincos: the samplers and the per-triangle frames)
  acos, asin    |x| <= 1         (make_tri_frame, sample_uniform; the exact environment-texel row)
  pow(p, 2.2f)  0 < p <= 1       (the tonemap, k_img_processing)

A binary64 pass in C with OpenMP (cr_hard_cases_scan.c, glibc, < 1 ulp) flags the inputs; mpmath at 200 bits
resolves each flagged one.  WINDOW = 64 exceeds the error of either binary64 library the project rounds from (CUDA's,
<= 2 ulp; glibc's, < 1 ulp) plus the guard the kernels and the oracle apply (oracle/cr_tie.h, CR_TIE_GUARD = 16),
so every input on which the kernels' guard fires is in the table.  Deterministic: a second run writes the same bytes.

usage: python tests/golden/make_cr_hard_cases.py [--check]   (--check: recompute and compare, write nothing)
"""
import ctypes
import io
import os
import subprocess
import sys
import tempfile
import time
import zipfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
NPZ = os.path.join(HERE, "cr_hard_cases.npz")
INC = os.path.join(ROOT, "ensem3a_openclraytracer_b200", "csrc", "cr_hard_cases.inc")
sys.path.insert(0, ROOT)
from tests.cr_reference import FUNCS, correctly_rounded  # noqa: E402

WINDOW = 64
KERNEL_TABLES = ["acos", "asin", "pow"]   # cr_sincos is checked input by input and needs no table (csrc/rt_math.cuh)

# name -> (scan code, bit-pattern ranges)
DOMAINS = {
    "sin": (0, [(0x00000000, 0x41000000), (0x80000000, 0xC1000000)]),
    "cos": (1, [(0x00000000, 0x41000000), (0x80000000, 0xC1000000)]),
    "acos": (2, [(0x00000000, 0x3F800000), (0x80000000, 0xBF800000)]),
    "asin": (3, [(0x00000000, 0x3F800000), (0x80000000, 0xBF800000)]),
    "pow": (4, [(0x00000001, 0x3F800000)]),
}
assert list(DOMAINS) == FUNCS


def _scanner(tmp):
    so = os.path.join(tmp, "cr_scan.so")
    subprocess.check_call(["gcc", "-O2", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-fopenmp", "-fPIC",
                           "-shared", os.path.join(HERE, "cr_hard_cases_scan.c"), "-o", so, "-lm"])
    lib = ctypes.CDLL(so)
    u32p = np.ctypeslib.ndpointer(np.uint32, flags="C_CONTIGUOUS")
    f32p = np.ctypeslib.ndpointer(np.float32, flags="C_CONTIGUOUS")
    lib.cr_scan.restype = ctypes.c_int64
    lib.cr_scan.argtypes = [ctypes.c_int, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_int64, u32p, ctypes.c_int64]
    lib.cr_eval.restype = None
    lib.cr_eval.argtypes = [ctypes.c_int, u32p, ctypes.c_int64, f32p]
    return lib


def compute(verbose=True):
    with tempfile.TemporaryDirectory() as tmp:
        lib = _scanner(tmp)
        fns, xs, ys, stats = [], [], [], {}
        for fn in FUNCS:
            code, ranges = DOMAINS[fn]
            t0 = time.time()
            found, total = [], 0
            for lo, hi in ranges:
                cap = 1 << 16
                buf = np.zeros(cap, np.uint32)
                n = lib.cr_scan(code, lo, hi, WINDOW, buf, cap)
                assert n <= cap, f"{fn}: {n} flagged inputs exceed the buffer"
                found.append(buf[:n])
                total += hi - lo + 1
            x = np.sort(np.concatenate(found))
            y = correctly_rounded(fn, x.view(np.float32))
            glibc = np.zeros(x.size, np.float32)
            lib.cr_eval(code, x, x.size, glibc)
            wrong = int((glibc.view(np.uint32) != y).sum())
            stats[fn] = (total, x.size, wrong)
            if verbose:
                print(f"{fn:5s}: {total} inputs, {x.size} within {WINDOW} binary64 ulps of a binary32 boundary, "
                      f"{wrong} of them rounded wrongly from glibc's binary64 value  ({time.time() - t0:.1f} s)")
            fns.append(np.full(x.size, FUNCS.index(fn), np.uint8))
            xs.append(x)
            ys.append(y)
    return np.concatenate(fns), np.concatenate(xs), np.concatenate(ys), stats


def npz_bytes(fn, x, y):
    """an .npz with fixed member times, so that the file depends on the arrays alone"""
    buf = io.BytesIO()
    with zipfile.ZipFile(buf, "w", zipfile.ZIP_DEFLATED) as z:
        for name, arr in (("fn", fn), ("x", x), ("y", y), ("names", np.array(FUNCS)), ("window", np.int64(WINDOW))):
            member = io.BytesIO()
            np.lib.format.write_array(member, np.asarray(arr), allow_pickle=False)
            info = zipfile.ZipInfo(name + ".npy", date_time=(1980, 1, 1, 0, 0, 0))
            info.compress_type = zipfile.ZIP_DEFLATED
            z.writestr(info, member.getvalue())
    return buf.getvalue()


def inc_text(fn, x, y):
    """the kernels' tables: one sorted {input bits, result bits} array per function in KERNEL_TABLES"""
    lines = ["// Generated by tests/golden/make_cr_hard_cases.py from tests/golden/cr_hard_cases.npz; do not edit.",
             "// Binary32 inputs whose binary64 value lies within %d binary64 ulps of a binary32 rounding boundary, with" % WINDOW,
             "// their correctly rounded results: {input bits, result bits}, sorted by input bits.",
             "#pragma once"]
    for name in KERNEL_TABLES:
        sel = fn == FUNCS.index(name)
        rows = [f"{{0x{a:08x}u, 0x{b:08x}u}}" for a, b in zip(x[sel].tolist(), y[sel].tolist())]
        lines.append(f"#define CR_HARD_{name.upper()}_N {len(rows)}")
        lines.append(f"__device__ const uint32_t cr_hard_{name}[{len(rows)}][2] = {{")
        for k in range(0, len(rows), 4):
            lines.append("    " + ", ".join(rows[k:k + 4]) + ",")
        lines.append("};")
    return "\n".join(lines) + "\n"


def main():
    fn, x, y, _ = compute()
    data, text = npz_bytes(fn, x, y), inc_text(fn, x, y)
    if "--check" in sys.argv:
        same = open(NPZ, "rb").read() == data and open(INC).read() == text
        print("committed files reproduced" if same else "committed files DIFFER")
        sys.exit(0 if same else 1)
    with open(NPZ, "wb") as f:
        f.write(data)
    with open(INC, "w") as f:
        f.write(text)
    print(f"wrote {NPZ} and {INC}: {x.size} entries")


if __name__ == "__main__":
    main()
