"""GPU: every binary32 input the kernels can give their correctly rounded transcendentals, device against oracle, bit
for bit; and the environment-texel chain at every texel boundary of the map sizes in use.

The renders are bit-identical to the oracle only if both round cos sin acos asin powr correctly (DESIGN.md
"Arithmetic contract").  Random samples reach about one input in a thousand of these domains; the sweeps below reach
all of them:

  sin / cos (cr_sincos)      every float with |a| <= 8, +-inf, NaN, and 2^24 random floats with |a| > 8
  acos, asin                 every float with |x| <= 2
  the tonemap kernel itself  every bit pattern with p <= 1 (-inf and the negative NaN-producing ones included),
                             NaN and a few values > 1

The inputs are enumerated as bit patterns in chunks of 2^26; the oracle's share of a chunk runs on a thread pool
(ctypes releases the GIL) while the GPU works on it.  Wherever the oracle's result is not NaN the bits must agree;
where it is NaN only NaN-ness counts.  Every disagreement is reported with the correctly rounded value (mpmath, 200
bits), which says which side is wrong."""
import os
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import oracle
from tests.cr_reference import correctly_rounded

pytestmark = pytest.mark.gpu

CHUNK = 1 << 26
THREADS = max(1, os.cpu_count() or 1)
REPORT = 20           # disagreements printed per function


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def pattern_ranges(lo, hi):
    """float32 views of the bit patterns lo..hi (inclusive), chunk by chunk"""
    for s in range(lo, hi + 1, CHUNK):
        yield np.arange(s, min(s + CHUNK, hi + 1), dtype=np.uint32).view(np.float32)


def differ(got, want):
    """bits differ where the oracle's value is a number; NaN-ness differs where it is NaN"""
    wn = np.isnan(want)
    return np.where(wn, ~np.isnan(got), bits(got) != bits(want))


def report(name, x, got, want):
    idx = np.nonzero(differ(got, want))[0]
    lines = []
    if idx.size:
        cr = correctly_rounded(name, x[idx[:REPORT]])
        for k, i in enumerate(idx[:REPORT]):
            who = "GPU" if bits(want[i:i + 1])[0] == cr[k] else "oracle" if bits(got[i:i + 1])[0] == cr[k] else "both"
            lines.append(f"  {name}(0x{bits(x[i:i + 1])[0]:08x} = {x[i]!r}): GPU 0x{bits(got[i:i + 1])[0]:08x}, "
                         f"oracle 0x{bits(want[i:i + 1])[0]:08x}, correctly rounded 0x{cr[k]:08x} -> {who} wrong")
    return idx.size, lines


def sweep(name, chunks, gpu, orc):
    """runs every chunk through gpu(x) and, on the thread pool, orc(x); returns (inputs, disagreements, report lines)"""
    t0 = time.time()
    total, bad, lines = 0, 0, []
    with ThreadPoolExecutor(THREADS) as pool:
        for x in chunks:
            futs = [pool.submit(orc, p) for p in np.array_split(x, THREADS)]
            got = gpu(x)
            want = np.concatenate([f.result() for f in futs])
            n, ln = report(name, x, got, want)
            total += x.size
            bad += n
            lines += ln[:max(0, REPORT - len(lines))]
    print(f"\n{name}: {total} inputs swept, {bad} GPU/oracle disagreements, {time.time() - t0:.1f} s")
    for ln in lines:
        print(ln)
    return total, bad


def sincos_inputs():
    for lo, hi in ((0x00000000, 0x41000000), (0x80000000, 0xC1000000)):
        yield from pattern_ranges(lo, hi)
    r = np.random.default_rng(12)
    big = r.integers(0x41000001, 0x7F800000, 1 << 24, dtype=np.uint32) | (r.integers(0, 2, 1 << 24, dtype=np.uint32) << 31)
    special = np.array([0x7F800000, 0xFF800000, 0x7FC00000, 0xFFC00000, 0x00000000, 0x80000000], np.uint32)
    yield np.concatenate([big, special]).view(np.float32)


@pytest.mark.parametrize("name,code", [("sin", 9), ("cos", 10)])
def test_sincos_every_input_up_to_8(gpu_ctx, name, code):
    total, bad = sweep(name, sincos_inputs(), lambda x: gpu_ctx.math_probe(code, x), lambda x: oracle.math_probe(name, x))
    assert total == 2 * 0x41000001 + (1 << 24) + 6
    assert bad == 0


@pytest.mark.parametrize("name,code", [("acos", 2), ("asin", 3)])
def test_acos_asin_every_input_up_to_2(gpu_ctx, name, code):
    chunks = (x for lo, hi in ((0x00000000, 0x40000000), (0x80000000, 0xC0000000)) for x in pattern_ranges(lo, hi))
    total, bad = sweep(name, chunks, lambda x: gpu_ctx.math_probe(code, x), lambda x: oracle.math_probe(name, x))
    assert total == 2 * 0x40000001
    assert bad == 0


def test_tonemap_kernel_every_input_up_to_1(gpu_ctx):
    def chunks():
        for lo, hi in ((0x00000000, 0x3F800000), (0x80000000, 0xFF800000)):
            yield from pattern_ranges(lo, hi)
        yield np.array([np.nan, -np.nan, np.inf, 1.0000001, 1.5, 2.0, 1e30], np.float32)

    def gpu(x):
        out = np.empty_like(x)
        return gpu_ctx.img_processing(x, out, x.size)

    total, bad = sweep("pow", chunks(), gpu, lambda x: oracle.img_processing(x, x.size))
    assert total == 0x3F800001 + 0x7F800001 + 7
    assert bad == 0


# ---- the environment-texel chain ---------------------------------------------------------------------------------
SIZES = [(600, 300), (16, 8), (1, 1), (8192, 4096), (601, 301)]   # (width, height)
U_INV, V_INV = np.float32(0.1591), np.float32(0.3183)
_max_ulp = {"atan2f": 0, "asinf": 0}


def texel(a, inv, extent):
    """rt_shade.cuh texel_coord in numpy binary32: trunc(RN(RN(RN(a * inv) + 0.5) * extent)), clamped"""
    a = np.asarray(a, np.float32)
    u = (a * inv).astype(np.float32) + np.float32(0.5)
    p = np.trunc((u * np.float32(extent)).astype(np.float32)).astype(np.int64)
    return np.clip(p, 0, extent - 1)


def ordered(f):
    """float32 -> integers in the order of the floats (adjacent floats differ by 1)"""
    i = bits(f).astype(np.int64)
    return np.where(i >= 0x80000000, 0x80000000 - i, i)


def from_ordered(o):
    o = np.asarray(o, np.int64)
    return np.where(o < 0, 0x80000000 - o, o).astype(np.uint32).view(np.float32)


def boundaries(inv, extent, lo, hi):
    """for every texel boundary j in 1..extent-1 the smallest binary32 angle in [lo, hi] whose texel is >= j"""
    j = np.arange(1, extent, dtype=np.int64)
    a, b = np.full(j.size, ordered(np.float32(lo))[()]), np.full(j.size, ordered(np.float32(hi))[()])
    while np.any(b - a > 1):
        m = (a + b) // 2
        up = texel(from_ordered(m), inv, extent) >= j
        b, a = np.where(up, m, b), np.where(up, a, m)
    return from_ordered(b)


def neighbourhood(centres, k):
    """every float within k floats of each centre"""
    o = ordered(np.asarray(centres, np.float32))[:, None] + np.arange(-k, k + 1)[None, :]
    return from_ordered(o.reshape(-1))


def binade_angles():
    """angles within 8 ulp of +-2^k, k = -10..1: there a -+ del crosses a binade"""
    p = np.float32(2.0) ** np.arange(-10, 2, dtype=np.float32)
    return neighbourhood(np.concatenate([p, -p]), 8)


def ulp_distance(a, b):
    return np.abs(ordered(a) - ordered(b))


def check_rows(gpu_ctx, h, y):
    fast, exact = gpu_ctx.math_probe(13, y, extent=h), gpu_ctx.math_probe(14, y, extent=h)
    assert np.array_equal(fast, exact), f"height {h}: fast and exact rows differ on {(fast != exact).sum()} inputs"
    want = texel(oracle.math_probe("asin", y), V_INV, h)
    assert np.array_equal(exact.astype(np.int64), want), f"height {h}: exact row differs from the oracle's chain"
    d = ulp_distance(gpu_ctx.math_probe(17, y), gpu_ctx.math_probe(3, y))
    _max_ulp["asinf"] = max(_max_ulp["asinf"], int(d.max()))


def check_columns(gpu_ctx, w, z, x):
    fast, exact = gpu_ctx.math_probe(11, z, x, extent=w), gpu_ctx.math_probe(12, z, x, extent=w)
    assert np.array_equal(fast, exact), f"width {w}: fast and exact columns differ on {(fast != exact).sum()} inputs"
    want = texel(oracle.math_probe("atan2", z, x), U_INV, w)
    assert np.array_equal(exact.astype(np.int64), want), f"width {w}: exact column differs from the oracle's chain"
    d = ulp_distance(gpu_ctx.math_probe(16, z, x), gpu_ctx.math_probe(4, z, x))
    _max_ulp["atan2f"] = max(_max_ulp["atan2f"], int(d.max()))


def row_inputs(h):
    """every float y whose asin lies within 2^12 ulp of a row-boundary angle, and y near sin(+-2^k)"""
    half_pi = np.float32(np.pi / 2)
    b = boundaries(V_INV, h, -half_pi, half_pi) if h > 1 else np.zeros(0, np.float32)
    o_lo = ordered(np.clip(np.sin(from_ordered(ordered(b) - 4096).astype(np.float64)), -1, 1).astype(np.float32)) - 1
    o_hi = ordered(np.clip(np.sin(from_ordered(ordered(b) + 4096).astype(np.float64)), -1, 1).astype(np.float32)) + 1
    ys = [from_ordered(np.arange(l_, h_ + 1)) for l_, h_ in zip(o_lo.tolist(), o_hi.tolist())]
    ys.append(neighbourhood(np.sin(binade_angles().astype(np.float64)).astype(np.float32), 16))
    y = np.concatenate(ys)
    return y[np.abs(y) <= 1]


MAGNITUDES = np.float64(2.0) ** np.array([-20, -10, -3, 0, 3, 10, 20])


def column_inputs(w):
    """directions (z, x) = m (sin a, cos a) for every angle a within 64 ulp of a column boundary, and within 8 ulp of
    +-2^k, at magnitudes m = +-2^-20 .. 2^20, rounded to binary32"""
    pi = np.float32(np.pi)
    b = boundaries(U_INV, w, -pi, pi) if w > 1 else np.zeros(0, np.float32)
    a = np.concatenate([neighbourhood(b, 64), binade_angles()]).astype(np.float64)
    m = np.concatenate([MAGNITUDES, -MAGNITUDES])
    z = (np.sin(a)[:, None] * m[None, :]).astype(np.float32).reshape(-1)
    x = (np.cos(a)[:, None] * m[None, :]).astype(np.float32).reshape(-1)
    return z, x


@pytest.mark.parametrize("w,h", SIZES)
def test_environment_texel_every_boundary(gpu_ctx, w, h):
    """rt_shade.cuh ibl_texel_u / ibl_texel_v pick their texel from atan2f / asinf and fall back to the correctly
    rounded angle only where a -+ del straddles a texel boundary.  At every boundary of a w x h map: the fast path
    selects the exact path's texel, and the exact path is the oracle's chain."""
    t0 = time.time()
    y = row_inputs(h)
    for s in range(0, y.size, CHUNK):
        check_rows(gpu_ctx, h, y[s:s + CHUNK])
    z, x = column_inputs(w)
    for s in range(0, z.size, CHUNK):
        check_columns(gpu_ctx, w, z[s:s + CHUNK], x[s:s + CHUNK])
    print(f"\n{w} x {h} map: {y.size} row inputs around {h - 1} boundaries, {z.size} column directions around "
          f"{w - 1} boundaries, {time.time() - t0:.1f} s; largest distance so far: atan2f {_max_ulp['atan2f']} ulp, "
          f"asinf {_max_ulp['asinf']} ulp from the correctly rounded angle")
    # del = |a| 2^-21 covers 4 ulp of the angle (rt_shade.cuh)
    assert _max_ulp["atan2f"] < 4 and _max_ulp["asinf"] < 4
