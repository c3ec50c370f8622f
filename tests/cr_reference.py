"""Correctly rounded binary32 values of the transcendentals the kernels round from binary64, by mpmath at 200 bits:
the reference that decides who is right when the kernels and the oracle disagree."""
import mpmath
import numpy as np

POW_EXP = float(np.float32(2.2))        # the tonemap's exponent, as the binary32 the kernels pass
FUNCS = ["sin", "cos", "acos", "asin", "pow"]


def mp_value(fn, x):
    """the exact function value at binary32 x, to 200 bits (pow: x ** 2.2f)"""
    with mpmath.workprec(200):
        a = mpmath.mpf(float(x))
        if fn == "sin":
            return mpmath.sin(a)
        if fn == "cos":
            return mpmath.cos(a)
        if fn == "acos":
            return mpmath.acos(a)
        if fn == "asin":
            return mpmath.asin(a)
        if fn == "pow":
            return mpmath.power(a, mpmath.mpf(POW_EXP))
        raise ValueError(fn)


def round_f32(v):
    """binary32 round-to-nearest-even of an mpmath value (subnormals included; no overflow on these domains)"""
    with mpmath.workprec(200):
        if v == 0:
            return np.float32(float(v))
        e = int(mpmath.floor(mpmath.log(abs(v), 2)))
        q = mpmath.ldexp(1, max(e, -126) - 23)
        n = v / q
        k = mpmath.floor(n)
        frac = n - k
        if frac > 0.5 or (frac == 0.5 and int(k) % 2):
            k += 1
        return np.float32(float(k * q))


def correctly_rounded(fn, x):
    """binary32 bits of fn at every binary32 x, correctly rounded; NaN where the function is undefined"""
    out = []
    for v in np.asarray(x, np.float32).reshape(-1):
        if not np.isfinite(v) or (fn in ("acos", "asin") and abs(v) > 1) or (fn == "pow" and v < 0):
            out.append(np.float32(np.nan))
        else:
            out.append(round_f32(mp_value(fn, v)))
    return np.array(out, np.float32).view(np.uint32)
