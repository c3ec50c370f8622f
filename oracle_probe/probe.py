"""TEST INFRASTRUCTURE — ctypes access to oracle_probe/_build/librt_oracle_probe.so: the oracle's per-hit shading rules
(oracle/rt_oracle.c and the oracle_smooth/, oracle_glass/, oracle_texture/ and oracle_rough/ modes, compiled in
unchanged) one record at a time, in the layout of include/b200rt.h's b200rt_rule_probe.  Only tests/ and tools/ may
import this; the product never does."""
import ctypes
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

# rule codes of b200rt_rule_probe
DIELECTRIC, ROUGH_DIELECTRIC, COSINE_FLAT, COSINE_SMOOTH, UNIFORM_FLAT, UNIFORM_SMOOTH = 0, 1, 2, 3, 4, 5
GLOSSY, GGX, LIGHT, SMOOTH_NORMAL, ALBEDO, TEXEL = 6, 7, 8, 9, 10, 11


def build(verbose=False):
    subprocess.check_call(["make", "-C", _HERE] + ([] if verbose else ["-s"]))


def _lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "_build", "librt_oracle_probe.so")
        if not os.path.exists(path):
            build()
        lib = ctypes.CDLL(path)
        lib.orc_rule_probe.restype = None
        vp = ctypes.c_void_p
        lib.orc_rule_probe.argtypes = [ctypes.c_int, vp, ctypes.c_int, vp, vp, vp, vp, vp, vp, ctypes.c_int, vp, vp,
                                       ctypes.c_int, vp, ctypes.c_int]
        _LIB = lib
    return _LIB


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def records(m):
    """m zeroed records as (m, 16) uint32: set float fields through .view(np.float32), integer fields and uniform words
    directly"""
    return np.zeros((m, 16), np.uint32)


def rule_probe(rule, recs, scene=None, tex=None, threads=1):
    """orc_rule_probe of the (m, 16) 4-byte records `recs` -> (m, 8) float32.  scene: a fixture dict (V_p, V_n, V_uv,
    faceData, materialData) for rules 8-10; tex: (texels uint8, dims int32 (w, h) per texture, mat_tex int32) as
    b200rt_set_textures takes them, for rules 10 and 11.  threads > 1 splits the records over a thread pool (ctypes
    releases the GIL)."""
    rec = np.ascontiguousarray(recs)
    assert rec.ndim == 2 and rec.shape[1] == 16 and rec.dtype.itemsize == 4
    rec = rec.view(np.float32)
    m = rec.shape[0]
    out = np.zeros((m, 8), np.float32)
    arrs = [None] * 5
    n_tri = 0
    if scene is not None:
        arrs = [np.ascontiguousarray(scene[k], t) for k, t in
                (("V_p", np.float32), ("V_n", np.float32), ("V_uv", np.float32), ("faceData", np.int32),
                 ("materialData", np.float32))]
        n_tri = arrs[3].size // 10
    texels = dims = mat_tex = None
    n_tex = n_mat = 0
    if tex is not None:
        texels, dims, mat_tex = (np.ascontiguousarray(a, t) for a, t in zip(tex, (np.uint8, np.int32, np.int32)))
        n_tex, n_mat = dims.size // 2, mat_tex.size
    lib = _lib()

    def run(lo, hi):
        lib.orc_rule_probe(int(rule), _p(rec[lo:hi]), hi - lo, _p(out[lo:hi]), *map(_p, arrs), n_tri, _p(texels),
                           _p(dims), n_tex, _p(mat_tex), n_mat)

    step = max(1, -(-m // max(1, threads)))
    with ThreadPoolExecutor(max(1, threads)) as ex:
        list(ex.map(lambda lo: run(lo, min(m, lo + step)), range(0, m, step)))
    return out
