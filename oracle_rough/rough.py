"""TEST INFRASTRUCTURE — ctypes access to oracle_rough/_build/librt_oracle_rough.so: the oracle (oracle/rt_oracle.c,
oracle_smooth/, oracle_glass/ and oracle_texture/, compiled in unchanged) in which sampling bits 128 | 2048 make a glass
surface of roughness > 0 the rough GGX interface of include/b200rt.h's B200RT_SAMPLING_ROUGH_GLASS.  One entry point
covers the plain, pixel-jitter (bit 8), smooth-shading (bit 32), refractive-glass (bit 128), texture (bit 512) and
adaptive renders.  Only tests/ and tools/ may import this; the product never does."""
import ctypes
import os
import subprocess

import numpy as np

from oracle.oracle import OrcOpts, _f32p, _i32p, _u8p
from oracle_adaptive.adaptive import OrcAdaptive
from oracle_texture.texture import pack

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(verbose=False):
    subprocess.check_call(["make", "-C", _HERE] + ([] if verbose else ["-s"]))


def _lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "_build", "librt_oracle_rough.so")
        if not os.path.exists(path):
            build()
        lib = ctypes.CDLL(path)
        lib.orc_render_rough.restype = None
        lib.orc_render_rough.argtypes = [_f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, _f32p, _f32p, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.c_int, _u8p, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.POINTER(OrcOpts),
                                         ctypes.POINTER(OrcAdaptive), _i32p, _f32p, ctypes.c_void_p,
                                         _u8p, _i32p, ctypes.c_int, _i32p, ctypes.c_int]
        lib.orc_rough_dielectric.restype = None
        lib.orc_rough_dielectric.argtypes = [ctypes.c_int, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p, _f32p,
                                             _i32p, _f32p]
        _LIB = lib
    return _LIB


def render(scene, cam, env, img_dim, spp, max_bounce, ibl_rgba, i0=0, i1=None, rng_mode=0, seed=0, stack_cap=20,
           s0=0, s1=0, raw_sums=False, nthreads=0, sampling=0, adaptive=None, textures=None):
    """oracle_texture.texture.render's arguments and result; `sampling` also takes bit 2048 (with 128)."""
    lib = _lib()
    i1 = img_dim if i1 is None else i1
    out = np.zeros(img_dim * 3, dtype=np.float32)
    spp_map = np.zeros(img_dim, dtype=np.int32)
    err_map = np.zeros(img_dim, dtype=np.float32)
    ibl = np.ascontiguousarray(ibl_rgba, dtype=np.uint8)
    h, w = ibl.shape[0], ibl.shape[1]
    light = np.ascontiguousarray(scene.get("lightData", np.zeros(0, np.int32)), dtype=np.int32)
    opts = OrcOpts(rng_mode, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF, stack_cap, s0, s1, 1 if raw_sums else 0,
                   nthreads, sampling, int(light.size), light.ctypes.data_as(ctypes.c_void_p) if light.size else None)
    ad = None
    if adaptive is not None:
        ad = ctypes.byref(OrcAdaptive(int(adaptive.get("min_spp", 16)), int(adaptive.get("check_every", 8)),
                                      float(adaptive["rel_error"]), float(adaptive.get("floor", 0.05))))
    cnt = (ctypes.c_ulonglong * 4)()
    face = scene["faceData"]
    texels, dims, n_tex, mat_tex, n_mat = pack(textures)
    lib.orc_render_rough(out, scene["V_p"], scene["V_n"], np.ascontiguousarray(scene["V_uv"], np.float32), face,
                         np.ascontiguousarray(scene["materialData"], np.float32), scene["BVH"],
                         np.ascontiguousarray(cam, np.float32), np.ascontiguousarray(env, np.float32),
                         face.size // 10, img_dim, spp, max_bounce, ibl.reshape(-1), w, h, i0, i1,
                         ctypes.byref(opts), ad, spp_map, err_map, ctypes.cast(cnt, ctypes.c_void_p),
                         texels, dims, n_tex, mat_tex, n_mat)
    counters = {"rays": cnt[0], "box_tests": cnt[1], "tri_tests": cnt[2], "rand_calls": cnt[3]}
    if adaptive is not None:
        return out, spp_map, err_map, counters
    return out, counters


def rough_dielectric(w, n, ior, r, uf, u1, u2):
    """the oracle's rough interface rule for m cases: w (m, 3) incoming directions, n (m, 3) unit normals, ior (m,) ior
    slots (not 1; 0 resolves to B200RT_GLASS_DEFAULT_IOR), r (m,) roughness > 0, uf u1 u2 (m,) uniforms ->
    (directions (m, 3) float32, reflected (m,) bool, weight (m,) float32)"""
    cols = [np.ascontiguousarray(a, np.float32).reshape(-1) for a in (w, n, ior, r, uf, u1, u2)]
    m = cols[2].size
    d = np.zeros(3 * m, np.float32)
    refl = np.zeros(m, np.int32)
    wt = np.zeros(m, np.float32)
    _lib().orc_rough_dielectric(m, *cols, d, refl, wt)
    return d.reshape(-1, 3), refl.astype(bool), wt
