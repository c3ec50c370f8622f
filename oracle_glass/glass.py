"""TEST INFRASTRUCTURE — ctypes access to oracle_glass/_build/librt_oracle_glass.so: the oracle (oracle/rt_oracle.c and
oracle_smooth/rt_oracle_smooth.c, compiled in unchanged) in which sampling bit 128 makes a type-3 surface the smooth
dielectric interface of include/b200rt.h's B200RT_SAMPLING_DIELECTRIC_GLASS.  One entry point covers the plain,
pixel-jitter (bit 8), smooth-shading (bit 32) and adaptive renders.  Only tests/ and tools/ may import this; the product
never does."""
import ctypes
import os
import subprocess

import numpy as np

from oracle.oracle import OrcOpts, _f32p, _i32p, _u8p
from oracle_adaptive.adaptive import OrcAdaptive

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(verbose=False):
    subprocess.check_call(["make", "-C", _HERE] + ([] if verbose else ["-s"]))


def _lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "_build", "librt_oracle_glass.so")
        if not os.path.exists(path):
            build()
        lib = ctypes.CDLL(path)
        lib.orc_render_glass.restype = None
        lib.orc_render_glass.argtypes = [_f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, _f32p, _f32p, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.c_int, _u8p, ctypes.c_int, ctypes.c_int,
                                         ctypes.c_int, ctypes.c_int, ctypes.POINTER(OrcOpts),
                                         ctypes.POINTER(OrcAdaptive), _i32p, _f32p, ctypes.c_void_p]
        lib.orc_dielectric.restype = None
        lib.orc_dielectric.argtypes = [ctypes.c_int, _f32p, _f32p, _f32p, _f32p, _f32p, _i32p, _f32p]
        _LIB = lib
    return _LIB


def render(scene, cam, env, img_dim, spp, max_bounce, ibl_rgba, i0=0, i1=None, rng_mode=0, seed=0, stack_cap=20,
           s0=0, s1=0, raw_sums=False, nthreads=0, sampling=0, adaptive=None):
    """oracle.render's arguments and result, (out[img_dim*3] float32, counters dict); `sampling` takes bits 0, 1, 8, 32
    and 128.  adaptive: a dict as oracle_adaptive.adaptive.render takes it; the result is then (out, spp_map,
    stderr_map, counters) as that function returns it."""
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
    lib.orc_render_glass(out, scene["V_p"], scene["V_n"], scene["V_uv"], face,
                         np.ascontiguousarray(scene["materialData"], np.float32), scene["BVH"],
                         np.ascontiguousarray(cam, np.float32), np.ascontiguousarray(env, np.float32),
                         face.size // 10, img_dim, spp, max_bounce, ibl.reshape(-1), w, h, i0, i1,
                         ctypes.byref(opts), ad, spp_map, err_map, ctypes.cast(cnt, ctypes.c_void_p))
    counters = {"rays": cnt[0], "box_tests": cnt[1], "tri_tests": cnt[2], "rand_calls": cnt[3]}
    if adaptive is not None:
        return out, spp_map, err_map, counters
    return out, counters


def dielectric(w, n, ior, u):
    """the oracle's interface rule for m cases: w (m, 3) incoming directions, n (m, 3) unit normals, ior (m,) ior slots
    (0 resolves to B200RT_GLASS_DEFAULT_IOR), u (m,) uniforms -> (directions (m, 3) float32, reflected (m,) bool,
    F (m,) float32, 1 on total internal reflection)"""
    w = np.ascontiguousarray(w, np.float32).reshape(-1)
    n = np.ascontiguousarray(n, np.float32).reshape(-1)
    ior = np.ascontiguousarray(ior, np.float32).reshape(-1)
    u = np.ascontiguousarray(u, np.float32).reshape(-1)
    m = ior.size
    d = np.zeros(3 * m, np.float32)
    refl = np.zeros(m, np.int32)
    F = np.zeros(m, np.float32)
    _lib().orc_dielectric(m, w, n, ior, u, d, refl, F)
    return d.reshape(-1, 3), refl.astype(bool), F
