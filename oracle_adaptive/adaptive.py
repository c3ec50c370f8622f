"""TEST INFRASTRUCTURE — ctypes access to oracle_adaptive/_build/librt_oracle_adaptive.so: the oracle
(oracle/rt_oracle.c, compiled in unchanged) with the adaptive-sampling rule of include/b200rt.h applied inside its
per-pixel sample loop.  Only tests/ may import this; the product never does."""
import ctypes
import os
import subprocess

import numpy as np

from oracle.oracle import OrcOpts, _f32p, _i32p, _u8p

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class OrcAdaptive(ctypes.Structure):
    _fields_ = [("min_spp", ctypes.c_int), ("check_every", ctypes.c_int), ("rel_error", ctypes.c_float),
                ("floor", ctypes.c_float)]


def build(verbose=False):
    subprocess.check_call(["make", "-C", _HERE] + ([] if verbose else ["-s"]))


def _lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "_build", "librt_oracle_adaptive.so")
        if not os.path.exists(path):
            build()
        lib = ctypes.CDLL(path)
        lib.orc_render_adaptive.restype = None
        lib.orc_render_adaptive.argtypes = [_f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, _f32p, _f32p, ctypes.c_int,
                                            ctypes.c_int, ctypes.c_int, ctypes.c_int, _u8p, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_int, ctypes.c_int, ctypes.POINTER(OrcOpts),
                                            ctypes.POINTER(OrcAdaptive), _i32p, _f32p, ctypes.c_void_p]
        _LIB = lib
    return _LIB


def render(scene, cam, env, img_dim, spp, max_bounce, ibl_rgba, adaptive, i0=0, i1=None, rng_mode=0, seed=0,
           stack_cap=20, nthreads=0, sampling=0):
    """adaptive: dict(rel_error, min_spp=16, check_every=8, floor=0.05), the fields of b200rt_adaptive.
    Returns (out[img_dim*3] float32, spp_map[img_dim] int32, stderr_map[img_dim] float32, counters dict); entries
    outside [i0, i1) are 0."""
    lib = _lib()
    i1 = img_dim if i1 is None else i1
    ad = OrcAdaptive(int(adaptive.get("min_spp", 16)), int(adaptive.get("check_every", 8)),
                     float(adaptive["rel_error"]), float(adaptive.get("floor", 0.05)))
    out = np.zeros(img_dim * 3, dtype=np.float32)
    spp_map = np.zeros(img_dim, dtype=np.int32)
    err_map = np.zeros(img_dim, dtype=np.float32)
    ibl = np.ascontiguousarray(ibl_rgba, dtype=np.uint8)
    h, w = ibl.shape[0], ibl.shape[1]
    light = np.ascontiguousarray(scene.get("lightData", np.zeros(0, np.int32)), dtype=np.int32)
    opts = OrcOpts(rng_mode, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF, stack_cap, 0, 0, 0, nthreads, sampling,
                   int(light.size), light.ctypes.data_as(ctypes.c_void_p) if light.size else None)
    cnt = (ctypes.c_ulonglong * 4)()
    face = scene["faceData"]
    lib.orc_render_adaptive(out, scene["V_p"], scene["V_n"], scene["V_uv"], face, scene["materialData"], scene["BVH"],
                            np.ascontiguousarray(cam, np.float32), np.ascontiguousarray(env, np.float32),
                            face.size // 10, img_dim, spp, max_bounce, ibl.reshape(-1), w, h, i0, i1,
                            ctypes.byref(opts), ctypes.byref(ad), spp_map, err_map, ctypes.cast(cnt, ctypes.c_void_p))
    return out, spp_map, err_map, {"rays": cnt[0], "box_tests": cnt[1], "tri_tests": cnt[2], "rand_calls": cnt[3]}
