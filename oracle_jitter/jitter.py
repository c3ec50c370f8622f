"""TEST INFRASTRUCTURE — ctypes access to oracle_jitter/_build/librt_oracle_jitter.so: the oracle (oracle/rt_oracle.c,
compiled in unchanged) in which every sample traces its own camera ray through a jittered point of its pixel, the rule
of include/b200rt.h's B200RT_SAMPLING_PIXEL_JITTER.  Only tests/ and tools/ may import this; the product never does."""
import ctypes
import os
import subprocess

import numpy as np

from oracle.oracle import OrcOpts, _f32p, _i32p, _u8p

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


def build(verbose=False):
    subprocess.check_call(["make", "-C", _HERE] + ([] if verbose else ["-s"]))


def _lib():
    global _LIB
    if _LIB is None:
        path = os.path.join(_HERE, "_build", "librt_oracle_jitter.so")
        if not os.path.exists(path):
            build()
        lib = ctypes.CDLL(path)
        lib.orc_render_jitter.restype = None
        lib.orc_render_jitter.argtypes = [_f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, _f32p, _f32p, ctypes.c_int,
                                          ctypes.c_int, ctypes.c_int, ctypes.c_int, _u8p, ctypes.c_int, ctypes.c_int,
                                          ctypes.c_int, ctypes.c_int, ctypes.POINTER(OrcOpts), ctypes.c_void_p]
        _LIB = lib
    return _LIB


def render(scene, cam, env, img_dim, spp, max_bounce, ibl_rgba, i0=0, i1=None, rng_mode=0, seed=0, stack_cap=20,
           s0=0, s1=0, raw_sums=False, nthreads=0, sampling=0):
    """oracle.render's arguments and result, (out[img_dim*3] float32, counters dict), with one jittered camera ray per
    sample; `sampling` takes bits 0 and 1 (the jitter is implied)."""
    lib = _lib()
    i1 = img_dim if i1 is None else i1
    out = np.zeros(img_dim * 3, dtype=np.float32)
    ibl = np.ascontiguousarray(ibl_rgba, dtype=np.uint8)
    h, w = ibl.shape[0], ibl.shape[1]
    light = np.ascontiguousarray(scene.get("lightData", np.zeros(0, np.int32)), dtype=np.int32)
    opts = OrcOpts(rng_mode, seed & 0xFFFFFFFF, (seed >> 32) & 0xFFFFFFFF, stack_cap, s0, s1, 1 if raw_sums else 0,
                   nthreads, sampling, int(light.size), light.ctypes.data_as(ctypes.c_void_p) if light.size else None)
    cnt = (ctypes.c_ulonglong * 4)()
    face = scene["faceData"]
    lib.orc_render_jitter(out, scene["V_p"], scene["V_n"], scene["V_uv"], face, scene["materialData"], scene["BVH"],
                          np.ascontiguousarray(cam, np.float32), np.ascontiguousarray(env, np.float32),
                          face.size // 10, img_dim, spp, max_bounce, ibl.reshape(-1), w, h, i0, i1,
                          ctypes.byref(opts), ctypes.cast(cnt, ctypes.c_void_p))
    return out, {"rays": cnt[0], "box_tests": cnt[1], "tri_tests": cnt[2], "rand_calls": cnt[3]}
