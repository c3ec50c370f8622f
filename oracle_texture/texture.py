"""TEST INFRASTRUCTURE — ctypes access to oracle_texture/_build/librt_oracle_texture.so: the oracle (oracle/rt_oracle.c,
oracle_smooth/ and oracle_glass/, compiled in unchanged) in which sampling bit 512 gives every diffuse or glossy hit the
albedo of include/b200rt.h's B200RT_SAMPLING_TEXTURES.  One entry point covers the plain, pixel-jitter (bit 8),
smooth-shading (bit 32), refractive-glass (bit 128) and adaptive renders.  Only tests/ and tools/ may import this; the
product never does."""
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
        path = os.path.join(_HERE, "_build", "librt_oracle_texture.so")
        if not os.path.exists(path):
            build()
        lib = ctypes.CDLL(path)
        lib.orc_render_tex.restype = None
        lib.orc_render_tex.argtypes = [_f32p, _f32p, _f32p, _f32p, _i32p, _f32p, _f32p, _f32p, _f32p, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_int, ctypes.c_int, _u8p, ctypes.c_int, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_int, ctypes.POINTER(OrcOpts),
                                       ctypes.POINTER(OrcAdaptive), _i32p, _f32p, ctypes.c_void_p,
                                       _u8p, _i32p, ctypes.c_int, _i32p, ctypes.c_int]
        lib.orc_gbuffer_albedo_tex.restype = None
        lib.orc_gbuffer_albedo_tex.argtypes = [_f32p, _f32p, _f32p, _i32p, _f32p, _f32p, ctypes.c_int, _i32p, _f32p,
                                               _u8p, _i32p, ctypes.c_int, _i32p, ctypes.c_int]
        lib.orc_texel.restype = None
        lib.orc_texel.argtypes = [_u8p, ctypes.c_int, ctypes.c_int, ctypes.c_int, _f32p, _f32p, _f32p]
        _LIB = lib
    return _LIB


def pack(textures):
    """(texels uint8, dims int32 (w, h) per texture, mat_tex int32) of a {material: (H, W, 4) uint8 RGBA} dict, one
    texture per distinct array object, the layout b200rt_set_textures takes"""
    images, index = [], {}
    for m, a in sorted((textures or {}).items()):
        k = next((i for i, b in enumerate(images) if b is a), None)
        if k is None:
            k = len(images)
            images.append(a)
        index[m] = k
    mat_tex = np.full(max(index) + 1 if index else 0, -1, np.int32)
    for m, k in index.items():
        mat_tex[m] = k
    texels = (np.concatenate([np.ascontiguousarray(a, np.uint8).reshape(-1) for a in images]) if images
              else np.zeros(4, np.uint8))
    dims = np.array([[a.shape[1], a.shape[0]] for a in images] or [[1, 1]], np.int32).reshape(-1)
    return texels, dims, len(images), mat_tex if mat_tex.size else np.full(1, -1, np.int32), int(mat_tex.size)


def render(scene, cam, env, img_dim, spp, max_bounce, ibl_rgba, i0=0, i1=None, rng_mode=0, seed=0, stack_cap=20,
           s0=0, s1=0, raw_sums=False, nthreads=0, sampling=0, adaptive=None, textures=None):
    """oracle_glass.glass.render's arguments and result; `sampling` takes bits 0, 1, 8, 32, 128 and 512, `textures` is
    a {material index: (H, W, 4) uint8 RGBA array} dict (None: nothing bound)."""
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
    lib.orc_render_tex(out, scene["V_p"], scene["V_n"], np.ascontiguousarray(scene["V_uv"], np.float32), face,
                       np.ascontiguousarray(scene["materialData"], np.float32), scene["BVH"],
                       np.ascontiguousarray(cam, np.float32), np.ascontiguousarray(env, np.float32),
                       face.size // 10, img_dim, spp, max_bounce, ibl.reshape(-1), w, h, i0, i1,
                       ctypes.byref(opts), ad, spp_map, err_map, ctypes.cast(cnt, ctypes.c_void_p),
                       texels, dims, n_tex, mat_tex, n_mat)
    counters = {"rays": cnt[0], "box_tests": cnt[1], "tri_tests": cnt[2], "rand_calls": cnt[3]}
    if adaptive is not None:
        return out, spp_map, err_map, counters
    return out, counters


def gbuffer_albedo(scene, cam, tri, k, textures=None):
    """(n, 3) float32: the G-buffer albedo of primary hits tri / k (n,) of the first n work-items"""
    tri = np.ascontiguousarray(tri, np.int32).reshape(-1)
    k = np.ascontiguousarray(k, np.float32).reshape(-1)
    out = np.zeros(tri.size * 3, np.float32)
    texels, dims, n_tex, mat_tex, n_mat = pack(textures)
    _lib().orc_gbuffer_albedo_tex(out, scene["V_p"], np.ascontiguousarray(scene["V_uv"], np.float32), scene["faceData"],
                                  np.ascontiguousarray(scene["materialData"], np.float32),
                                  np.ascontiguousarray(cam, np.float32), tri.size, tri, k, texels, dims, n_tex,
                                  mat_tex, n_mat)
    return out.reshape(-1, 3)


def texel(rgba, u, v):
    """(n, 3) float32: the texture factor of one (H, W, 4) uint8 texture at points (u, v) (n,)"""
    rgba = np.ascontiguousarray(rgba, np.uint8)
    u = np.ascontiguousarray(u, np.float32).reshape(-1)
    v = np.ascontiguousarray(v, np.float32).reshape(-1)
    out = np.zeros(u.size * 3, np.float32)
    _lib().orc_texel(rgba.reshape(-1), rgba.shape[1], rgba.shape[0], u.size, u, v, out)
    return out.reshape(-1, 3)
