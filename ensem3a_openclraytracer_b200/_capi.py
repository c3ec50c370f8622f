"""ctypes binding of include/b200rt.h (lib/libb200rt.so).

This module is the only place the package touches native code.  It raises if the library is
missing or the GPU cannot be used — there is no CPU, OpenCL or PyTorch fallback behind it.
"""
import ctypes
import os
import subprocess

import numpy as np

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "lib", "libb200rt.so")
CSRC = os.path.join(_PKG, "csrc")

RNG_REFERENCE, RNG_PHILOX = 0, 1
TRAVERSAL_FAST, TRAVERSAL_REFERENCE, TRAVERSAL_VERIFY = 0, 1, 2
OUT_FINAL, OUT_SUMS = 0, 1
SAMPLING_REFERENCE, SAMPLING_IMPORTANCE, SAMPLING_LIGHTS = 0, 1, 2


class B200RTError(RuntimeError):
    pass


class Opts(ctypes.Structure):
    _fields_ = [("rng_mode", ctypes.c_int32), ("traversal", ctypes.c_int32), ("stack_cap", ctypes.c_int32),
                ("output", ctypes.c_int32), ("sample_begin", ctypes.c_int32), ("sample_end", ctypes.c_int32),
                ("pixel_begin", ctypes.c_int32), ("pixel_end", ctypes.c_int32), ("seed", ctypes.c_uint64),
                ("collect_stats", ctypes.c_int32), ("time_kernels", ctypes.c_int32), ("tile_row_mod", ctypes.c_int32),
                ("tile_row_rem", ctypes.c_int32), ("sample_streams", ctypes.c_int32), ("sampling", ctypes.c_int32)]


class Stats(ctypes.Structure):
    _fields_ = [("rays", ctypes.c_uint64), ("box_tests", ctypes.c_uint64), ("tri_tests", ctypes.c_uint64),
                ("mismatches", ctypes.c_uint64), ("samples", ctypes.c_uint64), ("primary_ms", ctypes.c_float),
                ("trace_ms", ctypes.c_float), ("total_ms", ctypes.c_float), ("upload_ms", ctypes.c_float),
                ("kernel_launches", ctypes.c_int32), ("nodes", ctypes.c_int32), ("triangles", ctypes.c_int32),
                ("bvh_depth", ctypes.c_int32), ("scene_in_smem", ctypes.c_int32), ("revalidated", ctypes.c_int32),
                ("shade_kernel_ms", ctypes.c_float), ("trace_kernel_ms", ctypes.c_float), ("repack_ms", ctypes.c_float),
                ("ref_stack_need", ctypes.c_int32), ("exact_walks", ctypes.c_int32), ("wave_iterations", ctypes.c_int32),
                ("sample_streams", ctypes.c_int32), ("primary_rays", ctypes.c_uint64)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_ if not k.startswith("reserved")}


class Adaptive(ctypes.Structure):
    """b200rt_adaptive: the stopping rule of adaptive sampling (include/b200rt.h)."""
    _fields_ = [("min_spp", ctypes.c_int32), ("check_every", ctypes.c_int32), ("rel_error", ctypes.c_float),
                ("floor", ctypes.c_float)]


class Denoise(ctypes.Structure):
    """b200rt_denoise_params: the edge-avoiding à-trous filter's parameters (include/b200rt.h)."""
    _fields_ = [("passes", ctypes.c_int32), ("sigma_color", ctypes.c_float), ("sigma_normal", ctypes.c_float),
                ("sigma_position", ctypes.c_float)]


# B200RT_DENOISE_* of include/b200rt.h; sigma_position 0 = automatic (1 % of the scene's BVH root-box diagonal)
DENOISE_DEFAULTS = dict(passes=5, sigma_color=0.5, sigma_normal=0.2, sigma_position=0.0)


def _denoise_params(passes=DENOISE_DEFAULTS["passes"], sigma_color=DENOISE_DEFAULTS["sigma_color"],
                    sigma_normal=DENOISE_DEFAULTS["sigma_normal"], sigma_position=DENOISE_DEFAULTS["sigma_position"]):
    return Denoise(int(passes), float(sigma_color), float(sigma_normal), float(sigma_position))


# every symbol include/b200rt.h declares (tests/test_abi.py checks the header against this list)
SYMBOLS = [
    "b200rt_default_opts", "b200rt_create", "b200rt_destroy", "b200rt_last_error", "b200rt_set_scene",
    "b200rt_set_materials", "b200rt_set_ibl", "b200rt_render", "b200rt_render_adaptive", "b200rt_gbuffer", "b200rt_denoise", "b200rt_render_denoised", "b200rt_render_rgb8", "b200rt_render_device", "b200rt_finalize_device",
    "b200rt_reduce_finalize_device", "b200rt_sync", "b200rt_set_stream", "b200rt_invalidate", "b200rt_primary_hits", "b200rt_trace_rays",
    "b200rt_img_processing", "b200rt_get_stats", "b200rt_math_probe", "b200rt_philox_probe", "b200rt_alloc",
    "b200rt_free", "b200rt_ipc_export",
    "b200rt_ipc_open", "b200rt_ipc_close", "b200rt_build_bvh", "b200rt_repack_probe", "b200rt_version", "b200rt_device_count",
    "b200rt_multi_create", "b200rt_multi_destroy", "b200rt_multi_last_error", "b200rt_multi_device_count",
    "b200rt_multi_context", "b200rt_multi_set_scene", "b200rt_multi_set_ibl", "b200rt_multi_invalidate",
    "b200rt_multi_render", "b200rt_multi_render_denoised", "b200rt_multi_get_stats",
]

_lib = None


def build_library(verbose=False):
    """Compiles csrc/ for sm_100a into lib/libb200rt.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", CSRC] + ([] if verbose else ["-s"])
    subprocess.check_call(cmd)
    return LIB_PATH


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B200RTError(f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(or `make -C ensem3a_openclraytracer_b200/csrc`). There is no fallback renderer.")
    lib = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint32
    lib.b200rt_version.restype = ctypes.c_char_p
    lib.b200rt_last_error.restype = ctypes.c_char_p
    lib.b200rt_last_error.argtypes = [vp]
    lib.b200rt_default_opts.restype = None
    lib.b200rt_default_opts.argtypes = [ctypes.POINTER(Opts)]
    lib.b200rt_create.argtypes = [i32, ctypes.POINTER(vp)]
    lib.b200rt_destroy.restype = None
    lib.b200rt_destroy.argtypes = [vp]
    lib.b200rt_set_scene.argtypes = [vp, vp, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp, i64]
    lib.b200rt_set_materials.argtypes = [vp, vp, i64]
    lib.b200rt_set_ibl.argtypes = [vp, vp, i32, i32]
    lib.b200rt_render.argtypes = [vp, vp, vp, i32, i32, i32, i32, ctypes.POINTER(Opts), vp]
    lib.b200rt_render_adaptive.argtypes = [vp, vp, vp, i32, i32, i32, i32, ctypes.POINTER(Opts), ctypes.POINTER(Adaptive),
                                           vp, vp, vp]
    lib.b200rt_gbuffer.argtypes = [vp, vp, i32, i32, ctypes.POINTER(Opts), vp, vp, vp, vp]
    lib.b200rt_denoise.argtypes = [vp, vp, vp, vp, vp, vp, i32, i32, ctypes.POINTER(Denoise), vp]
    lib.b200rt_render_denoised.argtypes = [vp, vp, vp, i32, i32, i32, i32, ctypes.POINTER(Opts), ctypes.POINTER(Denoise),
                                           vp, vp]
    lib.b200rt_multi_render_denoised.argtypes = lib.b200rt_render_denoised.argtypes
    lib.b200rt_render_device.argtypes = [vp, vp, vp, i32, i32, i32, i32, ctypes.POINTER(Opts), vp]
    lib.b200rt_render_rgb8.argtypes = [vp, vp, vp, i32, i32, i32, i32, ctypes.POINTER(Opts), vp]
    lib.b200rt_finalize_device.argtypes = [vp, vp, vp, i64, i32]
    lib.b200rt_reduce_finalize_device.argtypes = [vp, ctypes.POINTER(vp), i32, vp, i64, i32]
    lib.b200rt_sync.argtypes = [vp]
    lib.b200rt_set_stream.argtypes = [vp, vp]
    lib.b200rt_invalidate.argtypes = [vp]
    lib.b200rt_primary_hits.argtypes = [vp, vp, i32, i32, ctypes.POINTER(Opts), vp, vp]
    lib.b200rt_trace_rays.argtypes = [vp, vp, i64, ctypes.POINTER(Opts), vp, vp]
    lib.b200rt_img_processing.argtypes = [vp, vp, vp, i64, i64]
    lib.b200rt_get_stats.argtypes = [vp, ctypes.POINTER(Stats)]
    lib.b200rt_math_probe.argtypes = [vp, i32, vp, vp, i64, vp]
    lib.b200rt_philox_probe.argtypes = [vp, ctypes.POINTER(u32 * 4), u32, u32, ctypes.POINTER(u32 * 4)]
    lib.b200rt_alloc.argtypes = [vp, i64, ctypes.POINTER(vp)]
    lib.b200rt_free.argtypes = [vp, vp]
    lib.b200rt_ipc_export.argtypes = [vp, vp, vp]
    lib.b200rt_ipc_open.argtypes = [vp, vp, ctypes.POINTER(vp)]
    lib.b200rt_ipc_close.argtypes = [vp, vp]
    lib.b200rt_build_bvh.argtypes = [vp, i64, vp, i64, vp, i64, ctypes.POINTER(ctypes.c_int32)]
    lib.b200rt_repack_probe.argtypes = [vp, i64, vp, i64, vp, i64, i64, vp, i64, vp, i64, vp, vp]
    lib.b200rt_multi_create.argtypes = [ctypes.POINTER(ctypes.c_int), i32, ctypes.POINTER(vp)]
    lib.b200rt_multi_destroy.restype = None
    lib.b200rt_multi_destroy.argtypes = [vp]
    lib.b200rt_multi_last_error.restype = ctypes.c_char_p
    lib.b200rt_multi_last_error.argtypes = [vp]
    lib.b200rt_multi_device_count.argtypes = [vp]
    lib.b200rt_multi_context.restype = vp
    lib.b200rt_multi_context.argtypes = [vp, i32]
    lib.b200rt_multi_set_scene.argtypes = [vp, vp, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp, i64]
    lib.b200rt_multi_set_ibl.argtypes = [vp, vp, i32, i32]
    lib.b200rt_multi_invalidate.argtypes = [vp]
    lib.b200rt_multi_render.argtypes = [vp, vp, vp, i32, i32, i32, i32, ctypes.POINTER(Opts), vp]
    lib.b200rt_multi_get_stats.argtypes = [vp, ctypes.POINTER(Stats)]
    for name in SYMBOLS:
        fn = getattr(lib, name)
        if name not in ("b200rt_version", "b200rt_last_error", "b200rt_default_opts", "b200rt_destroy",
                        "b200rt_multi_destroy", "b200rt_multi_last_error", "b200rt_multi_context"):
            fn.restype = ctypes.c_int
    _lib = lib
    return lib


def _ptr(a):
    return a.ctypes.data_as(ctypes.c_void_p) if a is not None else None


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32).reshape(-1)


def _i32(a):
    return np.ascontiguousarray(a, dtype=np.int32).reshape(-1)


def make_opts(rng_mode=RNG_REFERENCE, traversal=TRAVERSAL_FAST, stack_cap=20, output=OUT_FINAL, sample_begin=0,
              sample_end=0, pixel_begin=0, pixel_end=0, seed=0, collect_stats=False, time_kernels=False, tile_row_mod=0,
              tile_row_rem=0, sample_streams=0, sampling=SAMPLING_REFERENCE):
    o = Opts()
    o.rng_mode, o.traversal, o.stack_cap, o.output = rng_mode, traversal, stack_cap, output
    o.sample_begin, o.sample_end, o.pixel_begin, o.pixel_end = sample_begin, sample_end, pixel_begin, pixel_end
    o.seed = seed & 0xFFFFFFFFFFFFFFFF
    o.collect_stats = 1 if collect_stats else 0
    o.time_kernels = 1 if time_kernels else 0
    o.tile_row_mod, o.tile_row_rem = int(tile_row_mod), int(tile_row_rem)
    o.sample_streams = int(sample_streams)
    o.sampling = int(sampling)
    return o


def build_bvh(face_data, vertex_p, return_depth=False):
    """BVH.py's exportArray (float32, 9 per node) for the given faceData / V_p, built natively (host cores)."""
    lib = load_library()
    face, vp_ = _i32(face_data), _f32(vertex_p)
    if face.size == 0 or face.size % 10:
        raise B200RTError("faceData must hold 10 ints per triangle")
    out = np.empty((2 * (face.size // 10) - 1) * 9, dtype=np.float32)
    depth = ctypes.c_int32(0)
    rc = lib.b200rt_build_bvh(_ptr(vp_), vp_.size, _ptr(face), face.size, _ptr(out), out.size, ctypes.byref(depth))
    if rc != 0:
        raise B200RTError(f"b200rt_build_bvh failed ({rc}): malformed buffers, more than 2^23 triangles, or a node whose "
                          "centroids all fall on one side of their mean (BVH.py does not terminate on such input)")
    return (out, depth.value) if return_depth else out


def device_count():
    """CUDA devices visible to the process."""
    lib = load_library()
    return int(lib.b200rt_device_count())


def repack_probe(vertex_p, vertex_n, face_data, n_materials, bvh):
    """(nodes[n_inner, 8] uint32, info dict) — the interior-node records b200rt_set_scene would upload (host only)."""
    lib = load_library()
    vp_, vn_, face, bvh_ = _f32(vertex_p), _f32(vertex_n), _i32(face_data), _f32(bvh)
    info = np.zeros(24, np.float32)
    rc = lib.b200rt_repack_probe(_ptr(vp_), vp_.size, _ptr(vn_), vn_.size, _ptr(face), face.size, int(n_materials),
                                 _ptr(bvh_), bvh_.size, None, 0, None, _ptr(info))
    if rc != 0:
        raise B200RTError(f"b200rt_repack_probe failed ({rc})")
    nodes = np.zeros((int(info[0]), 8), np.uint32)
    ranks = np.zeros(face.size // 10, np.int32)
    rc = lib.b200rt_repack_probe(_ptr(vp_), vp_.size, _ptr(vn_), vn_.size, _ptr(face), face.size, int(n_materials),
                                 _ptr(bvh_), bvh_.size, _ptr(nodes), nodes.size, _ptr(ranks), _ptr(info))
    if rc != 0:
        raise B200RTError(f"b200rt_repack_probe failed ({rc})")
    d = dict(n_inner=int(info[0]), node_f4=int(info[1]), depth=int(info[2]), ref_stack_need=int(info[3]),
             canonical=bool(info[4]), fast_ok=bool(info[5]), cmax=float(info[6]), cull_abs=float(info[7]),
             grid_base=info[8:11].copy(), grid_pitch=info[11:14].copy(), root_qmin=info[14:17].copy(),
             root_qmax=info[17:20].copy(), ranks=ranks, ms_tris=float(info[20]), ms_walk=float(info[21]), ms_nodes=float(info[22]), cull_depth=int(info[23]))
    return nodes, d


class _Handle:
    """What Context and MultiContext share: the calls whose C symbols differ only in the prefix (`b200rt_` or
    `b200rt_multi_`), and errors reported with the prefix's last-error getter."""

    _prefix = "b200rt_"

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc, what):
        if rc != 0:
            err = getattr(self._lib, self._prefix + "last_error")(self._h).decode()
            raise B200RTError(f"{what} failed ({rc}): {err}")

    def _call(self, name, *args):
        fn = self._prefix + name
        self._check(getattr(self._lib, fn)(self._h, *args), fn)

    # ---- uploads -----------------------------------------------------------------------------------
    def set_scene(self, vertex_p, vertex_n, vertex_uv, face_data, material_data, light_data, bvh):
        vp_, vn_, vuv_ = _f32(vertex_p), _f32(vertex_n), _f32(vertex_uv)
        face, mat, bvh_ = _i32(face_data), _f32(material_data), _f32(bvh)
        light = _i32(light_data) if light_data is not None and len(light_data) else None
        self._call("set_scene", _ptr(vp_), vp_.size, _ptr(vn_), vn_.size, _ptr(vuv_), vuv_.size, _ptr(face), face.size,
                   _ptr(mat), mat.size, _ptr(light), 0 if light is None else light.size, _ptr(bvh_), bvh_.size)

    def set_ibl(self, rgba, width=None, height=None):
        """rgba: (H, W, 4) uint8 array, or bytes with explicit width/height."""
        if isinstance(rgba, (bytes, bytearray, memoryview)):
            arr = np.frombuffer(rgba, dtype=np.uint8)
        else:
            arr = np.ascontiguousarray(rgba, dtype=np.uint8)
            if width is None:
                height, width = arr.shape[0], arr.shape[1]
            arr = arr.reshape(-1)
        if arr.size != int(width) * int(height) * 4:
            raise B200RTError(f"environment map: {arr.size} bytes for {width}x{height} RGBA")
        self._call("set_ibl", _ptr(arr), int(width), int(height))

    def invalidate(self):
        self._call("invalidate")

    # ---- rendering ------------------------------------------------------------------------------------
    def render(self, cam, env, width, height, spp, max_bounce, out=None, opts=None):
        cam_, env_ = _f32(cam), _f32(env)
        if cam_.size != 10 or env_.size != 5:
            raise B200RTError("cam must hold 10 floats and envData 5 (main.py:59-61,72-73)")
        n = int(width) * int(height) * 3
        if out is None:
            out = np.zeros(n, dtype=np.float32)
        if out.dtype != np.float32 or not out.flags["C_CONTIGUOUS"] or out.size != n:
            raise B200RTError(f"out must be a C-contiguous float32 array of {n} elements")
        o = opts if opts is not None else make_opts()
        self._call("render", _ptr(cam_), _ptr(env_), int(width), int(height), int(spp), int(max_bounce), ctypes.byref(o),
                   _ptr(out))
        return out

    def render_denoised(self, cam, env, width, height, spp, max_bounce, opts=None, return_noisy=False, **denoise):
        """A render followed by the edge-avoiding à-trous filter of include/b200rt.h on the device (b200rt_render_denoised,
        or b200rt_multi_render_denoised).  denoise: passes, sigma_color, sigma_normal, sigma_position (0 = automatic),
        defaults DENOISE_DEFAULTS.  Returns the (H, W, 3) float32 image, and the undenoised one with return_noisy."""
        cam_, env_ = _f32(cam), _f32(env)
        if cam_.size != 10 or env_.size != 5:
            raise B200RTError("cam must hold 10 floats and envData 5 (main.py:59-61,72-73)")
        h, w = int(height), int(width)
        img = np.zeros((h, w, 3), dtype=np.float32)
        noisy = np.zeros((h, w, 3), dtype=np.float32) if return_noisy else None
        dn = _denoise_params(**denoise)
        o = opts if opts is not None else make_opts()
        self._call("render_denoised", _ptr(cam_), _ptr(env_), w, h, int(spp), int(max_bounce), ctypes.byref(o),
                   ctypes.byref(dn), _ptr(img), _ptr(noisy))
        return (img, noisy) if return_noisy else img

    def stats(self):
        s = Stats()
        self._call("get_stats", ctypes.byref(s))
        return s.as_dict()


class Context(_Handle):
    """One GPU.  Thin, 1:1 over the C ABI; numpy in, numpy out."""

    def __init__(self, device=0, _borrowed=None):
        self._lib = load_library()
        self._owned = _borrowed is None
        if _borrowed is not None:            # a context lent by a MultiContext (b200rt_multi_context)
            self._h = ctypes.c_void_p(_borrowed)
            self.device = int(device)
            return
        h = ctypes.c_void_p()
        rc = self._lib.b200rt_create(int(device), ctypes.byref(h))
        if rc != 0:
            raise B200RTError(f"b200rt_create({device}) failed ({rc}): {self._lib.b200rt_last_error(None).decode()}")
        self._h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "_h", None):
            if self._owned:
                self._lib.b200rt_destroy(self._h)
            self._h = None

    def set_materials(self, material_data):
        mat = _f32(material_data)
        self._check(self._lib.b200rt_set_materials(self._h, _ptr(mat), mat.size), "b200rt_set_materials")

    # ---- rendering ------------------------------------------------------------------------------------
    def render_adaptive(self, cam, env, width, height, spp, max_bounce, rel_error, min_spp=16, check_every=8, floor=0.05,
                        opts=None):
        """Adaptive sampling (b200rt_render_adaptive): every pixel takes at least min_spp and at most spp samples and
        stops once the standard error of its mean luminance is at most rel_error * max(min(mean, 1), floor).
        Returns (image (H, W, 3) float32, samples taken (H, W) int32, standard error (H, W) float32)."""
        cam_, env_ = _f32(cam), _f32(env)
        if cam_.size != 10 or env_.size != 5:
            raise B200RTError("cam must hold 10 floats and envData 5 (main.py:59-61,72-73)")
        h, w = int(height), int(width)
        img = np.zeros((h, w, 3), dtype=np.float32)
        spp_map = np.zeros((h, w), dtype=np.int32)
        err_map = np.zeros((h, w), dtype=np.float32)
        ad = Adaptive(int(min_spp), int(check_every), float(rel_error), float(floor))
        o = opts if opts is not None else make_opts()
        self._check(self._lib.b200rt_render_adaptive(self._h, _ptr(cam_), _ptr(env_), w, h, int(spp), int(max_bounce),
                                                     ctypes.byref(o), ctypes.byref(ad), _ptr(img), _ptr(spp_map),
                                                     _ptr(err_map)), "b200rt_render_adaptive")
        return img, spp_map, err_map

    def gbuffer(self, cam, width, height, opts=None):
        """The denoiser's G-buffer of the frame's primary hits (b200rt_gbuffer): a dict of albedo / normal / position
        (H, W, 3) float32 and kind (H, W) int32 (-1 miss, 0 emitter, 1 surface)."""
        cam_ = _f32(cam)
        h, w = int(height), int(width)
        gb = {k: np.zeros((h, w, 3), np.float32) for k in ("albedo", "normal", "position")}
        gb["kind"] = np.zeros((h, w), np.int32)
        o = opts if opts is not None else make_opts()
        self._check(self._lib.b200rt_gbuffer(self._h, _ptr(cam_), w, h, ctypes.byref(o), _ptr(gb["albedo"]),
                                             _ptr(gb["normal"]), _ptr(gb["position"]), _ptr(gb["kind"])), "b200rt_gbuffer")
        return gb

    def denoise(self, img, gb, **denoise):
        """The filter on its own (b200rt_denoise) over an (H, W, 3) image and a G-buffer as gbuffer() returns it;
        denoise as for render_denoised.  Returns a new (H, W, 3) float32 image."""
        kind = np.ascontiguousarray(gb["kind"], np.int32)
        h, w = kind.shape
        n = h * w * 3
        arrs = [_f32(a) for a in (img, gb["albedo"], gb["normal"], gb["position"])]
        if any(a.size != n for a in arrs):
            raise B200RTError(f"image and G-buffer must hold {n} floats each for a {w}x{h} kind map")
        out = np.zeros((h, w, 3), np.float32)
        dn = _denoise_params(**denoise)
        self._check(self._lib.b200rt_denoise(self._h, *[_ptr(a) for a in arrs], _ptr(kind), w, h, ctypes.byref(dn),
                                             _ptr(out)), "b200rt_denoise")
        return out

    def render_rgb8(self, cam, env, width, height, spp, max_bounce, opts=None):
        """(height, width, 3) uint8 image, quantised on the device like FileManager.saveImg does on the host."""
        cam_, env_ = _f32(cam), _f32(env)
        out = np.zeros((int(height), int(width), 3), dtype=np.uint8)
        o = opts if opts is not None else make_opts()
        self._check(self._lib.b200rt_render_rgb8(self._h, _ptr(cam_), _ptr(env_), int(width), int(height), int(spp),
                                                 int(max_bounce), ctypes.byref(o), _ptr(out)), "b200rt_render_rgb8")
        return out

    def render_device(self, cam, env, width, height, spp, max_bounce, d_out_ptr, opts=None):
        """Enqueue a render into device memory (raw pointer as int); returns immediately."""
        cam_, env_ = _f32(cam), _f32(env)
        o = opts if opts is not None else make_opts()
        self._check(self._lib.b200rt_render_device(self._h, _ptr(cam_), _ptr(env_), int(width), int(height), int(spp),
                                                   int(max_bounce), ctypes.byref(o), ctypes.c_void_p(int(d_out_ptr))),
                    "b200rt_render_device")

    def finalize_device(self, d_sums_ptr, d_out_ptr, n_pixels, spp):
        self._check(self._lib.b200rt_finalize_device(self._h, ctypes.c_void_p(int(d_sums_ptr)),
                                                     ctypes.c_void_p(int(d_out_ptr)), int(n_pixels), int(spp)),
                    "b200rt_finalize_device")

    def reduce_finalize_device(self, part_ptrs, d_out_ptr, n_pixels, spp):
        arr = (ctypes.c_void_p * len(part_ptrs))(*[ctypes.c_void_p(int(p)) for p in part_ptrs])
        self._check(self._lib.b200rt_reduce_finalize_device(self._h, arr, len(part_ptrs), ctypes.c_void_p(int(d_out_ptr)),
                                                            int(n_pixels), int(spp)), "b200rt_reduce_finalize_device")

    def sync(self):
        self._check(self._lib.b200rt_sync(self._h), "b200rt_sync")

    def set_stream(self, cuda_stream):
        """cuda_stream: raw cudaStream_t as int (e.g. torch.cuda.current_stream().cuda_stream); None restores
        the context's own stream.  0 (torch's default stream) is passed as cudaStreamLegacy (0x1), because a
        NULL handle means "restore" in the C ABI."""
        if cuda_stream is None:
            h = None
        else:
            h = ctypes.c_void_p(int(cuda_stream) or 1)
        self._check(self._lib.b200rt_set_stream(self._h, h), "b200rt_set_stream")

    def primary_hits(self, cam, width, height, opts=None):
        cam_ = _f32(cam)
        n = int(width) * int(height)
        tri = np.zeros(n, np.int32)
        k = np.zeros(n, np.float32)
        o = opts if opts is not None else make_opts()
        self._check(self._lib.b200rt_primary_hits(self._h, _ptr(cam_), int(width), int(height), ctypes.byref(o),
                                                  _ptr(tri), _ptr(k)), "b200rt_primary_hits")
        return tri, k

    def trace_rays(self, rays, opts=None):
        r = np.ascontiguousarray(rays, np.float32).reshape(-1, 6)
        n = r.shape[0]
        tri = np.zeros(n, np.int32)
        k = np.zeros(n, np.float32)
        o = opts if opts is not None else make_opts()
        self._check(self._lib.b200rt_trace_rays(self._h, _ptr(r), n, ctypes.byref(o), _ptr(tri), _ptr(k)),
                    "b200rt_trace_rays")
        return tri, k

    def img_processing(self, src, dst, n, global_size=None):
        src_ = _f32(src)
        if dst.dtype != np.float32 or not dst.flags["C_CONTIGUOUS"]:
            raise B200RTError("dst must be C-contiguous float32")
        g = src_.size if global_size is None else int(global_size)
        if dst.size < g or src_.size < g:
            raise B200RTError("src/dst smaller than the global size")
        self._check(self._lib.b200rt_img_processing(self._h, _ptr(src_), _ptr(dst), int(n), g), "b200rt_img_processing")
        return dst

    # ---- probes ---------------------------------------------------------------------------------------------
    def math_probe(self, fn, a, b=None):
        a_ = _f32(a)
        b_ = None if b is None else _f32(b)
        out = np.zeros_like(a_)
        self._check(self._lib.b200rt_math_probe(self._h, int(fn), _ptr(a_), _ptr(b_), a_.size, _ptr(out)),
                    "b200rt_math_probe")
        return out

    def philox_probe(self, ctr, key0, key1):
        c = (ctypes.c_uint32 * 4)(*[int(x) & 0xFFFFFFFF for x in ctr])
        o = (ctypes.c_uint32 * 4)()
        self._check(self._lib.b200rt_philox_probe(self._h, ctypes.byref(c), int(key0), int(key1), ctypes.byref(o)),
                    "b200rt_philox_probe")
        return np.array(list(o), dtype=np.uint32)

    # ---- CUDA IPC (multi-GPU peer reduce) -----------------------------------------------------------------------
    def alloc(self, nbytes):
        p = ctypes.c_void_p()
        self._check(self._lib.b200rt_alloc(self._h, int(nbytes), ctypes.byref(p)), "b200rt_alloc")
        return p.value

    def free(self, d_ptr):
        self._check(self._lib.b200rt_free(self._h, ctypes.c_void_p(int(d_ptr))), "b200rt_free")

    def ipc_export(self, d_ptr):
        buf = (ctypes.c_uint8 * 64)()
        self._check(self._lib.b200rt_ipc_export(self._h, ctypes.c_void_p(int(d_ptr)), buf), "b200rt_ipc_export")
        return bytes(buf)

    def ipc_open(self, handle):
        buf = (ctypes.c_uint8 * 64)(*handle)
        p = ctypes.c_void_p()
        self._check(self._lib.b200rt_ipc_open(self._h, buf, ctypes.byref(p)), "b200rt_ipc_open")
        return p.value

    def ipc_close(self, d_ptr):
        self._check(self._lib.b200rt_ipc_close(self._h, ctypes.c_void_p(int(d_ptr))), "b200rt_ipc_close")


class MultiContext(_Handle):
    """Several GPUs of one box behind one handle (b200rt_multi_*): same set_scene / set_ibl / render / stats surface as
    Context, the frame divided among the GPUs inside the library.  `contexts[i]` are the per-GPU contexts (lent)."""

    _prefix = "b200rt_multi_"

    def __init__(self, devices):
        self._lib = load_library()
        devs = [int(d) for d in devices]
        arr = (ctypes.c_int * len(devs))(*devs)
        h = ctypes.c_void_p()
        rc = self._lib.b200rt_multi_create(arr, len(devs), ctypes.byref(h))
        if rc != 0:
            raise B200RTError(f"b200rt_multi_create({devs}) failed ({rc}): {self._lib.b200rt_multi_last_error(None).decode()}")
        self._h = h
        self.devices = devs
        self.device = devs[0]
        self.contexts = [Context(d, _borrowed=self._lib.b200rt_multi_context(h, i)) for i, d in enumerate(devs)]

    def close(self):
        if getattr(self, "_h", None):
            for c in self.contexts:
                c.close()
            self._lib.b200rt_multi_destroy(self._h)
            self._h = None

    def img_processing(self, src, dst, n, global_size=None):
        return self.contexts[0].img_processing(src, dst, n, global_size)

    def primary_hits(self, cam, width, height, opts=None):
        return self.contexts[0].primary_hits(cam, width, height, opts)
