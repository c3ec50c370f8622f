"""B200-native (sm_100a) implementation of the path-tracing hot path of
QuentinHuan/ENSEM3A_OpenCLRaytracer behind the reference's KernelLauncher call surface.

    from ensem3a_openclraytracer_b200 import KernelLauncher      # drop-in class
    from ensem3a_openclraytracer_b200 import Context, make_opts   # 1:1 over include/b200rt.h
"""
from ._capi import (Adaptive, B200RTError, Context, Denoise, DENOISE_DEFAULTS, MultiContext, Opts, Stats, make_opts, build_library, build_bvh, device_count, load_library, LIB_PATH,
                    RNG_REFERENCE, RNG_PHILOX, TRAVERSAL_FAST, TRAVERSAL_REFERENCE, TRAVERSAL_VERIFY,
                    OUT_FINAL, OUT_SUMS, SAMPLING_REFERENCE, SAMPLING_IMPORTANCE, SAMPLING_LIGHTS,
                    SAMPLING_PIXEL_JITTER, SAMPLING_SMOOTH_NORMALS,
                    SAMPLING_DIELECTRIC_GLASS, SAMPLING_TEXTURES, SAMPLING_ROUGH_GLASS)
from .KernelLauncher import KernelLauncher
from .BVH import BVH
from .progressive import ProgressiveRender

__all__ = ["Adaptive", "B200RTError", "Context", "Denoise", "DENOISE_DEFAULTS", "MultiContext", "Opts", "Stats", "make_opts", "build_library", "load_library", "LIB_PATH",
           "KernelLauncher", "BVH", "ProgressiveRender", "build_bvh", "device_count", "RNG_REFERENCE", "RNG_PHILOX", "TRAVERSAL_FAST", "TRAVERSAL_REFERENCE",
           "TRAVERSAL_VERIFY", "OUT_FINAL", "OUT_SUMS", "SAMPLING_REFERENCE", "SAMPLING_IMPORTANCE", "SAMPLING_LIGHTS",
           "SAMPLING_PIXEL_JITTER", "SAMPLING_SMOOTH_NORMALS", "SAMPLING_DIELECTRIC_GLASS", "SAMPLING_TEXTURES",
           "SAMPLING_ROUGH_GLASS"]
