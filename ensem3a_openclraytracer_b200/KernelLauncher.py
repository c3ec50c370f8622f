"""Drop-in replacement for the reference's KernelLauncher.py (PyOpenCL) on B200.

Same class name, same three method signatures in the same positional order
(reference KernelLauncher.py:8, :33, :90), same in-place / synchronous behaviour:
`launch_Raytracing` fills the caller's `h_img_out` and returns None when the image is on the host
(the reference's blocking enqueue_copy, :78); `launch_ImgProcessing` fills `h_out`.  main.py and
UI.py therefore drive it unchanged (main.py:28,84-86).

The work is done by the CUDA kernels behind the C ABI of include/b200rt.h; there is no OpenCL,
CPU or PyTorch fallback: constructing a KernelLauncher without a usable B200 raises.

Differences a caller can observe (all documented in INTEGRATION.md):
  * the OpenCL objects passed to __init__ are accepted and ignored;
  * geometry / environment uploads are cached by content between calls (the UI re-creates
    identical arrays for every render, UI.py:98), materials are always refreshed;
  * non-square frames: width = int(cam[6]), height = imgDim // width, exactly what the reference
    kernel computes for such a launch (Raytracing.cl:21-29);
  * extra behaviour is opt-in through attributes (`rng_mode`, `traversal`, `seed`, ...) that the
    reference's callers never touch, so the default is the reference's result — including on trees whose
    walk needs more than the reference's 20 stack entries, where its stack silently drops pushes
    (stack.cl:21-26): for such a tree the default switches to the reference-order walk with that cap (slow,
    but the reference's image) and warns once; `deep_trees = "nodrop"` keeps the fast traversal, which visits
    everything (the geometrically correct image, not the reference's);
  * `cuda_devices=[0, 1, ...]` renders every frame on several GPUs of the box through the same call
    (b200rt_multi_*): bit-identical with the reference generator, equal up to the order of the float additions
    with `rng_mode = RNG_PHILOX`;
  * `adaptive = dict(rel_error=..., min_spp=16, check_every=8, floor=0.05)` (the keys of Context.render_adaptive) lets
    each pixel stop sampling once its estimated error is below the tolerance, with the caller's spp as the maximum;
    `last_spp` then holds the (height, width) map of samples taken.  B200RT_ADAPTIVE=rel_error[,min_spp[,check_every]]
    in the environment sets it for callers that never touch the attribute.  One GPU only;
  * `denoise = dict(passes=5, sigma_color=0.5, sigma_normal=0.2, sigma_position=0)` (the keywords of
    Context.render_denoised; missing keys take DENOISE_DEFAULTS) runs the edge-avoiding à-trous filter of include/b200rt.h
    over every frame, on one GPU or on `cuda_devices`.  B200RT_DENOISE=1 (the defaults) or
    B200RT_DENOISE=passes[,sigma_color[,sigma_normal[,sigma_position]]] sets it for callers that never touch the
    attribute.  It cannot be combined with `adaptive`.
"""
import math
import os
import warnings

import numpy as np

from . import _capi


def adaptive_from_env(text):
    """The `adaptive` dict that B200RT_ADAPTIVE=rel_error[,min_spp[,check_every]] stands for; ValueError if malformed."""
    usage = f"B200RT_ADAPTIVE={text!r}: expected rel_error[,min_spp[,check_every]], e.g. 0.02 or 0.02,16,8"
    parts = [p.strip() for p in str(text).split(",")]
    if not 1 <= len(parts) <= 3 or "" in parts:
        raise ValueError(usage)
    try:
        rel_error = float(parts[0])
        ints = [int(p) for p in parts[1:]]
    except ValueError:
        raise ValueError(usage) from None
    if not math.isfinite(rel_error) or rel_error < 0:
        raise ValueError(usage + " (rel_error must be finite and >= 0)")
    if ints and ints[0] < 2:
        raise ValueError(usage + " (min_spp must be >= 2)")
    if len(ints) > 1 and ints[1] < 1:
        raise ValueError(usage + " (check_every must be >= 1)")
    ad = {"rel_error": rel_error}
    ad.update(zip(("min_spp", "check_every"), ints))
    return ad


def denoise_from_env(text):
    """The `denoise` dict that B200RT_DENOISE=1 or =passes[,sigma_color[,sigma_normal[,sigma_position]]] stands for
    ("1" is the defaults); ValueError if malformed."""
    usage = (f"B200RT_DENOISE={text!r}: expected 1 (defaults) or passes[,sigma_color[,sigma_normal[,sigma_position]]], "
             "e.g. 5,0.5,0.2 (sigma_position <= 0: automatic)")
    parts = [p.strip() for p in str(text).split(",")]
    if not 1 <= len(parts) <= 4 or "" in parts:
        raise ValueError(usage)
    try:
        passes = int(parts[0])
        sigmas = [float(p) for p in parts[1:]]
    except ValueError:
        raise ValueError(usage) from None
    if not 1 <= passes <= 8:
        raise ValueError(usage + " (passes must be 1..8)")
    if not all(math.isfinite(x) for x in sigmas) or any(x <= 0 for x in sigmas[:2]):
        raise ValueError(usage + " (sigma_color and sigma_normal must be finite and > 0, sigma_position finite)")
    dn = dict(_capi.DENOISE_DEFAULTS)
    if parts == ["1"]:   # the switch, not a one-pass filter
        return dn
    dn["passes"] = passes
    dn.update(zip(("sigma_color", "sigma_normal", "sigma_position"), sigmas))
    return dn


class KernelLauncher(object):

    def __init__(self, context=None, platform=None, device=None, queue=None, cuda_device=0, cuda_devices=None):
        self.platform = platform
        self.device = device
        self.context = context
        self.queue = queue
        if cuda_devices is None and os.environ.get("B200RT_CUDA_DEVICES"):
            # main.py:28 constructs the launcher with the four OpenCL objects only; a deployment that wants several
            # GPUs behind the unchanged driver names them here, e.g. B200RT_CUDA_DEVICES=0,1,2,3,4,5,6,7
            cuda_devices = [int(x) for x in os.environ["B200RT_CUDA_DEVICES"].split(",") if x.strip() != ""]
        if cuda_devices is not None and len(cuda_devices) > 1:
            self._ctx = _capi.MultiContext(cuda_devices)
        else:
            self._ctx = _capi.Context(cuda_devices[0] if cuda_devices else cuda_device)
        # opt-in knobs; the defaults reproduce the reference's image
        self.rng_mode = _capi.RNG_REFERENCE
        self.traversal = _capi.TRAVERSAL_FAST
        self.seed = 0
        self.stack_cap = 20          # the reference's stack capacity (MathLib.cl:248); used by the reference-order walk
        self.deep_trees = "reference"  # "reference": trees needing > stack_cap entries are walked like the reference
        #                                 walks them (drops included); "nodrop": keep the fast, complete traversal
        self.sample_streams = 0      # RNG_PHILOX only: -1 automatic, N > 1 concurrent sample ranges on each GPU (b200rt.h)
        self.collect_stats = False
        # None: every pixel takes spp samples (the reference's image); a dict: adaptive sampling (module docstring)
        self.adaptive = adaptive_from_env(os.environ["B200RT_ADAPTIVE"]) if os.environ.get("B200RT_ADAPTIVE") else None
        # None: the render as it comes; a dict: denoised (module docstring)
        self.denoise = denoise_from_env(os.environ["B200RT_DENOISE"]) if os.environ.get("B200RT_DENOISE") else None
        self.last_spp = None
        self.last_stats = None
        self._warned_deep = False

    # reference KernelLauncher.py:33
    def launch_Raytracing(self, h_img_out, h_vertex_p, h_vertex_n, h_vertex_uv, h_face_data, h_material_data,
                          h_light_data, h_BVH, h_cam, h_envData, imgDim, spp, maxBounce, h_IBL):
        if self.adaptive is not None and self.denoise is not None:
            raise ValueError("adaptive sampling and denoising cannot be combined: set launcher.adaptive = None or "
                             "launcher.denoise = None")
        if self.adaptive is not None and isinstance(self._ctx, _capi.MultiContext):
            raise ValueError("adaptive sampling renders on one GPU: its stopping rule needs each pixel's samples in one "
                             f"sequence, which a split over cuda_devices={self._ctx.devices} would cut apart; set "
                             "launcher.adaptive = None or use one device")
        cam = np.ascontiguousarray(h_cam, dtype=np.float32).reshape(-1)
        if cam.size < 10:
            raise ValueError("h_cam must hold 10 floats (main.py:59-61)")
        width = int(cam[6])
        imgDim = int(imgDim)
        if width <= 0 or imgDim <= 0 or imgDim % width:
            raise ValueError(f"imgDim={imgDim} is not a whole number of rows of cam[6]={width} pixels")
        height = imgDim // width
        if not isinstance(h_img_out, np.ndarray) or h_img_out.dtype != np.float32 or not h_img_out.flags["C_CONTIGUOUS"]:
            raise TypeError("h_img_out must be a C-contiguous float32 numpy array (it is filled in place)")
        if h_img_out.size < imgDim * 3:
            raise ValueError(f"h_img_out has {h_img_out.size} elements, needs {imgDim * 3}")

        self._ctx.set_scene(h_vertex_p, h_vertex_n, h_vertex_uv, h_face_data, h_material_data, h_light_data, h_BVH)
        # h_IBL is a PIL RGBA image in the reference (uses .size and .tobytes(), KernelLauncher.py:72);
        # an (H, W, 4) uint8 array is accepted as well
        if hasattr(h_IBL, "tobytes") and hasattr(h_IBL, "size") and not isinstance(h_IBL, np.ndarray):
            w, h = h_IBL.size
            self._ctx.set_ibl(h_IBL.tobytes(), w, h)
        else:
            self._ctx.set_ibl(np.asarray(h_IBL))

        traversal = self.traversal
        need = self._ctx.stats()["ref_stack_need"]
        if traversal == _capi.TRAVERSAL_FAST and need > self.stack_cap and self.deep_trees == "reference":
            traversal = _capi.TRAVERSAL_REFERENCE
            if not self._warned_deep:
                warnings.warn(f"this BVH needs {need} traversal-stack entries; the reference's {self.stack_cap}-entry stack "
                              "drops pushes on it (stack.cl:21-26).  Rendering with the reference-order walk to reproduce its "
                              "image; set launcher.deep_trees = 'nodrop' for the fast traversal that visits everything.",
                              RuntimeWarning, stacklevel=2)
                self._warned_deep = True
        opts = _capi.make_opts(rng_mode=self.rng_mode, traversal=traversal, stack_cap=self.stack_cap,
                               seed=self.seed, collect_stats=self.collect_stats, sample_streams=self.sample_streams)
        out = h_img_out.reshape(-1)[:imgDim * 3]
        if self.adaptive is not None:
            img, self.last_spp, _ = self._ctx.render_adaptive(cam[:10], h_envData, width, height, int(spp), int(maxBounce),
                                                              opts=opts, **self.adaptive)
            out[:] = img.reshape(-1)
        elif self.denoise is not None:
            img = self._ctx.render_denoised(cam[:10], h_envData, width, height, int(spp), int(maxBounce), opts=opts,
                                            **self.denoise)
            out[:] = img.reshape(-1)
        else:
            self._ctx.render(cam[:10], h_envData, width, height, int(spp), int(maxBounce), out=out, opts=opts)
        self.last_stats = self._ctx.stats()

    # reference KernelLauncher.py:90
    def launch_ImgProcessing(self, h_src, h_out, SIZE):
        src = np.ascontiguousarray(h_src, dtype=np.float32)
        if not isinstance(h_out, np.ndarray) or h_out.dtype != np.float32 or not h_out.flags["C_CONTIGUOUS"]:
            raise TypeError("h_out must be a C-contiguous float32 numpy array (it is filled in place)")
        # global size = h_src.shape, N = SIZE*SIZE*3 (KernelLauncher.py:101-102)
        self._ctx.img_processing(src.reshape(-1), h_out.reshape(-1), int(SIZE) * int(SIZE) * 3, src.size)

    def close(self):
        self._ctx.close()
