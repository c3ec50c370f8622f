"""Progressive accumulation on top of the C ABI (SURVEY.md §8f-3): the frame's samples are rendered in slices
[s0, s1) (counter-based Philox, so a slice is independent of how the others are cut), each slice returns raw
per-pixel sums (B200RT_OUT_SUMS), and the running total gives a preview after every slice and a state that can
be saved and resumed (`sums`, `done`).  The reference renders all samples in one blocking kernel launch
(KernelLauncher.py:76-78) and has neither.

The final image equals the one-shot render up to the order of the float additions (slices are summed pairwise
instead of sample by sample): relative difference ~1e-7 per addition, far inside north_star's 1e-4.

`denoise` (a dict of Context.denoise's keywords, {} for the defaults) passes every preview and image() through the
edge-avoiding à-trous filter of include/b200rt.h, with the G-buffer computed once, on the first slice.  The saved state
(`sums`, `done`) stays undenoised, so a resumed render denoises the same way.
"""
import numpy as np

from . import _capi


def finalize(sums, samples):
    """clamp(sum / samples) as Raytracing.cl:211-219 (fmin/fmax drop NaNs, so a NaN pixel becomes 1)."""
    img = np.asarray(sums, np.float32) / np.float32(samples)
    return np.fmax(np.fmin(img, np.float32(1.0)), np.float32(0.0))


class ProgressiveRender:
    """Iterate to refine:  for preview in ProgressiveRender(ctx, cam, env, w, h, spp, bounce, slice_spp=16): ..."""

    def __init__(self, ctx, cam, env, width, height, spp, max_bounce, slice_spp=16, seed=0, sums=None, done=0,
                 denoise=None):
        if slice_spp <= 0 or spp <= 0:
            raise ValueError("spp and slice_spp must be positive")
        self.ctx, self.cam, self.env = ctx, cam, env
        self.width, self.height, self.spp, self.max_bounce = int(width), int(height), int(spp), int(max_bounce)
        self.slice_spp, self.seed = int(slice_spp), int(seed)
        n = self.width * self.height * 3
        self.sums = np.zeros(n, np.float32) if sums is None else np.ascontiguousarray(sums, np.float32).reshape(n).copy()
        self.done = int(done)          # samples accumulated so far — (sums, done) is the checkpoint
        self.denoise = denoise
        self._gb = None

    def _view(self, img):
        if self.denoise is None:
            return img
        if self._gb is None:
            self._gb = self.ctx.gbuffer(self.cam, self.width, self.height)
        return self.ctx.denoise(img, self._gb, **self.denoise).reshape(-1)

    def __iter__(self):
        return self

    def __next__(self):
        if self.done >= self.spp:
            raise StopIteration
        s0, s1 = self.done, min(self.done + self.slice_spp, self.spp)
        opts = _capi.make_opts(rng_mode=_capi.RNG_PHILOX, seed=self.seed, output=_capi.OUT_SUMS, sample_begin=s0,
                               sample_end=s1)
        part = self.ctx.render(self.cam, self.env, self.width, self.height, self.spp, self.max_bounce, opts=opts)
        self.sums += part
        self.done = s1
        return self._view(finalize(self.sums, self.done))

    def image(self):
        return self._view(finalize(self.sums, max(self.done, 1)))
