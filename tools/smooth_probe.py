#!/usr/bin/env python3
"""What smooth shading (B200RT_SAMPLING_SMOOTH_NORMALS) costs and what it buys, one JSON line per measurement.

- render: per scene (1920x1080, Philox, maxBounce 4, sample_streams -1) and sampling 0 / 32, the call time (best of
  `repeat`, host clock around the synchronous call), stats.total_ms, Mrays/s, then one render with time_kernels for the
  summed k_shade / k_trace device time (sums of durations over the sample streams, which overlap);
- upload: b200rt_set_scene + b200rt_set_ibl of the BASELINE config 5 height field (~5 M triangles, tests/synthetic.py),
  caches invalidated, best of 3: host seconds around both calls, and stats.repack_ms;
- quality: a 12 x 6 UV sphere (tests/smooth_scene.py) flat and smooth against a 192 x 96 one, RMSE over the pixels whose
  primary hits both lie on the sphere.
The card's name and power limit are read in the same call.  --lib times another build of libb200rt.so (e.g. the parent
commit's, for the upload stage).

usage: smooth_probe.py [--out profiles/r06_smooth.jsonl] [--spp 64] [--repeat 3] [--stages render,upload,quality]
                       [--scenes monkey_cfg2:preview,serre:preview] [--lib PATH] [--label NAME]"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_smooth.jsonl"))
    ap.add_argument("--spp", type=int, default=64)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--stages", default="render,upload,quality")
    ap.add_argument("--scenes", default="monkey_cfg2:preview,serre:preview")
    ap.add_argument("--lib", default=None)
    ap.add_argument("--label", default="this")
    a = ap.parse_args()
    from ensem3a_openclraytracer_b200 import _capi
    if a.lib:
        _capi.LIB_PATH = os.path.abspath(a.lib)
    import ensem3a_openclraytracer_b200 as rt
    from adaptive_probe import BOUNCE, H, W, card, timed
    from tests import fixtures, smooth_scene
    from tests.synthetic import height_field_scene

    name, power = card()
    out = open(a.out, "a")

    def emit(**kw):
        kw = dict(kw, lib=a.label, card=name, power_limit=power)
        line = json.dumps(kw)
        print(line, flush=True)
        out.write(line + "\n")

    ctx = rt.Context(0)
    stages = a.stages.split(",")
    if "render" in stages:
        for item in a.scenes.split(","):
            scene, ibl_name = item.split(":")
            sc = fixtures.load_scene(scene)
            fixtures.upload(ctx, sc, fixtures.load_ibl(ibl_name))
            cam, env = fixtures.cam_env(sc["params"], W, H)
            for sampling in (0, rt.SAMPLING_SMOOTH_NORMALS):
                o = rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=1, sample_streams=-1, sampling=sampling)
                ctx.render(cam, env, W, H, a.spp, BOUNCE, opts=o)   # warm-up
                ms, _ = timed(lambda: ctx.render(cam, env, W, H, a.spp, BOUNCE, opts=o), a.repeat)
                st = ctx.stats()
                o.time_kernels = 1
                ctx.render(cam, env, W, H, a.spp, BOUNCE, opts=o)
                tk = ctx.stats()
                emit(stage="render", scene=scene, ibl=ibl_name, width=W, height=H, spp=a.spp, bounce=BOUNCE,
                     sampling=sampling, call_ms=ms, total_ms=st["total_ms"], rays=st["rays"],
                     mrays_s=st["rays"] / ms / 1e3, streams=st["sample_streams"],
                     shade_kernel_ms=tk["shade_kernel_ms"], trace_kernel_ms=tk["trace_kernel_ms"])
    if "upload" in stages:
        sc = height_field_scene(1582, seed=0)
        sc["BVH"] = rt.build_bvh(sc["faceData"], sc["V_p"])
        ibl = fixtures.load_ibl("preview")
        best = None
        for _ in range(3):
            ctx.invalidate()
            t0 = time.perf_counter()
            fixtures.upload(ctx, sc, ibl)
            s = time.perf_counter() - t0
            st = ctx.stats()
            if best is None or s < best[0]:
                best = (s, st["repack_ms"])
        emit(stage="upload", scene="config5", triangles=int(sc["faceData"].size // 10), seconds=best[0],
             repack_ms=best[1])
    if "quality" in stages:
        Wq, spp = 512, 1024
        cam, env, ibl = smooth_scene.sphere_view(Wq)
        fine = smooth_scene.sphere(192, 96)
        fixtures.upload(ctx, fine, ibl)
        o = rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=4, sample_streams=-1)
        ref = ctx.render(cam, env, Wq, Wq, spp, 2, opts=o).reshape(-1, 3)
        mask = ctx.primary_hits(cam, Wq, Wq)[0] >= 0
        coarse = smooth_scene.sphere(12, 6)
        fixtures.upload(ctx, coarse, ibl)
        mask &= ctx.primary_hits(cam, Wq, Wq)[0] >= 0
        err = {}
        for sampling in (0, rt.SAMPLING_SMOOTH_NORMALS):
            o = rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=4, sample_streams=-1, sampling=sampling)
            img = ctx.render(cam, env, Wq, Wq, spp, 2, opts=o).reshape(-1, 3)
            err[sampling] = float(np.sqrt(np.mean((img[mask].astype(np.float64) - ref[mask]) ** 2)))
        emit(stage="quality", scene="uv_sphere_12x6_vs_192x96", width=Wq, spp=spp, bounce=2, pixels=int(mask.sum()),
             rmse_flat=err[0], rmse_smooth=err[rt.SAMPLING_SMOOTH_NORMALS],
             ratio=err[rt.SAMPLING_SMOOTH_NORMALS] / err[0])
    ctx.close()


if __name__ == "__main__":
    main()
