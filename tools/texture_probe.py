#!/usr/bin/env python3
"""What albedo textures (B200RT_SAMPLING_TEXTURES) cost, one JSON line per measurement.

- render: the bench scene (config 2, 1920x1080, Philox, maxBounce 4, sample_streams -1) with its monkey (material 4,
  glossy) and its walls (materials 0 and 2, diffuse) textured by seeded generated images of `size` x `size` texels
  (tests/texture_scene.py noise), for each size; masks 0 and 512 in the same call, their timed repeats alternating: the
  call time (best of `repeat`, host clock around the synchronous call), stats.total_ms of that best call, rays per
  sample, then one render with time_kernels for the summed k_shade / k_trace device time (sums of durations over the
  sample streams, which overlap);
- upload: b200rt_set_scene + b200rt_set_ibl of the BASELINE config 5 height field (~5 M triangles, tests/synthetic.py),
  caches invalidated, best of 3: host seconds around both calls, and stats.repack_ms.
The card's name and power limit are read in the same call.  --lib times another build of libb200rt.so (e.g. the parent
commit's, for the upload stage, which has no texture stage to run).

usage: texture_probe.py [--out profiles/r08_textures.jsonl] [--spp 64] [--repeat 3] [--sizes 1024,4096]
                        [--stages render,upload] [--lib PATH] [--label NAME]"""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_textures.jsonl"))
    ap.add_argument("--spp", type=int, default=64)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--sizes", default="1024,4096")
    ap.add_argument("--stages", default="render,upload")
    ap.add_argument("--lib", default=None)
    ap.add_argument("--label", default="this")
    a = ap.parse_args()
    from ensem3a_openclraytracer_b200 import _capi
    if a.lib:
        _capi.LIB_PATH = os.path.abspath(a.lib)
    import ensem3a_openclraytracer_b200 as rt
    from adaptive_probe import BOUNCE, H, W, card
    from tests import fixtures, texture_scene
    from tests.synthetic import height_field_scene

    name, power = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "a")

    def emit(**kw):
        kw = dict(kw, lib=a.label, card=name, power_limit=power)
        line = json.dumps(kw)
        print(line, flush=True)
        out.write(line + "\n")

    ctx = rt.Context(0)
    stages = a.stages.split(",")
    if "render" in stages:
        sc = fixtures.load_scene("monkey_cfg2")
        fixtures.upload(ctx, sc, fixtures.load_ibl("preview"))
        cam, env = fixtures.cam_env(sc["params"], W, H)
        masks = (0, rt.SAMPLING_TEXTURES)
        for size in (int(s) for s in a.sizes.split(",")):
            ctx.set_textures({m: texture_scene.noise(size, m) for m in (0, 2, 4)})
            opts = {m: rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=1, sample_streams=-1, sampling=m) for m in masks}
            best = {}
            for m in masks:
                ctx.render(cam, env, W, H, a.spp, BOUNCE, opts=opts[m])   # warm-up
            for _ in range(a.repeat):
                for m in masks:
                    t0 = time.perf_counter()
                    ctx.render(cam, env, W, H, a.spp, BOUNCE, opts=opts[m])
                    ms = (time.perf_counter() - t0) * 1e3
                    if m not in best or ms < best[m][0]:
                        best[m] = (ms, ctx.stats())
            for m in masks:
                ms, st = best[m]
                o = rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=1, sample_streams=-1, sampling=m)
                o.time_kernels = 1
                ctx.render(cam, env, W, H, a.spp, BOUNCE, opts=o)
                tk = ctx.stats()
                emit(stage="render", scene="monkey_cfg2", texture_size=size, width=W, height=H, spp=a.spp,
                     bounce=BOUNCE, sampling=m, call_ms=ms, total_ms=st["total_ms"], rays=st["rays"],
                     rays_per_sample=st["rays"] / (W * H * a.spp), streams=st["sample_streams"],
                     shade_kernel_ms=tk["shade_kernel_ms"], trace_kernel_ms=tk["trace_kernel_ms"])
        ctx.set_textures(None)
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
        emit(stage="upload", scene="config5", triangles=int(sc["faceData"].size // 10), uv_floats=int(sc["V_uv"].size),
             seconds=best[0], repack_ms=best[1])
    ctx.close()


if __name__ == "__main__":
    main()
