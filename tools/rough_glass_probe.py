#!/usr/bin/env python3
"""What rough glass (B200RT_SAMPLING_ROUGH_GLASS) costs, one JSON line per scene and sampling mask.

Per scene (1920x1080, Philox, maxBounce 4, sample_streams -1) the masks 128 (refractive glass) and 128 | 2048 (rough
glass) are measured in the same call, their timed repeats alternating: the call time (best of `repeat`, host clock
around the synchronous call), stats.total_ms of that best call, rays per sample, then one render with time_kernels for
the summed k_shade / k_trace device time (sums of durations over the sample streams, which overlap).  Scenes: config 2
with its glass wall at roughness 0.2 (tests/rough_glass_scene.py) and the proto scene as shipped (glass of roughness
0.1).  The card's name and power limit are read in the same call.

usage: rough_glass_probe.py [--out profiles/r09_rough_glass.jsonl] [--spp 64] [--repeat 3] [--scenes bench_rough,proto]"""
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_rough_glass.jsonl"))
    ap.add_argument("--spp", type=int, default=64)
    ap.add_argument("--repeat", type=int, default=3)
    ap.add_argument("--scenes", default="bench_rough,proto")
    a = ap.parse_args()
    import ensem3a_openclraytracer_b200 as rt
    from adaptive_probe import BOUNCE, H, W, card
    from tests import fixtures, rough_glass_scene

    name, power = card()
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    out = open(a.out, "a")

    def emit(**kw):
        kw = dict(kw, card=name, power_limit=power)
        line = json.dumps(kw)
        print(line, flush=True)
        out.write(line + "\n")

    ctx = rt.Context(0)
    masks = (rt.SAMPLING_DIELECTRIC_GLASS, rt.SAMPLING_DIELECTRIC_GLASS | rt.SAMPLING_ROUGH_GLASS)
    for scene in a.scenes.split(","):
        fixtures.upload(ctx, rough_glass_scene.load(scene), fixtures.load_ibl("preview"))
        cam, env = rough_glass_scene.view(scene, W, H)
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
            emit(stage="render", scene=scene, width=W, height=H, spp=a.spp, bounce=BOUNCE, sampling=m, call_ms=ms,
                 total_ms=st["total_ms"], rays=st["rays"], rays_per_sample=st["rays"] / (W * H * a.spp),
                 streams=st["sample_streams"], shade_kernel_ms=tk["shade_kernel_ms"],
                 trace_kernel_ms=tk["trace_kernel_ms"])
    ctx.close()


if __name__ == "__main__":
    main()
