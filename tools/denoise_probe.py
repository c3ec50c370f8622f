#!/usr/bin/env python3
"""The denoiser against fixed spp at equal error, on the 1920x1080 scenes and truth images of adaptive_probe.py (Philox,
maxBounce 4, sample_streams -1).

Per scene and N (spp): the render's call time (best of `repeat`, host clock around the synchronous call), the same for
render_denoised, the filter's device time (k_primary + k_gbuffer + k_atrous kernel time of one render_denoised under
torch.profiler, in a run of its own), RMSE and relative mean bias against the truth of the noisy and the denoised image,
and the smallest fixed spp (N doubled, measured up to --max-spp) whose RMSE is at most the denoised one, with its call
time.  Each scene's first line also carries the sigma sweep at the sweep's N (b200rt_denoise over the same noisy image).

usage: denoise_probe.py [--out profiles/r04_denoise.jsonl] [--truth-spp 8192] [--n 16,64,256] [--max-spp 4096]
                        [--scenes monkey_cfg2:preview,furnace_cfg3:grey,serre:8k]"""
import argparse
import itertools
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ensem3a_openclraytracer_b200 as rt  # noqa: E402
from adaptive_probe import BOUNCE, H, W, card, timed, truth_image  # noqa: E402
from tests import fixtures  # noqa: E402

SWEEP = dict(passes=(3, 5, 7), sigma_color=(0.25, 0.5, 1.0), sigma_normal=(0.1, 0.2, 0.5))


def rmse(img, truth):
    return float(np.sqrt(np.mean((np.asarray(img, np.float64).reshape(H, W, 3) - truth) ** 2)))


def bias(img, truth):
    return float((np.asarray(img, np.float64).mean() - truth.mean()) / truth.mean())


def filter_kernel_ms(ctx, cam, env, n, opts):
    """device time of the G-buffer and filter kernels of one render_denoised, from torch.profiler"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        ctx.render_denoised(cam, env, W, H, n, BOUNCE, opts=opts)
        torch.cuda.synchronize()
    us, names = 0.0, {}
    for e in prof.events():
        name = e.name
        # the PARITY instance of k_primary is the G-buffer's; the render's own k_primary is the non-PARITY one
        parity = "k_primary<" in name and name.split("k_primary<")[1].split(">")[0].split(", ")[2] == "true"
        if "k_gbuffer" in name or "k_atrous" in name or parity:
            t = e.device_time if hasattr(e, "device_time") else e.cuda_time
            us += t
            key = name.split("(")[0]
            names[key] = names.get(key, 0.0) + t / 1e3
    return us / 1e3, names


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_denoise.jsonl"))
    ap.add_argument("--truth-spp", type=int, default=8192)
    ap.add_argument("--n", default="16,64,256")
    ap.add_argument("--sweep-n", type=int, default=64)
    ap.add_argument("--max-spp", type=int, default=4096)
    ap.add_argument("--scenes", default="monkey_cfg2:preview,furnace_cfg3:grey,serre:8k")
    ap.add_argument("--repeat", type=int, default=3)
    a = ap.parse_args()
    name, power = card()
    ctx = rt.Context(0)
    o = rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=1, sample_streams=-1)
    with open(a.out, "a") as f:
        for entry in a.scenes.split(","):
            scene, ibl_name = entry.split(":")
            sc = fixtures.load_scene(scene)
            fixtures.upload(ctx, sc, fixtures.load_ibl(ibl_name))
            cam, env = fixtures.cam_env(sc["params"], W, H)
            t0 = time.perf_counter()
            truth = truth_image(ctx, cam, env, a.truth_spp)
            truth_s = time.perf_counter() - t0
            gb = ctx.gbuffer(cam, W, H, opts=o)
            sweep = []
            noisy = ctx.render(cam, env, W, H, a.sweep_n, BOUNCE, opts=o)
            for p, sc_, sn in itertools.product(*SWEEP.values()):
                img = ctx.denoise(noisy, gb, passes=p, sigma_color=sc_, sigma_normal=sn)
                sweep.append(dict(passes=p, sigma_color=sc_, sigma_normal=sn, rmse=rmse(img, truth)))
            for n in (int(x) for x in a.n.split(",")):
                r_ms, noisy = timed(lambda: ctx.render(cam, env, W, H, n, BOUNCE, opts=o), a.repeat)
                st_r = ctx.stats()
                d_ms, den = timed(lambda: ctx.render_denoised(cam, env, W, H, n, BOUNCE, opts=o), a.repeat)
                k_ms, per_kernel = filter_kernel_ms(ctx, cam, env, n, o)
                e_den = rmse(den, truth)
                match = None
                spp = n
                while spp < a.max_spp:
                    spp *= 2
                    ms, img = timed(lambda: ctx.render(cam, env, W, H, spp, BOUNCE, opts=o), 1)
                    e = rmse(img, truth)
                    if e <= e_den:
                        match = dict(spp=spp, call_ms=ms, rmse=e)
                        break
                line = dict(tool="denoise_probe", card=name, power_limit=power, scene=scene, ibl=ibl_name, width=W,
                            height=H, max_bounce=BOUNCE, truth_spp=a.truth_spp, truth_renders=4, truth_seconds=truth_s,
                            spp=n, defaults=rt.DENOISE_DEFAULTS, render_call_ms=r_ms, render_device_ms=st_r["total_ms"],
                            denoised_call_ms=d_ms, filter_host_ms=d_ms - r_ms, filter_kernel_ms=k_ms,
                            filter_kernels=per_kernel, rmse_noisy=rmse(noisy, truth), rmse_denoised=e_den,
                            bias_noisy=bias(noisy, truth), bias_denoised=bias(den, truth),
                            fixed_match=match, max_spp_tried=a.max_spp,
                            speedup_at_equal_rmse=(match["call_ms"] / d_ms) if match else None)
                if sweep:
                    line.update(sweep_spp=a.sweep_n, sweep=sorted(sweep, key=lambda r: r["rmse"]))
                    sweep = []
                print(json.dumps({k: v for k, v in line.items() if k != "sweep"}), flush=True)
                f.write(json.dumps(line) + "\n")
                f.flush()
    ctx.close()


if __name__ == "__main__":
    main()
