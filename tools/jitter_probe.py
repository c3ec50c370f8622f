#!/usr/bin/env python3
"""What pixel jitter (B200RT_SAMPLING_PIXEL_JITTER) costs and what it removes, on the 1920x1080 scenes of
adaptive_probe.py (Philox, maxBounce 4, sample_streams -1).

Per scene: the aliasing floor, i.e. the RMSE between the converged unjittered and jittered images (each the mean of
`renders` renders of --truth-spp, clamped to [0, 1]), over the whole frame and over the edge pixels (those whose primary
triangle differs from a 4-neighbour's, from b200rt_primary_hits); then, per N and mode, the call time (best of
`repeat`, host clock around the synchronous call), Mrays/s (stats.rays over that time), rays per sample and the RMSE
against that mode's own converged image.  The card's name and power limit are read in the same call.

usage: jitter_probe.py [--out profiles/r05_jitter.jsonl] [--truth-spp 4096] [--n 16,64,256]
                       [--scenes monkey_cfg2:preview,furnace_cfg3:grey,serre:8k]"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import ensem3a_openclraytracer_b200 as rt  # noqa: E402
from adaptive_probe import BOUNCE, H, W, card, timed  # noqa: E402
from tests import fixtures  # noqa: E402

MODES = {"point": rt.SAMPLING_REFERENCE, "jitter": rt.SAMPLING_PIXEL_JITTER}


def converged(ctx, cam, env, sampling, spp, renders):
    """(H, W, 3) float64: the mean of `renders` Philox renders (OUT_SUMS / spp), clamped to [0, 1]"""
    acc = np.zeros(W * H * 3)
    for seed in range(renders):
        o = rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=1000 + seed, output=rt.OUT_SUMS, sample_streams=-1,
                         sampling=sampling)
        acc += ctx.render(cam, env, W, H, spp, BOUNCE, opts=o).astype(np.float64) / spp
    return np.clip(acc / renders, 0.0, 1.0).reshape(H, W, 3)


def edge_mask(tri):
    tri = tri.reshape(H, W)
    e = np.zeros((H, W), bool)
    e[:, 1:] |= tri[:, 1:] != tri[:, :-1]
    e[:, :-1] |= tri[:, :-1] != tri[:, 1:]
    e[1:, :] |= tri[1:, :] != tri[:-1, :]
    e[:-1, :] |= tri[:-1, :] != tri[1:, :]
    return e


def rmse(a, b, mask=None):
    d = (np.asarray(a, np.float64).reshape(H, W, 3) - b) ** 2
    return float(np.sqrt(d[mask].mean() if mask is not None else d.mean()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_jitter.jsonl"))
    ap.add_argument("--truth-spp", type=int, default=4096)
    ap.add_argument("--renders", type=int, default=4)
    ap.add_argument("--n", default="16,64,256")
    ap.add_argument("--scenes", default="monkey_cfg2:preview,furnace_cfg3:grey,serre:8k")
    ap.add_argument("--repeat", type=int, default=3)
    a = ap.parse_args()
    name, power = card()
    ctx = rt.Context(0)
    with open(a.out, "a") as f:
        for entry in a.scenes.split(","):
            scene, ibl_name = entry.split(":")
            sc = fixtures.load_scene(scene)
            fixtures.upload(ctx, sc, fixtures.load_ibl(ibl_name))
            cam, env = fixtures.cam_env(sc["params"], W, H)
            tri, _ = ctx.primary_hits(cam, W, H)
            edges = edge_mask(tri)
            conv = {m: converged(ctx, cam, env, s, a.truth_spp, a.renders) for m, s in MODES.items()}
            line = dict(tool="jitter_probe", card=name, power_limit=power, scene=scene, ibl=ibl_name, width=W, height=H,
                        max_bounce=BOUNCE, truth_spp=a.truth_spp, truth_renders=a.renders,
                        edge_pixel_share=float(edges.mean()),
                        aliasing_rmse_frame=rmse(conv["point"], conv["jitter"]),
                        aliasing_rmse_edges=rmse(conv["point"], conv["jitter"], edges), runs=[])
            for n in (int(x) for x in a.n.split(",")):
                for m, s in MODES.items():
                    o = rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=7, sample_streams=-1, sampling=s)
                    ctx.render(cam, env, W, H, n, BOUNCE, opts=o)   # warm-up of this shape
                    ms, img = timed(lambda: ctx.render(cam, env, W, H, n, BOUNCE, opts=o), a.repeat)
                    st = ctx.stats()
                    line["runs"].append(dict(mode=m, spp=n, call_ms=ms, mrays_per_s=st["rays"] / (ms * 1e3),
                                             rays_per_sample=st["rays"] / (W * H * n), device_ms=st["total_ms"],
                                             rmse_vs_own_converged=rmse(img, conv[m]),
                                             rmse_edges_vs_own_converged=rmse(img, conv[m], edges)))
            f.write(json.dumps(line) + "\n")
            f.flush()
            print(json.dumps(line))
    ctx.close()


if __name__ == "__main__":
    main()
