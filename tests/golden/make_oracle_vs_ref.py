#!/usr/bin/env python3
"""Regenerates tests/golden/oracle_vs_ref.npz, the expected values of tests/test_oracle_vs_ref.py:

    python tests/golden/make_oracle_vs_ref.py          (after __graft_entry__.build())

The values are recorded from the reference's own kernels (oracle/_ref/libclref*.so) where oracle/build_ref.py has
built them from a checkout of the reference, and from the oracle restatement (oracle/rt_oracle.c) otherwise; the
file's `source` entry says which.  The inputs are the committed scene fixtures plus what is stored beside the outputs
(the random cameras and suns, the tonemap input), drawn here from fixed seeds.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from oracle import oracle, ref_lib  # noqa: E402
from tests import fixtures  # noqa: E402
from tests.test_oracle_vs_ref import (CAMERAS, COUNTERS, RENDERS, RNG_IMG, RNG_N, RNG_PIXELS, TONEMAP_N,  # noqa: E402
                                      VECTORS, render_inputs, render_key)


def main():
    ref = ref_lib.available() and ref_lib.available("libclref_count.so")
    v = {"source": np.array("reference" if ref else "oracle")}

    for name, res, spp, bounce in RENDERS:
        sc, cam, env, ibl = render_inputs(name, res)
        if ref:
            out, cnt = ref_lib.raytrace(sc, cam, env, res * res, spp, bounce, ibl, counters=True)
        else:
            out, cnt = oracle.render(sc, cam, env, res * res, spp, bounce, ibl)
        k = render_key(name, res, spp, bounce)
        v[k + "/out"] = out
        v[k + "/counters"] = np.array([cnt[c] for c in COUNTERS], np.uint64)

    rng = np.random.default_rng(11)
    sc = fixtures.load_scene("serre")
    ibl = fixtures.load_ibl()
    for i in range(CAMERAS):
        cam, env = fixtures.cam_env(sc["params"], 40)
        cam[0:3] += rng.uniform(-1, 1, 3).astype(np.float32)
        cam[3:6] = rng.uniform(-60, 60, 3).astype(np.float32)
        cam[9] = np.float32(rng.uniform(0.4, 1.6))
        env[0:3] = rng.uniform(-90, 90, 3).astype(np.float32)
        env[3:5] = rng.uniform(0, 2, 2).astype(np.float32)
        if ref:
            out, _ = ref_lib.raytrace(sc, cam, env, 40 * 40, 3, 3, ibl)
            p = ref_lib.primary(sc, cam, 40 * 40)
        else:
            out, _ = oracle.render(sc, cam, env, 40 * 40, 3, 3, ibl)
            p = oracle.primary(sc, cam, 40 * 40)
        k = f"camera/{i}"
        v.update({k + "/cam": cam, k + "/env": env, k + "/out": out, k + "/primary_tri": p["tri"],
                  k + "/primary_k": p["k"], k + "/primary_dir": p["dir"]})

    x = np.random.default_rng(0).uniform(-0.5, 2.0, 4096).astype(np.float32)
    v["tonemap/in"] = x
    v["tonemap/out"] = (ref_lib if ref else oracle).img_processing(x, TONEMAP_N)
    for px in RNG_PIXELS:
        v[f"rand/{px}"] = ref_lib.rand_stream(px, RNG_IMG, RNG_N) if ref else oracle.rand_stream(0, px, RNG_IMG, RNG_N)

    np.savez_compressed(VECTORS, **v)
    print(VECTORS, "source:", v["source"], os.path.getsize(VECTORS), "bytes")


if __name__ == "__main__":
    main()
