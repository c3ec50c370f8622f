"""CPU: the restatement oracle on configurations test_oracle_golden.py does not hold — other resolutions, bounce
counts 0 / 1 / 3, random cameras and suns, a pixel range of a launch, a long generator stream, a tonemap over 4 000
values — bit for bit against stored vectors.

tests/golden/oracle_vs_ref.npz (written by tests/golden/make_oracle_vs_ref.py) holds what these tests expect; its
`source` entry says whether it was recorded from the reference's own kernels (oracle/_ref/libclref.so, the .cl text
compiled by g++, oracle/build_ref.py) or from the oracle.  Where oracle/_ref is built, every test also runs the
reference live and requires it to give the same bits, so the stored vectors are checked against the reference there.
The pixel-range test compares with the reference's full launch stored in tests/golden/golden_ref.npz."""
import os

import numpy as np
import pytest

from oracle import oracle, ref_lib
from tests import fixtures

VECTORS = os.path.join(fixtures.GOLDEN, "oracle_vs_ref.npz")
RENDERS = [("cornell", 80, 5, 4), ("cornell", 33, 3, 0), ("monkey_cfg2", 40, 3, 4), ("serre", 56, 3, 3),
           ("furnace_cfg3", 48, 4, 4), ("proto", 50, 3, 1), ("single", 40, 2, 4)]
CAMERAS = 4                        # random cameras / suns on Serre, 40 x 40, 3 spp, maxBounce 3
RNG_PIXELS, RNG_IMG, RNG_N = (3, 1000, 123456), 1 << 20, 500
TONEMAP_N = 4000                   # of the 4 096 stored inputs
COUNTERS = ("rays", "box_tests", "tri_tests", "rand_calls")
_vectors = {}


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def vectors():
    if not _vectors:
        z = np.load(VECTORS)
        _vectors.update({k: z[k] for k in z.files})
    return _vectors


def render_key(name, res, spp, bounce):
    return f"render/{name}/{res}x{spp}x{bounce}"


def render_inputs(name, res):
    sc = fixtures.load_scene(name)
    cam, env = fixtures.cam_env(sc["params"], res)
    return sc, cam, env, fixtures.load_ibl("grey" if name == "furnace_cfg3" else "preview")


@pytest.mark.parametrize("name,res,spp,bounce", RENDERS)
def test_render_bit_exact(name, res, spp, bounce):
    v, k = vectors(), render_key(name, res, spp, bounce)
    sc, cam, env, ibl = render_inputs(name, res)
    got, gc = oracle.render(sc, cam, env, res * res, spp, bounce, ibl)
    assert np.array_equal(bits(got), bits(v[k + "/out"]))
    assert [gc[c] for c in COUNTERS] == [int(x) for x in v[k + "/counters"]]
    if ref_lib.available():
        want, wc = ref_lib.raytrace(sc, cam, env, res * res, spp, bounce, ibl, counters=True)
        assert np.array_equal(bits(got), bits(want))
        assert gc == wc


def test_random_cameras_bit_exact():
    v = vectors()
    sc = fixtures.load_scene("serre")
    ibl = fixtures.load_ibl()
    for i in range(CAMERAS):
        k = f"camera/{i}"
        cam, env = v[k + "/cam"], v[k + "/env"]
        got, _ = oracle.render(sc, cam, env, 40 * 40, 3, 3, ibl)
        p = oracle.primary(sc, cam, 40 * 40)
        assert np.array_equal(bits(got), bits(v[k + "/out"]))
        assert np.array_equal(p["tri"], v[k + "/primary_tri"])
        assert np.array_equal(bits(p["k"]), bits(v[k + "/primary_k"]))
        assert np.array_equal(bits(p["dir"]), bits(v[k + "/primary_dir"]))
        if ref_lib.available():
            want, _ = ref_lib.raytrace(sc, cam, env, 40 * 40, 3, 3, ibl)
            assert np.array_equal(bits(got), bits(want))
            p_ref = ref_lib.primary(sc, cam, 40 * 40)
            assert np.array_equal(p["tri"], p_ref["tri"])
            assert np.array_equal(bits(p["k"]), bits(p_ref["k"]))
            assert np.array_equal(bits(p["dir"]), bits(p_ref["dir"]))


def test_pixel_subrange_matches_full_launch():
    g = fixtures.golden()
    full = g["cornell/render"]          # the reference's launch over all 64 x 64 pixels, 8 spp, maxBounce 4
    part, _ = oracle.render(fixtures.load_scene("cornell"), g["cornell/cam"], g["cornell/env"], 64 * 64, 8, 4,
                            fixtures.load_ibl(), i0=500, i1=900)
    assert np.array_equal(bits(part[1500:2700]), bits(full[1500:2700]))
    assert np.all(part[:1500] == 0) and np.all(part[2700:] == 0)


def test_tonemap_and_rng_live():
    v = vectors()
    x = v["tonemap/in"]
    got = oracle.img_processing(x, TONEMAP_N)
    assert np.array_equal(bits(got), bits(v["tonemap/out"]))
    if ref_lib.available():
        assert np.array_equal(bits(got), bits(ref_lib.img_processing(x, TONEMAP_N)))
    for px in RNG_PIXELS:
        got = oracle.rand_stream(0, px, RNG_IMG, RNG_N)
        assert np.array_equal(bits(got), bits(v[f"rand/{px}"]))
        if ref_lib.available():
            assert np.array_equal(bits(got), bits(ref_lib.rand_stream(px, RNG_IMG, RNG_N)))
