"""GPU: opt-in pixel jitter (B200RT_SAMPLING_PIXEL_JITTER) against the jitter oracle, bit for bit, statistics included,
through every path that carries the sampling mask: pixel ranges, tile rows, partial sample ranges, sample streams, the
multi-GPU handle, render_rgb8, render_denoised, the launcher and progressive slices; its refusals; and the coverage
of an edge at a high sample count."""
import numpy as np
import pytest

import ensem3a_openclraytracer_b200 as rt
from oracle import oracle
from oracle_jitter import jitter
from tests import fixtures, jitter_scene

pytestmark = pytest.mark.gpu

J = rt.SAMPLING_PIXEL_JITTER


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def lit_cornell():
    """the Cornell box with its lamp switched on and no sun"""
    sc = dict(fixtures.load_scene("cornell"))
    m = sc["materialData"].copy().reshape(-1, 6)
    m[3, 4] = 5.0
    sc["materialData"] = m.reshape(-1)
    sc["params"] = dict(sc["params"], sun_Power="0")
    return sc


def setup(ctx, name, ibl_name, w, h=None):
    sc = lit_cornell() if name == "lit_cornell" else fixtures.load_scene(name)
    ibl = fixtures.load_ibl(ibl_name)
    fixtures.upload(ctx, sc, ibl)
    cam, env = fixtures.cam_env(sc["params"], w, h)
    return sc, ibl, cam, env


def parts_image(sc, ibl, cam, env, n_pix, spp, n, rng, seed):
    """the oracle's raw sums of the n contiguous sample ranges the library cuts [0, spp) into (sizes differing by at
    most one, the longer first), added in part order and finalised; and the oracle's ray count"""
    base, extra = divmod(spp, n)
    total, rays, s0 = None, 0, 0
    for k in range(n):
        s1 = s0 + base + (1 if k < extra else 0)
        part, cnt = jitter.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=rng, seed=seed, s0=s0, s1=s1, raw_sums=True,
                                  sampling=J)
        total = part if total is None else total + part
        rays += cnt["rays"]
        s0 = s1
    return np.fmax(np.fmin(total / np.float32(spp), np.float32(1)), np.float32(0)), rays


def per_sample(sampling, bounce, nee):
    return (2 * (bounce + 1) + 1 if nee else bounce + 2) + 1


@pytest.mark.parametrize("name,ibl_name,res,rows,sampling", [
    ("cornell", "preview", 64, None, J),
    ("cornell", "preview", 64, None, J | 3),
    ("monkey_cfg2", "preview", 72, None, J),
    ("monkey_cfg2", "preview", 72, None, J | 3),
    ("furnace_cfg3", "grey", 64, None, J),
    ("furnace_cfg3", "grey", 64, None, J | 3),
    ("serre", "preview", 96, (30, 50), J),
    ("serre", "preview", 96, (30, 50), J | 3),
    ("lit_cornell", "preview", 64, None, J | rt.SAMPLING_LIGHTS),
])
@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_jitter_equals_the_oracle_bit_for_bit(gpu_ctx, name, ibl_name, res, rows, sampling, rng):
    sc, ibl, cam, env = setup(gpu_ctx, name, ibl_name, res)
    spp, n_pix = 5, res * res
    i0, i1 = (rows[0] * res, rows[1] * res) if rows else (0, n_pix)
    nee = bool(sampling & rt.SAMPLING_LIGHTS) and sc["lightData"].size > 0
    for trav, bounce in ((rt.TRAVERSAL_FAST, 4), (rt.TRAVERSAL_REFERENCE, 0)):
        want, cnt = jitter.render(sc, cam, env, n_pix, spp, bounce, ibl, i0=i0, i1=i1, rng_mode=rng, seed=31,
                                  sampling=sampling)
        o = rt.make_opts(rng_mode=rng, seed=31, sampling=sampling, traversal=trav, collect_stats=False,
                         pixel_begin=i0 if rows else 0, pixel_end=i1 if rows else 0)
        got = gpu_ctx.render(cam, env, res, res, spp, bounce, opts=o)
        assert np.array_equal(bits(got[3 * i0:3 * i1]), bits(want[3 * i0:3 * i1]))
        st = gpu_ctx.stats()
        assert st["rays"] == cnt["rays"]
        assert st["primary_rays"] == 0
        assert st["samples"] == (i1 - i0) * spp
        assert st["wave_iterations"] == spp * per_sample(sampling, bounce, nee)
        it = st["wave_iterations"]
        compactions = sum(1 for k in range(it) if (k + 1) % 4 == 0)
        assert st["kernel_launches"] == 3 + (it + 1) + compactions + it
    # jitter moves the image off the reference's
    plain, _ = oracle.render(sc, cam, env, n_pix, spp, 4, ibl, i0=i0, i1=i1, rng_mode=rng, seed=31,
                             sampling=sampling & 3)
    assert not np.array_equal(bits(plain[3 * i0:3 * i1]), bits(want[3 * i0:3 * i1]))


def test_tile_rows_and_pixel_range_reference_generator(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 72, 50)
    W, H, spp = 72, 50, 6
    want, _ = jitter.render(sc, cam, env, W * H, spp, 4, ibl, sampling=J)
    img = gpu_ctx.render(cam, env, W, H, spp, 4, opts=rt.make_opts(sampling=J, tile_row_mod=3, tile_row_rem=1))
    img = img.reshape(H, W, 3)
    rows = (np.arange(H) // 4) % 3 == 1
    assert np.array_equal(bits(img[rows]), bits(want.reshape(H, W, 3)[rows])) and not img[~rows].any()
    assert gpu_ctx.stats()["samples"] == rows.sum() * W * spp
    got = gpu_ctx.render(cam, env, W, H, spp, 4, opts=rt.make_opts(sampling=J, pixel_begin=700, pixel_end=1900))
    assert np.array_equal(bits(got[3 * 700:3 * 1900]), bits(want[3 * 700:3 * 1900]))


def test_partial_sample_range_sums(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", "preview", 64)
    want, cnt = jitter.render(sc, cam, env, 64 * 64, 8, 4, ibl, rng_mode=1, seed=3, s0=2, s1=7, raw_sums=True,
                              sampling=J | 1)
    got = gpu_ctx.render(cam, env, 64, 64, 8, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3, sampling=J | 1,
                                                                   output=rt.OUT_SUMS, sample_begin=2, sample_end=7))
    assert np.array_equal(bits(got), bits(want))
    assert gpu_ctx.stats()["rays"] == cnt["rays"]


@pytest.mark.parametrize("streams", [3, -1])
def test_sample_streams_add_the_parts_in_order(gpu_ctx, streams):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 64)
    spp = 8
    got = gpu_ctx.render(cam, env, 64, 64, spp, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=6, sampling=J,
                                                                     sample_streams=streams))
    st = gpu_ctx.stats()
    n = st["sample_streams"]
    assert n > 1
    want, rays = parts_image(sc, ibl, cam, env, 64 * 64, spp, n, 1, 6)
    assert np.array_equal(bits(got), bits(want))
    assert st["rays"] == rays and st["primary_rays"] == 0


@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_multi_handle_on_one_gpu(rng):
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    cam, env = fixtures.cam_env(sc["params"], 64, 48)
    if rng == rt.RNG_REFERENCE:   # tile rows: every pixel's samples on one GPU
        want, cnt = jitter.render(sc, cam, env, 64 * 48, 6, 4, ibl, rng_mode=rng, seed=8, sampling=J)
        rays = cnt["rays"]
    else:                         # sample ranges, added in GPU order
        want, rays = parts_image(sc, ibl, cam, env, 64 * 48, 6, 3, rng, 8)
    m = rt.MultiContext([0, 0, 0])
    try:
        fixtures.upload(m, sc, ibl)
        got = m.render(cam, env, 64, 48, 6, 4, opts=rt.make_opts(rng_mode=rng, seed=8, sampling=J))
        assert np.array_equal(bits(got.reshape(-1)), bits(want))
        assert m.stats()["rays"] == rays
    finally:
        m.close()


def test_rgb8_and_denoised(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 80, 60)
    for o in (rt.make_opts(sampling=J), rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=2, sampling=J | 3, sample_streams=4)):
        img = gpu_ctx.render(cam, env, 80, 60, 8, 4, opts=o)
        q = gpu_ctx.render_rgb8(cam, env, 80, 60, 8, 4, opts=o)
        assert np.array_equal(q.reshape(-1), (img * np.float32(255)).astype(np.uint8))
        st0 = gpu_ctx.stats()
        den = gpu_ctx.render_denoised(cam, env, 80, 60, 8, 4, opts=o)
        st1 = gpu_ctx.stats()
        gb = gpu_ctx.gbuffer(cam, 80, 60, opts=o)
        assert np.array_equal(bits(den), bits(gpu_ctx.denoise(img.reshape(60, 80, 3), gb)))
        assert st1["rays"] == st0["rays"] + 80 * 60 and st1["primary_rays"] == 80 * 60
        # the G-buffer is the unjittered primary hit
        assert np.array_equal(bits(gb["position"]), bits(gpu_ctx.gbuffer(cam, 80, 60)["position"]))


def test_coverage_of_an_edge_at_high_sample_count(gpu_ctx):
    W = H = 256
    spp = 1024
    sc, cam, env, ibl = jitter_scene.scene(W, H)
    fixtures.upload(gpu_ctx, sc, ibl)
    f = jitter_scene.coverage(W, H)
    img = gpu_ctx.render(cam, env, W, H, spp, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=13, sampling=J))
    img = img.reshape(H, W, 3)[..., 0]
    assert np.all(np.abs(img - f) <= 5.0 * np.sqrt(f * (1.0 - f) / spp) + 2e-3)
    plain = gpu_ctx.render(cam, env, W, H, 4, 4)
    assert set(np.unique(plain)) == {0.0, 1.0}


def test_refusals(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 32)
    for bad in (4, 12, 16, 24, -8):
        with pytest.raises(rt.B200RTError, match="sampling"):
            gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=bad))
    with pytest.raises(rt.B200RTError, match="PIXEL_JITTER"):
        gpu_ctx.render_adaptive(cam, env, 32, 32, 8, 4, rel_error=0.1, min_spp=4, check_every=4,
                                opts=rt.make_opts(sampling=J))
    kl = rt.KernelLauncher(None, None, None, None)
    kl.pixel_jitter = True
    kl.adaptive = dict(rel_error=0.1)
    out = np.zeros(32 * 32 * 3, np.float32)
    with pytest.raises(ValueError, match="cannot be combined"):
        kl.launch_Raytracing(out, sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"],
                             sc["BVH"], cam, env, 32 * 32, 2, 4, ibl)
    kl.close()


def test_a_default_render_after_a_jittered_one(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", "preview", 64)
    gpu_ctx.render(cam, env, 64, 64, 4, 4, opts=rt.make_opts(sampling=J | 2))
    want, cnt = oracle.render(sc, cam, env, 64 * 64, 4, 4, ibl)
    got = gpu_ctx.render(cam, env, 64, 64, 4, 4)
    assert np.array_equal(bits(got), bits(want))
    st = gpu_ctx.stats()
    assert st["rays"] == cnt["rays"] and st["primary_rays"] == 64 * 64


def test_launcher_attribute_and_environment(monkeypatch):
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    res, spp = 64, 6
    cam, env = fixtures.cam_env(sc["params"], res)
    args = (sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"], sc["BVH"], cam, env,
            res * res, spp, 4, ibl)
    for var in ("B200RT_ADAPTIVE", "B200RT_DENOISE", "B200RT_CUDA_DEVICES"):
        monkeypatch.delenv(var, raising=False)
    ctx = rt.Context(0)
    fixtures.upload(ctx, sc, ibl)
    want = ctx.render(cam, env, res, res, spp, 4, opts=rt.make_opts(sampling=J))
    plain = ctx.render(cam, env, res, res, spp, 4)
    monkeypatch.setenv("B200RT_PIXEL_JITTER", "1")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.pixel_jitter is True
    out = np.zeros(res * res * 3, np.float32)
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(want))
    kl.pixel_jitter = False
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(plain))
    kl.close()
    monkeypatch.setenv("B200RT_PIXEL_JITTER", "0")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.pixel_jitter is False
    kl.pixel_jitter = True
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(want))
    kl.close()
    monkeypatch.setenv("B200RT_PIXEL_JITTER", "on")
    with pytest.raises(ValueError):
        rt.KernelLauncher(None, None, None, None)
    ctx.close()


def test_progressive_slices(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 64, 48)
    pr = rt.ProgressiveRender(gpu_ctx, cam, env, 64, 48, 40, 4, slice_spp=16, seed=3, sampling=J)
    for _ in pr:
        pass
    one = gpu_ctx.render(cam, env, 64, 48, 40, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3, sampling=J))
    rel = np.abs(pr.image() - one) / np.maximum(np.abs(one), 1e-3)
    assert rel.max() <= 1e-4
    plain = rt.ProgressiveRender(gpu_ctx, cam, env, 64, 48, 40, 4, slice_spp=16, seed=3)
    for _ in plain:
        pass
    assert not np.array_equal(bits(plain.image()), bits(pr.image()))
