"""GPU: opt-in refractive glass (B200RT_SAMPLING_DIELECTRIC_GLASS) against the glass oracle, bit for bit, ray counts
included, on config 2 (its glass wall), config 2 with a glass monkey and Serre; every path that carries the sampling
mask (pixel ranges, tile rows, partial sample ranges, sample streams, the multi-GPU handle, render_rgb8,
render_adaptive, render_denoised, the launcher and progressive slices); unchanged cases and the furnace; the refusals;
no state left behind."""
import numpy as np
import pytest

import ensem3a_openclraytracer_b200 as rt
from oracle import oracle
from oracle_denoise import denoise as D
from oracle_glass import glass
from tests import fixtures, glass_scene as gs

pytestmark = pytest.mark.gpu

G = rt.SAMPLING_DIELECTRIC_GLASS
S = rt.SAMPLING_SMOOTH_NORMALS
J = rt.SAMPLING_PIXEL_JITTER


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def setup(ctx, name, w, h=None):
    sc = gs.load(name)
    ibl = fixtures.load_ibl()
    fixtures.upload(ctx, sc, ibl)
    cam, env = fixtures.cam_env(fixtures.load_scene("serre" if name == "serre" else "monkey_cfg2")["params"], w, h)
    return sc, ibl, cam, env


def parts_image(sc, ibl, cam, env, n_pix, spp, n, seed, sampling):
    """the oracle's raw sums of the n contiguous sample ranges the library cuts [0, spp) into, added in part order and
    finalised; and the oracle's ray count"""
    base, extra = divmod(spp, n)
    total, rays, s0 = None, 0, 0
    for k in range(n):
        s1 = s0 + base + (1 if k < extra else 0)
        part, cnt = glass.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=1, seed=seed, s0=s0, s1=s1, raw_sums=True,
                                 sampling=sampling)
        total = part if total is None else total + part
        rays += cnt["rays"] - (n_pix if k > 0 else 0)   # every part traces the primary rays; `rays` counts them once
        s0 = s1
    return np.fmax(np.fmin(total / np.float32(spp), np.float32(1)), np.float32(0)), rays


@pytest.mark.parametrize("name,res", [("monkey_cfg2", 48), ("monkey_glass", 48), ("serre", 40)])
@pytest.mark.parametrize("sampling", [G, G | 1, G | 2, G | 3, G | J, G | S, G | S | 2])
@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_glass_equals_the_oracle_bit_for_bit(gpu_ctx, name, res, sampling, rng):
    sc, ibl, cam, env = setup(gpu_ctx, name, res)
    spp, n_pix = 4, res * res
    for trav, bounce in ((rt.TRAVERSAL_FAST, 4), (rt.TRAVERSAL_REFERENCE, 1), (rt.TRAVERSAL_VERIFY, 2)):
        want, cnt = glass.render(sc, cam, env, n_pix, spp, bounce, ibl, rng_mode=rng, seed=17, sampling=sampling)
        got = gpu_ctx.render(cam, env, res, res, spp, bounce,
                             opts=rt.make_opts(rng_mode=rng, seed=17, sampling=sampling, traversal=trav))
        assert np.array_equal(bits(got), bits(want))
        st = gpu_ctx.stats()
        assert st["rays"] == cnt["rays"]
        if trav == rt.TRAVERSAL_VERIFY:
            assert st["mismatches"] == 0
    # the bit moves the image off the pass-through one
    plain, _ = glass.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=rng, seed=17, sampling=sampling & ~G)
    want, _ = glass.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=rng, seed=17, sampling=sampling)
    assert not np.array_equal(bits(plain), bits(want))


def test_tile_rows_and_pixel_range(gpu_ctx):
    W, H, spp = 72, 50, 5
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_glass", W, H)
    want, _ = glass.render(sc, cam, env, W * H, spp, 4, ibl, sampling=G)
    img = gpu_ctx.render(cam, env, W, H, spp, 4, opts=rt.make_opts(sampling=G, tile_row_mod=3, tile_row_rem=1))
    img = img.reshape(H, W, 3)
    rows = (np.arange(H) // 4) % 3 == 1
    assert np.array_equal(bits(img[rows]), bits(want.reshape(H, W, 3)[rows])) and not img[~rows].any()
    for rng in (rt.RNG_REFERENCE, rt.RNG_PHILOX):
        got = gpu_ctx.render(cam, env, W, H, spp, 4, opts=rt.make_opts(rng_mode=rng, seed=1, sampling=G | 2,
                                                                       pixel_begin=700, pixel_end=1900))
        want2, _ = glass.render(sc, cam, env, W * H, spp, 4, ibl, rng_mode=rng, seed=1, sampling=G | 2, i0=700, i1=1900)
        assert np.array_equal(bits(got[3 * 700:3 * 1900]), bits(want2[3 * 700:3 * 1900]))


def test_partial_sample_range_sums(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_glass", 48)
    for sampling in (G | 1, G | J, G | S):
        want, cnt = glass.render(sc, cam, env, 48 * 48, 8, 4, ibl, rng_mode=1, seed=3, s0=2, s1=7, raw_sums=True,
                                 sampling=sampling)
        got = gpu_ctx.render(cam, env, 48, 48, 8, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3, sampling=sampling,
                                                                       output=rt.OUT_SUMS, sample_begin=2, sample_end=7))
        assert np.array_equal(bits(got), bits(want))
        assert gpu_ctx.stats()["rays"] == cnt["rays"]


@pytest.mark.parametrize("streams", [3, -1])
def test_sample_streams_add_the_parts_in_order(gpu_ctx, streams):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_glass", 48)
    spp = 8
    got = gpu_ctx.render(cam, env, 48, 48, spp, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=6, sampling=G | 2,
                                                                     sample_streams=streams))
    st = gpu_ctx.stats()
    n = st["sample_streams"]
    assert n > 1
    want, rays = parts_image(sc, ibl, cam, env, 48 * 48, spp, n, 6, G | 2)
    assert np.array_equal(bits(got), bits(want))
    assert st["rays"] == rays


@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_multi_handle(rng):
    """MultiContext over every visible GPU, or three entries on GPU 0 when there is one; and a device listed twice"""
    sc, ibl = gs.glass_monkey(), fixtures.load_ibl()
    cam, env = fixtures.cam_env(fixtures.load_scene("monkey_cfg2")["params"], 64, 48)
    n = rt.device_count()
    for devices in ([*range(n)] if n >= 2 else [0, 0, 0], [0, 0]):
        if rng == rt.RNG_REFERENCE:   # tile rows: every pixel's samples on one GPU
            want, _ = glass.render(sc, cam, env, 64 * 48, 6, 4, ibl, rng_mode=rng, seed=8, sampling=G)
        else:                         # sample ranges, added in GPU order
            want, _ = parts_image(sc, ibl, cam, env, 64 * 48, 6, min(len(devices), 6), 8, G)
        m = rt.MultiContext(devices)
        try:
            fixtures.upload(m, sc, ibl)
            got = m.render(cam, env, 64, 48, 6, 4, opts=rt.make_opts(rng_mode=rng, seed=8, sampling=G))
            assert np.array_equal(bits(got.reshape(-1)), bits(want))
        finally:
            m.close()


def test_rgb8_adaptive_and_denoised(gpu_ctx):
    W, H = 64, 48
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_glass", W, H)
    o = rt.make_opts(sampling=G | 1)
    img = gpu_ctx.render(cam, env, W, H, 6, 4, opts=o)
    q = gpu_ctx.render_rgb8(cam, env, W, H, 6, 4, opts=o)
    assert np.array_equal(q.reshape(-1), (img * np.float32(255)).astype(np.uint8))
    ad = dict(rel_error=0.2, min_spp=4, check_every=2)
    for rng, sampling in ((rt.RNG_REFERENCE, G), (rt.RNG_PHILOX, G | S | 2)):
        want, n_want, err_want, cnt = glass.render(sc, cam, env, W * H, 16, 4, ibl, rng_mode=rng, seed=4,
                                                   sampling=sampling, adaptive=ad)
        got, n_got, err_got = gpu_ctx.render_adaptive(cam, env, W, H, 16, 4, opts=rt.make_opts(rng_mode=rng, seed=4,
                                                                                             sampling=sampling), **ad)
        assert np.array_equal(bits(got.reshape(-1)), bits(want))
        assert np.array_equal(n_got.reshape(-1), n_want) and np.array_equal(bits(err_got.reshape(-1)), bits(err_want))
        assert gpu_ctx.stats()["rays"] == cnt["rays"]
        assert (n_want < 16).any()
    with pytest.raises(rt.B200RTError, match="PIXEL_JITTER"):
        gpu_ctx.render_adaptive(cam, env, W, H, 8, 4, opts=rt.make_opts(sampling=G | J), **ad)
    gb = D.gbuffer(sc, cam, W, H)   # the G-buffer ignores the bit: it describes the glass surface
    for o in (rt.make_opts(sampling=G), rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=2, sampling=G | 3, sample_streams=3)):
        den, noisy = gpu_ctx.render_denoised(cam, env, W, H, 6, 4, opts=o, return_noisy=True)
        assert np.array_equal(bits(noisy).reshape(-1), bits(gpu_ctx.render(cam, env, W, H, 6, 4, opts=o)).reshape(-1))
        ref = D.atrous(noisy.reshape(H, W, 3), gb, bvh=sc["BVH"], **rt.DENOISE_DEFAULTS)
        assert np.array_equal(bits(den).reshape(-1), bits(ref).reshape(-1))


def test_launcher_attribute_and_environment(monkeypatch):
    sc, ibl = gs.glass_monkey(), fixtures.load_ibl()
    res, spp = 48, 4
    cam, env = fixtures.cam_env(fixtures.load_scene("monkey_cfg2")["params"], res)
    args = (sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"], sc["BVH"], cam, env,
            res * res, spp, 4, ibl)
    for var in ("B200RT_ADAPTIVE", "B200RT_DENOISE", "B200RT_CUDA_DEVICES", "B200RT_PIXEL_JITTER",
                "B200RT_SMOOTH_NORMALS"):
        monkeypatch.delenv(var, raising=False)
    want, _ = glass.render(sc, cam, env, res * res, spp, 4, ibl, sampling=G)
    both, _ = glass.render(sc, cam, env, res * res, spp, 4, ibl, sampling=G | S)
    plain, _ = glass.render(sc, cam, env, res * res, spp, 4, ibl, sampling=0)
    monkeypatch.setenv("B200RT_DIELECTRIC_GLASS", "1")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.dielectric_glass is True
    out = np.zeros(res * res * 3, np.float32)
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(want))
    kl.smooth_normals = True
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(both))
    kl.smooth_normals = False
    kl.dielectric_glass = False
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(plain))
    kl.close()
    monkeypatch.setenv("B200RT_DIELECTRIC_GLASS", "0")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.dielectric_glass is False
    kl.close()
    monkeypatch.setenv("B200RT_DIELECTRIC_GLASS", "yes")
    with pytest.raises(ValueError):
        rt.KernelLauncher(None, None, None, None)


def test_progressive_slices(gpu_ctx):
    W, H = 64, 48
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_glass", W, H)
    pr = rt.ProgressiveRender(gpu_ctx, cam, env, W, H, 40, 4, slice_spp=16, seed=3, sampling=G)
    for _ in pr:
        pass
    one = gpu_ctx.render(cam, env, W, H, 40, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3, sampling=G))
    rel = np.abs(pr.image() - one) / np.maximum(np.abs(one), 1e-3)
    assert rel.max() <= 1e-4
    plain = gpu_ctx.render(cam, env, W, H, 40, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3))
    assert not np.array_equal(bits(one), bits(plain))


@pytest.mark.parametrize("name", ["monkey_cfg2", "serre", "monkey_glass", "cornell"])
def test_ior_one_and_glass_free_scenes_render_the_same(gpu_ctx, name):
    sc = gs.glass_ior(gs.load(name), 1.0)
    ibl = fixtures.load_ibl()
    fixtures.upload(gpu_ctx, sc, ibl)
    cam, env = fixtures.cam_env(fixtures.load_scene("monkey_cfg2" if name == "monkey_glass" else name)["params"], 64)
    for base in (0, 3, J, S):
        for rng in (rt.RNG_REFERENCE, rt.RNG_PHILOX):
            a = gpu_ctx.render(cam, env, 64, 64, 4, 4, opts=rt.make_opts(rng_mode=rng, seed=3, sampling=base))
            ra = gpu_ctx.stats()["rays"]
            b = gpu_ctx.render(cam, env, 64, 64, 4, 4, opts=rt.make_opts(rng_mode=rng, seed=3, sampling=base | G))
            assert np.array_equal(bits(a), bits(b)) and gpu_ctx.stats()["rays"] == ra


def test_furnace(gpu_ctx):
    W, spp = 32, 8
    sc = gs.glass_sphere()
    cam, env, grey = gs.grey_view(W)
    fixtures.upload(gpu_ctx, sc, grey)
    hit = oracle.primary(sc, cam, W * W)["tri"] >= 0
    for rng in (rt.RNG_REFERENCE, rt.RNG_PHILOX):
        o = gpu_ctx.render(cam, env, W, W, spp, 8, opts=rt.make_opts(rng_mode=rng, seed=5, sampling=G | S,
                                                                     sample_streams=1)).reshape(-1, 3)
        assert np.array_equal(bits(o), bits(np.broadcast_to(o[~hit][0], o.shape)))
        want, _ = glass.render(sc, cam, env, W * W, spp, 8, grey, rng_mode=rng, seed=5, sampling=G)
        got = gpu_ctx.render(cam, env, W, W, spp, 8, opts=rt.make_opts(rng_mode=rng, seed=5, sampling=G))
        assert np.array_equal(bits(got), bits(want))


def test_refusals_and_no_leaked_state(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "serre", 32)
    for bad in (G | 64, 64, 4 | G, 256, -128):
        with pytest.raises(rt.B200RTError, match="sampling"):
            gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=bad))
    want_plain, cnt_plain = oracle.render(sc, cam, env, 32 * 32, 2, 4, ibl)
    for v in (-1.0, np.nan, np.inf):
        bad = gs.glass_ior(sc, v)   # Serre's glass is material 13
        fixtures.upload(gpu_ctx, bad, ibl)
        assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4)), bits(want_plain))
        gpu_ctx.primary_hits(cam, 32, 32, opts=rt.make_opts(sampling=G))
        gpu_ctx.gbuffer(cam, 32, 32, opts=rt.make_opts(sampling=G))
        calls = (lambda o: gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=o),
                 lambda o: gpu_ctx.render_rgb8(cam, env, 32, 32, 2, 4, opts=o),
                 lambda o: gpu_ctx.render_adaptive(cam, env, 32, 32, 4, 4, opts=o, rel_error=0.1, min_spp=2),
                 lambda o: gpu_ctx.render_denoised(cam, env, 32, 32, 2, 4, opts=o),
                 lambda o: gpu_ctx.render(cam, env, 32, 32, 4, 4, opts=rt.make_opts(
                     rng_mode=rt.RNG_PHILOX, sampling=o.sampling, sample_streams=2)))
        for call in calls:
            with pytest.raises(rt.B200RTError, match="material 13"):
                call(rt.make_opts(sampling=G))
        gpu_ctx.set_materials(sc["materialData"])   # fixed by a material edit alone
        want, _ = glass.render(sc, cam, env, 32 * 32, 2, 4, ibl, sampling=G)
        assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=G))), bits(want))
        gpu_ctx.set_materials(bad["materialData"])   # and broken again, the sample-stream helpers included
        with pytest.raises(rt.B200RTError, match="material 13"):
            gpu_ctx.render(cam, env, 32, 32, 4, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, sampling=G,
                                                                     sample_streams=2))
        m = rt.MultiContext([0, 0])
        try:
            fixtures.upload(m, bad, ibl)
            with pytest.raises(rt.B200RTError, match="material 13"):
                m.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=G))
            fixtures.upload(m, sc, ibl)
            m.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=G))
        finally:
            m.close()
    # a NaN ior on a diffuse material is never read
    nan_diffuse = gs.with_materials(sc, lambda mt: (mt.__setitem__((0, 5), np.nan), mt)[1])
    fixtures.upload(gpu_ctx, nan_diffuse, ibl)
    want, _ = glass.render(nan_diffuse, cam, env, 32 * 32, 2, 4, ibl, sampling=G)
    assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=G))), bits(want))
    # no leaked state: a default render after a glass render is the plain oracle's, ray count included
    fixtures.upload(gpu_ctx, sc, ibl)
    gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=G | S | 2))
    assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4)), bits(want_plain))
    assert gpu_ctx.stats()["rays"] == cnt_plain["rays"]
