"""GPU: opt-in rough glass (B200RT_SAMPLING_ROUGH_GLASS) against the rough-glass oracle, bit for bit, in image, rays,
samples, wave_iterations and kernel_launches, on config 2 with its glass wall at roughness 0.2, the proto scene as shipped
(glass of roughness 0.1) and the mixed scene (a rough and a smooth glass material in one frame); every path that carries
the sampling mask (pixel ranges, tile rows, partial sample ranges, sample streams, the multi-GPU handle, render_rgb8,
render_adaptive, render_denoised, the launcher and progressive slices); the refusals; no state left behind."""
import numpy as np
import pytest

import ensem3a_openclraytracer_b200 as rt
from oracle import oracle
from oracle_denoise import denoise as D
from oracle_rough import rough
from tests import fixtures, glass_scene as gs, rough_glass_scene as rs

pytestmark = pytest.mark.gpu

G = rt.SAMPLING_DIELECTRIC_GLASS
R = rt.SAMPLING_ROUGH_GLASS
GR = G | R
S = rt.SAMPLING_SMOOTH_NORMALS
J = rt.SAMPLING_PIXEL_JITTER
T = rt.SAMPLING_TEXTURES


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def setup(ctx, name, w, h=None):
    sc = rs.load(name)
    ibl = fixtures.load_ibl()
    fixtures.upload(ctx, sc, ibl)
    cam, env = rs.view(name, w, h)
    return sc, ibl, cam, env


def parts_image(sc, ibl, cam, env, n_pix, spp, n, seed, sampling):
    """the oracle's raw sums of the n contiguous sample ranges the library cuts [0, spp) into, added in part order and
    finalised; and the oracle's ray count"""
    base, extra = divmod(spp, n)
    total, rays, s0 = None, 0, 0
    for k in range(n):
        s1 = s0 + base + (1 if k < extra else 0)
        part, cnt = rough.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=1, seed=seed, s0=s0, s1=s1, raw_sums=True,
                                 sampling=sampling)
        total = part if total is None else total + part
        rays += cnt["rays"] - (n_pix if k > 0 else 0)   # every part traces the primary rays; `rays` counts them once
        s0 = s1
    return np.fmax(np.fmin(total / np.float32(spp), np.float32(1)), np.float32(0)), rays


def _checker(n=64):
    yy, xx = np.mgrid[0:n, 0:n]
    c = ((yy // 8 + xx // 8) % 2).astype(np.uint8) * 200 + 40
    return np.ascontiguousarray(np.stack([c, c // 2, 255 - c, np.full_like(c, 255)], axis=2))


@pytest.mark.parametrize("name,res", [("bench_rough", 48), ("proto", 48), ("mixed", 48)])
@pytest.mark.parametrize("sampling", [GR, GR | 1, GR | 2, GR | 3, GR | J, GR | S, GR | S | 2, GR | T])
@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_rough_glass_equals_the_oracle_bit_for_bit(gpu_ctx, name, res, sampling, rng):
    sc, ibl, cam, env = setup(gpu_ctx, name, res)
    tex = {0: _checker()} if sampling & T else None
    if tex:
        gpu_ctx.set_textures(tex)
    spp, n_pix = 4, res * res
    try:
        for trav, bounce in ((rt.TRAVERSAL_FAST, 4), (rt.TRAVERSAL_REFERENCE, 1), (rt.TRAVERSAL_VERIFY, 2)):
            want, cnt = rough.render(sc, cam, env, n_pix, spp, bounce, ibl, rng_mode=rng, seed=17, sampling=sampling,
                                     textures=tex)
            got = gpu_ctx.render(cam, env, res, res, spp, bounce,
                                 opts=rt.make_opts(rng_mode=rng, seed=17, sampling=sampling, traversal=trav))
            assert np.array_equal(bits(got), bits(want))
            st = gpu_ctx.stats()
            assert st["rays"] == cnt["rays"]
            if trav == rt.TRAVERSAL_VERIFY:
                assert st["mismatches"] == 0
            # samples, wave_iterations and kernel_launches follow the rough glass's formulas, which are bit 128's
            b = gpu_ctx.render(cam, env, res, res, spp, bounce,
                               opts=rt.make_opts(rng_mode=rng, seed=17, sampling=sampling & ~R, traversal=trav))
            sb = gpu_ctx.stats()
            for key in ("samples", "wave_iterations", "kernel_launches"):
                assert st[key] == sb[key], key
        # the bit moves the image off the smooth-glass one
        smooth, _ = rough.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=rng, seed=17, sampling=sampling & ~R,
                                 textures=tex)
        want, _ = rough.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=rng, seed=17, sampling=sampling, textures=tex)
        assert not np.array_equal(bits(smooth), bits(want))
    finally:
        if tex:
            gpu_ctx.set_textures(None)


def test_tile_rows_and_pixel_range(gpu_ctx):
    W, H, spp = 72, 50, 5
    sc, ibl, cam, env = setup(gpu_ctx, "mixed", W, H)
    want, _ = rough.render(sc, cam, env, W * H, spp, 4, ibl, sampling=GR)
    img = gpu_ctx.render(cam, env, W, H, spp, 4, opts=rt.make_opts(sampling=GR, tile_row_mod=3, tile_row_rem=1))
    img = img.reshape(H, W, 3)
    rows = (np.arange(H) // 4) % 3 == 1
    assert np.array_equal(bits(img[rows]), bits(want.reshape(H, W, 3)[rows])) and not img[~rows].any()
    for rng in (rt.RNG_REFERENCE, rt.RNG_PHILOX):
        got = gpu_ctx.render(cam, env, W, H, spp, 4, opts=rt.make_opts(rng_mode=rng, seed=1, sampling=GR | 2,
                                                                       pixel_begin=700, pixel_end=1900))
        want2, _ = rough.render(sc, cam, env, W * H, spp, 4, ibl, rng_mode=rng, seed=1, sampling=GR | 2, i0=700, i1=1900)
        assert np.array_equal(bits(got[3 * 700:3 * 1900]), bits(want2[3 * 700:3 * 1900]))


def test_partial_sample_range_sums(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "bench_rough", 48)
    for sampling in (GR | 1, GR | J, GR | S):
        want, cnt = rough.render(sc, cam, env, 48 * 48, 8, 4, ibl, rng_mode=1, seed=3, s0=2, s1=7, raw_sums=True,
                                 sampling=sampling)
        got = gpu_ctx.render(cam, env, 48, 48, 8, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3, sampling=sampling,
                                                                       output=rt.OUT_SUMS, sample_begin=2, sample_end=7))
        assert np.array_equal(bits(got), bits(want))
        assert gpu_ctx.stats()["rays"] == cnt["rays"]


@pytest.mark.parametrize("streams", [3, -1])
def test_sample_streams_add_the_parts_in_order(gpu_ctx, streams):
    sc, ibl, cam, env = setup(gpu_ctx, "mixed", 48)
    spp = 8
    got = gpu_ctx.render(cam, env, 48, 48, spp, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=6, sampling=GR | 2,
                                                                     sample_streams=streams))
    st = gpu_ctx.stats()
    n = st["sample_streams"]
    assert n > 1
    want, rays = parts_image(sc, ibl, cam, env, 48 * 48, spp, n, 6, GR | 2)
    assert np.array_equal(bits(got), bits(want))
    assert st["rays"] == rays


@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_multi_handle(rng):
    """MultiContext over every visible GPU, or three entries on GPU 0 when there is one; and a device listed twice"""
    sc, ibl = rs.mixed(), fixtures.load_ibl()
    cam, env = rs.view("mixed", 64, 48)
    n = rt.device_count()
    for devices in ([*range(n)] if n >= 2 else [0, 0, 0], [0, 0]):
        if rng == rt.RNG_REFERENCE:   # tile rows: every pixel's samples on one GPU
            want, _ = rough.render(sc, cam, env, 64 * 48, 6, 4, ibl, rng_mode=rng, seed=8, sampling=GR)
        else:                         # sample ranges, added in GPU order
            want, _ = parts_image(sc, ibl, cam, env, 64 * 48, 6, min(len(devices), 6), 8, GR)
        m = rt.MultiContext(devices)
        try:
            fixtures.upload(m, sc, ibl)
            got = m.render(cam, env, 64, 48, 6, 4, opts=rt.make_opts(rng_mode=rng, seed=8, sampling=GR))
            assert np.array_equal(bits(got.reshape(-1)), bits(want))
        finally:
            m.close()


def test_rgb8_adaptive_and_denoised(gpu_ctx):
    W, H = 64, 48
    sc, ibl, cam, env = setup(gpu_ctx, "bench_rough", W, H)
    o = rt.make_opts(sampling=GR | 1)
    img = gpu_ctx.render(cam, env, W, H, 6, 4, opts=o)
    q = gpu_ctx.render_rgb8(cam, env, W, H, 6, 4, opts=o)
    assert np.array_equal(q.reshape(-1), (img * np.float32(255)).astype(np.uint8))
    ad = dict(rel_error=0.2, min_spp=4, check_every=2)
    for rng, sampling in ((rt.RNG_REFERENCE, GR), (rt.RNG_PHILOX, GR | S | 2)):
        want, n_want, err_want, cnt = rough.render(sc, cam, env, W * H, 16, 4, ibl, rng_mode=rng, seed=4,
                                                   sampling=sampling, adaptive=ad)
        got, n_got, err_got = gpu_ctx.render_adaptive(cam, env, W, H, 16, 4, opts=rt.make_opts(rng_mode=rng, seed=4,
                                                                                             sampling=sampling), **ad)
        assert np.array_equal(bits(got.reshape(-1)), bits(want))
        assert np.array_equal(n_got.reshape(-1), n_want) and np.array_equal(bits(err_got.reshape(-1)), bits(err_want))
        assert gpu_ctx.stats()["rays"] == cnt["rays"]
        assert (n_want < 16).any()
    with pytest.raises(rt.B200RTError, match="PIXEL_JITTER"):
        gpu_ctx.render_adaptive(cam, env, W, H, 8, 4, opts=rt.make_opts(sampling=GR | J), **ad)
    gb = D.gbuffer(sc, cam, W, H)   # the G-buffer ignores the bit: it describes the glass surface
    for o in (rt.make_opts(sampling=GR), rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=2, sampling=GR | 3, sample_streams=3)):
        den, noisy = gpu_ctx.render_denoised(cam, env, W, H, 6, 4, opts=o, return_noisy=True)
        assert np.array_equal(bits(noisy).reshape(-1), bits(gpu_ctx.render(cam, env, W, H, 6, 4, opts=o)).reshape(-1))
        ref = D.atrous(noisy.reshape(H, W, 3), gb, bvh=sc["BVH"], **rt.DENOISE_DEFAULTS)
        assert np.array_equal(bits(den).reshape(-1), bits(ref).reshape(-1))


def test_launcher_attribute_and_environment(monkeypatch):
    sc, ibl = rs.mixed(), fixtures.load_ibl()
    res, spp = 48, 4
    cam, env = rs.view("mixed", res)
    args = (sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"], sc["BVH"], cam, env,
            res * res, spp, 4, ibl)
    for var in ("B200RT_ADAPTIVE", "B200RT_DENOISE", "B200RT_CUDA_DEVICES", "B200RT_PIXEL_JITTER",
                "B200RT_SMOOTH_NORMALS", "B200RT_TEXTURES", "B200RT_DIELECTRIC_GLASS"):
        monkeypatch.delenv(var, raising=False)
    want, _ = rough.render(sc, cam, env, res * res, spp, 4, ibl, sampling=GR)
    smooth, _ = rough.render(sc, cam, env, res * res, spp, 4, ibl, sampling=G)
    monkeypatch.setenv("B200RT_ROUGH_GLASS", "1")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.rough_glass is True and kl.dielectric_glass is False
    out = np.zeros(res * res * 3, np.float32)
    with pytest.raises(ValueError, match="dielectric_glass"):
        kl.launch_Raytracing(out, *args)
    kl.dielectric_glass = True
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(want))
    kl.rough_glass = False
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(smooth))
    kl.close()
    monkeypatch.setenv("B200RT_ROUGH_GLASS", "0")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.rough_glass is False
    kl.close()
    monkeypatch.setenv("B200RT_ROUGH_GLASS", "yes")
    with pytest.raises(ValueError):
        rt.KernelLauncher(None, None, None, None)


def test_progressive_slices(gpu_ctx):
    W, H = 64, 48
    sc, ibl, cam, env = setup(gpu_ctx, "proto", W, H)
    pr = rt.ProgressiveRender(gpu_ctx, cam, env, W, H, 40, 4, slice_spp=16, seed=3, sampling=GR)
    for _ in pr:
        pass
    one = gpu_ctx.render(cam, env, W, H, 40, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3, sampling=GR))
    rel = np.abs(pr.image() - one) / np.maximum(np.abs(one), 1e-3)
    assert rel.max() <= 1e-4
    smooth = gpu_ctx.render(cam, env, W, H, 40, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3, sampling=G))
    assert not np.array_equal(bits(one), bits(smooth))


def test_zero_roughness_and_ior_one_render_as_smooth_glass(gpu_ctx):
    """every glass at roughness 0 (the refractive-glass kernels run) or at ior 1 (pass-through): the bit changes nothing"""
    for sc in (rs.glass_roughness(fixtures.load_scene("proto"), 0.0), gs.glass_ior(fixtures.load_scene("proto"), 1.0)):
        fixtures.upload(gpu_ctx, sc, fixtures.load_ibl())
        cam, env = rs.view("proto", 48)
        for base in (G, G | 2, G | J, G | S):
            for rng in (rt.RNG_REFERENCE, rt.RNG_PHILOX):
                a = gpu_ctx.render(cam, env, 48, 48, 4, 4, opts=rt.make_opts(rng_mode=rng, seed=3, sampling=base))
                ra = gpu_ctx.stats()["rays"]
                b = gpu_ctx.render(cam, env, 48, 48, 4, 4, opts=rt.make_opts(rng_mode=rng, seed=3, sampling=base | R))
                assert np.array_equal(bits(a), bits(b)) and gpu_ctx.stats()["rays"] == ra


def test_refusals_and_no_leaked_state(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "proto", 32)   # the proto scene's glass is material 1
    calls = (lambda o: gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=o),
             lambda o: gpu_ctx.render_rgb8(cam, env, 32, 32, 2, 4, opts=o),
             lambda o: gpu_ctx.render_adaptive(cam, env, 32, 32, 4, 4, opts=o, rel_error=0.1, min_spp=2),
             lambda o: gpu_ctx.render_denoised(cam, env, 32, 32, 2, 4, opts=o),
             lambda o: gpu_ctx.render(cam, env, 32, 32, 4, 4, opts=rt.make_opts(
                 rng_mode=rt.RNG_PHILOX, sampling=o.sampling, sample_streams=2)))
    for bad in (R, R | 2, R | S, R | 1024, 1024 | GR, 4096 | GR):
        for call in calls:
            with pytest.raises(rt.B200RTError, match="sampling"):
                call(rt.make_opts(sampling=bad))
    m = rt.MultiContext([0, 0])
    try:
        fixtures.upload(m, sc, ibl)
        with pytest.raises(rt.B200RTError, match="DIELECTRIC_GLASS"):
            m.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=R))
    finally:
        m.close()
    want_smooth, _ = rough.render(sc, cam, env, 32 * 32, 2, 4, ibl, sampling=G)
    for v in (-0.5, np.nan, np.inf):
        bad = rs.glass_roughness(sc, v)
        fixtures.upload(gpu_ctx, bad, ibl)
        # bit 128 alone never reads the roughness
        assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=G))),
                              bits(want_smooth))
        gpu_ctx.primary_hits(cam, 32, 32, opts=rt.make_opts(sampling=GR))
        gpu_ctx.gbuffer(cam, 32, 32, opts=rt.make_opts(sampling=GR))
        for call in calls:
            with pytest.raises(rt.B200RTError, match="material 1 "):
                call(rt.make_opts(sampling=GR))
        gpu_ctx.set_materials(sc["materialData"])   # fixed by a material edit alone
        want, _ = rough.render(sc, cam, env, 32 * 32, 2, 4, ibl, sampling=GR)
        assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=GR))), bits(want))
        gpu_ctx.set_materials(bad["materialData"])   # and broken again, the sample-stream helpers included
        with pytest.raises(rt.B200RTError, match="material 1 "):
            gpu_ctx.render(cam, env, 32, 32, 4, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, sampling=GR,
                                                                     sample_streams=2))
        m = rt.MultiContext([0, 0])
        try:
            fixtures.upload(m, bad, ibl)
            with pytest.raises(rt.B200RTError, match="material 1 "):
                m.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=GR))
            fixtures.upload(m, sc, ibl)
            m.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=GR))
        finally:
            m.close()
        # a bad roughness on pass-through glass (ior 1) is never read
        fixtures.upload(gpu_ctx, gs.glass_ior(bad, 1.0), ibl)
        gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=GR))
    # no leaked state: a render without the bit after one with it equals a fresh render without it, counters included
    fixtures.upload(gpu_ctx, sc, ibl)
    for base in (0, G | S | 2):
        fresh = rt.Context(0)
        try:
            fixtures.upload(fresh, sc, ibl)
            a = fresh.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=base))
            sa = fresh.stats()
        finally:
            fresh.close()
        gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=GR | S | 2))
        b = gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=base))
        sb = gpu_ctx.stats()
        assert np.array_equal(bits(a), bits(b))
        for key in ("rays", "samples", "wave_iterations", "kernel_launches"):
            assert sa[key] == sb[key], key
    want_plain, cnt_plain = oracle.render(sc, cam, env, 32 * 32, 2, 4, ibl)
    assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4)), bits(want_plain))
    assert gpu_ctx.stats()["rays"] == cnt_plain["rays"]
