"""GPU: opt-in smooth shading (B200RT_SAMPLING_SMOOTH_NORMALS) against the oracle, bit for bit, statistics included, on
the two fixture scenes with curved triangles; flat scenes unchanged; the G-buffer normal and the denoised render; every
path that carries the sampling mask (pixel ranges, tile rows, partial sample ranges, sample streams, the multi-GPU
handle, render_rgb8, render_adaptive, the launcher and progressive slices); its refusals."""
import numpy as np
import pytest

import ensem3a_openclraytracer_b200 as rt
from ensem3a_openclraytracer_b200.progressive import finalize
from oracle import oracle
from oracle_denoise import denoise as D
from oracle_smooth import smooth
from tests import fixtures, smooth_scene as ss

pytestmark = pytest.mark.gpu

S = rt.SAMPLING_SMOOTH_NORMALS
J = rt.SAMPLING_PIXEL_JITTER


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def setup(ctx, name, w, h=None):
    sc = fixtures.load_scene(name)
    ibl = fixtures.load_ibl()
    fixtures.upload(ctx, sc, ibl)
    cam, env = fixtures.cam_env(sc["params"], w, h)
    return sc, ibl, cam, env


def want_image(sc, cam, env, n_pix, spp, bounce, ibl, sampling, **kw):
    """the smooth oracle, which also states bits 0, 1 and 8"""
    return smooth.render(sc, cam, env, n_pix, spp, bounce, ibl, sampling=sampling, **kw)


def parts_image(sc, ibl, cam, env, n_pix, spp, n, seed, sampling):
    """the oracle's raw sums of the n contiguous sample ranges the library cuts [0, spp) into, added in part order and
    finalised; and the oracle's ray count"""
    base, extra = divmod(spp, n)
    total, rays, s0 = None, 0, 0
    for k in range(n):
        s1 = s0 + base + (1 if k < extra else 0)
        part, cnt = smooth.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=1, seed=seed, s0=s0, s1=s1, raw_sums=True,
                                  sampling=sampling)
        total = part if total is None else total + part
        rays += cnt["rays"] - (n_pix if k > 0 else 0)   # every part traces the primary rays; `rays` counts them once
        s0 = s1
    return np.fmax(np.fmin(total / np.float32(spp), np.float32(1)), np.float32(0)), rays


@pytest.mark.parametrize("name,res,rows", [("monkey_cfg2", 48, None), ("serre", 64, (24, 44))])
@pytest.mark.parametrize("sampling", [S, S | 1, S | 2, S | 3, S | J])
@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_smooth_equals_the_oracle_bit_for_bit(gpu_ctx, name, res, rows, sampling, rng):
    sc, ibl, cam, env = setup(gpu_ctx, name, res)
    spp, n_pix = 4, res * res
    i0, i1 = (rows[0] * res, rows[1] * res) if rows else (0, n_pix)
    for trav, bounce in ((rt.TRAVERSAL_FAST, 4), (rt.TRAVERSAL_REFERENCE, 1), (rt.TRAVERSAL_VERIFY, 2)):
        want, cnt = want_image(sc, cam, env, n_pix, spp, bounce, ibl, sampling, i0=i0, i1=i1, rng_mode=rng, seed=17)
        o = rt.make_opts(rng_mode=rng, seed=17, sampling=sampling, traversal=trav, pixel_begin=i0 if rows else 0,
                         pixel_end=i1 if rows else 0)
        got = gpu_ctx.render(cam, env, res, res, spp, bounce, opts=o)
        assert np.array_equal(bits(got[3 * i0:3 * i1]), bits(want[3 * i0:3 * i1]))
        st = gpu_ctx.stats()
        assert st["rays"] == cnt["rays"]
    # the bit moves the image off the faceted one
    plain, _ = want_image(sc, cam, env, n_pix, spp, 4, ibl, sampling & ~S, i0=i0, i1=i1, rng_mode=rng, seed=17)
    assert not np.array_equal(bits(plain[3 * i0:3 * i1]), bits(want[3 * i0:3 * i1]))


@pytest.mark.parametrize("name,ibl_name", [("cornell", "preview"), ("furnace_cfg3", "grey")])
def test_flat_scenes_render_the_same(gpu_ctx, name, ibl_name):
    sc, ibl = fixtures.load_scene(name), fixtures.load_ibl(ibl_name)
    fixtures.upload(gpu_ctx, sc, ibl)
    cam, env = fixtures.cam_env(sc["params"], 64)
    for base in (0, 3, J):
        for rng in (rt.RNG_REFERENCE, rt.RNG_PHILOX):
            a = gpu_ctx.render(cam, env, 64, 64, 4, 4, opts=rt.make_opts(rng_mode=rng, seed=3, sampling=base))
            b = gpu_ctx.render(cam, env, 64, 64, 4, 4, opts=rt.make_opts(rng_mode=rng, seed=3, sampling=base | S))
            assert np.array_equal(bits(a), bits(b))


@pytest.mark.parametrize("name", ["monkey_cfg2", "serre"])
def test_gbuffer_and_denoised_render(gpu_ctx, name):
    W, H = 80, 60
    sc, ibl, cam, env = setup(gpu_ctx, name, W, H)
    want = ss.gbuffer(sc, cam, W, H)
    for trav in (rt.TRAVERSAL_FAST, rt.TRAVERSAL_REFERENCE):
        gb = gpu_ctx.gbuffer(cam, W, H, opts=rt.make_opts(sampling=S, traversal=trav))
        for key in ("albedo", "normal", "position", "kind"):
            assert np.array_equal(np.asarray(gb[key]).view(np.uint32), np.asarray(want[key]).view(np.uint32)), key
    plain = gpu_ctx.gbuffer(cam, W, H)
    assert not np.array_equal(bits(plain["normal"]), bits(want["normal"]))
    assert np.array_equal(bits(gpu_ctx.gbuffer(cam, W, H, opts=rt.make_opts(sampling=J))["normal"]), bits(plain["normal"]))
    for o in (rt.make_opts(sampling=S), rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=2, sampling=S | 3, sample_streams=3)):
        den, noisy = gpu_ctx.render_denoised(cam, env, W, H, 6, 4, opts=o, return_noisy=True)
        assert np.array_equal(bits(noisy).reshape(-1), bits(gpu_ctx.render(cam, env, W, H, 6, 4, opts=o)).reshape(-1))
        ref = D.atrous(noisy.reshape(H, W, 3), want, bvh=sc["BVH"], **rt.DENOISE_DEFAULTS)
        assert np.array_equal(bits(den).reshape(-1), bits(ref).reshape(-1))


def test_tile_rows_and_pixel_range_reference_generator(gpu_ctx):
    W, H, spp = 72, 50, 5
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", W, H)
    want, _ = smooth.render(sc, cam, env, W * H, spp, 4, ibl, sampling=S)
    img = gpu_ctx.render(cam, env, W, H, spp, 4, opts=rt.make_opts(sampling=S, tile_row_mod=3, tile_row_rem=1))
    img = img.reshape(H, W, 3)
    rows = (np.arange(H) // 4) % 3 == 1
    assert np.array_equal(bits(img[rows]), bits(want.reshape(H, W, 3)[rows])) and not img[~rows].any()
    got = gpu_ctx.render(cam, env, W, H, spp, 4, opts=rt.make_opts(sampling=S | 2, pixel_begin=700, pixel_end=1900))
    want2, _ = smooth.render(sc, cam, env, W * H, spp, 4, ibl, sampling=S | 2, i0=700, i1=1900)
    assert np.array_equal(bits(got[3 * 700:3 * 1900]), bits(want2[3 * 700:3 * 1900]))


def test_partial_sample_range_sums(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", 48)
    for sampling in (S | 1, S | J):
        want, cnt = want_image(sc, cam, env, 48 * 48, 8, 4, ibl, sampling, rng_mode=1, seed=3, s0=2, s1=7,
                               raw_sums=True)
        got = gpu_ctx.render(cam, env, 48, 48, 8, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3, sampling=sampling,
                                                                       output=rt.OUT_SUMS, sample_begin=2, sample_end=7))
        assert np.array_equal(bits(got), bits(want))
        assert gpu_ctx.stats()["rays"] == cnt["rays"]


@pytest.mark.parametrize("streams", [3, -1])
def test_sample_streams_add_the_parts_in_order(gpu_ctx, streams):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", 48)
    spp = 8
    got = gpu_ctx.render(cam, env, 48, 48, spp, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=6, sampling=S | 2,
                                                                     sample_streams=streams))
    st = gpu_ctx.stats()
    n = st["sample_streams"]
    assert n > 1
    want, rays = parts_image(sc, ibl, cam, env, 48 * 48, spp, n, 6, S | 2)
    assert np.array_equal(bits(got), bits(want))
    assert st["rays"] == rays


@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_multi_handle(rng):
    """MultiContext over every visible GPU, or three entries on GPU 0 when there is one"""
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    cam, env = fixtures.cam_env(sc["params"], 64, 48)
    n = rt.device_count()
    devices = list(range(n)) if n >= 2 else [0, 0, 0]
    if rng == rt.RNG_REFERENCE:   # tile rows: every pixel's samples on one GPU
        want, _ = smooth.render(sc, cam, env, 64 * 48, 6, 4, ibl, rng_mode=rng, seed=8, sampling=S)
    else:                         # sample ranges, added in GPU order
        want, _ = parts_image(sc, ibl, cam, env, 64 * 48, 6, min(len(devices), 6), 8, S)
    m = rt.MultiContext(devices)
    try:
        fixtures.upload(m, sc, ibl)
        got = m.render(cam, env, 64, 48, 6, 4, opts=rt.make_opts(rng_mode=rng, seed=8, sampling=S))
        assert np.array_equal(bits(got.reshape(-1)), bits(want))
    finally:
        m.close()


def test_rgb8_and_adaptive(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", 64)
    o = rt.make_opts(sampling=S | 1)
    img = gpu_ctx.render(cam, env, 64, 64, 6, 4, opts=o)
    q = gpu_ctx.render_rgb8(cam, env, 64, 64, 6, 4, opts=o)
    assert np.array_equal(q.reshape(-1), (img * np.float32(255)).astype(np.uint8))
    ad = dict(rel_error=0.2, min_spp=4, check_every=2)
    for rng, sampling in ((rt.RNG_REFERENCE, S), (rt.RNG_PHILOX, S | 2)):
        want, n_want, err_want, cnt = smooth.render(sc, cam, env, 64 * 64, 16, 4, ibl, rng_mode=rng, seed=4,
                                                    sampling=sampling, adaptive=ad)
        got, n_got, err_got = gpu_ctx.render_adaptive(cam, env, 64, 64, 16, 4, opts=rt.make_opts(rng_mode=rng, seed=4,
                                                                                               sampling=sampling), **ad)
        assert np.array_equal(bits(got.reshape(-1)), bits(want))
        assert np.array_equal(n_got.reshape(-1), n_want) and np.array_equal(bits(err_got.reshape(-1)), bits(err_want))
        assert gpu_ctx.stats()["rays"] == cnt["rays"]
        assert (n_want < 16).any()
    with pytest.raises(rt.B200RTError, match="PIXEL_JITTER"):
        gpu_ctx.render_adaptive(cam, env, 64, 64, 8, 4, opts=rt.make_opts(sampling=S | J), **ad)


def test_launcher_attribute_and_environment(monkeypatch):
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    res, spp = 48, 4
    cam, env = fixtures.cam_env(sc["params"], res)
    args = (sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"], sc["BVH"], cam, env,
            res * res, spp, 4, ibl)
    for var in ("B200RT_ADAPTIVE", "B200RT_DENOISE", "B200RT_CUDA_DEVICES", "B200RT_PIXEL_JITTER"):
        monkeypatch.delenv(var, raising=False)
    ctx = rt.Context(0)
    fixtures.upload(ctx, sc, ibl)
    want = ctx.render(cam, env, res, res, spp, 4, opts=rt.make_opts(sampling=S))
    plain = ctx.render(cam, env, res, res, spp, 4)
    both = ctx.render(cam, env, res, res, spp, 4, opts=rt.make_opts(sampling=S | J))
    ctx.close()
    monkeypatch.setenv("B200RT_SMOOTH_NORMALS", "1")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.smooth_normals is True
    out = np.zeros(res * res * 3, np.float32)
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(want))
    kl.pixel_jitter = True
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(both))
    kl.pixel_jitter = False
    kl.smooth_normals = False
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(plain))
    kl.smooth_normals = True
    kl.denoise = {}
    kl.launch_Raytracing(out, *args)
    assert kl.last_stats["kernel_launches"] > 0 and not np.array_equal(bits(out), bits(want))
    kl.close()
    monkeypatch.setenv("B200RT_SMOOTH_NORMALS", "0")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.smooth_normals is False
    kl.close()
    monkeypatch.setenv("B200RT_SMOOTH_NORMALS", "yes")
    with pytest.raises(ValueError):
        rt.KernelLauncher(None, None, None, None)


def test_progressive_slices(gpu_ctx):
    W, H = 64, 48
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", W, H)
    pr = rt.ProgressiveRender(gpu_ctx, cam, env, W, H, 40, 4, slice_spp=16, seed=3, sampling=S)
    for _ in pr:
        pass
    one = gpu_ctx.render(cam, env, W, H, 40, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3, sampling=S))
    rel = np.abs(pr.image() - one) / np.maximum(np.abs(one), 1e-3)
    assert rel.max() <= 1e-4
    pd = rt.ProgressiveRender(gpu_ctx, cam, env, W, H, 16, 4, slice_spp=16, seed=3, sampling=S, denoise={})
    img = next(pd)
    want = gpu_ctx.denoise(finalize(pd.sums, 16).reshape(H, W, 3), ss.gbuffer(sc, cam, W, H))
    assert np.array_equal(bits(img), bits(want.reshape(-1)))


def test_refusals(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", 32)
    for bad in (16, 48, 36, 64, -32):
        with pytest.raises(rt.B200RTError, match="sampling"):
            gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=bad))
    # an out-of-range n1 index: the scene loads and renders plainly; only a smooth-shaded frame refuses it
    bad = dict(sc)
    face = sc["faceData"].copy().reshape(-1, 10)
    face[123, 5] = sc["V_n"].size // 3 + 7
    face[300, 6] = -1
    bad["faceData"] = face.reshape(-1)
    fixtures.upload(gpu_ctx, bad, ibl)
    want, _ = oracle.render(sc, cam, env, 32 * 32, 2, 4, ibl)
    assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4)), bits(want))
    gpu_ctx.primary_hits(cam, 32, 32, opts=rt.make_opts(sampling=S))
    for call in (lambda o: gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=o),
                 lambda o: gpu_ctx.gbuffer(cam, 32, 32, opts=o),
                 lambda o: gpu_ctx.render_denoised(cam, env, 32, 32, 2, 4, opts=o)):
        with pytest.raises(rt.B200RTError, match="triangle 123"):
            call(rt.make_opts(sampling=S))
    fixtures.upload(gpu_ctx, sc, ibl)
    gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=S))
