"""GPU: opt-in albedo textures (B200RT_SAMPLING_TEXTURES) against the texture oracle, bit for bit, ray counts included,
on the bench scene (config 2) and the Cornell box with generated textures on every diffuse and glossy material; adaptive
renders, sample streams, the multi-GPU handle, the G-buffer and the denoised render; the refusals; no state left
behind; the launcher and progressive slices."""
import ctypes

import numpy as np
import pytest

import ensem3a_openclraytracer_b200 as rt
from oracle import oracle
from oracle_denoise import denoise as D
from oracle_texture import texture
from tests import fixtures, texture_scene as ts

pytestmark = pytest.mark.gpu

X = rt.SAMPLING_TEXTURES
G = rt.SAMPLING_DIELECTRIC_GLASS
S = rt.SAMPLING_SMOOTH_NORMALS
J = rt.SAMPLING_PIXEL_JITTER


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def setup(ctx, name, w, h=None, size=32):
    sc = fixtures.load_scene(name)
    ibl = fixtures.load_ibl()
    fixtures.upload(ctx, sc, ibl)
    tex = ts.textured(sc, size)
    ctx.set_textures(tex)
    cam, env = fixtures.cam_env(sc["params"], w, h)
    return sc, ibl, tex, cam, env


def parts_image(sc, ibl, tex, cam, env, n_pix, spp, n, seed, sampling):
    """the oracle's raw sums of the n contiguous sample ranges the library cuts [0, spp) into, added in part order and
    finalised; and the oracle's ray count"""
    base, extra = divmod(spp, n)
    total, rays, s0 = None, 0, 0
    for k in range(n):
        s1 = s0 + base + (1 if k < extra else 0)
        part, cnt = texture.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=1, seed=seed, s0=s0, s1=s1, raw_sums=True,
                                   sampling=sampling, textures=tex)
        total = part if total is None else total + part
        rays += cnt["rays"] - (n_pix if k > 0 else 0)   # every part traces the primary rays; `rays` counts them once
        s0 = s1
    return np.fmax(np.fmin(total / np.float32(spp), np.float32(1)), np.float32(0)), rays


@pytest.mark.parametrize("name,res", [("monkey_cfg2", 48), ("cornell", 40)])
@pytest.mark.parametrize("sampling", [X, X | 1, X | 2, X | 3, X | J, X | S, X | G, X | S | G | 2])
@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_textures_equal_the_oracle_bit_for_bit(gpu_ctx, name, res, sampling, rng):
    sc, ibl, tex, cam, env = setup(gpu_ctx, name, res)
    spp, n_pix = 4, res * res
    for trav, bounce in ((rt.TRAVERSAL_FAST, 4), (rt.TRAVERSAL_REFERENCE, 1)):
        want, cnt = texture.render(sc, cam, env, n_pix, spp, bounce, ibl, rng_mode=rng, seed=17, sampling=sampling,
                                   textures=tex)
        got = gpu_ctx.render(cam, env, res, res, spp, bounce,
                             opts=rt.make_opts(rng_mode=rng, seed=17, sampling=sampling, traversal=trav))
        assert np.array_equal(bits(got), bits(want))
        assert gpu_ctx.stats()["rays"] == cnt["rays"]
    # the textures move the image; the counters stay
    plain = gpu_ctx.render(cam, env, res, res, spp, 4, opts=rt.make_opts(rng_mode=rng, seed=17, sampling=sampling & ~X))
    want4, cnt4 = texture.render(sc, cam, env, n_pix, spp, 4, ibl, rng_mode=rng, seed=17, sampling=sampling, textures=tex)
    assert not np.array_equal(bits(plain), bits(want4))
    assert gpu_ctx.stats()["rays"] == cnt4["rays"]


def test_nothing_bound_renders_as_without_the_bit(gpu_ctx):
    sc, ibl, tex, cam, env = setup(gpu_ctx, "monkey_cfg2", 48)
    gpu_ctx.set_textures(None)
    for base in (0, 3, J, S | G):
        a = gpu_ctx.render(cam, env, 48, 48, 4, 4, opts=rt.make_opts(rng_mode=1, seed=3, sampling=base))
        ra = gpu_ctx.stats()["rays"]
        b = gpu_ctx.render(cam, env, 48, 48, 4, 4, opts=rt.make_opts(rng_mode=1, seed=3, sampling=base | X))
        assert np.array_equal(bits(a), bits(b)) and gpu_ctx.stats()["rays"] == ra
    gpu_ctx.set_textures(tex)   # bindings survive scene and material uploads
    fixtures.upload(gpu_ctx, sc, ibl)
    gpu_ctx.set_materials(sc["materialData"])
    want, _ = texture.render(sc, cam, env, 48 * 48, 4, 4, ibl, rng_mode=1, seed=3, sampling=X, textures=tex)
    got = gpu_ctx.render(cam, env, 48, 48, 4, 4, opts=rt.make_opts(rng_mode=1, seed=3, sampling=X))
    assert np.array_equal(bits(got), bits(want))


@pytest.mark.parametrize("streams", [3, -1])
def test_sample_streams_add_the_parts_in_order(gpu_ctx, streams):
    sc, ibl, tex, cam, env = setup(gpu_ctx, "monkey_cfg2", 48)
    spp = 8
    got = gpu_ctx.render(cam, env, 48, 48, spp, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=6, sampling=X | 2,
                                                                     sample_streams=streams))
    st = gpu_ctx.stats()
    n = st["sample_streams"]
    assert n > 1
    want, rays = parts_image(sc, ibl, tex, cam, env, 48 * 48, spp, n, 6, X | 2)
    assert np.array_equal(bits(got), bits(want))
    assert st["rays"] == rays


@pytest.mark.parametrize("rng", [rt.RNG_REFERENCE, rt.RNG_PHILOX])
def test_multi_handle(rng):
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    tex = ts.textured(sc, 32)
    cam, env = fixtures.cam_env(sc["params"], 64, 48)
    if rng == rt.RNG_REFERENCE:   # tile rows: every pixel's samples on one GPU
        want, _ = texture.render(sc, cam, env, 64 * 48, 6, 4, ibl, rng_mode=rng, seed=8, sampling=X, textures=tex)
    else:                         # sample ranges, added in GPU order
        want, _ = parts_image(sc, ibl, tex, cam, env, 64 * 48, 6, 2, 8, X)
    m = rt.MultiContext([0, 0])
    try:
        fixtures.upload(m, sc, ibl)
        m.set_textures(tex)
        got = m.render(cam, env, 64, 48, 6, 4, opts=rt.make_opts(rng_mode=rng, seed=8, sampling=X))
        assert np.array_equal(bits(got.reshape(-1)), bits(want))
        gb = D.gbuffer(sc, cam, 64, 48)
        p = oracle.primary(sc, cam, 64 * 48)
        gb["albedo"] = texture.gbuffer_albedo(sc, cam, p["tri"], p["k"], tex).reshape(48, 64, 3)
        den, noisy = m.render_denoised(cam, env, 64, 48, 6, 4, opts=rt.make_opts(rng_mode=rng, seed=8, sampling=X),
                                       return_noisy=True)
        assert np.array_equal(bits(noisy.reshape(-1)), bits(want))
        ref = D.atrous(noisy, gb, bvh=sc["BVH"], **rt.DENOISE_DEFAULTS)
        assert np.array_equal(bits(den), bits(ref))
    finally:
        m.close()


def test_adaptive_gbuffer_and_denoised(gpu_ctx):
    W, H = 64, 48
    sc, ibl, tex, cam, env = setup(gpu_ctx, "monkey_cfg2", W, H)
    ad = dict(rel_error=0.2, min_spp=4, check_every=2)
    for rng, sampling in ((rt.RNG_REFERENCE, X), (rt.RNG_PHILOX, X | S | G | 2)):
        want, n_want, err_want, cnt = texture.render(sc, cam, env, W * H, 16, 4, ibl, rng_mode=rng, seed=4,
                                                     sampling=sampling, adaptive=ad, textures=tex)
        got, n_got, err_got = gpu_ctx.render_adaptive(cam, env, W, H, 16, 4, opts=rt.make_opts(rng_mode=rng, seed=4,
                                                                                             sampling=sampling), **ad)
        assert np.array_equal(bits(got.reshape(-1)), bits(want))
        assert np.array_equal(n_got.reshape(-1), n_want) and np.array_equal(bits(err_got.reshape(-1)), bits(err_want))
        assert gpu_ctx.stats()["rays"] == cnt["rays"]
    gb = D.gbuffer(sc, cam, W, H)
    p = oracle.primary(sc, cam, W * H)
    alb = texture.gbuffer_albedo(sc, cam, p["tri"], p["k"], tex).reshape(H, W, 3)
    got = gpu_ctx.gbuffer(cam, W, H, opts=rt.make_opts(sampling=X))
    assert np.array_equal(bits(got["albedo"]), bits(alb))
    assert not np.array_equal(bits(alb), bits(gb["albedo"]))
    plain = gpu_ctx.gbuffer(cam, W, H)
    assert np.array_equal(bits(plain["albedo"]), bits(gb["albedo"]))
    gb["albedo"] = alb
    for o in (rt.make_opts(sampling=X), rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=2, sampling=X | 3, sample_streams=3)):
        den, noisy = gpu_ctx.render_denoised(cam, env, W, H, 6, 4, opts=o, return_noisy=True)
        assert np.array_equal(bits(noisy).reshape(-1), bits(gpu_ctx.render(cam, env, W, H, 6, 4, opts=o)).reshape(-1))
        ref = D.atrous(noisy.reshape(H, W, 3), gb, bvh=sc["BVH"], **rt.DENOISE_DEFAULTS)
        assert np.array_equal(bits(den).reshape(-1), bits(ref).reshape(-1))
    q = gpu_ctx.render_rgb8(cam, env, W, H, 6, 4, opts=rt.make_opts(sampling=X))
    img = gpu_ctx.render(cam, env, W, H, 6, 4, opts=rt.make_opts(sampling=X))
    assert np.array_equal(q.reshape(-1), (img * np.float32(255)).astype(np.uint8))


def _raw_set_textures(ctx, texels, n_bytes, dims, n_tex, mat_tex, n_mat):
    lib = ctx._lib
    p = lambda a: None if a is None else a.ctypes.data_as(ctypes.c_void_p)
    rc = lib.b200rt_set_textures(ctx._h, p(texels), n_bytes, p(dims), n_tex, p(mat_tex), n_mat)
    return rc, lib.b200rt_last_error(ctx._h).decode()


def test_refusals_and_no_leaked_state(gpu_ctx):
    sc, ibl, tex, cam, env = setup(gpu_ctx, "cornell", 32)
    px = np.zeros(2 * 3 * 4, np.uint8)
    dims = np.array([2, 3], np.int32)
    mt = np.array([0, -1], np.int32)
    assert _raw_set_textures(gpu_ctx, px, px.size, dims, 1, mt, 2)[0] == 0
    for args, code, msg in (
            ((None, 24, dims, 1, mt, 2), -1, "NULL"),
            ((px, 24, None, 1, mt, 2), -1, "NULL"),
            ((px, 24, dims, 1, None, 2), -1, "NULL"),
            ((px, 24, dims, -1, mt, 2), -1, "negative"),
            ((px, 20, dims, 1, mt, 2), -1, "texel bytes"),
            ((px, 24, np.array([0, 3], np.int32), 1, mt, 2), -1, "0 x 3"),
            ((px, 24, dims, 1, np.array([1, -1], np.int32), 2), -1, "material 0"),
            ((px, 24, dims, 1, np.array([0, -2], np.int32), 2), -1, "material 1"),
            ((px, 24, np.array([1 << 25, 1], np.int32), 1, mt, 2), -4, "2^24"),
            ((px, 24, np.array([1 << 24, 1 << 8], np.int32), 1, mt, 2), -4, "2^31")):
        rc, err = _raw_set_textures(gpu_ctx, *args)
        assert rc == code and msg in err, (args, rc, err)
    for bad in (np.zeros((2, 2), np.uint8), np.zeros((2, 2, 4), np.float32), np.zeros((0, 2, 4), np.uint8)):
        with pytest.raises(rt.B200RTError):
            gpu_ctx.set_textures({0: bad})
    with pytest.raises(rt.B200RTError):
        gpu_ctx.set_textures({-1: np.zeros((2, 2, 4), np.uint8)})
    # a scene with an out-of-range UV index loads and renders without the bit, and is refused with it
    want_plain, cnt_plain = oracle.render(sc, cam, env, 32 * 32, 2, 4, ibl)
    bad = dict(sc, faceData=sc["faceData"].copy())
    bad["faceData"][10 * 7 + 2] = sc["V_uv"].size // 2
    gpu_ctx.set_textures(tex)
    fixtures.upload(gpu_ctx, bad, ibl)
    assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4)), bits(want_plain))
    gpu_ctx.primary_hits(cam, 32, 32, opts=rt.make_opts(sampling=X))
    calls = (lambda o: gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=o),
             lambda o: gpu_ctx.render_rgb8(cam, env, 32, 32, 2, 4, opts=o),
             lambda o: gpu_ctx.render_adaptive(cam, env, 32, 32, 4, 4, opts=o, rel_error=0.1, min_spp=2),
             lambda o: gpu_ctx.render_denoised(cam, env, 32, 32, 2, 4, opts=o),
             lambda o: gpu_ctx.gbuffer(cam, 32, 32, opts=o),
             lambda o: gpu_ctx.render(cam, env, 32, 32, 4, 4, opts=rt.make_opts(
                 rng_mode=rt.RNG_PHILOX, sampling=o.sampling, sample_streams=2)))
    for call in calls:
        with pytest.raises(rt.B200RTError, match="triangle 7"):
            call(rt.make_opts(sampling=X))
    m = rt.MultiContext([0, 0])
    try:
        fixtures.upload(m, bad, ibl)
        with pytest.raises(rt.B200RTError, match="triangle 7"):
            m.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=X))
        fixtures.upload(m, sc, ibl)
        m.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=X))
    finally:
        m.close()
    # no leaked state: a default render after a textured one is the plain oracle's, ray count included
    fixtures.upload(gpu_ctx, sc, ibl)
    want, _ = texture.render(sc, cam, env, 32 * 32, 2, 4, ibl, sampling=X | 2, textures=tex)
    assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4, opts=rt.make_opts(sampling=X | 2))), bits(want))
    assert np.array_equal(bits(gpu_ctx.render(cam, env, 32, 32, 2, 4)), bits(want_plain))
    assert gpu_ctx.stats()["rays"] == cnt_plain["rays"]


def test_launcher_and_progressive(gpu_ctx, monkeypatch, tmp_path):
    from PIL import Image
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    res, spp = 48, 4
    cam, env = fixtures.cam_env(sc["params"], res)
    args = (sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"], sc["BVH"], cam, env,
            res * res, spp, 4, ibl)
    for var in ("B200RT_ADAPTIVE", "B200RT_DENOISE", "B200RT_CUDA_DEVICES", "B200RT_PIXEL_JITTER",
                "B200RT_SMOOTH_NORMALS", "B200RT_DIELECTRIC_GLASS", "B200RT_TEXTURES"):
        monkeypatch.delenv(var, raising=False)
    tex = {0: ts.noise(32, 1), 4: ts.noise(16, 2)}
    Image.fromarray(tex[0]).save(tmp_path / "a.png")
    Image.fromarray(tex[4][..., :3]).save(tmp_path / "b.png")
    want, _ = texture.render(sc, cam, env, res * res, spp, 4, ibl, sampling=X, textures=tex)
    plain, _ = oracle.render(sc, cam, env, res * res, spp, 4, ibl)
    monkeypatch.setenv("B200RT_TEXTURES", f"0={tmp_path / 'a.png'},4={tmp_path / 'b.png'}")
    kl = rt.KernelLauncher(None, None, None, None)
    out = np.zeros(res * res * 3, np.float32)
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(want))
    kl.textures = None   # unbinds: the reference's image again
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(plain))
    kl.close()
    W, H = 64, 48
    cam, env = fixtures.cam_env(sc["params"], W, H)
    fixtures.upload(gpu_ctx, sc, ibl)
    gpu_ctx.set_textures(tex)
    pr = rt.ProgressiveRender(gpu_ctx, cam, env, W, H, 8, 4, slice_spp=8, seed=3, sampling=X)
    for _ in pr:
        pass
    want, _ = texture.render(sc, cam, env, W * H, 8, 4, ibl, rng_mode=1, seed=3, sampling=X, textures=tex)
    assert np.array_equal(bits(pr.image()), bits(want))
