"""GPU: the denoiser (b200rt_gbuffer, b200rt_denoise, b200rt_render_denoised, b200rt_multi_render_denoised) against its
numpy restatement (oracle_denoise/), bit for bit — G-buffers of every fixture scene, the filter over rendered and random
images, odd frame sizes and every pass count; the fused render against denoise(render, gbuffer) with its statistics; the
refused arguments; the error it removes; the multi-GPU handle; the launcher and progressive previews."""
import ctypes

import numpy as np
import pytest

import ensem3a_openclraytracer_b200 as rt
from oracle_denoise import denoise as D
from tests import fixtures

pytestmark = pytest.mark.gpu

VARIANTS = ["cornell", "monkey", "monkey_cfg2", "furnace", "furnace_cfg3", "serre", "proto", "single"]
DEFAULTS = rt.DENOISE_DEFAULTS
OTHER = dict(passes=3, sigma_color=0.2, sigma_normal=0.5, sigma_position=0.05)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def setup(ctx, name, ibl_name, w, h=None):
    sc, ibl = fixtures.load_scene(name), fixtures.load_ibl(ibl_name)
    fixtures.upload(ctx, sc, ibl)
    cam, env = fixtures.cam_env(sc["params"], w, h)
    return sc, ibl, cam, env


def assert_same_gbuffer(got, want):
    assert np.array_equal(got["kind"], want["kind"])
    for k in ("albedo", "normal", "position"):
        assert np.array_equal(bits(got[k]), bits(want[k])), k


@pytest.mark.parametrize("trav", [rt.TRAVERSAL_FAST, rt.TRAVERSAL_REFERENCE])
@pytest.mark.parametrize("name", VARIANTS)
def test_gbuffer_equals_the_restatement(gpu_ctx, name, trav):
    sc, ibl, cam, env = setup(gpu_ctx, name, "preview", 96, 64)
    gb = gpu_ctx.gbuffer(cam, 96, 64, opts=rt.make_opts(traversal=trav))
    assert_same_gbuffer(gb, D.gbuffer(sc, cam, 96, 64))
    st = gpu_ctx.stats()
    assert st["kernel_launches"] == 2 and st["rays"] == 96 * 64 and st["primary_rays"] == 96 * 64


@pytest.mark.parametrize("name,ibl_name,w,h", [("cornell", "preview", 128, 96), ("monkey_cfg2", "preview", 120, 90),
                                               ("furnace_cfg3", "grey", 100, 80), ("serre", "preview", 112, 84)])
def test_denoise_of_a_render_equals_the_restatement(gpu_ctx, name, ibl_name, w, h):
    sc, ibl, cam, env = setup(gpu_ctx, name, ibl_name, w, h)
    img = gpu_ctx.render(cam, env, w, h, 8, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=3)).reshape(h, w, 3)
    gb = gpu_ctx.gbuffer(cam, w, h)
    for params in (DEFAULTS, OTHER):
        got = gpu_ctx.denoise(img, gb, **params)
        assert gpu_ctx.stats()["kernel_launches"] == params["passes"]
        assert np.array_equal(bits(got), bits(D.atrous(img, gb, bvh=sc["BVH"], **params)))
        assert not np.array_equal(bits(got), bits(img))


def random_case(seed, w, h):
    rng = np.random.default_rng(seed)
    kind = rng.choice([-1, 0, 1, 1, 1, 1], size=(h, w)).astype(np.int32)
    n = rng.normal(size=(h, w, 3)).astype(np.float32)
    n /= np.linalg.norm(n, axis=2, keepdims=True).astype(np.float32)
    n[rng.random((h, w)) < 0.05] = np.nan
    albedo = rng.random((h, w, 3), dtype=np.float32)
    albedo[rng.random((h, w)) < 0.05] = 0
    img = (rng.random((h, w, 3), dtype=np.float32) * np.float32(1.2)).astype(np.float32)
    img[rng.random((h, w)) < 0.01] = np.nan
    pos = (rng.random((h, w, 3), dtype=np.float32) * np.float32(4)).astype(np.float32)
    return img, {"kind": kind, "albedo": albedo, "normal": n, "position": pos}


@pytest.mark.parametrize("w,h", [(97, 61), (33, 5), (1, 1), (3, 130)])
def test_denoise_of_random_images_equals_the_restatement(gpu_ctx, w, h):
    img, gb = random_case(w * 1000 + h, w, h)
    for params in (dict(DEFAULTS, sigma_position=0.3), OTHER, dict(passes=2, sigma_color=1e3, sigma_normal=1e-3, sigma_position=1e-4)):
        got = gpu_ctx.denoise(img, gb, **params)
        assert np.array_equal(bits(got), bits(D.atrous(img, gb, **params)))


@pytest.mark.parametrize("passes", range(1, 9))
def test_every_pass_count_including_steps_wider_than_the_frame(gpu_ctx, passes):
    img, gb = random_case(passes, 97, 61)
    params = dict(passes=passes, sigma_color=0.7, sigma_normal=0.3, sigma_position=0.5)
    got = gpu_ctx.denoise(img, gb, **params)
    assert np.array_equal(bits(got), bits(D.atrous(img, gb, **params)))


@pytest.mark.parametrize("rng,sampling,streams,trav", [
    (rt.RNG_REFERENCE, 0, 0, rt.TRAVERSAL_FAST),
    (rt.RNG_REFERENCE, 1, 0, rt.TRAVERSAL_REFERENCE),
    (rt.RNG_PHILOX, 2, -1, rt.TRAVERSAL_FAST),
    (rt.RNG_PHILOX, 3, -1, rt.TRAVERSAL_REFERENCE),
    (rt.RNG_PHILOX, 0, 4, rt.TRAVERSAL_FAST),
])
def test_render_denoised_is_denoise_of_render(gpu_ctx, rng, sampling, streams, trav):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", "preview", 80, 60)
    o = rt.make_opts(rng_mode=rng, seed=9, sampling=sampling, sample_streams=streams, traversal=trav)
    plain = gpu_ctx.render(cam, env, 80, 60, 8, 4, opts=o)
    st0 = gpu_ctx.stats()
    img, noisy = gpu_ctx.render_denoised(cam, env, 80, 60, 8, 4, opts=o, return_noisy=True)
    st1 = gpu_ctx.stats()
    assert np.array_equal(bits(noisy.reshape(-1)), bits(plain))
    assert st1["kernel_launches"] == st0["kernel_launches"] + 2 + DEFAULTS["passes"]
    assert st1["rays"] == st0["rays"] + 80 * 60
    assert st1["primary_rays"] == st0["primary_rays"] + 80 * 60
    assert st1["samples"] == st0["samples"] and st1["sample_streams"] == st0["sample_streams"]
    gb = gpu_ctx.gbuffer(cam, 80, 60, opts=o)
    assert np.array_equal(bits(img), bits(gpu_ctx.denoise(plain.reshape(60, 80, 3), gb)))
    assert np.array_equal(bits(img), bits(gpu_ctx.render_denoised(cam, env, 80, 60, 8, 4, opts=o)))
    # a plain render after a denoised one is unchanged, launches included
    again = gpu_ctx.render(cam, env, 80, 60, 8, 4, opts=o)
    assert np.array_equal(bits(again), bits(plain))
    assert gpu_ctx.stats()["kernel_launches"] == st0["kernel_launches"]


def test_refused_arguments(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 32)
    bad_opts = [rt.make_opts(output=rt.OUT_SUMS),
                rt.make_opts(rng_mode=rt.RNG_PHILOX, output=rt.OUT_SUMS, sample_begin=0, sample_end=8),
                rt.make_opts(rng_mode=rt.RNG_PHILOX, sample_begin=4, sample_end=16),
                rt.make_opts(pixel_begin=0, pixel_end=100),
                rt.make_opts(tile_row_mod=2, tile_row_rem=1)]
    for o in bad_opts:
        with pytest.raises(rt.B200RTError, match="b200rt_render_denoised"):
            gpu_ctx.render_denoised(cam, env, 32, 32, 16, 4, opts=o)
    nan, inf = float("nan"), float("inf")
    bad_params = [dict(passes=0), dict(passes=9), dict(sigma_color=0), dict(sigma_color=-1), dict(sigma_color=nan),
                  dict(sigma_color=inf), dict(sigma_normal=0), dict(sigma_normal=nan), dict(sigma_normal=inf),
                  dict(sigma_position=nan), dict(sigma_position=inf), dict(sigma_position=-inf)]
    for p in bad_params:
        with pytest.raises(rt.B200RTError, match="b200rt_render_denoised"):
            gpu_ctx.render_denoised(cam, env, 32, 32, 16, 4, **p)
    for o in bad_opts[3:]:
        with pytest.raises(rt.B200RTError, match="b200rt_gbuffer"):
            gpu_ctx.gbuffer(cam, 32, 32, opts=o)
    gb = gpu_ctx.gbuffer(cam, 32, 32)
    img = np.zeros((32, 32, 3), np.float32)
    for p in bad_params:
        with pytest.raises(rt.B200RTError, match="b200rt_denoise"):
            gpu_ctx.denoise(img, gb, **p)
    for k in (2, -2):
        bad = dict(gb, kind=gb["kind"].copy())
        bad["kind"][3, 4] = k
        with pytest.raises(rt.B200RTError, match="kind"):
            gpu_ctx.denoise(img, bad)
    lib = rt.load_library()
    out = np.zeros(32 * 32 * 3, np.float32)
    cam_, env_ = np.ascontiguousarray(cam), np.ascontiguousarray(env)
    o = rt.make_opts()
    rc = lib.b200rt_render_denoised(gpu_ctx._h, cam_.ctypes.data_as(ctypes.c_void_p), env_.ctypes.data_as(ctypes.c_void_p),
                                    32, 32, 16, 4, ctypes.byref(o), None, out.ctypes.data_as(ctypes.c_void_p), None)
    assert rc == -1 and b"NULL" in lib.b200rt_last_error(gpu_ctx._h)
    # the whole sample range spelled out is accepted, and the filter may write over its input
    gpu_ctx.render_denoised(cam, env, 32, 32, 16, 4, opts=rt.make_opts(sample_begin=0, sample_end=16))
    src = gpu_ctx.render(cam, env, 32, 32, 4, 2).reshape(32, 32, 3)
    want = gpu_ctx.denoise(src, gb)
    dn = rt.Denoise(5, 0.5, 0.2, 0.0)
    k = np.ascontiguousarray(gb["kind"])
    ptr = [np.ascontiguousarray(a).ctypes.data_as(ctypes.c_void_p) for a in (src, gb["albedo"], gb["normal"], gb["position"], k)]
    assert lib.b200rt_denoise(gpu_ctx._h, *ptr, 32, 32, ctypes.byref(dn), ptr[0]) == 0
    assert np.array_equal(bits(src), bits(want))


def test_denoised_is_closer_to_the_converged_image(gpu_ctx):
    """Cornell 128x128, 16 spp Philox, against a 2048-spp render, default parameters: RMSE noisy 0.0429, denoised 0.0147
    (measured on one NVIDIA B200 at a 1 000 W power limit)."""
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 128)
    truth = gpu_ctx.render(cam, env, 128, 128, 2048, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=100, sample_streams=-1))
    img, noisy = gpu_ctx.render_denoised(cam, env, 128, 128, 16, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=1),
                                         return_noisy=True)
    rmse_noisy = float(np.sqrt(np.mean((noisy.reshape(-1) - truth) ** 2)))
    rmse_den = float(np.sqrt(np.mean((img.reshape(-1) - truth) ** 2)))
    print(f"cornell 128^2 16 spp: RMSE noisy {rmse_noisy:.4f}, denoised {rmse_den:.4f}")
    assert rmse_den < 0.75 * rmse_noisy


def test_multi_gpu_handle_equals_denoise_of_its_render():
    if rt.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    m = rt.MultiContext([0, 1])
    fixtures.upload(m, sc, ibl)
    cam, env = fixtures.cam_env(sc["params"], 72, 56)
    for o in (rt.make_opts(), rt.make_opts(rng_mode=rt.RNG_PHILOX, seed=4, sampling=3)):
        plain = m.render(cam, env, 72, 56, 8, 4, opts=o)
        st0 = m.stats()
        img, noisy = m.render_denoised(cam, env, 72, 56, 8, 4, opts=o, return_noisy=True, **OTHER)
        st1 = m.stats()
        assert np.array_equal(bits(noisy.reshape(-1)), bits(plain))
        assert st1["kernel_launches"] == st0["kernel_launches"] + 2 + OTHER["passes"]
        assert st1["rays"] == st0["rays"] + 72 * 56
        gb = m.contexts[0].gbuffer(cam, 72, 56, opts=o)
        assert np.array_equal(bits(img), bits(m.contexts[0].denoise(plain.reshape(56, 72, 3), gb, **OTHER)))
    with pytest.raises(rt.B200RTError, match="b200rt_multi_render_denoised"):
        m.render_denoised(cam, env, 72, 56, 8, 4, opts=rt.make_opts(pixel_begin=0, pixel_end=10))
    m.close()


def test_kernel_launcher_denoise(monkeypatch):
    sc = fixtures.load_scene("monkey_cfg2")
    ibl = fixtures.load_ibl()
    res, spp = 64, 8
    cam, env = fixtures.cam_env(sc["params"], res)
    monkeypatch.delenv("B200RT_ADAPTIVE", raising=False)
    monkeypatch.setenv("B200RT_DENOISE", "3,0.4")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.denoise == dict(DEFAULTS, passes=3, sigma_color=0.4)
    out = np.zeros(res * res * 3, np.float32)
    args = (sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"], sc["BVH"], cam, env,
            res * res, spp, 4, ibl)
    kl.launch_Raytracing(out, *args)
    ctx = rt.Context(0)
    fixtures.upload(ctx, sc, ibl)
    want = ctx.render_denoised(cam, env, res, res, spp, 4, passes=3, sigma_color=0.4)
    assert np.array_equal(bits(out), bits(want.reshape(-1)))
    assert kl.last_stats["kernel_launches"] == ctx.stats()["kernel_launches"]
    kl.adaptive = dict(rel_error=0.1)
    with pytest.raises(ValueError, match="cannot be combined"):
        kl.launch_Raytracing(out, *args)
    kl.adaptive = None
    kl.denoise = None
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(ctx.render(cam, env, res, res, spp, 4)))
    monkeypatch.setenv("B200RT_DENOISE", "1")
    assert rt.KernelLauncher(None, None, None, None).denoise == DEFAULTS
    ctx.close()
    kl.close()


def test_progressive_previews(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 64, 48)
    den = rt.ProgressiveRender(gpu_ctx, cam, env, 64, 48, 40, 4, slice_spp=16, denoise=dict(passes=4))
    plain = rt.ProgressiveRender(gpu_ctx, cam, env, 64, 48, 40, 4, slice_spp=16)
    gb = gpu_ctx.gbuffer(cam, 64, 48)
    n = 0
    for a, b in zip(den, plain):
        assert np.array_equal(bits(a), bits(gpu_ctx.denoise(b, gb, passes=4).reshape(-1)))
        n += 1
    assert n == 3 and den.done == plain.done == 40
    assert np.array_equal(bits(den.sums), bits(plain.sums))
    assert np.array_equal(bits(den.image()), bits(gpu_ctx.denoise(plain.image(), gb, passes=4).reshape(-1)))
