"""GPU: adaptive sampling (b200rt_render_adaptive) against the oracle's adaptive mode, bit for bit — image, sample map
and standard-error map — over scenes, generators, estimators, traversals, pixel ranges and tile rows; its early end
of the launch loop; its argument checks; and the launcher's `adaptive` attribute."""
import ctypes

import numpy as np
import pytest

import ensem3a_openclraytracer_b200 as rt
from ensem3a_openclraytracer_b200 import _capi
from oracle import oracle
from oracle_adaptive import adaptive
from tests import fixtures

pytestmark = pytest.mark.gpu

AD = dict(rel_error=0.1, min_spp=4, check_every=4, floor=0.05)


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def setup(ctx, name, ibl_name, w, h=None):
    sc, ibl = fixtures.load_scene(name), fixtures.load_ibl(ibl_name)
    fixtures.upload(ctx, sc, ibl)
    cam, env = fixtures.cam_env(sc["params"], w, h)
    return sc, ibl, cam, env


def live_pixels(ctx, sc, cam, w, h):
    """pixels whose samples need rays (not a primary miss, not an emitter)"""
    tri, _ = ctx.primary_hits(cam, w, h)
    mat = sc["faceData"][10 * np.maximum(tri, 0)]
    return (tri >= 0) & (sc["materialData"][6 * mat].astype(np.int32) != 0)


@pytest.mark.parametrize("name,ibl_name,res,rows,rng,sampling,trav", [
    ("cornell", "preview", 64, None, rt.RNG_REFERENCE, 0, rt.TRAVERSAL_FAST),
    ("cornell", "preview", 64, None, rt.RNG_PHILOX, 1, rt.TRAVERSAL_REFERENCE),
    ("monkey_cfg2", "preview", 72, None, rt.RNG_REFERENCE, 2, rt.TRAVERSAL_FAST),
    ("monkey_cfg2", "preview", 72, None, rt.RNG_PHILOX, 3, rt.TRAVERSAL_FAST),
    ("furnace_cfg3", "grey", 64, None, rt.RNG_PHILOX, 0, rt.TRAVERSAL_REFERENCE),
    ("furnace_cfg3", "grey", 64, None, rt.RNG_REFERENCE, 1, rt.TRAVERSAL_FAST),
    ("serre", "preview", 96, (30, 50), rt.RNG_PHILOX, 0, rt.TRAVERSAL_FAST),
    ("serre", "preview", 96, (30, 50), rt.RNG_REFERENCE, 3, rt.TRAVERSAL_REFERENCE),
])
def test_adaptive_equals_the_oracle_bit_for_bit(gpu_ctx, name, ibl_name, res, rows, rng, sampling, trav):
    sc, ibl, cam, env = setup(gpu_ctx, name, ibl_name, res)
    spp, n_pix = 32, res * res
    i0, i1 = (rows[0] * res, rows[1] * res) if rows else (0, n_pix)
    want, n_want, err_want, cnt = adaptive.render(sc, cam, env, n_pix, spp, 4, ibl, AD, i0=i0, i1=i1, rng_mode=rng,
                                                  seed=77, sampling=sampling)
    o = rt.make_opts(rng_mode=rng, seed=77, sampling=sampling, traversal=trav,
                     pixel_begin=i0 if rows else 0, pixel_end=i1 if rows else 0)
    img, n, err = gpu_ctx.render_adaptive(cam, env, res, res, spp, 4, opts=o, **AD)
    assert np.array_equal(n.reshape(-1), n_want)
    assert np.array_equal(bits(img.reshape(-1)), bits(want))
    assert np.array_equal(bits(err.reshape(-1)), bits(err_want))
    assert 0 < np.mean(n_want[i0:i1] < spp) < 1
    st = gpu_ctx.stats()
    assert st["rays"] == cnt["rays"]
    assert st["sample_streams"] == 1


def test_tile_rows(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 72, 50)
    W, H, spp = 72, 50, 24
    want, n_want, err_want, _ = adaptive.render(sc, cam, env, W * H, spp, 4, ibl, AD, rng_mode=rt.RNG_REFERENCE)
    img, n, err = gpu_ctx.render_adaptive(cam, env, W, H, spp, 4, opts=rt.make_opts(tile_row_mod=3, tile_row_rem=1), **AD)
    rows = (np.arange(H) // 4) % 3 == 1
    assert np.array_equal(n[rows], n_want.reshape(H, W)[rows]) and not n[~rows].any()
    assert np.array_equal(bits(img[rows]), bits(want.reshape(H, W, 3)[rows])) and not img[~rows].any()
    assert np.array_equal(bits(err[rows]), bits(err_want.reshape(H, W)[rows])) and not err[~rows].any()


@pytest.mark.parametrize("rng,sampling", [(rt.RNG_REFERENCE, 0), (rt.RNG_PHILOX, 3)])
def test_min_spp_equal_to_spp_is_b200rt_render(gpu_ctx, rng, sampling):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", "preview", 80)
    o = rt.make_opts(rng_mode=rng, seed=5, sampling=sampling)
    plain = gpu_ctx.render(cam, env, 80, 80, 12, 4, opts=o)
    rays = gpu_ctx.stats()["rays"]
    img, n, err = gpu_ctx.render_adaptive(cam, env, 80, 80, 12, 4, rel_error=1e30, min_spp=12, opts=o)
    assert np.array_equal(bits(img.reshape(-1)), bits(plain))
    assert np.all(n == 12)
    assert gpu_ctx.stats()["rays"] == rays


def test_samples_counts_what_the_map_says(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "monkey_cfg2", "preview", 96)
    _, n, _ = gpu_ctx.render_adaptive(cam, env, 96, 96, 64, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX), **AD)
    st = gpu_ctx.stats()
    live = live_pixels(gpu_ctx, sc, cam, 96, 96).reshape(96, 96)
    assert st["samples"] == int(n[live].sum())
    assert st["samples"] < 64 * int(live.sum())
    assert np.all(n[~live] == 64)


def test_a_frame_that_stops_at_min_spp_ends_the_launch_loop_early(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 96)
    spp, bounce, ad = 256, 4, dict(rel_error=1e30, min_spp=4, check_every=4)
    img, n, err = gpu_ctx.render_adaptive(cam, env, 96, 96, spp, bounce, **ad)
    st = gpu_ctx.stats()
    live = live_pixels(gpu_ctx, sc, cam, 96, 96).reshape(96, 96)
    assert np.all(n[live] == 4) and np.all(n[~live] == spp)
    assert st["wave_iterations"] <= 4 * (bounce + 2) + 2 * 32
    assert st["wave_iterations"] * 10 < spp * (bounce + 2)
    assert st["kernel_launches"] < 3 * st["wave_iterations"] + 8
    want, n_want, err_want, _ = adaptive.render(sc, cam, env, 96 * 96, spp, bounce, ibl, ad)
    assert np.array_equal(bits(img.reshape(-1)), bits(want))
    assert np.array_equal(n.reshape(-1), n_want)
    assert np.array_equal(bits(err.reshape(-1)), bits(err_want))


def test_rejected_arguments(gpu_ctx):
    sc, ibl, cam, env = setup(gpu_ctx, "cornell", "preview", 32)

    def call(spp=16, opts=None, **kw):
        return gpu_ctx.render_adaptive(cam, env, 32, 32, spp, 4, opts=opts, **dict(AD, **kw))

    bad = [dict(min_spp=1), dict(min_spp=17), dict(check_every=0), dict(rel_error=-0.1), dict(rel_error=float("nan")),
           dict(rel_error=float("inf")), dict(floor=0.0), dict(floor=float("nan")), dict(floor=float("inf")),
           dict(opts=rt.make_opts(output=rt.OUT_SUMS)),
           dict(opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, output=rt.OUT_SUMS, sample_begin=0, sample_end=8)),
           dict(opts=rt.make_opts(sample_begin=0, sample_end=8)),
           dict(opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, sample_streams=2)),
           dict(opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, sample_streams=-2))]
    for kw in bad:
        with pytest.raises(rt.B200RTError, match="b200rt_render_adaptive"):
            call(**kw)
    lib = rt.load_library()
    out = np.zeros(32 * 32 * 3, np.float32)
    cam_, env_ = np.ascontiguousarray(cam), np.ascontiguousarray(env)
    o = rt.make_opts()
    rc = lib.b200rt_render_adaptive(gpu_ctx._h, cam_.ctypes.data_as(ctypes.c_void_p), env_.ctypes.data_as(ctypes.c_void_p),
                                    32, 32, 16, 4, ctypes.byref(o), None, out.ctypes.data_as(ctypes.c_void_p), None, None)
    assert rc == -1 and b"NULL" in lib.b200rt_last_error(gpu_ctx._h)
    # the whole range, spelled out, is accepted; automatic sample streams resolve to one
    call(opts=rt.make_opts(sample_begin=0, sample_end=16))
    call(opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, sample_streams=-1))
    assert gpu_ctx.stats()["sample_streams"] == 1


def test_kernel_launcher_adaptive(monkeypatch):
    sc = fixtures.load_scene("monkey_cfg2")
    ibl = fixtures.load_ibl()
    res, spp = 64, 32
    cam, env = fixtures.cam_env(sc["params"], res)
    monkeypatch.setenv("B200RT_ADAPTIVE", "0.1,4,4")
    kl = rt.KernelLauncher(None, None, None, None)
    assert kl.adaptive == {"rel_error": 0.1, "min_spp": 4, "check_every": 4}
    out = np.zeros(res * res * 3, np.float32)
    args = (sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"], sc["BVH"], cam, env,
            res * res, spp, 4, ibl)
    kl.launch_Raytracing(out, *args)
    ctx = rt.Context(0)
    fixtures.upload(ctx, sc, ibl)
    img, n, _ = ctx.render_adaptive(cam, env, res, res, spp, 4, rel_error=0.1, min_spp=4, check_every=4)
    assert np.array_equal(bits(out), bits(img.reshape(-1)))
    assert np.array_equal(kl.last_spp, n) and kl.last_spp.min() < spp
    kl.adaptive = None
    kl.launch_Raytracing(out, *args)
    assert np.array_equal(bits(out), bits(ctx.render(cam, env, res, res, spp, 4)))
    ctx.close()
    # several GPUs: refused before anything is rendered (a stand-in MultiContext where the box has one GPU)
    kl.adaptive = dict(rel_error=0.1)
    fake = object.__new__(_capi.MultiContext)
    fake.devices = [0, 1]
    kl._ctx, real = fake, kl._ctx
    with pytest.raises(ValueError, match="one GPU"):
        kl.launch_Raytracing(out, *args)
    kl._ctx = real
    kl.close()
