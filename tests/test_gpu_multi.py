"""The multi-GPU handle (b200rt_multi_*, KernelLauncher(cuda_devices=...)): one host process drives several GPUs of
the box through the reference-facing call.  With one visible GPU the one-device handle still exercises the whole
path (share computation, partial sums, reduce + finalize kernel); the two-device tests need `gpurun --gpus 2`."""
import numpy as np
import pytest

import ensem3a_openclraytracer_b200 as rt
from oracle import oracle
from tests import fixtures

pytestmark = pytest.mark.gpu


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def devices(n):
    if rt.device_count() < n:
        pytest.skip(f"needs {n} visible GPUs")
    return list(range(n))


@pytest.mark.parametrize("name,res", [("cornell", 128), ("monkey_cfg2", 96)])
def test_one_device_handle_equals_the_plain_context(gpu_ctx, name, res):
    sc, ibl = fixtures.load_scene(name), fixtures.load_ibl()
    cam, env = fixtures.cam_env(sc["params"], res)
    fixtures.upload(gpu_ctx, sc, ibl)
    m = rt.MultiContext([0])
    try:
        fixtures.upload(m, sc, ibl)
        for rng in (rt.RNG_REFERENCE, rt.RNG_PHILOX):
            o = rt.make_opts(rng_mode=rng, seed=5)
            want = gpu_ctx.render(cam, env, res, res, 6, 4, opts=o)
            got = m.render(cam, env, res, res, 6, 4, opts=rt.make_opts(rng_mode=rng, seed=5))
            assert np.array_equal(bits(got), bits(want))
            assert m.stats()["rays"] == gpu_ctx.stats()["rays"]
    finally:
        m.close()


def test_handle_rejects_a_caller_side_partition(gpu_ctx):
    sc, ibl = fixtures.load_scene("cornell"), fixtures.load_ibl()
    cam, env = fixtures.cam_env(sc["params"], 32)
    m = rt.MultiContext([0])
    try:
        fixtures.upload(m, sc, ibl)
        with pytest.raises(rt.B200RTError):
            m.render(cam, env, 32, 32, 4, 4, opts=rt.make_opts(rng_mode=rt.RNG_PHILOX, output=rt.OUT_SUMS, sample_begin=0, sample_end=2))
        with pytest.raises(rt.B200RTError):
            rt.MultiContext([])
    finally:
        m.close()


@pytest.mark.parametrize("n", [2, 4, 8])
def test_n_devices_reference_generator_is_bit_identical(gpu_ctx, n):
    """Tile-row split: disjoint pixels per GPU, so the image is the one-GPU image bit for bit — and the oracle's."""
    devs = devices(n)
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    res = 160
    cam, env = fixtures.cam_env(sc["params"], res)
    fixtures.upload(gpu_ctx, sc, ibl)
    want = gpu_ctx.render(cam, env, res, res, 5, 4, opts=rt.make_opts(rng_mode=rt.RNG_REFERENCE))
    m = rt.MultiContext(devs)
    try:
        fixtures.upload(m, sc, ibl)
        got = m.render(cam, env, res, res, 5, 4, opts=rt.make_opts(rng_mode=rt.RNG_REFERENCE))
        assert np.array_equal(bits(got), bits(want))
        assert m.stats()["samples"] == gpu_ctx.stats()["samples"]
    finally:
        m.close()
    ref, _ = oracle.render(sc, cam, env, res * res, 5, 4, ibl)
    assert np.array_equal(bits(got), bits(ref))


@pytest.mark.parametrize("n", [2, 8])
def test_n_devices_philox_sample_ranges(gpu_ctx, n):
    """Sample-range split: same samples, summed per GPU and then across GPUs — within 1e-4 relative (north_star) of the
    one-GPU image; an spp that does not divide evenly and one smaller than the GPU count (idle GPUs) included."""
    devs = devices(n)
    sc, ibl = fixtures.load_scene("serre"), fixtures.load_ibl()
    res = 128
    cam, env = fixtures.cam_env(sc["params"], res)
    fixtures.upload(gpu_ctx, sc, ibl)
    m = rt.MultiContext(devs)
    try:
        fixtures.upload(m, sc, ibl)
        for spp in (11, 1):
            o = dict(rng_mode=rt.RNG_PHILOX, seed=3)
            want = gpu_ctx.render(cam, env, res, res, spp, 4, opts=rt.make_opts(**o))
            got = m.render(cam, env, res, res, spp, 4, opts=rt.make_opts(**o))
            rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-3)
            assert np.array_equal(np.isnan(got), np.isnan(want))
            assert np.nanmax(rel) <= 1e-4
            assert m.stats()["samples"] == gpu_ctx.stats()["samples"]
    finally:
        m.close()


WORK = ("rays", "samples", "box_tests", "tri_tests", "mismatches", "revalidated", "exact_walks", "kernel_launches")


@pytest.mark.parametrize("rng,spp,height", [(rt.RNG_PHILOX, 2, 32), (rt.RNG_REFERENCE, 3, 8)])
def test_idle_entry_reports_no_work_of_an_earlier_frame(gpu_ctx, rng, spp, height):
    """A frame in which an entry has nothing to render (Philox with spp below the entry count; two tile rows for three
    entries) reports the statistics it reports on a fresh handle: the idle entry adds nothing from the frame before."""
    sc, ibl = fixtures.load_scene("cornell"), fixtures.load_ibl()
    width = 32
    o = dict(rng_mode=rng, traversal=rt.TRAVERSAL_REFERENCE, collect_stats=True, seed=7)
    cam_a, env_a = fixtures.cam_env(sc["params"], width, 32)
    cam_b, env_b = fixtures.cam_env(sc["params"], width, height)

    def frame_b(m):
        img = m.render(cam_b, env_b, width, height, spp, 4, opts=rt.make_opts(**o))
        return img, {k: m.stats()[k] for k in WORK}

    used, fresh = rt.MultiContext([0, 0, 0]), rt.MultiContext([0, 0, 0])
    try:
        fixtures.upload(used, sc, ibl)
        fixtures.upload(fresh, sc, ibl)
        used.render(cam_a, env_a, width, 32, 6, 4, opts=rt.make_opts(**o))
        assert used.stats()["box_tests"] > 0
        got_img, got = frame_b(used)
        want_img, want = frame_b(fresh)
        assert got == want
        assert np.array_equal(bits(got_img), bits(want_img))
    finally:
        used.close()
        fresh.close()


def test_launcher_drives_two_gpus_through_the_reference_call():
    """KernelLauncher(cuda_devices=[0, 1]).launch_Raytracing — the call main.py makes (main.py:84-86) — on two GPUs."""
    devs = devices(2)
    sc, ibl = fixtures.load_scene("cornell"), fixtures.load_ibl()
    res = 128
    cam, env = fixtures.cam_env(sc["params"], res)
    one = rt.KernelLauncher(None, None, None, None)
    two = rt.KernelLauncher(None, None, None, None, cuda_devices=devs)
    a, b = np.zeros(res * res * 3, np.float32), np.zeros(res * res * 3, np.float32)
    args = (sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"], sc["BVH"], cam, env,
            res * res, 8, 4, ibl)
    one.launch_Raytracing(a, *args)
    two.launch_Raytracing(b, *args)
    assert np.array_equal(bits(a), bits(b))
    tone_a, tone_b = np.zeros_like(a), np.zeros_like(b)
    one.launch_ImgProcessing(a, tone_a, res)
    two.launch_ImgProcessing(b, tone_b, res)
    assert np.array_equal(bits(tone_a), bits(tone_b))
    one.close()
    two.close()
