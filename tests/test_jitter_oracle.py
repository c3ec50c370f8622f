"""CPU: the pixel-jitter rule of include/b200rt.h (B200RT_SAMPLING_PIXEL_JITTER) as the jitter oracle states it
integrates the pixel's area; the unchanged oracle ignores the bit; the launcher's environment switch."""
import numpy as np
import pytest

from ensem3a_openclraytracer_b200.KernelLauncher import pixel_jitter_from_env
from oracle import oracle
from oracle_jitter import jitter
from tests import jitter_scene

W, H, SPP = 64, 48, 256


@pytest.fixture(scope="module")
def case():
    sc, cam, env, ibl = jitter_scene.scene(W, H)
    return sc, cam, env, ibl, jitter_scene.coverage(W, H)


def test_philox_pixels_converge_to_their_coverage(case):
    sc, cam, env, ibl, f = case
    img, cnt = jitter.render(sc, cam, env, W * H, SPP, 4, ibl, rng_mode=oracle.RNG_PHILOX, seed=11)
    img = img.reshape(H, W, 3)
    assert np.array_equal(img[..., 0], img[..., 1]) and np.array_equal(img[..., 0], img[..., 2])
    tol = 5.0 * np.sqrt(f * (1.0 - f) / SPP) + 2e-3
    assert np.all(np.abs(img[..., 0] - f) <= tol)
    assert cnt["rays"] == W * H * SPP            # one camera ray per sample; nothing scatters
    assert cnt["rand_calls"] == 2 * W * H * SPP


@pytest.mark.parametrize("rng", [oracle.RNG_REFERENCE, oracle.RNG_PHILOX])
def test_frame_mean_is_the_mean_coverage(case, rng):
    """the reference generator gets no per-pixel bound: its per-pixel streams fall into a few short cycles (DESIGN §5)"""
    sc, cam, env, ibl, f = case
    img, _ = jitter.render(sc, cam, env, W * H, SPP, 4, ibl, rng_mode=rng, seed=5)
    se = np.sqrt(np.sum(f * (1.0 - f)) / SPP) / f.size
    assert abs(img.reshape(H, W, 3)[..., 0].mean(dtype=np.float64) - f.mean()) <= 4.0 * se


def test_the_unjittered_image_is_a_step_the_jittered_one_is_not(case):
    sc, cam, env, ibl, f = case
    plain, _ = oracle.render(sc, cam, env, W * H, SPP, 4, ibl, rng_mode=oracle.RNG_PHILOX, seed=11)
    assert set(np.unique(plain)) == {0.0, 1.0}
    jit, _ = jitter.render(sc, cam, env, W * H, SPP, 4, ibl, rng_mode=oracle.RNG_PHILOX, seed=11)
    jit = jit.reshape(H, W, 3)[..., 0]
    edge = (f > 0.05) & (f < 0.95)
    assert edge.sum() >= 40
    assert np.all((jit[edge] > 0.0) & (jit[edge] < 1.0))


@pytest.mark.parametrize("rng", [oracle.RNG_REFERENCE, oracle.RNG_PHILOX])
def test_the_oracle_ignores_the_jitter_bit(rng):
    from tests import fixtures
    sc, ibl = fixtures.load_scene("cornell"), fixtures.load_ibl()
    cam, env = fixtures.cam_env(sc["params"], 32)
    for base in (0, 3):
        a, ca = oracle.render(sc, cam, env, 32 * 32, 4, 4, ibl, rng_mode=rng, seed=2, sampling=base)
        b, cb = oracle.render(sc, cam, env, 32 * 32, 4, 4, ibl, rng_mode=rng, seed=2, sampling=base | 8)
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32)) and ca == cb


def test_pixel_jitter_from_env():
    assert pixel_jitter_from_env("1") is True
    assert pixel_jitter_from_env("0") is False
    assert pixel_jitter_from_env(" 1 ") is True
    for bad in ("", "2", "yes", "true", "1,0", "-1"):
        with pytest.raises(ValueError, match="B200RT_PIXEL_JITTER"):
            pixel_jitter_from_env(bad)
