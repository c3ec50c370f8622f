"""CPU: the restatement of the denoiser (oracle_denoise/, include/b200rt.h) — pass-through of ray-free pixels, a constant
image, the plain masked B3-spline à-trous it reduces to with very large sigmas, the edge stop at a crease, NaN normals and
zero albedo, the automatic position scale, which pixels its G-buffer calls ray-free, and B200RT_DENOISE parsing."""
import numpy as np
import pytest
from scipy import ndimage

from ensem3a_openclraytracer_b200.KernelLauncher import denoise_from_env
from oracle import oracle
from oracle_denoise import denoise as D
from tests import fixtures

f32 = np.float32


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def random_gbuffer(rng, H, W, p_live=0.8):
    kind = np.where(rng.random((H, W)) < p_live, 1, rng.choice([-1, 0], size=(H, W))).astype(np.int32)
    n = rng.normal(size=(H, W, 3)).astype(f32)
    n /= np.linalg.norm(n, axis=2, keepdims=True).astype(f32)
    return {"kind": kind, "albedo": rng.random((H, W, 3), dtype=f32), "normal": n,
            "position": rng.random((H, W, 3), dtype=f32)}


def test_ray_free_pixels_pass_through_bit_for_bit():
    rng = np.random.default_rng(1)
    gb = random_gbuffer(rng, 40, 56, p_live=0.6)
    img = rng.random((40, 56, 3), dtype=f32) * f32(3)   # above 1 too: a ray-free pixel is not clamped again
    img[0, 0] = np.nan
    gb["kind"][0, 0] = -1
    out = D.atrous(img, gb, 4, 0.5, 0.2, 0.1)
    free = gb["kind"] != 1
    assert np.array_equal(bits(out[free]), bits(img[free]))
    assert np.all(np.isfinite(out[~free])) and out[~free].min() >= 0 and out[~free].max() <= 1


@pytest.mark.parametrize("passes", [1, 5])
def test_constant_demodulated_image_stays_within_a_few_ulp(passes):
    """Demodulated, the image is 0.7 up to one rounding; each pass is a normalised sum of 25 such values, which keeps it
    within a few ulp (rounding of the sums), so after `passes` passes within 8 * passes ulp (relative)."""
    rng = np.random.default_rng(2)
    gb = random_gbuffer(rng, 33, 47, p_live=0.9)
    gb["albedo"] = (f32(0.05) + f32(0.9) * rng.random((33, 47, 3), dtype=f32)).astype(f32)
    img = (f32(0.7) * gb["albedo"]).astype(f32)
    out = D.atrous(img, gb, passes, 0.5, 0.2, 0.1)
    live = gb["kind"] == 1
    assert np.abs(out[live] / img[live] - 1).max() <= 8 * passes * 2.0**-24


def reference_atrous(img, gb, passes):
    """masked, normalised B3-spline à-trous in float64 with scipy.ndimage (no edge stopping)"""
    live = (gb["kind"] == 1).astype(np.float64)
    a = np.maximum(gb["albedo"].astype(np.float64), 0.01)
    c = img.astype(np.float64) / a
    k1 = np.array([1, 4, 6, 4, 1]) / 16.0
    for l in range(passes):
        h = 1 << l
        k = np.zeros(4 * h + 1)
        k[::h] = k1
        kern = np.outer(k, k)
        num = np.stack([ndimage.correlate(c[..., ch] * live, kern, mode="constant") for ch in range(3)], axis=-1)
        den = ndimage.correlate(live, kern, mode="constant")
        c = np.where(live[..., None] > 0, num / np.maximum(den, 1e-300)[..., None], c)
    out = np.clip(c * a, 0, 1)
    return np.where(live[..., None] > 0, out, img)


@pytest.mark.parametrize("passes", [1, 3, 6])
def test_very_large_sigmas_give_the_plain_masked_atrous(passes):
    rng = np.random.default_rng(3 + passes)
    gb = random_gbuffer(rng, 37, 53)
    img = rng.random((37, 53, 3), dtype=f32)
    out = D.atrous(img, gb, passes, 1e15, 1e15, 1e15)
    assert np.abs(out - reference_atrous(img, gb, passes)).max() <= 1e-6


def test_crease_between_two_planes_leaks_less_than_the_weights_allow():
    """Left half faces +x with colour 0, right half faces +y with colour 1 (albedo 1, one position).  The centre tap
    weighs k1[2]^2 and a tap across the crease at most f(2, s_n) of its spatial weight, whose sum is 1: each pass moves a
    pixel at most f(2, s_n) / k1[2]^2 towards the other side."""
    H, W, passes, sn = 24, 32, 5, 0.02
    n = np.zeros((H, W, 3), f32)
    n[:, : W // 2, 0] = 1
    n[:, W // 2:, 1] = 1
    gb = {"kind": np.ones((H, W), np.int32), "albedo": np.ones((H, W, 3), f32), "normal": n,
          "position": np.zeros((H, W, 3), f32)}
    img = np.zeros((H, W, 3), f32)
    img[:, W // 2:] = 1
    bound = passes * (1 / (1 + 2 / sn**2)) / (3 / 8) ** 2
    out = D.atrous(img, gb, passes, 1e6, sn, 1.0)
    assert out[:, : W // 2].max() <= bound and 1 - out[:, W // 2:].min() <= bound
    assert out[:, W // 2 - 1].max() > 0   # the filter does reach across, as little as the weights say
    blurred = D.atrous(img, gb, passes, 1e6, 1e6, 1.0)
    assert blurred[:, W // 2 - 1].min() > 0.3 > 40 * bound   # without the normal's edge stop the crease blurs


def test_nan_normals_and_zero_albedo():
    rng = np.random.default_rng(5)
    gb = random_gbuffer(rng, 30, 30, p_live=1.0)
    gb["normal"][5:10, 5:10] = np.nan
    gb["albedo"][12:20, 3:9] = 0
    img = rng.random((30, 30, 3), dtype=f32)
    img[12:20, 3:9] *= f32(0.01)
    out = D.atrous(img, gb, 4, 0.5, 0.2, 0.1)
    assert np.all(np.isfinite(out)) and out.min() >= 0 and out.max() <= 1
    # every tap of a NaN-normal pixel has a NaN weight: it keeps its own colour (demodulated and remodulated)
    nan_px = out[5:10, 5:10]
    assert np.all(np.abs(nan_px - img[5:10, 5:10]) <= 2 * np.spacing(img[5:10, 5:10]))
    # and it is no tap of its neighbours: the result does not depend on its colour
    img2 = img.copy()
    img2[5:10, 5:10] = 0.5
    out2 = D.atrous(img2, gb, 4, 0.5, 0.2, 0.1)
    mask = np.ones((30, 30), bool)
    mask[5:10, 5:10] = False
    assert np.array_equal(bits(out[mask]), bits(out2[mask]))


def test_automatic_sigma_position_is_one_percent_of_the_root_diagonal():
    for name in ("cornell", "monkey", "serre"):
        bvh = fixtures.load_scene(name)["BVH"]
        lo, hi = bvh[2:5].astype(np.float64), bvh[5:8].astype(np.float64)
        want = 0.01 * np.sqrt(((hi - lo) ** 2).sum())
        got = D.auto_sigma_position(bvh)
        assert got.dtype == np.float32 and abs(got - want) <= 1e-6 * want
    gb = random_gbuffer(np.random.default_rng(6), 20, 20)
    img = np.random.default_rng(7).random((20, 20, 3), dtype=f32)
    bvh = fixtures.load_scene("cornell")["BVH"]
    assert np.array_equal(bits(D.atrous(img, gb, 3, 0.5, 0.2, 0, bvh)),
                          bits(D.atrous(img, gb, 3, 0.5, 0.2, float(D.auto_sigma_position(bvh)))))


@pytest.mark.parametrize("name", ["cornell", "monkey_cfg2"])
def test_kind_matches_the_pixels_the_oracle_renders_without_a_ray(name):
    """The oracle traces a ray-free pixel's primary ray once and nothing else; any other pixel traces more."""
    sc = fixtures.load_scene(name)
    W, H, spp = 16, 12, 2
    cam, env = fixtures.cam_env(sc["params"], W, H)
    gb = D.gbuffer(sc, cam, W, H)
    ibl = fixtures.load_ibl()
    rays = np.array([oracle.render(sc, cam, env, W * H, spp, 2, ibl, i0=i, i1=i + 1)[1]["rays"] for i in range(W * H)])
    assert np.array_equal(gb["kind"].reshape(-1) != 1, rays == 1)
    assert (gb["kind"] == 1).any() and (gb["kind"] != 1).any()
    free = gb["kind"].reshape(-1) != 1
    assert np.all(gb["albedo"].reshape(-1, 3)[free] == 1)
    assert np.all(gb["position"].reshape(-1, 3)[gb["kind"].reshape(-1) == -1] == 0)


def test_denoise_from_env():
    defaults = {"passes": 5, "sigma_color": 0.5, "sigma_normal": 0.2, "sigma_position": 0.0}
    assert denoise_from_env("1") == defaults
    assert denoise_from_env("3") == dict(defaults, passes=3)
    assert denoise_from_env(" 4 , 0.3") == dict(defaults, passes=4, sigma_color=0.3)
    assert denoise_from_env("2,0.3,0.1,0.05") == {"passes": 2, "sigma_color": 0.3, "sigma_normal": 0.1, "sigma_position": 0.05}
    assert denoise_from_env("5,0.5,0.2,-1")["sigma_position"] == -1.0
    for bad in ["", "0", "9", "x", "1.5", "5,0", "5,-1", "5,0.5,0", "5,nan", "5,0.5,0.2,inf", "5,0.5,0.2,0,1", "5,,0.2"]:
        with pytest.raises(ValueError, match="B200RT_DENOISE"):
            denoise_from_env(bad)
