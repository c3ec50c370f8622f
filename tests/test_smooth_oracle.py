"""CPU: the smooth-shading rule of include/b200rt.h (B200RT_SAMPLING_SMOOTH_NORMALS) as the smooth oracle (oracle_smooth/)
states it — equal, bit for bit, to a numpy restatement, fallbacks included; without the bit that oracle is the plain,
jitter and adaptive oracles bit for bit; flat scenes unchanged by the bit; the quality it buys on a coarse sphere; the
launcher's environment switch."""
import numpy as np
import pytest

from ensem3a_openclraytracer_b200.KernelLauncher import smooth_normals_from_env
from oracle import oracle
from oracle_adaptive import adaptive
from oracle_jitter import jitter
from oracle_smooth import smooth
from tests import fixtures, smooth_scene as ss

f32 = np.float32
SMOOTH = ss.SMOOTH


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


def random_points(scene, tris, rng):
    """points inside the given triangles (barycentric weights drawn in binary64, the point rounded to binary32)"""
    vp = scene["V_p"].reshape(-1, 3).astype(np.float64)
    face = scene["faceData"].reshape(-1, 10)[tris]
    u, v = rng.random(tris.size), rng.random(tris.size)
    flip = u + v > 1
    u[flip], v[flip] = 1 - u[flip], 1 - v[flip]
    A, B, C = vp[face[:, 7]], vp[face[:, 8]], vp[face[:, 9]]
    return (A + (B - A) * u[:, None] + (C - A) * v[:, None]).astype(f32)


@pytest.mark.parametrize("name", ["monkey", "serre"])
def test_oracle_equals_the_restatement(name):
    sc = fixtures.load_scene(name)
    rng = np.random.default_rng(7)
    cur = np.nonzero(ss.curved(sc))[0]
    tris = np.concatenate([rng.choice(cur, 3000), rng.integers(0, sc["faceData"].size // 10, 1000)]).astype(np.int32)
    x = random_points(sc, tris, rng)
    got = smooth.smooth_normal(sc, tris, x)
    want = ss.smooth_normal(sc, tris, x)
    assert np.array_equal(bits(got), bits(want))
    n0 = sc["V_n"].reshape(-1, 3)[sc["faceData"].reshape(-1, 10)[tris, 4]]
    moved = ~(bits(got) == bits(n0)).all(axis=1)
    assert moved[:3000].mean() > 0.99 and not moved[3000:][~ss.curved(sc)[tris[3000:]]].any()
    assert np.abs(np.linalg.norm(got[moved], axis=1) - 1).max() < 1e-6


def fallback_scene():
    """three triangles of (0,0,0), (2,0,0), (0,2,0) or a degenerate one, with awkward normals"""
    vp = np.array([0, 0, 0, 2, 0, 0, 0, 2, 0, 1, 0, 0, 3, 0, 0], f32)
    vn = np.array([0, 0, 1, 0, 0, -1, 1, 0, 0, np.nan, 0, 0, 0, 1, 0], f32)
    faces = [
        [0, 0, 0, 0, 0, 1, 2, 0, 1, 2],   # n0 = -n1: zero sum at x = (1, 0, 0) (b0 = b1 = 1/2, b2 = 0)
        [0, 0, 0, 0, 0, 2, 3, 0, 1, 2],   # NaN n2
        [0, 0, 0, 0, 0, 4, 2, 0, 3, 4],   # collinear vertices: den = 0
        [0, 0, 0, 0, 0, 4, 2, 0, 1, 2],   # an ordinary curved triangle
    ]
    return {"V_p": vp, "V_n": vn, "faceData": np.array(faces, np.int32).reshape(-1)}


def test_fallbacks_give_the_first_vertex_normal():
    sc = fallback_scene()
    tris = np.array([0, 1, 2, 3], np.int32)
    x = np.array([[1, 0, 0], [0.5, 0.5, 0], [2, 0, 0], [0.5, 0.5, 0]], f32)
    got = smooth.smooth_normal(sc, tris, x)
    assert np.array_equal(bits(got), bits(ss.smooth_normal(sc, tris, x)))
    assert np.array_equal(got[:3], np.array([[0, 0, 1]] * 3, f32))
    assert not np.array_equal(got[3], np.array([0, 0, 1], f32)) and np.isfinite(got[3]).all()


@pytest.mark.parametrize("name", ["cornell", "furnace_cfg3", "proto"])
@pytest.mark.parametrize("base", [0, 3])
def test_flat_scenes_render_the_same(name, base):
    sc = fixtures.load_scene(name)
    assert not ss.curved(sc).any()
    ibl = fixtures.load_ibl("grey" if name.startswith("furnace") else "preview")
    cam, env = fixtures.cam_env(sc["params"], 40)
    a, ca = oracle.render(sc, cam, env, 40 * 40, 3, 4, ibl, rng_mode=1, seed=5, sampling=base)
    b, cb = smooth.render(sc, cam, env, 40 * 40, 3, 4, ibl, rng_mode=1, seed=5, sampling=base | SMOOTH)
    assert np.array_equal(bits(a), bits(b)) and ca == cb


def test_smooth_shading_approaches_the_fine_sphere():
    """a 12 x 6 UV sphere under a vertically graded environment against a 192 x 96 one, RMSE over the pixels whose
    primary hits both lie on the sphere: 0.0078 smooth against 0.046 flat at this setting (64 px, 256 spp, seeds 4 and 9)"""
    W, spp = 64, 256
    cam, env, ibl = ss.sphere_view(W)
    coarse, fine = ss.sphere(12, 6), ss.sphere(192, 96)
    ref, _ = oracle.render(fine, cam, env, W * W, spp, 2, ibl, rng_mode=1, seed=4)
    mask = (oracle.primary(coarse, cam, W * W)["tri"] >= 0) & (oracle.primary(fine, cam, W * W)["tri"] >= 0)
    assert mask.sum() > 1000
    err = {}
    for s in (0, SMOOTH):
        img, _ = smooth.render(coarse, cam, env, W * W, spp, 2, ibl, rng_mode=1, seed=4, sampling=s)
        d = (img.reshape(-1, 3) - ref.reshape(-1, 3))[mask]
        err[s] = np.sqrt(np.mean(d.astype(np.float64) ** 2))
    assert err[SMOOTH] < 0.35 * err[0], err


@pytest.mark.parametrize("rng", [oracle.RNG_REFERENCE, oracle.RNG_PHILOX])
def test_without_the_bit_the_smooth_oracle_is_the_other_oracles(rng):
    """oracle_smooth restates path_sample and the per-pixel loops of oracle/, oracle_jitter/ and oracle_adaptive/; without
    bit 32 it must be each of them bit for bit, counters included"""
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    cam, env = fixtures.cam_env(sc["params"], 32)
    n = 32 * 32
    for sampling in (0, 1, 2, 3):
        want = oracle.render(sc, cam, env, n, 4, 4, ibl, rng_mode=rng, seed=9, sampling=sampling, i0=100, i1=900)
        got = smooth.render(sc, cam, env, n, 4, 4, ibl, rng_mode=rng, seed=9, sampling=sampling, i0=100, i1=900)
        assert np.array_equal(bits(got[0]), bits(want[0])) and got[1] == want[1]
        want = jitter.render(sc, cam, env, n, 4, 4, ibl, rng_mode=rng, seed=9, sampling=sampling)
        got = smooth.render(sc, cam, env, n, 4, 4, ibl, rng_mode=rng, seed=9, sampling=sampling | 8)
        assert np.array_equal(bits(got[0]), bits(want[0])) and got[1] == want[1]
        ad = dict(rel_error=0.2, min_spp=4, check_every=2)
        want = adaptive.render(sc, cam, env, n, 12, 4, ibl, ad, rng_mode=rng, seed=9, sampling=sampling)
        got = smooth.render(sc, cam, env, n, 12, 4, ibl, rng_mode=rng, seed=9, sampling=sampling, adaptive=ad)
        assert np.array_equal(bits(got[0]), bits(want[0])) and np.array_equal(got[1], want[1])
        assert np.array_equal(bits(got[2]), bits(want[2])) and got[3] == want[3]
    if rng == oracle.RNG_PHILOX:
        want = oracle.render(sc, cam, env, n, 8, 4, ibl, rng_mode=rng, seed=9, s0=3, s1=7, raw_sums=True)
        got = smooth.render(sc, cam, env, n, 8, 4, ibl, rng_mode=rng, seed=9, s0=3, s1=7, raw_sums=True)
        assert np.array_equal(bits(got[0]), bits(want[0])) and got[1] == want[1]
    # and the bit changes the image of a curved mesh
    a, _ = smooth.render(sc, cam, env, n, 4, 4, ibl, rng_mode=rng, seed=9, sampling=SMOOTH)
    assert not np.array_equal(bits(a), bits(oracle.render(sc, cam, env, n, 4, 4, ibl, rng_mode=rng, seed=9)[0]))


def test_environment_switch():
    assert smooth_normals_from_env("1") is True
    assert smooth_normals_from_env(" 0 ") is False
    for bad in ("on", "", "2", "true"):
        with pytest.raises(ValueError, match="B200RT_SMOOTH_NORMALS"):
            smooth_normals_from_env(bad)
