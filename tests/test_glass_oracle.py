"""CPU: opt-in refractive glass (B200RT_SAMPLING_DIELECTRIC_GLASS).  The oracle's interface rule against a numpy
restatement, bit for bit, and against the float64 physics; without the bit the glass oracle is the smooth oracle, bit
for bit, counters included; ior-1 and glass-free scenes do not change with the bit; the white-glass furnace; the ball
lens turns the environment upside down; the launcher's environment variable."""
import numpy as np
import pytest

from ensem3a_openclraytracer_b200.KernelLauncher import dielectric_glass_from_env
from oracle import oracle
from oracle_glass import glass
from oracle_smooth import smooth
from tests import fixtures, glass_scene as gs, smooth_scene as ss

f32 = np.float32
G = gs.GLASS


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


def unit_rows(a):
    a = np.asarray(a, f32)
    return (a / np.sqrt(gs._dot(a, a))[:, None]).astype(f32)


def same_rule(w, n, v, u):
    d, r, F = glass.dielectric(w, n, v, u)
    d2, r2, F2 = gs.dielectric(w, n, v, u)
    assert np.array_equal(r, r2)
    assert np.array_equal(bits(F), bits(F2))
    assert np.array_equal(bits(d), bits(d2))
    return d, r, F


def critical_cases(ior):
    """leaving directions (x, 0, z) around the critical angle of ior against n = +z: the float32 z at which k first
    becomes >= 0 and its neighbours (k < 0 just past the critical angle, k > 0 just before)"""
    zc = np.sqrt(1.0 - 1.0 / (ior * ior))
    z = f32(zc)
    for _ in range(64):
        z = np.nextafter(z, f32(0))
    zs = [z]
    for _ in range(128):
        zs.append(np.nextafter(zs[-1], f32(1)))
    zs = np.array(zs, f32)
    w = np.stack([np.sqrt(f32(1) - zs * zs), np.zeros_like(zs), zs], axis=1).astype(f32)
    ww = unit_rows(w)
    ci = ww[:, 2]
    eta = f32(ior)
    k = f32(1) - (eta * eta) * (f32(1) - ci * ci)
    first = int(np.argmax(k >= 0))
    assert 0 < first and k[first - 1] < 0
    return w[first - 3:first + 3], k[first - 3:first + 3]


def test_rule_bit_for_bit_random():
    rng = np.random.default_rng(7)
    m = 100_000
    w = rng.normal(size=(m, 3)).astype(f32) * rng.uniform(0.2, 3.0, size=(m, 1)).astype(f32)
    n = unit_rows(rng.normal(size=(m, 3)))
    v = rng.uniform(0.3, 3.0, size=m).astype(f32)
    v[::7] = 0.0
    v[1::11] = f32(1.5)
    u = rng.random(m, dtype=np.float32)
    d, r, F = same_rule(w, n, v, u)
    assert 0.02 < r.mean() < 0.6   # both outcomes occur
    assert np.isfinite(d).all()


def test_rule_bit_for_bit_edge_cases():
    z = np.array([[0, 0, 1]], f32)
    u = f32(0.5)
    # normal incidence, entering and leaving
    for w in (-z, z):
        d, r, F = same_rule(w, z, [1.5], [u])
        assert not r[0] and np.array_equal(d, w)
    # grazing: ci = 0 (c = 0 counts as leaving): total internal reflection for ior > 1, F = 1 below 1
    x = np.array([[1, 0, 0]], f32)
    for ior in (1.5, 0.75):
        d, r, F = same_rule(x, z, [ior], [f32(0.999)])
        assert r[0] and F[0] == 1 and np.array_equal(d, x)
    # at and just past the critical angle
    for ior in (1.5, 2.0, 1.33):
        w, k = critical_cases(ior)
        d, r, F = same_rule(w, np.repeat(z, len(w), axis=0), np.full(len(w), ior, f32), np.full(len(w), 0.999, f32))
        assert (r[k < 0]).all() and (F[k < 0] == 1).all()
        assert (F[k >= 0] <= 1).all()
    # ior < 1: a bubble; entering behaves like leaving glass of 1 / ior
    rng = np.random.default_rng(3)
    w = unit_rows(rng.normal(size=(2000, 3)))
    nn = np.repeat(z, 2000, axis=0)
    u = rng.random(2000, dtype=np.float32)
    same_rule(w, nn, np.full(2000, 0.75, f32), u)
    # ior slot 0 resolves to the default, 1.5
    d0, r0, F0 = same_rule(w, nn, np.zeros(2000, f32), u)
    d1, r1, F1 = glass.dielectric(w, nn, np.full(2000, 1.5, f32), u)
    assert np.array_equal(bits(d0), bits(d1)) and np.array_equal(r0, r1) and np.array_equal(bits(F0), bits(F1))


def _angles(m, seed, ior):
    """m entering directions at angles of incidence in [0, 85] degrees against n = +z (closer to grazing, binary32
    loses digits of F to the cancellation in 1 - ci * ci)"""
    rng = np.random.default_rng(seed)
    th = np.radians(rng.uniform(0.0, 85.0, m))
    ph = rng.uniform(0.0, 2 * np.pi, m)
    w = np.stack([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), -np.cos(th)], axis=1).astype(f32)
    return unit_rows(w), np.repeat(np.array([[0, 0, 1]], f32), m, axis=0), np.full(m, ior, f32)


@pytest.mark.parametrize("ior", [1.5, 1.33, 2.4, 0.75])
def test_physics_against_float64(ior):
    m = 4000
    w, n, v = _angles(m, 11, ior)
    w64, n64 = w.astype(np.float64), n.astype(np.float64)
    top = np.full(m, np.nextafter(f32(1), f32(0)), f32)   # u just below 1: refracts unless F = 1
    dt, rt_, Ft = glass.dielectric(w, n, v, top)
    assert ((Ft >= 0) & (Ft <= 1)).all()
    sin_i = np.linalg.norm(np.cross(w64, n64), axis=1)
    ok = ~rt_   # refracted (entering glass of ior > 1 never reflects totally; a bubble does past its critical angle)
    if ior > 1:
        assert ok.all()
    sin_t = np.linalg.norm(np.cross(dt.astype(np.float64), n64), axis=1)
    assert np.allclose(sin_t[ok], sin_i[ok] / ior, atol=1e-5)
    # both outgoing directions are unit vectors; the reflection is the mirror image, the refraction on the far side
    d_refl, r_all, _ = glass.dielectric(w, n, v, np.full(m, -1.0, f32))   # u < 0 <= F: always reflects
    assert r_all.all()
    for d in (dt, d_refl):
        assert np.allclose(np.linalg.norm(d.astype(np.float64), axis=1), 1.0, atol=1e-6)
    assert (dt[ok, 2] < 0).all() and (d_refl[:, 2] > 0).all()
    mirror = w64 - 2.0 * np.sum(w64 * n64, axis=1)[:, None] * n64
    assert np.allclose(d_refl, mirror, atol=1e-6)
    # F at normal incidence
    d0, r0, F0 = glass.dielectric([[0, 0, -1]], [[0, 0, 1]], [ior], [0.5])
    assert np.isclose(F0[0], ((ior - 1) / (ior + 1)) ** 2, rtol=1e-6, atol=1e-9)
    # Stokes: F entering at theta_i equals F leaving at theta_t; a slab (parallel faces) keeps the direction
    if ior > 1:
        d_out, r_out, F_out = glass.dielectric(dt, -n, v, top)   # the exit face's outward normal is -n
        assert not r_out.any()
        assert np.allclose(F_out, Ft, atol=2e-5)
        assert np.allclose(d_out, w, atol=1e-5)


def _smooth_and_glass(name, res, sampling, rng, adaptive=None):
    sc = fixtures.load_scene(name)
    ibl = fixtures.load_ibl()
    cam, env = fixtures.cam_env(sc["params"], res)
    kw = dict(rng_mode=rng, seed=9, sampling=sampling, adaptive=adaptive)
    return (smooth.render(sc, cam, env, res * res, 6, 4, ibl, **kw),
            glass.render(sc, cam, env, res * res, 6, 4, ibl, **kw))


@pytest.mark.parametrize("name", ["cornell", "monkey_cfg2", "serre"])
@pytest.mark.parametrize("sampling", [0, 1, 2, 3, 8, 32])
def test_without_the_bit_equals_the_smooth_oracle(name, sampling):
    for rng in (0, 1):
        (a, ca), (b, cb) = _smooth_and_glass(name, 24, sampling, rng)
        assert np.array_equal(bits(a), bits(b)) and ca == cb


@pytest.mark.parametrize("name", ["monkey_cfg2", "serre"])
def test_without_the_bit_equals_the_smooth_oracle_adaptive(name):
    ad = dict(rel_error=0.2, min_spp=2, check_every=2)
    for rng, sampling in ((0, 0), (1, 34)):
        a, b = _smooth_and_glass(name, 24, sampling, rng, adaptive=ad)
        for x, y in zip(a[:3], b[:3]):
            assert np.array_equal(np.asarray(x).view(np.uint32), np.asarray(y).view(np.uint32))
        assert a[3] == b[3]


@pytest.mark.parametrize("name", ["monkey_cfg2", "serre", "monkey_glass", "cornell"])
def test_ior_one_and_glass_free_scenes_do_not_change(name):
    sc = gs.glass_ior(gs.load(name), 1.0)
    ibl = fixtures.load_ibl()
    cam, env = fixtures.cam_env(fixtures.load_scene("serre" if name == "serre" else
                                                    "cornell" if name == "cornell" else "monkey_cfg2")["params"], 24)
    for base in (0, 3, 8, 32):
        for rng in (0, 1):
            a, ca = glass.render(sc, cam, env, 24 * 24, 4, 4, ibl, rng_mode=rng, seed=2, sampling=base)
            b, cb = glass.render(sc, cam, env, 24 * 24, 4, 4, ibl, rng_mode=rng, seed=2, sampling=base | G)
            assert np.array_equal(bits(a), bits(b)) and ca == cb
    # and the bit does change a scene with glass of another ior
    if name != "cornell":
        sc = gs.glass_ior(sc, 0.0)
        a, _ = glass.render(sc, cam, env, 24 * 24, 4, 4, ibl, sampling=0)
        b, _ = glass.render(sc, cam, env, 24 * 24, 4, 4, ibl, sampling=G)
        assert not np.array_equal(bits(a), bits(b))


@pytest.mark.parametrize("rng", [0, 1])
def test_white_glass_furnace(rng):
    """every sample of a white glass sphere keeps throughput 1 until it escapes into the uniform map: a sphere pixel adds
    the value a background pixel adds, as often and in the same order, unless a path was cut at maxBounce"""
    W, spp = 32, 8
    sc = gs.glass_sphere()
    cam, env, grey = gs.grey_view(W)
    hit = oracle.primary(sc, cam, W * W)["tri"] >= 0
    assert hit.sum() > 200
    # smooth shading: no path is cut at maxBounce 8, every pixel equals the background bit for bit
    out, cnt = glass.render(sc, cam, env, W * W, spp, 8, grey, rng_mode=rng, seed=5, sampling=G | 32)
    o = out.reshape(-1, 3)
    bg = o[~hit][0]
    assert np.array_equal(bits(o), bits(np.broadcast_to(bg, o.shape)))
    # flat shading (the first vertex's normal): a few paths run into maxBounce; those pixels lose exactly the samples
    # that were cut, and no other pixel changes
    out, _ = glass.render(sc, cam, env, W * W, spp, 8, grey, rng_mode=rng, seed=5, sampling=G)
    o = out.reshape(-1, 3)
    one = o[~hit][0][0]   # what every sample that escapes adds
    allowed = [np.float32(np.float32(sum([one] * n, np.float32(0))) / np.float32(spp)) for n in range(spp + 1)]
    assert np.isin(o, allowed).all()
    assert 0 < (o[:, 0] != o[~hit][0][0]).sum() < 0.1 * hit.sum()


def test_ball_lens_turns_the_environment_upside_down():
    W = 32
    sc = gs.glass_sphere()
    cam, env, graded = ss.sphere_view(W)
    mask = (oracle.primary(sc, cam, W * W)["tri"] >= 0).reshape(W, W)
    rows = np.where(mask.any(axis=1))[0]
    r = np.arange(W)[:, None] + np.zeros((1, W))
    top, bottom = mask & (r < (rows[0] + rows[-1]) / 2), mask & (r > (rows[0] + rows[-1]) / 2)

    def gradient(scene, sampling):
        out, _ = glass.render(scene, cam, env, W * W, 32, 8, graded, rng_mode=1, seed=2, sampling=sampling)
        lum = out.reshape(W, W, 3).mean(axis=2)
        return lum[top].mean() - lum[bottom].mean()

    assert gradient(sc, 0) > 0.05                          # pass-through: the sky above, the ground below
    assert gradient(gs.glass_sphere(ior=1.0), G) > 0.05    # an ior of 1 passes through with the bit too
    assert gradient(sc, G) < -0.05                         # a ball lens inverts the image behind it


def test_environment_variable_parsing():
    assert dielectric_glass_from_env("1") is True and dielectric_glass_from_env(" 0 ") is False
    for bad in ("", "2", "yes", "true"):
        with pytest.raises(ValueError):
            dielectric_glass_from_env(bad)
