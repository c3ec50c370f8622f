"""CPU: the oracle's adaptive-sampling mode (oracle_adaptive/, the rule include/b200rt.h states for b200rt_adaptive)
against the plain oracle and against a numpy restatement of the rule, and the launcher's B200RT_ADAPTIVE parsing."""
import numpy as np
import pytest

from ensem3a_openclraytracer_b200.KernelLauncher import adaptive_from_env
from oracle import oracle
from oracle_adaptive import adaptive
from tests import fixtures

RNGS = [oracle.RNG_REFERENCE, oracle.RNG_PHILOX]


def bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.uint32)


def ray_free(sc, cam, img_dim, i0, i1):
    """pixels of [i0, i1) whose samples need no ray: primary miss or emitter (what the GPU's primary-hit kernel finishes)"""
    p = oracle.primary(sc, cam, img_dim, i0, i1)
    mat_type = sc["materialData"][6 * np.maximum(p["mat"], 0)].astype(np.int32)
    return (p["tri"] < 0) | (mat_type == 0)


@pytest.mark.parametrize("rng", RNGS)
@pytest.mark.parametrize("name,sampling", [("cornell", 0), ("monkey_cfg2", 3)])
def test_min_spp_equal_to_spp_is_the_plain_render(name, sampling, rng):
    sc, ibl = fixtures.load_scene(name), fixtures.load_ibl()
    res, spp = 40, 8
    cam, env = fixtures.cam_env(sc["params"], res)
    want, cnt = oracle.render(sc, cam, env, res * res, spp, 4, ibl, rng_mode=rng, seed=11, sampling=sampling)
    got, n, err, acnt = adaptive.render(sc, cam, env, res * res, spp, 4, ibl, dict(rel_error=1e30, min_spp=spp),
                                        rng_mode=rng, seed=11, sampling=sampling)
    assert np.array_equal(bits(got), bits(want))
    assert np.all(n == spp)
    assert acnt["rays"] == cnt["rays"]
    free = ray_free(sc, cam, res * res, 0, res * res)
    assert free.any() and not free.all()
    assert np.all(err[free] == 0) and np.mean(err[~free] > 0) > 0.5


@pytest.mark.parametrize("rng", RNGS)
@pytest.mark.parametrize("name,res,rows", [("cornell", 64, (20, 36)), ("monkey_cfg2", 96, (40, 52))])
def test_a_pixel_that_stops_after_n_samples_is_the_render_at_spp_n(name, res, rows, rng):
    """prefix-mean semantics: every pixel equals, bit for bit, the plain render of that pixel at spp = its sample count"""
    sc, ibl = fixtures.load_scene(name), fixtures.load_ibl()
    spp = 32
    cam, env = fixtures.cam_env(sc["params"], res)
    i0, i1 = rows[0] * res, rows[1] * res
    got, n, err, _ = adaptive.render(sc, cam, env, res * res, spp, 4, ibl, dict(rel_error=0.2, min_spp=4, check_every=4),
                                     i0=i0, i1=i1, rng_mode=rng, seed=3)
    band = slice(i0, i1)
    assert np.all(n[:i0] == 0) and np.all(n[i1:] == 0) and np.all(got[:3 * i0] == 0)
    nb = n[band]
    assert np.mean(nb < spp) > 0.5, "the tolerance should stop most pixels early"
    assert len(np.unique(nb)) > 2
    assert set(np.unique(nb)) <= set(range(4, spp, 4)) | {spp}
    img = got.reshape(-1, 3)
    for k in np.unique(nb):
        want, _ = oracle.render(sc, cam, env, res * res, int(k), 4, ibl, i0=i0, i1=i1, rng_mode=rng, seed=3)
        sel = np.nonzero(n == k)[0]
        assert np.array_equal(bits(img[sel]), bits(want.reshape(-1, 3)[sel])), f"pixels that took {k} samples"
    free = ray_free(sc, cam, res * res, i0, i1)
    assert np.all(nb[free] == spp) and np.all(err[band][free] == 0)


def restated_rule(y, min_spp, check_every, rel_error, floor, exempt):
    """the rule of b200rt.h in numpy float32 (every operation rounded to binary32; fmin / fmax ignore a NaN like C's)"""
    spp, npix = y.shape
    f = np.float32
    mean, m2 = np.zeros(npix, f), np.zeros(npix, f)
    n = np.full(npix, spp, np.int32)
    running = ~exempt
    for k in range(1, spp + 1):
        delta = y[k - 1] - mean
        new_mean = mean + delta / f(k)
        new_m2 = m2 + delta * (y[k - 1] - new_mean)
        mean = np.where(running, new_mean, mean)
        m2 = np.where(running, new_m2, m2)
        if k >= min_spp and (k - min_spp) % check_every == 0 and k < spp:
            v = (m2 / f(k - 1)) / f(k)
            e = f(rel_error) * np.fmax(np.fmin(mean, f(1.0)), f(floor))
            with np.errstate(invalid="ignore"):
                stop = running & (v <= e * e)
            n[stop] = k
            running &= ~stop
    with np.errstate(invalid="ignore"):
        err = np.sqrt((m2 / (n - 1).astype(f)) / n.astype(f))
    return n, np.where(exempt, f(0.0), err).astype(f)


def single_samples(sc, cam, env, img_dim, spp, ibl, i0, i1, **kw):
    """each sample's own contribution: Philox sample ranges [s, s+1) as raw sums"""
    out = []
    for s in range(spp):
        r, _ = oracle.render(sc, cam, env, img_dim, spp, 4, ibl, i0=i0, i1=i1, rng_mode=oracle.RNG_PHILOX, s0=s,
                             s1=s + 1, raw_sums=True, **kw)
        out.append(r.reshape(-1, 3)[i0:i1])
    return np.stack(out)


def luminance(c):
    f = np.float32
    return (f(0.2126) * c[..., 0] + f(0.7152) * c[..., 1]) + f(0.0722) * c[..., 2]


@pytest.mark.parametrize("name,rel_error,floor", [("cornell", 0.15, 0.05), ("monkey_cfg2", 0.3, 0.2)])
def test_numpy_restatement_finds_the_same_counts_and_errors(name, rel_error, floor):
    sc, ibl = fixtures.load_scene(name), fixtures.load_ibl()
    res, spp, min_spp, every = 48, 24, 5, 3
    cam, env = fixtures.cam_env(sc["params"], res)
    i0, i1 = 16 * res, 28 * res
    y = luminance(single_samples(sc, cam, env, res * res, spp, ibl, i0, i1, seed=21))
    n_want, err_want = restated_rule(y, min_spp, every, rel_error, floor, ray_free(sc, cam, res * res, i0, i1))
    _, n, err, _ = adaptive.render(sc, cam, env, res * res, spp, 4, ibl,
                                   dict(rel_error=rel_error, min_spp=min_spp, check_every=every, floor=floor),
                                   i0=i0, i1=i1, rng_mode=oracle.RNG_PHILOX, seed=21)
    assert len(np.unique(n_want)) > 2
    assert np.array_equal(n[i0:i1], n_want)
    assert np.array_equal(bits(err[i0:i1]), bits(err_want))


def test_non_finite_samples_never_stop_early():
    """an infinite environment makes escaped paths Inf or NaN: such a pixel runs to spp whatever the tolerance"""
    sc, ibl = fixtures.load_scene("cornell"), fixtures.load_ibl()
    res, spp, min_spp = 32, 12, 3
    cam, env = fixtures.cam_env(sc["params"], res)
    env = env.copy()
    env[4] = np.inf
    c = single_samples(sc, cam, env, res * res, min_spp, ibl, 0, res * res)
    bad_early = ~np.all(np.isfinite(c), axis=(0, 2))
    free = ray_free(sc, cam, res * res, 0, res * res)
    _, n, err, _ = adaptive.render(sc, cam, env, res * res, spp, 4, ibl, dict(rel_error=1e30, min_spp=min_spp, check_every=1),
                                   rng_mode=oracle.RNG_PHILOX, seed=0)
    assert (bad_early & ~free).any() and (~bad_early & ~free).any()
    assert np.all(n[bad_early] == spp)
    assert np.all(n[~bad_early & ~free] == min_spp)   # a huge tolerance stops every finite pixel at once
    assert np.all(n[free] == spp) and np.all(err[free] == 0)


def test_b200rt_adaptive_environment_variable():
    assert adaptive_from_env("0.02") == {"rel_error": 0.02}
    assert adaptive_from_env(" 0.05 , 32 ") == {"rel_error": 0.05, "min_spp": 32}
    assert adaptive_from_env("0,2,1") == {"rel_error": 0.0, "min_spp": 2, "check_every": 1}
    for bad in ("", "x", "0.02,", "0.02,16,8,4", "-0.1", "nan", "inf", "0.02,1", "0.02,16,0", "0.02,1.5", "0.02,,8"):
        with pytest.raises(ValueError, match="B200RT_ADAPTIVE"):
            adaptive_from_env(bad)
