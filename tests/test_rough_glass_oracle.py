"""CPU: opt-in rough glass (B200RT_SAMPLING_ROUGH_GLASS).  The oracle's rough interface rule against a numpy
restatement, bit for bit, on random and edge cases; the estimator against a float64 quadrature of Walter et al.'s
microfacet BSDF, bin by bin; roughness 0 and ior 1 render as without the bit, bit for bit; the image converges to the
smooth-glass one as the roughness goes to 0; the white furnace; a rough slab blurs the checker behind it; the launcher's
environment variable."""
import numpy as np
import pytest
from scipy.special import roots_legendre

from ensem3a_openclraytracer_b200.KernelLauncher import rough_glass_from_env
from oracle import oracle
from oracle_rough import rough
from oracle_texture import texture
from tests import fixtures, glass_scene as gs, rough_glass_scene as rs

f32 = np.float32
G, R = rs.GLASS, rs.ROUGH
GR = G | R


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


def same_bits(a, b):
    """bit for bit, every NaN counting as one value (the sign of a NaN is not part of the rule)"""
    a, b = np.asarray(a, f32), np.asarray(b, f32)
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(bits(a)[~np.isnan(a)], bits(b)[~np.isnan(b)])


def unit_rows(a):
    a = np.asarray(a, f32)
    return (a / np.sqrt(gs._dot(a, a))[:, None]).astype(f32)


def same_rule(w, n, v, r, uf, u1, u2):
    d, refl, wt = rough.rough_dielectric(w, n, v, r, uf, u1, u2)
    d2, refl2, wt2 = rs.rough_dielectric(w, n, v, r, uf, u1, u2)
    assert np.array_equal(refl, refl2)
    assert same_bits(wt, wt2)
    assert same_bits(d, d2)
    return d, refl, wt


def test_rule_bit_for_bit_random():
    rng = np.random.default_rng(17)
    m = 100_000
    w = rng.normal(size=(m, 3)).astype(f32) * rng.uniform(0.2, 3.0, size=(m, 1)).astype(f32)
    n = unit_rows(rng.normal(size=(m, 3)))
    v = rng.uniform(0.3, 3.0, size=m).astype(f32)
    v[::7] = 0.0
    r = np.exp(rng.uniform(np.log(1e-3), np.log(2.0), size=m)).astype(f32)
    uf, u1, u2 = (rng.random(m, dtype=np.float32) for _ in range(3))
    d, refl, wt = same_rule(w, n, v, r, uf, u1, u2)
    assert 0.02 < refl.mean() < 0.6   # both outcomes occur
    assert 0.01 < (wt == 0).mean() < 0.3 and ((wt >= 0) & (wt <= 1)).all()   # some go to the wrong side
    assert np.isfinite(d).all()


def test_rule_bit_for_bit_edge_cases():
    rng = np.random.default_rng(5)
    m = 4000
    z = np.repeat(np.array([[0, 0, 1]], f32), m, axis=0)
    uf, u1, u2 = (rng.random(m, dtype=np.float32) for _ in range(3))
    w = unit_rows(rng.normal(size=(m, 3)))
    # tiny and large roughness, ior < 1 (a bubble) and > 1, slot 0 (the default)
    for r in (1e-6, 1e-3, 0.05, 1.0, 5.0, 1e3):
        for v in (0.0, 1.5, 0.75, 2.4):
            d, refl, wt = same_rule(w, z, np.full(m, v, f32), np.full(m, r, f32), uf, u1, u2)
            assert np.isfinite(d).all()
    # a tiny roughness scatters like the smooth interface (same uf)
    d, refl, wt = same_rule(w, z, np.full(m, 1.5, f32), np.full(m, 1e-6, f32), uf, u1, u2)
    d0, r0, _ = gs.dielectric(w, z, np.full(m, 1.5, f32), uf)
    assert (refl == r0).mean() > 0.999 and np.abs(d - d0).max() < 1e-3 and (wt > 0.999).all()
    # grazing incidence, both sides, just off c == 0
    gz = np.stack([np.ones(m), np.zeros(m), rng.choice([-1, 1], m) * 10.0 ** rng.uniform(-7, -1, m)], axis=1)
    same_rule(gz, z, np.full(m, 1.5, f32), np.full(m, 0.3, f32), uf, u1, u2)
    # c == 0 exactly, a non-finite normal, a roughness whose h underflows or overflows: bit 128's rule with uf, weight 1
    x = np.repeat(np.array([[1, 0, 0]], f32), m, axis=0)
    bad_n = np.array([[np.nan, 0, 1], [np.inf, 0, 0], [0, 0, np.nan]], f32)
    for ww, nn, r in ((x, z, 0.3), (w[:3], bad_n, 0.3), (w, z, 1e-38)):
        k = len(ww)
        v = np.full(k, 1.5, f32)
        d, refl, wt = same_rule(ww, nn, v, np.full(k, r, f32), uf[:k], u1[:k], u2[:k])
        d0, r0, _ = gs.dielectric(ww, nn, v, uf[:k])
        with np.errstate(all="ignore"):
            fb = ~np.isfinite(rs.visible_normal(np.full(k, r, f32), nn, -ww, u1[:k], u2[:k])).all(axis=1)
        if r < 1e-30:
            assert fb.any() and (~fb).any()   # a roughness of 1e-38 underflows h for some draws only
        fb |= r == 0.3
        assert (wt[fb] == 1).all() and np.array_equal(refl[fb], r0[fb]) and same_bits(d[fb], d0[fb])
    # a roughness of 3e38 overflows the visible-normal statements: still the rule, with finite weights in [0, 1]
    d, refl, wt = same_rule(w, z, np.full(m, 1.5, f32), np.full(m, 3e38, f32), uf, u1, u2)
    assert ((wt >= 0) & (wt <= 1)).all() and (wt == 0).any()
    # total internal reflection: leaving glass of 1.5 at 60 degrees from the normal (critical angle 42) nearly always reflects
    lv = np.repeat(np.array([[np.sin(1.05), 0, np.cos(1.05)]], f32), m, axis=0)
    d, refl, wt = same_rule(lv, z, np.full(m, 1.5, f32), np.full(m, 0.05, f32), uf, u1, u2)
    assert refl.mean() > 0.99
    # the weight-0 branches: reflections below and refractions above the macro surface, at high roughness and grazing
    # incidence on a medium of lower index (ior 0.8)
    gr = unit_rows(np.stack([np.ones(m), np.zeros(m), -np.full(m, 0.05)], axis=1))
    d, refl, wt = same_rule(gr, z, np.full(m, 0.8, f32), np.full(m, 1.0, f32), uf, u1, u2)
    assert (wt[refl] == 0).any() and (wt[~refl] == 0).any()
    assert ((d[refl & (wt == 0), 2] <= 0)).all() and ((d[~refl & (wt == 0), 2] >= 0)).all()


# ---- the estimator against float64 quadrature of Walter et al.'s BSDF --------------------------------------------------
def _g1(a2, c):
    c = np.abs(c)
    return 2 * c / (c + np.sqrt(a2 + (1 - a2) * c * c))


def _fresnel(eta, ci):
    k = 1 - eta * eta * (1 - ci * ci)
    ct = np.sqrt(np.maximum(k, 0))
    rs_ = (eta * ci - ct) / (eta * ci + ct)
    rp = (ci - eta * ct) / (ci + eta * ct)
    return np.where(k >= 0, 0.5 * (rs_ * rs_ + rp * rp), 1.0)


def walter_cos(i, l, al, eta):
    """float64: f(i, l) |l.m| of Walter et al. (2007), m = +z the normal on the incident side, i the unit direction
    towards the viewer, eta = n_incident / n_transmitted, separable Smith G2 = G1(i) G1(l), the rule's Fresnel formula"""
    a2 = al * al

    def D(h):
        c = h[..., 2]
        return np.where(c > 0, a2 / (np.pi * (c * c * (a2 - 1) + 1) ** 2), 0.0)

    ci_m = i[2]
    lz = l[..., 2]
    g2 = _g1(a2, ci_m) * _g1(a2, lz)
    hr = i + l
    hr = hr / np.linalg.norm(hr, axis=-1, keepdims=True)
    ih = hr @ i
    refl = np.where((lz > 0) & (ih > 0), _fresnel(eta, ih) * D(hr) * g2 / (4 * ci_m), 0.0)
    ht = -(eta * i + l)
    ht = ht / np.linalg.norm(ht, axis=-1, keepdims=True)
    ht = np.where(ht[..., 2:3] < 0, -ht, ht)
    ih, lh = ht @ i, np.sum(l * ht, axis=-1)
    ok = (lz < 0) & (ih > 0) & (lh < 0)
    tr = np.where(ok, np.abs(ih * lh) * (1 - _fresnel(eta, ih)) * D(ht) * g2 / (ci_m * (eta * ih + lh) ** 2), 0.0)
    return refl + tr


N_TH, N_PH, Q = 36, 12, 24


def _bins_quadrature(i, al, eta):
    x, wq = roots_legendre(Q)
    th_e = np.linspace(0, np.pi, N_TH + 1)
    ph_e = np.linspace(-np.pi, np.pi, N_PH + 1)
    out = np.zeros((N_TH, N_PH))
    for a in range(N_TH):
        th = 0.5 * (th_e[a + 1] - th_e[a]) * x + 0.5 * (th_e[a + 1] + th_e[a])
        wt = 0.5 * (th_e[a + 1] - th_e[a]) * wq * np.sin(th)
        for b in range(N_PH):
            ph = 0.5 * (ph_e[b + 1] - ph_e[b]) * x + 0.5 * (ph_e[b + 1] + ph_e[b])
            wp = 0.5 * (ph_e[b + 1] - ph_e[b]) * wq
            T, P = np.meshgrid(th, ph, indexing="ij")
            l = np.stack([np.sin(T) * np.cos(P), np.sin(T) * np.sin(P), np.cos(T)], axis=-1)
            out[a, b] = np.sum(walter_cos(i, l, al, eta) * np.outer(wt, wp))
    return out


@pytest.mark.parametrize("r", [0.05, 0.3, 1.0])
@pytest.mark.parametrize("ior", [1.5, 0.8])
@pytest.mark.parametrize("enter", [True, False])
def test_estimator_matches_walter_bsdf_bin_by_bin(r, ior, enter):
    """the mean of weight * 1{nd in bin} over 10^6 draws of the rule equals the float64 integral of f |cos| over the bin,
    within 5 sigma (plus a small absolute tolerance); both reflection and transmission are binned"""
    th_i = 0.6
    i = np.array([np.sin(th_i), 0.0, np.cos(th_i)])   # towards the viewer, m = +z on the incident side
    n_draw = 1_000_000
    rng = np.random.default_rng(11)
    w = np.repeat((-i)[None, :].astype(f32), n_draw, axis=0)
    # entering: un faces the viewer; leaving: un points away from it; m, the normal on the incident side, is +z either way
    un = np.repeat(np.array([[0, 0, 1 if enter else -1]], f32), n_draw, axis=0)
    uf, u1, u2 = (rng.random(n_draw, dtype=np.float32) for _ in range(3))
    d, refl, wt = rough.rough_dielectric(w, un, np.full(n_draw, ior, f32), np.full(n_draw, r, f32), uf, u1, u2)
    eta = 1.0 / ior if enter else ior
    d = d.astype(np.float64)
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    th = np.arccos(np.clip(d[:, 2], -1, 1))
    ph = np.arctan2(d[:, 1], d[:, 0])
    a = np.minimum((th / np.pi * N_TH).astype(int), N_TH - 1)
    b = np.minimum(((ph + np.pi) / (2 * np.pi) * N_PH).astype(int), N_PH - 1)
    k = a * N_PH + b
    wt64 = wt.astype(np.float64)
    s1 = np.bincount(k, wt64, N_TH * N_PH) / n_draw
    s2 = np.bincount(k, wt64 * wt64, N_TH * N_PH) / n_draw
    sigma = np.sqrt(np.maximum(s2 - s1 * s1, 0) / n_draw)
    want = _bins_quadrature(i, r, eta).reshape(-1)
    assert want.sum() > 0.3 and refl.any() and (~refl).any()
    upper = np.arange(N_TH * N_PH) // N_PH < N_TH // 2
    assert want[upper].sum() > 0.002 and want[~upper].sum() > 0.002   # reflection and transmission both weigh
    tol = 5 * sigma + 2e-5 + 1e-3 * want
    bad = np.abs(s1 - want) > tol
    assert not bad.any(), (np.where(bad)[0], s1[bad], want[bad], sigma[bad])
    assert abs(s1.sum() - want.sum()) < 5 * np.sqrt(np.var(wt64) / n_draw) + 1e-3


# ---- renders --------------------------------------------------------------------------------------------------------------
def _renders(sc, name, res, sampling_tex, sampling_rough, rng, spp=4, bounce=4, seed=9):
    ibl = fixtures.load_ibl()
    cam, env = rs.view(name, res)
    kw = dict(rng_mode=rng, seed=seed)
    return (texture.render(sc, cam, env, res * res, spp, bounce, ibl, sampling=sampling_tex, **kw),
            rough.render(sc, cam, env, res * res, spp, bounce, ibl, sampling=sampling_rough, **kw))


@pytest.mark.parametrize("name", ["monkey_cfg2", "proto"])
@pytest.mark.parametrize("base", [0, 2, 8, 32])
def test_zero_roughness_is_the_smooth_interface(name, base):
    sc = rs.glass_roughness(fixtures.load_scene(name), 0.0)
    for rng in (0, 1):
        (a, ca), (b, cb) = _renders(sc, name, 24, G | base, GR | base, rng)
        assert np.array_equal(bits(a), bits(b)) and ca == cb


@pytest.mark.parametrize("name", ["monkey_cfg2", "proto"])
def test_without_the_bit_and_at_ior_one_nothing_changes(name):
    sc = rs.glass_roughness(fixtures.load_scene(name), 0.5)
    for rng in (0, 1):
        for base in (0, G, G | 32):
            (a, ca), (b, cb) = _renders(sc, name, 24, base, base, rng)
            assert np.array_equal(bits(a), bits(b)) and ca == cb
        pane = gs.glass_ior(sc, 1.0)   # an ior-1 pane stays a pass-through at any roughness
        (a, ca), (b, cb) = _renders(pane, name, 24, G, GR, rng)
        assert np.array_equal(bits(a), bits(b)) and ca == cb
    # and a rough glass material does change the image
    (a, _), (b, _) = _renders(sc, name, 24, G, GR, 1)
    assert not np.array_equal(bits(a), bits(b))


def test_converges_to_smooth_glass_as_roughness_goes_to_zero():
    """proto at roughness 1e-3 against the smooth interface: the difference of two independent renders is the noise of
    two smooth renders (another seed)"""
    name, res, spp = "proto", 32, 32
    sc = fixtures.load_scene(name)
    ibl = fixtures.load_ibl()
    cam, env = rs.view(name, res)

    def img(scene, sampling, seed):
        return rough.render(scene, cam, env, res * res, spp, 4, ibl, rng_mode=1, seed=seed, sampling=sampling)[0]

    def rmse(a, b):
        return float(np.sqrt(np.mean((a.astype(np.float64) - b) ** 2)))

    smooth_a, smooth_b = img(sc, G, 1), img(sc, G, 2)
    noise = rmse(smooth_a, smooth_b)
    assert rmse(img(rs.glass_roughness(sc, 1e-3), GR, 2), smooth_a) < 1.1 * noise


FURNACE_R = (0.0, 0.1, 0.3, 0.6, 1.0)
# Measured on the oracle (white sphere, 32 x 32, 64 spp, Philox seed 5, smooth shading, maxBounce 12), loss of energy
# against the background at FURNACE_R: 0, 0.073, 0.280, 0.524, 0.703 (standard errors 0.004 - 0.007).  Most of it is the
# single-scattering Smith term seen from inside the glass: one exit at normal incidence keeps 0.989 of the throughput at
# roughness 0.1 and 0.417 at roughness 1 (entering: 0.999 and 0.893).
FURNACE_MIN_LOSS_AT_1 = 0.65


def test_white_rough_glass_furnace():
    """a white rough glass sphere in the uniform grey map: no pixel gains energy (the mean over the sphere is at most the
    background within noise), and the loss of energy (single-scattering Smith term, paths cut at maxBounce) does not
    decrease as the roughness grows"""
    W, spp = 32, 64
    cam, env, grey = gs.grey_view(W)
    loss = []
    for r in FURNACE_R:
        sc = rs.glass_roughness(gs.glass_sphere(), r)
        hit = oracle.primary(sc, cam, W * W)["tri"] >= 0
        out, _ = rough.render(sc, cam, env, W * W, spp, 12, grey, rng_mode=1, seed=5, sampling=GR | 32)
        o = out.reshape(-1, 3)[:, 0].astype(np.float64)
        bg = o[~hit][0]
        mean = o[hit].mean()
        se = o[hit].std() / np.sqrt(hit.sum())
        assert mean <= bg + 3 * se + 1e-6
        loss.append((1 - mean / bg, se / bg))
    for (l0, s0), (l1, s1) in zip(loss, loss[1:]):
        assert l1 >= l0 - 3 * np.hypot(s0, s1)
    assert loss[0][0] < 1e-6 and loss[-1][0] > FURNACE_MIN_LOSS_AT_1


def test_rough_slab_blurs_the_checker_behind_it():
    """the checker seen through a glass slab loses contrast monotonically with the roughness: the amplitude of the
    smooth slab's image in each rough image (its projection on the zero-mean smooth image) decreases"""
    W, spp = 32, 64
    cam, env, checker = rs.checker_view(W)
    imgs = []
    for r in (0.0, 0.05, 0.2, 0.5):
        out, _ = rough.render(rs.slab(r), cam, env, W * W, spp, 8, checker, rng_mode=1, seed=3, sampling=GR)
        imgs.append(out.reshape(-1, 3).mean(axis=1).astype(np.float64))
    ref = imgs[0] - imgs[0].mean()
    assert ref.std() > 0.3   # the smooth slab shows the checker
    amp = [float(np.dot(x - x.mean(), ref) / np.dot(ref, ref)) for x in imgs]
    assert all(a1 < a0 for a0, a1 in zip(amp, amp[1:])), amp
    assert amp[-1] < 0.6 * amp[0], amp


def test_environment_variable_parsing():
    assert rough_glass_from_env("1") is True and rough_glass_from_env(" 0 ") is False
    for bad in ("", "2", "yes", "true"):
        with pytest.raises(ValueError):
            rough_glass_from_env(bad)
