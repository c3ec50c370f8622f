"""CPU: the oracle's rule probe (oracle_probe/, the record layout of b200rt_rule_probe) calls the same rules as the
oracle's existing per-rule exports — orc_dielectric, orc_rough_dielectric, orc_texel and orc_smooth_normal — and agrees
with them bit for bit on the edge families of tests/rule_probe_cases.py; its uniform words reach the rules as
bits_to_unit(word)."""
import numpy as np
import pytest

from oracle import oracle
from oracle_glass import glass
from oracle_probe import probe as P
from oracle_rough import rough
from oracle_smooth import smooth
from oracle_texture import texture
from tests import fixtures, rule_probe_cases as C, smooth_scene as ss

f32 = np.float32


def same_bits(a, b):
    a, b = np.asarray(a, f32), np.asarray(b, f32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32))


def unit_word(w):
    """bits_to_unit of rt_oracle.c"""
    return (((np.asarray(w, np.uint32) & np.uint32(0x7FFFFF)) | np.uint32(0x40000000)).view(f32) - f32(2)) / f32(2)


def cr(fn, a):
    """the oracle's correctly rounded binary32 function fn at a"""
    return oracle.math_probe(fn, np.asarray(a, f32))


def dot(a, b):
    return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]


@pytest.mark.parametrize("nz", [1.0, -1.0])
def test_fed_samplers_equal_a_restatement_at_z(nz):
    """rules 2-5 at n = +-z (the samplers' z-aligned branch, l = local * n.z) against numpy float32 statements of
    rt_oracle.c's sample_cosine and sample_uniform, fed bits_to_unit of words 12 and 13: the probe's uniforms arrive in
    order and converted as the device converts them"""
    g = np.random.default_rng(7)
    m = 20000
    W = C.word_sets(g, m)
    n = np.tile(f32([0, 0, nz]), (m, 1))
    r = C.pack(np.zeros((m, 3), f32), n, W)
    u, u2 = unit_word(W[:, 0]), unit_word(W[:, 1])
    with np.errstate(all="ignore"):
        theta = (u2 * f32(2)) * f32(3.14)
        rad = np.sqrt(u)
        local = np.stack([rad * cr("cos", theta), rad * cr("sin", theta), np.sqrt(np.maximum(f32(0), f32(1) - u))], 1)
        l = local * f32(nz)
        inv = f32(3.14) / np.maximum(dot(l, n), f32(0))
    for rule in (P.COSINE_FLAT, P.COSINE_SMOOTH):
        out = P.rule_probe(rule, r)
        assert same_bits(out[:, :3], l) and same_bits(out[:, 3], inv)
    phi = f32(2 * f32(3.14)) * u
    th = cr("acos", f32(1) - u2)
    st = cr("sin", th)
    l = np.stack([cr("cos", phi) * st, st * cr("sin", phi), cr("cos", th)], 1) * f32(nz)
    for rule in (P.UNIFORM_FLAT, P.UNIFORM_SMOOTH):
        out = P.rule_probe(rule, r)
        assert same_bits(out[:, :3], l) and (out[:, 3] == f32(2) * f32(3.14)).all()


def ipow(x, k):
    r = np.ones_like(x)
    for _ in range(k):
        r = r * x
    return r


def test_ggx_equals_a_restatement():
    """rule 7 against numpy float32 statements of rt_oracle.c's bsdf_ggx (MathLib.cl:461-500)"""
    g = np.random.default_rng(8)
    r = C.scatter_random(g, P.GGX, 50000)
    f = r.view(f32)
    v, n, l, col, rough = f[:, 0:3], f[:, 3:6], f[:, 6:9], f[:, 9:12], f[:, 12]
    with np.errstate(all="ignore"):
        hs = l + v
        h = hs / np.sqrt(dot(hs, hs))[:, None]
        a2 = ipow(rough, 2)
        D = a2 / (f32(3.14) * ipow(ipow(np.maximum(dot(n, h), f32(0)), 2) * (a2 - f32(1)) + f32(1), 2))
        ndv = np.maximum(dot(n, v), f32(0))
        kk = rough * np.sqrt(f32(2) / f32(3.14))
        g1 = ndv / (ndv * (f32(1) - kk) + kk)
        ndl = np.maximum(dot(n, l), f32(0))
        g2 = ndl / (ndl * (f32(1) - kk) + kk)
        G = g1 * g2
        F = f32(0.04) + (f32(1) - f32(0.04)) * ipow(f32(1) - np.maximum(dot(h, v), f32(0)), 5)
        spec = ((F * G) * D) * (f32(1) / np.maximum((f32(4) * np.maximum(dot(v, n), f32(0))) * np.maximum(dot(l, n), f32(0)),
                                                    f32(0.001)))
        kd = (f32(1) - F) * (f32(1) - f32(0.5))
        want = (col * kd[:, None]) / f32(3.14) + spec[:, None]
    assert same_bits(P.rule_probe(P.GGX, r)[:, :3], want)


def test_light_sample_picks_the_given_emitter_and_point():
    """rule 8: the shadow-ray direction w = y - x to the point (ua, ub) folded into the triangle and the light density
    against numpy float32 statements; the emitter is the record's whatever word 12 and the number of emitters are"""
    sc = fixtures.load_scene("cornell")
    g = np.random.default_rng(9)
    m = 20000
    light = sc["lightData"]
    t = light[g.integers(0, light.size, m)]
    x = g.uniform(-1, 1, (m, 3)).astype(f32)
    W = C.word_sets(g, m)
    r = C.pack(C.sphere(g, m), C.sphere(g, m), W, x=x, i9=t, i10=np.zeros(m), i11=np.full(m, 2))
    out = P.rule_probe(P.LIGHT, r, scene=sc)
    vp = sc["V_p"].reshape(-1, 3)
    face = sc["faceData"].reshape(-1, 10)[t]
    A = vp[face[:, 7]]
    e1, e2 = vp[face[:, 8]] - A, vp[face[:, 9]] - A
    ua, ub = unit_word(W[:, 1]), unit_word(W[:, 2])
    fold = ua + ub > f32(1)
    ua, ub = np.where(fold, f32(1) - ua, ua), np.where(fold, f32(1) - ub, ub)
    w = ((A + e1 * ua[:, None]) + e2 * ub[:, None]) - x
    assert same_bits(out[:, 3:6], w)
    dist2 = dot(w, w)
    wi = w / np.sqrt(dist2)[:, None]
    nl = np.stack([e1[:, 1] * e2[:, 2] - e1[:, 2] * e2[:, 1], e1[:, 2] * e2[:, 0] - e1[:, 0] * e2[:, 2],
                   e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0]], 1)
    area2 = np.sqrt(dot(nl, nl))
    cosl = np.abs(dot(nl, wi)) / area2

    def pl(n_light):
        with np.errstate(all="ignore"):
            return np.where((cosl > 0) & (area2 > 0), dist2 / ((cosl * (f32(n_light) * f32(0.5))) * area2), f32(0))
    assert same_bits(out[:, 6], pl(2))
    r2 = r.copy()
    r2[:, 12] = g.integers(0, 1 << 32, m, dtype=np.uint64).astype(np.uint32)
    r2[:, 11] = 7
    out2 = P.rule_probe(P.LIGHT, r2, scene=sc)
    assert same_bits(out2[:, 3:6], out[:, 3:6]) and same_bits(out2[:, 6], pl(7)) and same_bits(out2[:, 7], out[:, 7])


def test_dielectric_equals_orc_dielectric():
    g = np.random.default_rng(1)
    r = np.concatenate([C.scatter_edges(g, P.DIELECTRIC), C.scatter_random(g, P.DIELECTRIC, 20000)])
    f = r.view(f32)
    f[:, 6] = np.where(f[:, 6] == 0, f32(1.5), f[:, 6])   # orc_dielectric resolves slot 0 to the default ior first
    out = P.rule_probe(P.DIELECTRIC, r, threads=4)
    d, refl, _ = glass.dielectric(f[:, 0:3], f[:, 3:6], f[:, 6], unit_word(r[:, 12]))
    assert same_bits(out[:, :3], d) and np.array_equal(out[:, 3] == 1, refl.astype(bool))


def test_rough_dielectric_equals_orc_rough_dielectric():
    g = np.random.default_rng(2)
    r = np.concatenate([C.scatter_edges(g, P.ROUGH_DIELECTRIC), C.scatter_random(g, P.ROUGH_DIELECTRIC, 20000)])
    f = r.view(f32)
    f[:, 6] = np.where(f[:, 6] == 0, f32(1.5), f[:, 6])
    out = P.rule_probe(P.ROUGH_DIELECTRIC, r, threads=4)
    d, refl, wt = rough.rough_dielectric(f[:, 0:3], f[:, 3:6], f[:, 6], f[:, 7], *(unit_word(r[:, k]) for k in (12, 13, 14)))
    assert same_bits(out[:, :3], d) and np.array_equal(out[:, 3] == 1, refl) and same_bits(out[:, 4], wt)


def test_texel_equals_orc_texel():
    g = np.random.default_rng(3)
    shapes = [(1, 1), (1, 7), (7, 1), (5, 3), (64, 33)]
    imgs = [g.integers(0, 256, (h, w, 4), dtype=np.uint8) for w, h in shapes]
    texels = np.concatenate([a.reshape(-1) for a in imgs])
    dims = np.array(shapes, np.int32).reshape(-1)
    u, v = C.uv_cases(g, 4000)
    for k, img in enumerate(imgs):
        x = np.zeros((u.size, 3), f32)
        x[:, 0], x[:, 1] = u, v
        r = C.pack(np.zeros_like(x), np.zeros_like(x), x=x, i9=np.full(u.size, k))
        out = P.rule_probe(P.TEXEL, r, tex=(texels, dims, np.zeros(1, np.int32)))
        assert same_bits(out[:, :3], texture.texel(img, u, v))


def test_smooth_normal_equals_orc_smooth_normal():
    g = np.random.default_rng(4)
    for sc in (fixtures.load_scene("monkey"), ss.sphere(16, 8)):
        nt = sc["faceData"].size // 10
        x, t = C.points_on(sc, g.integers(0, nt, 2000).astype(np.int32), g)
        r = C.pack(np.zeros((len(t), 3), f32), np.zeros((len(t), 3), f32), x=x, i9=t)
        out = P.rule_probe(P.SMOOTH_NORMAL, r, scene=sc)
        assert same_bits(out[:, :3], smooth.smooth_normal(sc, t, x))
        assert np.array_equal(out[:, 3] == 1, ss.curved(sc)[t])
