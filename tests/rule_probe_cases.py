"""Records for b200rt_rule_probe / orc_rule_probe (layout in include/b200rt.h): random ones and the edge families where
the per-hit rules go wrong — axis vectors with signed zeros, normals at and within a few ulp of +-z, denormal, non-unit
and non-finite components, grazing directions, the critical angle, extreme iors and roughnesses, and the uniform words at
the ends and the branch point of [0, 1)."""
import numpy as np

from oracle_probe import probe as P
from tests.test_texture_oracle import _cases

f32 = np.float32

IORS = np.array([0, 1, 0.8, 1.5, 2.4, 1e-30, 1e30], f32)
ROUGHNESS = np.array([1e-38, 1e-6, 1e-3, 0.05, 1, 5, 1e3, 3e38], f32)
# words whose bits_to_unit is 0, 2^-23, 0.5 - 2^-23, 0.5 (the glossy mixture's branch point) and 1 - 2^-23
WORDS = np.array([0, 1, (1 << 22) - 1, 1 << 22, (1 << 23) - 1], np.uint32)


def unit(a):
    a = np.asarray(a, np.float64)
    return (a / np.linalg.norm(a, axis=-1, keepdims=True)).astype(f32)


def sphere(g, m):
    return unit(g.normal(size=(m, 3)))


def axes():
    """the six axis vectors, each with every sign of zero in its other components"""
    out = []
    for k in range(3):
        for s in (1.0, -1.0):
            for z1 in (0.0, -0.0):
                for z2 in (0.0, -0.0):
                    v = [z1, z2]
                    v.insert(k, s)
                    out.append(v)
    return np.array(out, f32)


def near_z():
    """normals within 1 to 4 ulp of +-z, on both sides of |unit(n).z| == 1: a tiny tangential part, or z a few ulp
    below 1 with or without the tangential part that would make them unit"""
    out = []
    for s in (1.0, -1.0):
        for k in range(1, 5):
            z = f32(1) - f32(k) * f32(2.0 ** -24)
            out += [[0, 0, s * z], [np.sqrt(1 - float(z) ** 2), 0, s * z], [k * 2.0 ** -12, 0, s],
                    [0, -k * 2.0 ** -12.5, s], [k * 2.0 ** -13, k * 2.0 ** -13, s]]
    return np.array(out, f32)


def odd_normals():
    """denormal, non-unit (length 0.5 and 2) and non-finite components"""
    d = [[1e-40, 0, 1], [0, -1e-45, -1], [1e-40, 1e-40, 1e-40], [-1e-39, 1, 0], [1e-45, 0, 0]]
    nu = [[0, 0, 0.5], [0, 0, -2], [0.3, 0.4, 0], [1.2, -1.6, 0], [0.5 * 0.6, 0, 0.5 * 0.8], [2 * 0.6, 0, -2 * 0.8]]
    nf = [[np.nan, 0, 1], [0, 0, np.nan], [np.inf, 0, 1], [0, -np.inf, 0], [np.inf, np.inf, np.inf], [0, 0, 0]]
    return np.array(d + nu + nf, f32)


def normals(g, m=24):
    return np.concatenate([axes(), near_z(), odd_normals(), sphere(g, m)])


def grazing(n):
    """directions at cosine c to the unit normal n (per row of n): c == 0 exactly, and |c| from 1e-7 to 1e-1 on both
    sides"""
    n = np.asarray(n, np.float64)
    t = np.cross(n, [0.3, 0.5, 0.7])
    t /= np.linalg.norm(t, axis=1, keepdims=True)
    out = [t.astype(f32)]
    for c in (1e-7, 1e-5, 1e-3, 1e-1):
        for s in (1, -1):
            out.append((t * np.sqrt(1 - c * c) + n * (s * c)).astype(f32))
    return np.concatenate(out)


def directions(g, m=24):
    ax = axes()
    return np.concatenate([ax, near_z(), odd_normals(), grazing(unit(np.array([[0, 0, 1], [0.6, 0, 0.8],
                                                                              [0.48, -0.6, 0.64]]))), sphere(g, m)])


def critical(ior, n=np.array([0, 0, 1], f32), steps=160):
    """directions leaving a medium of index ior (> 1) across the unit normal n whose cosine is swept ulp by ulp through
    the critical angle, so that k = 1 - eta^2 (1 - c^2) passes through 0"""
    cz = np.float32(np.sqrt(1 - 1 / float(ior) ** 2))
    z = cz.view(np.uint32).astype(np.int64) + np.arange(-steps, steps + 1)
    z = z.astype(np.uint32).view(f32)
    x = np.sqrt(np.maximum(0, 1 - z.astype(np.float64) ** 2)).astype(f32)
    d = np.stack([x, np.zeros_like(x), z], 1)
    return d, np.tile(n, (d.shape[0], 1))


def pack(d, n, words=None, x=None, i9=None, i10=None, i11=None, f6=None, f7=None, f12=None, w15=None):
    """records from per-record columns (broadcast); words (m, 3) or a scalar word for all three slots"""
    cols = [np.atleast_1d(np.asarray(a)) for a in (d, n) if a is not None]
    m = max(c.shape[0] for c in cols)
    r = P.records(m)
    f = r.view(f32)
    f[:, 0:3] = d
    f[:, 3:6] = n
    if x is not None:
        f[:, 6:9] = x
    if f6 is not None:
        f[:, 6] = f6
    if f7 is not None:
        f[:, 7] = f7
    if f12 is not None:
        f[:, 12] = f12
    for k, v in ((9, i9), (10, i10), (11, i11), (15, w15)):
        if v is not None:
            r[:, k] = np.asarray(v).astype(np.int64).astype(np.uint32)
    if words is not None:
        r[:, 12:15] = words
    return r


def cross_rows(a, b):
    """every row of a with every row of b"""
    return np.repeat(a, b.shape[0], axis=0), np.tile(b, (a.shape[0], 1))


def word_sets(g, m):
    """m triples of uniform words: the WORDS in every slot combination, then random words"""
    fixed = np.array(np.meshgrid(WORDS, WORDS, WORDS)).reshape(3, -1).T.astype(np.uint32)
    return np.concatenate([fixed, g.integers(0, 1 << 32, (max(0, m - fixed.shape[0]), 3), dtype=np.uint64)
                           .astype(np.uint32)])[:m]


def scatter_edges(g, rule):
    """edge records of the dielectric (0), rough dielectric (1) and the direction samplers (2-6)"""
    d, n = cross_rows(directions(g), normals(g))
    m = d.shape[0]
    W = word_sets(g, m)
    recs = []
    if rule in (0, 1):
        dc, nc = zip(*[critical(v) for v in (1.5, 2.4, 1e30)] + [critical(1.5, unit([[0.3, -0.4, 0.5]])[0])])
        d = np.concatenate([d] + list(dc))
        n = np.concatenate([n] + list(nc))
        m = d.shape[0]
        W = word_sets(g, m)
        for k, ior in enumerate(IORS):
            if rule == 0:
                recs.append(pack(d, n, W, f6=ior))
            else:
                for al in ROUGHNESS:
                    sel = slice(k % 4, None, 4)   # a quarter of the pairs per (ior, roughness)
                    recs.append(pack(d[sel], n[sel], W[sel], f6=ior, f7=al))
    elif rule == P.GLOSSY:
        for al in ROUGHNESS:
            recs.append(pack(d, n, W, f6=al))
    else:
        recs.append(pack(d, n, W))
    return np.concatenate(recs)


def scatter_random(g, rule, m):
    d, n = sphere(g, m), sphere(g, m)
    W = g.integers(0, 1 << 32, (m, 3), dtype=np.uint64).astype(np.uint32)
    if rule == 0:
        return pack(d, n, W, f6=g.choice(np.concatenate([IORS, g.uniform(0.3, 3, 8).astype(f32)]), m))
    if rule == 1:
        al = np.where(g.random(m) < 0.5, g.choice(ROUGHNESS, m), g.uniform(0, 1.5, m)).astype(f32)
        return pack(d, n, W, f6=g.choice(IORS[IORS != 1], m), f7=al)
    if rule == P.GLOSSY:
        return pack(d, n, W, f6=np.where(g.random(m) < 0.5, g.choice(ROUGHNESS, m), g.uniform(0, 1.5, m)).astype(f32))
    if rule == P.GGX:
        col = g.uniform(0, 1, (m, 3)).astype(f32)
        r = pack(d, n, x=sphere(g, m), f12=np.where(g.random(m) < 0.3, g.choice(ROUGHNESS, m),
                                                     g.uniform(0, 1.5, m)).astype(f32))
        r.view(f32)[:, 9:12] = col
        return r
    return pack(d, n, W)


def ggx_edges(g):
    v, n = cross_rows(directions(g, 8), normals(g, 8))
    l = np.roll(v, 7, axis=0)
    recs = []
    for al in np.concatenate([ROUGHNESS, [0, 0.3]]).astype(f32):
        r = pack(v, n, x=l, f12=al)
        r.view(f32)[:, 9:12] = [0.8, 0.5, 0.2]
        recs.append(r)
    return np.concatenate(recs)


def points_on(scene, tris, g):
    """per triangle: inside, at each vertex, on each edge's midpoint and just outside (b < 0), as float32"""
    vp = scene["V_p"].reshape(-1, 3).astype(np.float64)
    face = scene["faceData"].reshape(-1, 10)[tris]
    A, B, Cc = vp[face[:, 7]], vp[face[:, 8]], vp[face[:, 9]]
    u, v = g.random(len(tris)), g.random(len(tris))
    flip = u + v > 1
    u[flip], v[flip] = 1 - u[flip], 1 - v[flip]
    pts = [A + (B - A) * u[:, None] + (Cc - A) * v[:, None], A, B, Cc, (A + B) / 2, (B + Cc) / 2, (A + Cc) / 2,
           A - 1e-3 * (B - A) - 1e-3 * (Cc - A), B + 0.02 * (B - Cc)]
    return np.concatenate(pts).astype(f32), np.tile(tris, len(pts)).astype(np.int32)


def uv_cases(g, m):
    """the UVs of tests/test_texture_oracle._cases, |u| from 2^23 to 2^30 (fu == 0), -2^-149, and u just below an
    integer, where u - floorf(u) rounds to 1"""
    u, v = _cases(g, m)
    big = np.concatenate([2.0 ** np.arange(23, 31), -(2.0 ** np.arange(23, 31)), 2.0 ** np.arange(23, 31) + 1]).astype(f32)
    below = np.nextafter(np.array([1, 2, -1, 0, 7, -3, 1e4], f32), f32(-np.inf))
    tiny = np.array([-2.0 ** -149, 2.0 ** -149, -0.0, 0.0], f32)
    extra = np.concatenate([big, below, tiny])
    eu = np.repeat(extra, extra.size)
    ev = np.tile(extra, extra.size)
    return np.concatenate([u, eu, ev[: eu.size // 2], g.uniform(-3, 3, eu.size // 2).astype(f32)]), \
        np.concatenate([v, ev, g.uniform(-3, 3, eu.size // 2).astype(f32), eu[: eu.size // 2]])
