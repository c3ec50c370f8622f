"""GPU: the per-hit shading rules of k_shade one record at a time (b200rt_rule_probe).

Part A — device against oracle (oracle_probe/), bit for bit (NaN counts as one value, flags exactly): 2^22 random records
per rule and the edge families of tests/rule_probe_cases.py — signed-zero axis vectors, normals at and within a few ulp
of +-z, denormal, non-unit and non-finite components, grazing directions, the critical angle, extreme iors and
roughnesses, the uniform words at the ends and the branch point of [0, 1); shading normals and albedos on triangles of
monkey_cfg2, serre and a UV sphere at their vertices, edges, insides and just outside; texels of sizes 1x1 to 2^24 x 1
bound together, and one binding of 2^31 - 1 texels; light samples on the lit Cornell box and monkey_cfg2.

Part B — the densities, no oracle involved: 10^8 device draws per case histogrammed in float64.  For the cosine and
uniform samplers the mean of inv_pdf 1{l in bin} must be the solid angle above the surface of the bin in the samplers'
own frame, whose phi stops at 2 * 3.14; for the glossy sampler (3.14 / pi) times the bin's solid angle;
for the light sampler the mean of g(wi) / p_light must be the float64 quadrature of g cosL / dist^2 over the emitters;
for rough glass the mean of weight 1{nd in bin} must be the quadrature of Walter et al.'s BSDF times |cos|.  Tolerance:
5 sigma of the sample mean plus the quadrature error (Q against 2Q nodes).  About 4 minutes on one B200."""
import os
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest
from scipy.special import roots_legendre

import ensem3a_openclraytracer_b200 as rt
from oracle_probe import probe as P
from tests import fixtures, rule_probe_cases as C, smooth_scene as ss, texture_scene as ts
from tests.test_rough_glass_oracle import walter_cos

pytestmark = pytest.mark.gpu

f32 = np.float32
THREADS = max(1, os.cpu_count() or 1)
POOL = min(THREADS, 8)      # part B: chunks in flight on the host (each holds about 0.5 GB)
N_RANDOM = 1 << 22
CHUNK = 1 << 22
N_DRAW = 100_000_000


@pytest.fixture(scope="module")
def ctx():
    c = rt.Context(0)
    yield c
    c.close()


def same_bits(a, b):
    """bit for bit, every NaN counting as one value"""
    a, b = np.asarray(a, f32), np.asarray(b, f32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32))


def agree(ctx, rule, recs, scene=None, tex=None):
    got = ctx.rule_probe(rule, recs)
    want = P.rule_probe(rule, recs, scene, tex, THREADS)
    if not same_bits(got, want):
        bad = ~((got.view(np.uint32) == want.view(np.uint32)) | (np.isnan(got) & np.isnan(want))).all(axis=1)
        i = np.nonzero(bad)[0]
        raise AssertionError(f"rule {rule}: {i.size} of {len(recs)} records differ, first {i[:4]}\n"
                             f"in {recs[i[:4]].view(f32)}\ndevice {got[i[:4]]}\noracle {want[i[:4]]}")
    return got


# ---- part A: device = oracle ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("rule", [P.DIELECTRIC, P.ROUGH_DIELECTRIC, P.COSINE_FLAT, P.COSINE_SMOOTH, P.UNIFORM_FLAT,
                                  P.UNIFORM_SMOOTH, P.GLOSSY, P.GGX])
def test_scatter_rules_equal_the_oracle(ctx, rule):
    g = np.random.default_rng(100 + rule)
    recs = [C.scatter_random(g, rule, N_RANDOM), C.ggx_edges(g) if rule == P.GGX else C.scatter_edges(g, rule)]
    agree(ctx, rule, np.concatenate(recs))


def test_dielectric_with_a_nan_fresnel_term_reflects(ctx):
    """ior 1 at c == 0: k = 0, ct = 0 and F = 0/0; the rule's !(u >= F) reflects"""
    ax = C.axes()
    d, n = C.cross_rows(ax, ax)
    perp = (np.abs(d) * np.abs(n)).sum(axis=1) == 0
    d, n = d[perp], n[perp]
    out = agree(ctx, P.DIELECTRIC, C.pack(d, n, C.word_sets(np.random.default_rng(2), len(d)), f6=f32(1)))
    assert len(d) > 100 and (out[:, 3] == 1).all()


def test_signed_zero_cosines(ctx):
    """A -0 at a clamp whose sign reaches an output.  The samplers' fmaxf(dot(l, n), 0) never sees a zero (the sampled
    l has l.z >= sqrt(2^-23) in the sampler's frame), and BSDF_GGX adds its clamped terms to the diffuse one, which
    turns -0 into +0.  The light sample's surface density of a diffuse surface is fmaxf(dot(un, wi), 0) / pi, returned
    as it is: with x on the lamp's plane (z = 0.983449) wi.z is +0, and a normal of zero components (+-0, +-0, +-1)
    makes every product of the dot +-0, so the dot is -0 for about half of the records.  C leaves the sign of
    fmaxf(-0, +0) unspecified; both sides return +0 there, so a -0 cosine gives a density of +0, as +0 does."""
    sc = scene("lit_cornell")
    upload(ctx, sc)
    g = np.random.default_rng(12)
    zs = np.array([[sx, sy, sz] for sx in (0.0, -0.0) for sy in (0.0, -0.0) for sz in (1.0, -1.0)], f32)
    m = 4096
    n = zs[g.integers(0, len(zs), m)]
    x = np.stack([g.uniform(-1, 1, m), g.uniform(-1, 1, m), np.full(m, 0.983449)], 1).astype(f32)
    light = sc["lightData"]
    r = C.pack(C.sphere(g, m), n, C.word_sets(g, m), x=x, i9=light[g.integers(0, light.size, m)], i10=np.zeros(m),
               i11=np.full(m, light.size))
    out = agree(ctx, P.LIGHT, r, sc)
    w = out[:, 3:6]
    wi = w / np.sqrt((w[:, 0] * w[:, 0] + w[:, 1] * w[:, 1]) + w[:, 2] * w[:, 2])[:, None]
    ndl = (n[:, 0] * wi[:, 0] + n[:, 1] * wi[:, 1]) + n[:, 2] * wi[:, 2]
    neg = (ndl == 0) & np.signbit(ndl)
    assert neg.sum() > 200 and (~neg & (ndl == 0)).sum() > 200
    assert (out[ndl == 0, 7] == 0).all() and not np.signbit(out[ndl == 0, 7]).any()


def fallback_scene():
    """the smooth oracle's awkward triangles (tests/test_smooth_oracle.fallback_scene: a zero sum of the vertex normals, a
    NaN normal, collinear vertices) and an ordinary one, each moved to its own place so that the scene has a tree"""
    corners = np.array([[0, 0, 0], [2, 0, 0], [0, 2, 0], [1, 0, 0], [3, 0, 0]], f32)
    vn = np.array([0, 0, 1, 0, 0, -1, 1, 0, 0, np.nan, 0, 0, 0, 1, 0], f32)
    tris = [((0, 1, 2), (0, 1, 2)), ((0, 2, 3), (0, 1, 2)), ((0, 4, 2), (0, 3, 4)), ((0, 4, 2), (0, 1, 2))]
    vp, faces = [], []
    for t, (nrm, pos) in enumerate(tris):
        faces.append([0, 0, 0, 0, *nrm, 3 * t, 3 * t + 1, 3 * t + 2])
        vp += [corners[p] + f32(10 * t) * np.array([1, 1, 1], f32) for p in pos]
    sc = {"V_p": np.array(vp, f32).reshape(-1), "V_n": vn, "V_uv": np.array([0, 0, 1, 0, 0, 1], f32),
          "faceData": np.array(faces, np.int32).reshape(-1), "materialData": np.array([1, 0.8, 0.8, 0.8, 0.5, 1], f32),
          "lightData": np.zeros(0, np.int32)}
    sc["BVH"] = rt.BVH(sc["faceData"], sc["V_p"]).exportArray
    return sc


def scene(name):
    if name == "sphere":
        return ss.sphere(24, 12)
    if name == "fallback":
        return fallback_scene()
    if name == "lit_cornell":   # tests/test_gpu_parity.py's: the lamp at power 5 (the shipped .ini has power 0)
        sc = dict(fixtures.load_scene("cornell"))
        m = sc["materialData"].copy().reshape(-1, 6)
        m[3, 4] = 5.0
        sc["materialData"] = m.reshape(-1)
        return sc
    if name.startswith("textured_"):
        sc = dict(fixtures.load_scene(name[len("textured_"):]))
        uv = np.random.default_rng(1).uniform(-3, 3, sc["V_uv"].size).astype(f32)   # wrapped UVs
        sc["V_uv"] = uv
        return sc
    return fixtures.load_scene(name)


def upload(ctx, sc):
    ctx.set_scene(sc["V_p"], sc["V_n"], sc["V_uv"], sc["faceData"], sc["materialData"], sc["lightData"], sc["BVH"])


@pytest.mark.parametrize("name", ["monkey_cfg2", "serre", "sphere", "fallback"])
def test_smooth_normal_equals_the_oracle(ctx, name):
    sc = scene(name)
    upload(ctx, sc)
    g = np.random.default_rng(3)
    nt = sc["faceData"].size // 10
    tris = np.arange(nt, dtype=np.int32) if nt < 5000 else g.integers(0, nt, 5000).astype(np.int32)
    x, t = C.points_on(sc, tris, g)
    out = agree(ctx, P.SMOOTH_NORMAL, C.pack(np.zeros((len(t), 3), f32), np.zeros((len(t), 3), f32), x=x, i9=t), sc)
    assert np.array_equal(out[:, 3] == 1, ss.curved(sc)[t])


def packed(textures):
    images = list(textures.values())
    texels = np.concatenate([a.reshape(-1) for a in images])
    dims = np.array([[a.shape[1], a.shape[0]] for a in images], np.int32).reshape(-1)
    return texels, dims


@pytest.mark.parametrize("name", ["cornell", "monkey_cfg2", "serre"])
def test_albedo_equals_the_oracle(ctx, name):
    sc = scene("textured_" + name)
    upload(ctx, sc)
    tex = ts.textured(sc, 33, seed=4)
    ctx.set_textures(tex)
    texels, dims = packed(tex)
    mat_tex = np.full(sc["materialData"].size // 6, -1, np.int32)
    for k, m in enumerate(tex):
        mat_tex[m] = k
    g = np.random.default_rng(5)
    nt = sc["faceData"].size // 10
    tris = np.arange(nt, dtype=np.int32) if nt < 5000 else g.integers(0, nt, 5000).astype(np.int32)
    x, t = C.points_on(sc, tris, g)
    mat = sc["faceData"].reshape(-1, 10)[t, 0]
    col = g.uniform(0, 1, (len(t), 3)).astype(f32)
    out = agree(ctx, P.ALBEDO, C.pack(col, np.zeros((len(t), 3), f32), x=x, i9=t, i10=mat), sc, (texels, dims, mat_tex))
    assert not same_bits(out[:, :3], col)
    ctx.set_textures(None)


def texel_records(g, n_tex, m):
    u, v = C.uv_cases(g, m)
    recs = []
    for k in range(n_tex):
        x = np.zeros((u.size, 3), f32)
        x[:, 0], x[:, 1] = u, v
        recs.append(C.pack(np.zeros_like(x), np.zeros_like(x), x=x, i9=np.full(u.size, k)))
    return np.concatenate(recs)


def test_texel_equals_the_oracle_at_every_size(ctx):
    """1x1 to 4096x4096, 2^24 x 1 and 1 x 2^24 bound together: later textures start at large first-texel indices"""
    g = np.random.default_rng(6)
    shapes = [(1, 1), (1, 7), (7, 1), (5, 3), (64, 33), (4096, 4096), (1, 1 << 24), (1 << 24, 1), (3, 5)]   # (w, h)
    imgs = [g.integers(0, 256, (h, w, 4), dtype=np.uint8) for w, h in shapes]
    texels = np.concatenate([a.reshape(-1) for a in imgs])
    dims = np.array(shapes, np.int32).reshape(-1)
    mat_tex = np.arange(len(shapes), dtype=np.int32)
    ctx._call("set_textures", rt._capi._ptr(texels), texels.size, rt._capi._ptr(dims), len(shapes), rt._capi._ptr(mat_tex),
              mat_tex.size)
    agree(ctx, P.TEXEL, texel_records(g, len(shapes), 4000), None, (texels, dims, mat_tex))
    ctx.set_textures(None)


def test_texel_at_the_binding_limit(ctx):
    """2^31 - 1 texels in all (8.6 GB): the last small textures start above index 2^31 - 2^24, where the int32 texel
    index arithmetic of b200rt_set_textures' limit is at its edge"""
    small = [(1, 1), (5, 3), (7, 1), (1, 7), (64, 33)]
    rest = (1 << 31) - 1 - sum(w * h for w, h in small)
    big = [(1 << 24, 1)] * (rest // (1 << 24))
    last = rest - len(big) * (1 << 24)
    shapes = big + [(last, 1)] + small
    total = sum(w * h for w, h in shapes)
    assert total == (1 << 31) - 1
    texels = np.zeros(4 * total, np.uint8)
    g = np.random.default_rng(8)
    tail = sum(w * h for w, h in small) + 4096
    texels[-4 * tail:] = g.integers(0, 256, 4 * tail, dtype=np.uint8)
    first = np.cumsum([0] + [w * h for w, h in shapes])[:-1]
    assert first[-len(small)] > (1 << 31) - (1 << 24)
    dims = np.array(shapes, np.int32).reshape(-1)
    mat_tex = np.zeros(1, np.int32)
    ctx._call("set_textures", rt._capi._ptr(texels), texels.size, rt._capi._ptr(dims), len(shapes), rt._capi._ptr(mat_tex),
              mat_tex.size)
    recs = texel_records(g, len(shapes), 2000)
    keep = recs[:, 9] >= len(big)   # the last big texture and the small ones
    agree(ctx, P.TEXEL, recs[keep], None, (texels, dims, mat_tex))
    ctx.set_textures(None)


def test_hit_rules_random(ctx):
    """2^22 random records each of the shading normal and the albedo (random points on random triangles of the textured
    monkey_cfg2, their vertices, edges and just outside) and of the texel rule (random UVs on nine textures bound
    together)"""
    sc = scene("textured_monkey_cfg2")
    upload(ctx, sc)
    tex = ts.textured(sc, 47, seed=6)
    ctx.set_textures(tex)
    texels, dims = packed(tex)
    mat_tex = np.full(sc["materialData"].size // 6, -1, np.int32)
    for k, m in enumerate(tex):
        mat_tex[m] = k
    g = np.random.default_rng(14)
    nt = sc["faceData"].size // 10
    x, t = C.points_on(sc, g.integers(0, nt, N_RANDOM // 9 + 1).astype(np.int32), g)
    x, t = x[:N_RANDOM], t[:N_RANDOM]
    z = np.zeros((len(t), 3), f32)
    agree(ctx, P.SMOOTH_NORMAL, C.pack(z, z, x=x, i9=t), sc)
    col = g.uniform(0, 1, (len(t), 3)).astype(f32)
    agree(ctx, P.ALBEDO, C.pack(col, z, x=x, i9=t, i10=sc["faceData"].reshape(-1, 10)[t, 0]), sc,
          (texels, dims, mat_tex))

    shapes = [(1, 1), (1, 7), (7, 1), (5, 3), (64, 33), (4096, 4096), (1, 1 << 24), (1 << 24, 1), (3, 5)]   # (w, h)
    imgs = [g.integers(0, 256, (h, w, 4), dtype=np.uint8) for w, h in shapes]
    texels = np.concatenate([a.reshape(-1) for a in imgs])
    dims = np.array(shapes, np.int32).reshape(-1)
    mat_tex = np.arange(len(shapes), dtype=np.int32)
    ctx._call("set_textures", rt._capi._ptr(texels), texels.size, rt._capi._ptr(dims), len(shapes), rt._capi._ptr(mat_tex),
              mat_tex.size)
    uv = np.where(g.random((N_RANDOM, 2)) < 0.8, g.uniform(-4, 4, (N_RANDOM, 2)),
                  g.uniform(-1, 1, (N_RANDOM, 2)) * 2.0 ** g.integers(-30, 31, (N_RANDOM, 2))).astype(f32)
    xt = np.zeros((N_RANDOM, 3), f32)
    xt[:, :2] = uv
    agree(ctx, P.TEXEL, C.pack(xt, xt, x=xt, i9=g.integers(0, len(shapes), N_RANDOM)), None, (texels, dims, mat_tex))
    ctx.set_textures(None)


def light_records(sc, g, m, pts, sampling):
    """light samples from the points pts (k, 3) with the surface normals facing towards and away from the emitters,
    every emitter of sc, diffuse and glossy surface materials, random and edge uniform words"""
    light = sc["lightData"]
    types = sc["materialData"].reshape(-1, 6)[:, 0]
    mats = np.nonzero((types == 1) | (types == 2))[0]
    k = g.integers(0, len(pts), m)
    x = pts[k]
    n = C.sphere(g, m)
    d = C.sphere(g, m)
    W = C.word_sets(g, m)
    return C.pack(d, n, W, x=x, i9=light[g.integers(0, light.size, m)], i10=mats[g.integers(0, mats.size, m)],
                  i11=np.full(m, light.size), w15=np.full(m, sampling))


def emitter_points(sc):
    """points on the emitters' planes (cosL = 0), on the emitters (dist2 = 0: a vertex and the point of ua = ub = 1/2,
    where ua + ub == 1 exactly), and a little away from them"""
    vp = sc["V_p"].reshape(-1, 3)
    face = sc["faceData"].reshape(-1, 10)
    out = []
    for t in sc["lightData"]:
        A, B, Cc = vp[face[t, 7]], vp[face[t, 8]], vp[face[t, 9]]
        out += [A, B, Cc, A + (B - A) * f32(0.5) + (Cc - A) * f32(0.5), A + (B - A) * f32(3), (A + B + Cc) / f32(3) +
                np.cross(B - A, Cc - A).astype(f32) * f32(0.1)]
    return np.array(out, f32)


@pytest.mark.parametrize("name", ["lit_cornell", "monkey_cfg2"])
def test_light_sample_equals_the_oracle(ctx, name):
    sc = scene(name)
    upload(ctx, sc)
    g = np.random.default_rng(9)
    vp = sc["V_p"].reshape(-1, 3)
    face = sc["faceData"].reshape(-1, 10)
    nt = face.shape[0]
    tris = g.integers(0, nt, 64)
    cent = ((vp[face[tris, 7]] + vp[face[tris, 8]] + vp[face[tris, 9]]) / 3).astype(f32)
    pts = np.concatenate([cent, emitter_points(sc)])
    for sampling in (0, 1):
        recs = light_records(sc, g, N_RANDOM // 4, pts, sampling)
        ep = emitter_points(sc)
        e = light_records(sc, g, 20000, ep, sampling)
        e.view(f32)[:, 3:6] = np.where(g.random((20000, 1)) < 0.5, 1, -1) * e.view(f32)[:, 3:6]
        e[:, 13:15] = np.array([[1 << 22, 1 << 22], [0, 0], [(1 << 23) - 1, (1 << 23) - 1], [1 << 22, 0]],
                               np.uint32)[g.integers(0, 4, 20000)]
        out = agree(ctx, P.LIGHT, np.concatenate([recs, e]), sc)
        assert (out[:, 6] > 0).mean() > 0.2 and (out[:, 0] > 0).any() and (out[:, 0] == 0).any()


def test_refusals(ctx):
    upload(ctx, scene("cornell"))
    ctx.set_textures(None)
    r = C.pack(np.zeros((1, 3), f32), np.zeros((1, 3), f32), i9=[36], i10=[0], i11=[1])
    for rule, bad in ((P.SMOOTH_NORMAL, {9: 36}), (P.SMOOTH_NORMAL, {9: -1}), (P.ALBEDO, {9: 0, 10: 4}),
                      (P.LIGHT, {9: 0, 10: 0, 11: 0}), (P.LIGHT, {9: 0, 10: -1, 11: 1}), (P.TEXEL, {9: 0})):
        rr = r.copy()
        for k, v in bad.items():
            rr[0, k] = np.uint32(v & 0xFFFFFFFF)
        with pytest.raises(rt.B200RTError):
            ctx.rule_probe(rule, rr)
    with pytest.raises(rt.B200RTError):
        ctx.rule_probe(12, r)


# ---- part B: densities -----------------------------------------------------------------------------------------------------
def frame(n):
    n = np.asarray(n, np.float64)
    n = n / np.linalg.norm(n)
    t = np.cross(n, [0.37, -0.51, 0.77])
    t /= np.linalg.norm(t)
    return n, t, np.cross(n, t)


_DEVICE = threading.Lock()


def accumulate(ctx, rule, make, reduce, n_draw=None, seed=0):
    """the sum over chunks of reduce(device output) for n_draw (default N_DRAW) records, CHUNK at a time; make(g, m) ->
    m records.  Chunks are made and reduced on a thread pool (numpy releases the GIL) while the device takes them one at a
    time; chunk k draws from its own generator, so the result does not depend on the scheduling."""
    n_draw = N_DRAW if n_draw is None else n_draw

    def one(k):
        recs = make(np.random.default_rng([seed, rule, k]), min(CHUNK, n_draw - k * CHUNK))
        with _DEVICE:
            out = ctx.rule_probe(rule, recs)
        return reduce(out)
    with ThreadPoolExecutor(POOL) as ex:
        return sum(ex.map(one, range(-(-n_draw // CHUNK))))


N_TH, N_PH = 18, 24


def to_local(n, l):
    """float64: the unit directions l in the frame the cosine and uniform samplers rotate +z onto n with (scaled by n.z
    when n is +-z, else the rotation by acos(n.z) about z x n)"""
    n = np.asarray(n, np.float64)
    if abs(n[2]) == 1:
        return l / n[2]
    k = np.cross([0.0, 0.0, 1.0], n)
    k /= np.linalg.norm(k)
    a = -np.arccos(n[2])
    return l * np.cos(a) + np.cross(k, l) * np.sin(a) + np.outer(l @ k, k) * (1 - np.cos(a))


def hemisphere_bins(ctx, rule, n, make, local=None, seed=0):
    """mean and sigma of inv_pdf 1{l in bin} over (theta, phi) bins about n and their expectation.  local: bin in the
    samplers' own frame (to_local), whose phi stops at 2 * 3.14 — there every bin's expectation is its solid angle above
    the surface, except the last phi bin's, which loses the wedge [2 * 3.14, 2 pi) (on the whole hemisphere that is
    the factor 3.14 / pi of rt_shade.cuh).  Otherwise (the glossy sampler, whose phi covers the circle): any frame about
    n, expectation (3.14 / pi) times the solid angle."""
    nn, t, b = frame(n)

    def reduce(out):
        l = out[:, :3].astype(np.float64)
        w = out[:, 3].astype(np.float64)
        l /= np.linalg.norm(l, axis=1, keepdims=True)
        if local:
            q = to_local(n, l)
            th = np.arccos(np.clip(q[:, 2], -1, 1))
            ph = np.mod(np.arctan2(q[:, 1], q[:, 0]), 2 * np.pi)
        else:
            th = np.arccos(np.clip(l @ nn, -1, 1))
            ph = np.arctan2(l @ b, l @ t) + np.pi
        k = np.minimum((th / np.pi * N_TH).astype(int), N_TH - 1) * N_PH + \
            np.minimum((ph / (2 * np.pi) * N_PH).astype(int), N_PH - 1)
        return np.stack([np.bincount(k, w, N_TH * N_PH), np.bincount(k, w * w, N_TH * N_PH)])
    s1, s2 = accumulate(ctx, rule, make, reduce, seed=seed)
    mean = s1 / N_DRAW
    sigma = np.sqrt(np.maximum(s2 / N_DRAW - mean * mean, 0) / N_DRAW)
    th_e = np.linspace(0, np.pi, N_TH + 1)
    ph_w = np.full(N_PH, 2 * np.pi / N_PH)
    if local:
        ph_w[-1] -= 2 * np.pi - 2 * 3.14
    want = np.outer(np.cos(th_e[:-1]) - np.cos(th_e[1:]), ph_w) * (1.0 if local else 3.14 / np.pi)
    want[N_TH // 2:] = 0
    return mean, sigma, want.reshape(-1)


def check_bins(mean, sigma, want, quad_err=0.0):
    bad = np.abs(mean - want) > 5 * sigma + quad_err
    assert not bad.any(), (np.nonzero(bad)[0], mean[bad], want[bad], sigma[bad])


NORMALS = {"+z": [0, 0, 1], "-z": [0, 0, -1], "near+z": C.unit([1e-3, -2e-3, 1]), "random": C.unit([0.48, -0.6, 0.64])}


@pytest.mark.parametrize("rule", [P.COSINE_FLAT, P.UNIFORM_FLAT])
@pytest.mark.parametrize("normal", list(NORMALS))
def test_sampler_density(ctx, rule, normal):
    n = np.array(NORMALS[normal], f32)

    def make(g, m):
        return C.pack(np.zeros(3, f32), np.tile(n, (m, 1)),
                      g.integers(0, 1 << 32, (m, 3), dtype=np.uint64).astype(np.uint32))
    check_bins(*hemisphere_bins(ctx, rule, n, make, local=True))


@pytest.mark.parametrize("rule", [P.COSINE_SMOOTH, P.UNIFORM_SMOOTH])
def test_sampler_density_smooth_frame(ctx, rule):
    n = np.array(NORMALS["random"], f32)

    def make(g, m):
        return C.pack(np.zeros(3, f32), np.tile(n, (m, 1)),
                      g.integers(0, 1 << 32, (m, 3), dtype=np.uint64).astype(np.uint32))
    check_bins(*hemisphere_bins(ctx, rule, n, make, local=True))


GLOSSY_CASES = [("random", al, view) for al in (0.05, 0.3, 1.0) for view in (0, 60, 85, 120)] + \
    [(normal, 0.3, view) for normal in ("+z", "-z", "near+z") for view in (0, 60, 85, 120)]


@pytest.mark.parametrize("normal,al,view", GLOSSY_CASES)   # view 120: the viewer below the surface, cosine lobe only
def test_glossy_importance_density(ctx, normal, al, view):
    """every branch of basis_duff (N.z > 0, N.z < 0, N = +-z) and of the mixture"""
    nn, t, _ = frame(NORMALS[normal])
    n = np.asarray(NORMALS[normal], f32)
    v = np.cos(np.radians(view)) * nn + np.sin(np.radians(view)) * t   # towards the viewer
    d = (-v).astype(f32)

    def make(g, m):
        return C.pack(np.tile(d, (m, 1)), np.tile(n, (m, 1)),
                      g.integers(0, 1 << 32, (m, 3), dtype=np.uint64).astype(np.uint32), f6=f32(al))
    check_bins(*hemisphere_bins(ctx, P.GLOSSY, n, make, seed=view))


def tri_quadrature(A, e1, e2, x, q):
    """float64 integrals of (1, wx, wy, wz) over the solid angle of triangle (A, e1, e2) seen from x, by Gauss-Legendre
    on the collapsed square (q x q nodes)"""
    s, ws = roots_legendre(q)
    s, ws = 0.5 * (s + 1), 0.5 * ws
    S, T = np.meshgrid(s, s, indexing="ij")
    W = np.outer(ws, ws) * (1 - S)
    y = A + S[..., None] * e1 + ((1 - S) * T)[..., None] * e2
    w = y - x
    dist2 = np.sum(w * w, axis=-1)
    wi = w / np.sqrt(dist2)[..., None]
    nl = np.cross(e1, e2)
    area2 = np.linalg.norm(nl)
    cosl = np.abs(wi @ nl) / area2
    f = W * area2 * cosl / dist2
    return np.array([f.sum(), (f * wi[..., 0]).sum(), (f * wi[..., 1]).sum(), (f * wi[..., 2]).sum()])


def test_light_sampler_density(ctx):
    sc = scene("lit_cornell")
    upload(ctx, sc)
    vp = sc["V_p"].reshape(-1, 3).astype(np.float64)
    face = sc["faceData"].reshape(-1, 10)
    light = sc["lightData"]
    la = np.concatenate([vp[face[light, j]] for j in (7, 8, 9)])
    lo, hi = la.min(axis=0), la.max(axis=0)
    # surface points of the box away from the emitters' plane: centroids of triangles of the floor and the walls
    A0 = vp[face[light[0], 7]]
    nl = np.cross(vp[face[light[0], 8]] - A0, vp[face[light[0], 9]] - A0)
    nl /= np.linalg.norm(nl)
    scale = np.ptp(vp, axis=0).max()
    cents = (vp[face[:, 7]] + vp[face[:, 8]] + vp[face[:, 9]]) / 3
    pts = [c for c in cents if abs((c - A0) @ nl) > 0.05 * scale][::3][:4]
    assert len(pts) == 4
    per = N_DRAW // len(pts)
    for j, x in enumerate(pts):
        x32 = x.astype(f32)

        def make(g, m):
            return C.pack(C.sphere(g, m), np.tile(f32([0, 0, 1]), (m, 1)),
                          g.integers(0, 1 << 32, (m, 3), dtype=np.uint64).astype(np.uint32), x=np.tile(x32, (m, 1)),
                          i9=light[g.integers(0, light.size, m)], i10=np.zeros(m), i11=np.full(m, light.size))
        def reduce(out):
            w = out[:, 3:6].astype(np.float64)
            wi = w / np.linalg.norm(w, axis=1, keepdims=True)
            pl = out[:, 6].astype(np.float64)
            ok = pl > 0
            v = np.zeros((len(pl), 4))
            v[ok, 0] = 1 / pl[ok]
            v[ok, 1:] = wi[ok] / pl[ok, None]
            return np.stack([v.sum(axis=0), (v * v).sum(axis=0)])
        s1, s2 = accumulate(ctx, P.LIGHT, make, reduce, per, seed=j)
        mean = s1 / per
        sigma = np.sqrt(np.maximum(s2 / per - mean * mean, 0) / per)
        want_q = np.zeros(4)
        want_2q = np.zeros(4)
        for t in light:
            A = vp[face[t, 7]]
            e1, e2 = vp[face[t, 8]] - A, vp[face[t, 9]] - A
            want_q += tri_quadrature(A, e1, e2, x, 16)
            want_2q += tri_quadrature(A, e1, e2, x, 32)
        assert want_2q[0] > 1e-3
        err = np.abs(mean - want_2q)
        assert (err <= 5 * sigma + np.abs(want_q - want_2q)).all(), (x, mean, want_2q, sigma)


def gauss_nodes(lo, hi, n_sub, q=8):
    """composite Gauss-Legendre on [lo, hi]: n_sub cells of q nodes (the BSDF has kinks and steps inside some bins, where
    one rule of many nodes converges too slowly for its error to show between Q and 2Q nodes)"""
    x, w = roots_legendre(q)
    e = np.linspace(lo, hi, n_sub + 1)
    h = np.diff(e)[:, None]
    return (0.5 * h * x + 0.5 * (e[:-1, None] + e[1:, None])).ravel(), (0.5 * h * w).ravel()


def walter_bins(i, al, eta, n_sub, n_th=36, n_ph=12):
    """float64 integral of Walter's f |cos| over each (theta, phi) bin"""
    th_e = np.linspace(0, np.pi, n_th + 1)
    ph_e = np.linspace(-np.pi, np.pi, n_ph + 1)
    out = np.zeros((n_th, n_ph))
    for a in range(n_th):
        th, wt = gauss_nodes(th_e[a], th_e[a + 1], n_sub)
        wt = wt * np.sin(th)
        for b in range(n_ph):
            ph, wp = gauss_nodes(ph_e[b], ph_e[b + 1], n_sub)
            T, Ph = np.meshgrid(th, ph, indexing="ij")
            l = np.stack([np.sin(T) * np.cos(Ph), np.sin(T) * np.sin(Ph), np.cos(T)], axis=-1)
            out[a, b] = np.sum(walter_cos(i, l, al, eta) * np.outer(wt, wp))
    return out.reshape(-1)


@pytest.mark.parametrize("r", [0.05, 0.3, 1.0])
@pytest.mark.parametrize("ior", [1.5, 0.8])
@pytest.mark.parametrize("enter", [True, False])
def test_rough_glass_matches_walter_bsdf_bin_by_bin(ctx, r, ior, enter):
    """tests/test_rough_glass_oracle.py's bin test on 10^8 device draws"""
    th_i = 0.6
    i = np.array([np.sin(th_i), 0.0, np.cos(th_i)])
    d = (-i).astype(f32)
    un = f32([0, 0, 1 if enter else -1])
    eta = 1.0 / ior if enter else ior
    n_th, n_ph = 36, 12

    def make(g, m):
        return C.pack(np.tile(d, (m, 1)), np.tile(un, (m, 1)),
                      g.integers(0, 1 << 32, (m, 3), dtype=np.uint64).astype(np.uint32), f6=f32(ior), f7=f32(r))

    def reduce(out):
        nd = out[:, :3].astype(np.float64)
        nd /= np.linalg.norm(nd, axis=1, keepdims=True)
        th = np.arccos(np.clip(nd[:, 2], -1, 1))
        ph = np.arctan2(nd[:, 1], nd[:, 0])
        k = np.minimum((th / np.pi * n_th).astype(int), n_th - 1) * n_ph + \
            np.minimum(((ph + np.pi) / (2 * np.pi) * n_ph).astype(int), n_ph - 1)
        w = out[:, 4].astype(np.float64)
        return np.stack([np.bincount(k, w, n_th * n_ph), np.bincount(k, w * w, n_th * n_ph)])
    s1, s2 = accumulate(ctx, P.ROUGH_DIELECTRIC, make, reduce, seed=int(enter) * 100 + int(r * 100) + int(ior * 10))
    mean = s1 / N_DRAW
    want_q, want_2q = walter_bins(i, r, eta, 12), walter_bins(i, r, eta, 24)
    # the weights lie in [0, 1], so a bin's variance is at most its mean.  That bound is used where it exceeds the sample
    # variance: in a bin that few or no draws reach (the quadrature gives such bins 1e-6 or less), the sample variance
    # of a handful of draws understates the true one
    var = np.maximum(np.maximum(s2 / N_DRAW - mean * mean, 0), want_2q)
    sigma = np.sqrt(var / N_DRAW)
    check_bins(mean, sigma, want_2q, np.abs(want_q - want_2q))
