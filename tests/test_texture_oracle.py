"""CPU: opt-in albedo textures (B200RT_SAMPLING_TEXTURES) in the texture oracle — the texel rule against a numpy
restatement, equality with the glass oracle when nothing is bound, white and constant textures, the orientation of the
image, the reproduction of a checker, what the textured G-buffer buys the denoiser, and B200RT_TEXTURES."""
import numpy as np
import pytest

from ensem3a_openclraytracer_b200.KernelLauncher import textures_from_env
from oracle import oracle
from oracle_denoise import denoise as D
from oracle_glass import glass
from oracle_texture import texture
from tests import fixtures, glass_scene as gs, texture_scene as ts

f32 = np.float32
T = ts.TEX


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


def _cases(g, n):
    """n (u, v) pairs: uniform over [-3, 3], texel boundaries of extents 1..8, exact integers and halves, and
    non-finite values"""
    u = g.uniform(-3, 3, n).astype(f32)
    v = g.uniform(-3, 3, n).astype(f32)
    k = n // 4
    ext = g.integers(1, 9, k)
    u[:k] = (g.integers(-20, 40, k) + f32(0.5)) / ext.astype(f32)   # texel centres and boundaries
    v[:k] = g.integers(-20, 40, k).astype(f32) / ext.astype(f32)
    u[k:k + 64] = np.repeat(np.array([0, 1, -1, 2, 0.5, -0.5, 1e-30, -1e-30], f32), 8)
    v[k:k + 64] = np.tile(np.array([0, 1, -1, 2, 0.5, -0.5, 1e-30, -1e-30], f32), 8)
    bad = np.array([np.nan, np.inf, -np.inf, 0.25], f32)
    u[k + 64:k + 80] = np.repeat(bad, 4)
    v[k + 64:k + 80] = np.tile(bad, 4)
    return u, v


@pytest.mark.parametrize("shape", [(1, 1), (1, 7), (7, 1), (4, 4), (5, 3), (64, 33)])
def test_texel_rule_equals_the_restatement(shape):
    g = np.random.default_rng(shape[0] * 100 + shape[1])
    img = g.integers(0, 256, shape + (4,)).astype(np.uint8)
    u, v = _cases(g, 20000)
    got = texture.texel(img, u, v)
    want = ts.texel(img, u, v)
    assert np.array_equal(bits(got), bits(want))
    nonfinite = ~(np.isfinite(u) & np.isfinite(v))
    assert nonfinite.sum() == 15 and (got[nonfinite] == f32(1)).all()


def test_uniform_textures_return_their_value_exactly():
    u, v = _cases(np.random.default_rng(5), 4000)
    ok = np.isfinite(u) & np.isfinite(v)
    for c in (0, 1, 77, 128, 254, 255):
        img = np.full((3, 5, 4), c, np.uint8)
        assert (texture.texel(img, u[ok], v[ok]) == f32(c) / f32(255)).all()


@pytest.mark.parametrize("sampling", [0, 1, 2, 3, 8, 32, 32 | 2, 128, 128 | 32 | 2])
@pytest.mark.parametrize("rng", [oracle.RNG_REFERENCE, oracle.RNG_PHILOX])
def test_nothing_bound_equals_the_glass_oracle(sampling, rng):
    sc, ibl = fixtures.load_scene("monkey_cfg2"), fixtures.load_ibl()
    cam, env = fixtures.cam_env(sc["params"], 24)
    want, cw = glass.render(sc, cam, env, 24 * 24, 2, 4, ibl, rng_mode=rng, seed=3, sampling=sampling)
    for s in (sampling, sampling | T):
        got, cg = texture.render(sc, cam, env, 24 * 24, 2, 4, ibl, rng_mode=rng, seed=3, sampling=s)
        assert np.array_equal(bits(got), bits(want)) and cg == cw
    # a bound texture without the bit is not read either
    got, cg = texture.render(sc, cam, env, 24 * 24, 2, 4, ibl, rng_mode=rng, seed=3, sampling=sampling,
                             textures=ts.textured(sc, 8))
    assert np.array_equal(bits(got), bits(want)) and cg == cw


@pytest.mark.parametrize("name", ["monkey_cfg2", "cornell"])
def test_white_and_constant_textures(name):
    sc, ibl = fixtures.load_scene(name), fixtures.load_ibl()
    cam, env = fixtures.cam_env(sc["params"], 24)
    n_mat = sc["materialData"].size // 6
    for sampling in (T, T | 2, T | 128 | 32):
        plain, cp = texture.render(sc, cam, env, 24 * 24, 3, 4, ibl, rng_mode=1, seed=9, sampling=sampling & ~T)
        white = np.full((4, 4, 4), 255, np.uint8)
        got, cg = texture.render(sc, cam, env, 24 * 24, 3, 4, ibl, rng_mode=1, seed=9, sampling=sampling,
                                 textures={m: white for m in range(n_mat)})
        assert np.array_equal(bits(got), bits(plain)) and cg == cp
        c = np.array([200, 90, 30], np.uint8)
        const = ts.rgba(np.broadcast_to(c, (3, 2, 3)))
        scaled = gs.with_materials(sc, lambda mt: np.where((np.isin(mt[:, 0], (1, 2)))[:, None],
                                                          np.concatenate([mt[:, :1], mt[:, 1:4] * (c.astype(f32) / f32(255)),
                                                                          mt[:, 4:]], axis=1), mt))
        want, cw = texture.render(scaled, cam, env, 24 * 24, 3, 4, ibl, rng_mode=1, seed=9, sampling=sampling & ~T)
        got, cg = texture.render(sc, cam, env, 24 * 24, 3, 4, ibl, rng_mode=1, seed=9, sampling=sampling,
                                 textures={m: const for m in range(n_mat)})
        assert np.array_equal(bits(got), bits(want)) and cg == cw
        # any texture leaves the counters alone
        _, cn = texture.render(sc, cam, env, 24 * 24, 3, 4, ibl, rng_mode=1, seed=9, sampling=sampling,
                               textures=ts.textured(sc, 16))
        assert cn == cp


def test_orientation_red_half_on_top():
    W = 32
    sc = ts.quad(half=2.0, uv_max=1.0)
    cam, env, grey = ts.view(W)
    img, _ = texture.render(sc, cam, env, W * W, 2, 1, grey, sampling=T, textures={0: ts.orientation()})
    img = img.reshape(W, W, 3)
    top, bottom = img[: W // 2 - 2], img[W // 2 + 2:]
    assert (top[..., 0] > 0.3).all() and (top[..., 2] < 0.05).all()
    assert (bottom[..., 2] > 0.3).all() and (bottom[..., 0] < 0.05).all()


def test_checker_is_reproduced():
    W, spp = 64, 8
    sc = ts.quad()
    cam, env, grey = ts.view(W)
    tex = ts.checker()
    img, _ = texture.render(sc, cam, env, W * W, spp, 1, grey, rng_mode=1, seed=2, sampling=T, textures={0: tex})
    img = img.reshape(-1, 3)
    u, v = ts.quad_uv(W)
    n = tex.shape[0]
    tx, ty = (u % 1.0) * n, (1.0 - v % 1.0) * n       # texel coordinates, float64
    cell_x, cell_y = np.floor(tx / 16).astype(int), np.floor(ty / 16).astype(int)
    # pixels whose four bilinear taps lie in one cell
    inner = ((tx - 0.5) % 16 > 0.01) & ((tx - 0.5) % 16 < 14.99) & ((ty - 0.5) % 16 > 0.01) & ((ty - 0.5) % 16 < 14.99)
    light = (cell_x + cell_y) % 2 == 0
    assert inner.sum() > W * W // 2 and (inner & light).any() and (inner & ~light).any()
    mean_light = img[inner & light].mean(axis=0)
    ratio = img[inner] / mean_light
    want = np.where(light[inner][:, None], 1.0, np.array([40, 60, 80]) / np.array([230, 200, 170]))
    assert np.abs(ratio - want).max() < 0.02


def test_textured_gbuffer_helps_the_denoiser():
    W = 48
    sc = ts.quad()
    cam, env, ibl = ts.view(W, graded=True)
    tex = {0: ts.checker(cells=4, cell_px=8)}
    conv, _ = texture.render(sc, cam, env, W * W, 1024, 1, ibl, rng_mode=1, seed=1, sampling=T, textures=tex)
    noisy, _ = texture.render(sc, cam, env, W * W, 16, 1, ibl, rng_mode=1, seed=7, sampling=T, textures=tex)
    gb = D.gbuffer(sc, cam, W, W)
    p = oracle.primary(sc, cam, W * W)
    gbt = dict(gb, albedo=texture.gbuffer_albedo(sc, cam, p["tri"], p["k"], tex).reshape(W, W, 3))
    assert not np.array_equal(gbt["albedo"], gb["albedo"])
    conv = conv.reshape(W, W, 3)
    errs = []
    for g in (gb, gbt):
        out = D.atrous(noisy.reshape(W, W, 3), g, passes=5, sigma_color=0.5, sigma_normal=0.2, sigma_position=0.0,
                       bvh=sc["BVH"])
        errs.append(np.sqrt(np.mean((out - conv) ** 2)))
    assert errs[1] < 0.7 * errs[0], errs


def test_gbuffer_albedo_without_textures_is_the_material_colour():
    sc = fixtures.load_scene("monkey_cfg2")
    cam, _ = fixtures.cam_env(sc["params"], 32)
    p = oracle.primary(sc, cam, 32 * 32)
    gb = D.gbuffer(sc, cam, 32, 32)
    got = texture.gbuffer_albedo(sc, cam, p["tri"], p["k"])
    glass_px = (p["tri"] >= 0) & (sc["materialData"].reshape(-1, 6)[sc["faceData"].reshape(-1, 10)[np.maximum(p["tri"], 0), 0], 0] == 3)
    assert np.array_equal(bits(got), bits(gb["albedo"].reshape(-1, 3)))
    assert glass_px.any()


def test_environment_variable(tmp_path):
    from PIL import Image
    a = ts.noise(8, 1)
    Image.fromarray(a).save(tmp_path / "a.png")
    Image.fromarray(a[..., :3]).save(tmp_path / "b.png")
    got = textures_from_env(f"4={tmp_path / 'a.png'}, 0 = {tmp_path / 'b.png'}")
    assert sorted(got) == [0, 4]
    assert np.array_equal(np.asarray(got[4]), a) and np.array_equal(np.asarray(got[0]), a)
    for bad in ("", "a.png", "x=a.png", "=a.png", "1=", "-1=a.png", "1.5=a.png",
                f"1={tmp_path / 'a.png'},1={tmp_path / 'b.png'}", f"1={tmp_path / 'a.png'},"):
        with pytest.raises(ValueError):
            textures_from_env(bad)
    with pytest.raises(OSError):
        textures_from_env(f"0={tmp_path / 'missing.png'}")
