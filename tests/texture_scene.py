"""Albedo textures (include/b200rt.h, B200RT_SAMPLING_TEXTURES) for the tests: a numpy float32 restatement of the texel
rule, a front-facing textured quad, seeded checker / orientation / noise textures, and a helper that textures every
diffuse and glossy material of a fixture scene.  Every step of the restatement is one elementwise binary32 operation in
the header's order (numpy never fuses two of them)."""
import numpy as np

import ensem3a_openclraytracer_b200 as rt
from tests import fixtures

f32 = np.float32
TEX = rt.SAMPLING_TEXTURES


def texel(rgba, u, v):
    """(n, 3) float32: the header's texture factor of one (H, W, 4) uint8 texture at points (u, v) (n,)"""
    rgba = np.asarray(rgba, np.uint8)
    h, w = rgba.shape[:2]
    u, v = np.asarray(u, f32).reshape(-1), np.asarray(v, f32).reshape(-1)
    ok = np.isfinite(u) & np.isfinite(v)
    u, v = np.where(ok, u, f32(0)), np.where(ok, v, f32(0))
    fu, fv = u - np.floor(u), v - np.floor(v)
    tx, ty = fu * f32(w) - f32(0.5), (f32(1) - fv) * f32(h) - f32(0.5)
    x0, y0 = np.floor(tx).astype(np.int64), np.floor(ty).astype(np.int64)
    ax, ay = (tx - x0.astype(f32))[:, None], (ty - y0.astype(f32))[:, None]
    c = rgba[..., :3].astype(f32) / f32(255)
    xa, xb, ya, yb = x0 % w, (x0 + 1) % w, y0 % h, (y0 + 1) % h

    def lerp(a, b, t):
        return a + (b - a) * t

    f = lerp(lerp(c[ya, xa], c[ya, xb], ax), lerp(c[yb, xa], c[yb, xb], ax), ay)
    return np.where(ok[:, None], f, f32(1)).astype(f32)


# ---- the quad ---------------------------------------------------------------------------------------------------------
Y = 3.0   # the quad's plane, in front of an unrotated camera at the origin, which looks along +y with +z up


def quad(half=2.0, uv_max=2.0, colour=(1.0, 1.0, 1.0)):
    """a square of half-width `half` in the plane y = Y, facing the camera (normal -y), one diffuse material; u runs from
    0 at x = -half to uv_max at x = +half, v from 0 at the bottom (z = -half) to uv_max at the top"""
    pos = np.array([[-half, Y, -half], [half, Y, -half], [half, Y, half], [-half, Y, half]], f32)
    uv = np.array([[0, 0], [uv_max, 0], [uv_max, uv_max], [0, uv_max]], f32)
    fd = np.array([[0, 0, 1, 2, 0, 0, 0, 0, 1, 2], [0, 0, 2, 3, 0, 0, 0, 0, 2, 3]], np.int32)
    sc = {"V_p": pos.reshape(-1), "V_n": np.array([0, -1, 0], f32), "V_uv": uv.reshape(-1), "faceData": fd.reshape(-1),
          "materialData": np.array([1, *colour, 0.5, 0], f32), "lightData": np.zeros(0, np.int32)}
    sc["BVH"] = rt.BVH(sc["faceData"], sc["V_p"]).exportArray
    return sc


def view(width, graded=False):
    """cam, env (no sun, environment power 1) for the quad, and a uniform grey environment map (or, graded, one whose
    rows go from bright at the top to dark, which makes the quad's samples noisy)"""
    cam = np.array([0, 0, 0, 0, 0, 0, width, width, 1, 60.0 * (3.14 / 180)], f32)
    env = np.array([0, 0, 0, 0, 1], f32)
    if not graded:
        return cam, env, fixtures.load_ibl("grey")
    rows = np.linspace(255, 0, 64).round().astype(np.uint8)
    ibl = np.zeros((64, 128, 4), np.uint8)
    ibl[..., 0] = ibl[..., 1] = ibl[..., 2] = rows[:, None]
    ibl[..., 3] = 255
    return cam, env, ibl


def quad_uv(width):
    """(u, v) of the reference's camera ray of every pixel on quad() (uv_max 2, half 2), by ray-plane intersection in
    float64, row-major (H*W,)"""
    i = np.arange(width * width)
    col = (i + 1) % width
    row = np.fix((i - col) / width).astype(np.int64)   # C's truncating division (Raytracing.cl:21-22)
    step = 1.0 / width
    f = 1.0 / (2.0 * np.tan(60.0 * (3.14 / 180) / 2.0))
    d = np.stack([col * step - 0.5, np.full(i.shape, f), 0.5 - row * step], axis=1)
    p = d * (Y / d[:, 1:2])
    return (p[:, 0] + 2.0) / 2.0, (p[:, 2] + 2.0) / 2.0


# ---- textures ---------------------------------------------------------------------------------------------------------
def rgba(rgb):
    """(H, W, 4) uint8 with alpha 255 from (H, W, 3)"""
    rgb = np.asarray(rgb, np.uint8)
    return np.concatenate([rgb, np.full(rgb.shape[:2] + (1,), 255, np.uint8)], axis=2)


def checker(cells=8, cell_px=16, light=(230, 200, 170), dark=(40, 60, 80)):
    """cells x cells squares of cell_px texels, light where (row + column) of the cell is even"""
    n = cells * cell_px
    r, c = np.mgrid[0:n, 0:n] // cell_px
    return rgba(np.where(((r + c) % 2 == 0)[..., None], np.array(light, np.uint8), np.array(dark, np.uint8)))


def orientation(w=64, h=64):
    """red top half, blue bottom half"""
    img = np.zeros((h, w, 3), np.uint8)
    img[: h // 2, :, 0] = 255
    img[h // 2:, :, 2] = 255
    return rgba(img)


def noise(size, seed):
    """seeded (size, size, 4) texture: a smooth gradient with uniform noise, every channel in [16, 255]"""
    g = np.random.default_rng(seed)
    y, x = np.mgrid[0:size, 0:size] / max(size - 1, 1)
    base = np.stack([x, y, 1 - x * y], axis=2) * 160 + 16
    return rgba(np.clip(base + g.integers(0, 80, (size, size, 3)), 16, 255).astype(np.uint8))


def textured(sc, size=64, seed=0):
    """{material: texture} for every diffuse (type 1) and glossy (type 2) material of scene sc, one seeded noise texture
    each (material m uses seed + m)"""
    types = sc["materialData"].reshape(-1, 6)[:, 0].astype(int)
    return {m: noise(size, seed + m) for m in range(types.size) if types[m] in (1, 2)}
