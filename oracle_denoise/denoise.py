"""TEST INFRASTRUCTURE — a numpy float32 restatement of the denoiser of include/b200rt.h: the G-buffer of the primary
hits, built from oracle.primary (the CPU restatement of the reference's hit) and the scene arrays, and the edge-avoiding
à-trous filter.  Every step is one elementwise binary32 operation in the header's order (numpy never fuses two of them),
so the result is meant to equal the GPU's bit for bit.  Only tests/ and tools/ may import this; the product never does."""
import numpy as np

from oracle import oracle

f32 = np.float32
K1 = [f32(1 / 16), f32(1 / 4), f32(3 / 8), f32(1 / 4), f32(1 / 16)]


def gbuffer(scene, cam, width, height, stack_cap=20):
    """dict of albedo / normal / position (H, W, 3) float32 and kind (H, W) int32, as b200rt_gbuffer returns it."""
    p = oracle.primary(scene, cam, width * height, stack_cap=stack_cap)
    tri, d, k = p["tri"], p["dir"], p["k"]
    face = scene["faceData"].reshape(-1, 10)
    mats = scene["materialData"].reshape(-1, 6)
    hit = tri >= 0
    t = np.maximum(tri, 0)
    m = mats[face[t, 0]]
    mtype = m[:, 0].astype(np.int32)
    kind = np.where(hit, np.where(mtype == 0, 0, 1), -1).astype(np.int32)
    albedo = np.where((kind == 1)[:, None], m[:, 1:4], f32(1)).astype(f32)
    n = scene["V_n"].reshape(-1, 3)[face[t, 4]].astype(f32)
    with np.errstate(all="ignore"):
        un = n / np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2])[:, None]
        pos = np.asarray(cam[:3], f32)[None, :] + d * k[:, None]
    normal = np.where((hit & np.isfinite(un).all(axis=1))[:, None], un, f32(0)).astype(f32)
    position = np.where(hit[:, None], pos, f32(0)).astype(f32)
    shape = (height, width, 3)
    return {"albedo": albedo.reshape(shape), "normal": normal.reshape(shape), "position": position.reshape(shape),
            "kind": kind.reshape(height, width)}


def auto_sigma_position(bvh):
    """0.01f * the binary32 diagonal of the BVH root box bvh[2..7]"""
    b = np.asarray(bvh, f32)[2:8]
    dx, dy, dz = b[3] - b[0], b[4] - b[1], b[5] - b[2]
    return f32(0.01) * np.sqrt((dx * dx + dy * dy) + dz * dz)


def clamp01(x):
    """the reference's fmax(fmin(x, 1), 0): a NaN becomes 1"""
    return np.where(np.isnan(x), f32(1), np.fmax(np.fmin(x, f32(1)), f32(0))).astype(f32)


def _d2(a, b):
    D = b - a
    return (D[..., 0] * D[..., 0] + D[..., 1] * D[..., 1]) + D[..., 2] * D[..., 2]


def _f(d2, s):
    return f32(1) / (f32(1) + d2 / s)


def atrous(img, gb, passes, sigma_color, sigma_normal, sigma_position, bvh=None):
    """The filter over an (H, W, 3) image and G-buffer; sigma_position <= 0 takes auto_sigma_position(bvh)."""
    kind = np.asarray(gb["kind"])
    H, W = kind.shape
    I = np.asarray(img, f32).reshape(H, W, 3)
    a = np.fmax(np.asarray(gb["albedo"], f32).reshape(H, W, 3), f32(0.01))   # fmaxf: a NaN albedo gives 0.01
    n = np.asarray(gb["normal"], f32).reshape(H, W, 3)
    x = np.asarray(gb["position"], f32).reshape(H, W, 3)
    live = kind == 1
    sp = f32(sigma_position) if sigma_position > 0 else auto_sigma_position(bvh)
    s_n, s_x = f32(sigma_normal) * f32(sigma_normal), sp * sp
    Y, X = np.mgrid[0:H, 0:W]
    with np.errstate(all="ignore"):
        c = I / a
        for l in range(passes):
            h = 1 << l
            s_c = (f32(sigma_color) * f32(sigma_color)) * f32(2.0 ** (-2 * l))
            sx = np.zeros((H, W, 3), f32)
            sw = np.zeros((H, W), f32)
            for j in range(-2, 3):
                for i in range(-2, 3):
                    if i == 0 and j == 0:
                        w = np.full((H, W), K1[2] * K1[2], f32)
                        cq = c
                        take = np.ones((H, W), bool)
                    else:
                        yq, xq = Y + h * j, X + h * i
                        inside = (yq >= 0) & (yq < H) & (xq >= 0) & (xq < W)
                        yq, xq = np.clip(yq, 0, H - 1), np.clip(xq, 0, W - 1)
                        cq = c[yq, xq]
                        w = (((K1[j + 2] * K1[i + 2]) * _f(_d2(c, cq), s_c)) * _f(_d2(n, n[yq, xq]), s_n)) * \
                            _f(_d2(x, x[yq, xq]), s_x)
                        take = inside & live[yq, xq] & (w > 0)
                    sx = np.where(take[..., None], sx + w[..., None] * cq, sx)
                    sw = np.where(take, sw + w, sw)
            c = np.where(live[..., None], sx / sw[..., None], c)
        out = clamp01(c * a)
    return np.where(live[..., None], out, I).astype(f32)
