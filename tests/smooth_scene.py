"""Smooth shading (include/b200rt.h, B200RT_SAMPLING_SMOOTH_NORMALS) for the tests: a numpy float32 restatement of the
rule, the denoiser's G-buffer with the smooth normal, and a
UV sphere with exact vertex normals under a vertically graded environment.  Every step of the restatement is one
elementwise binary32 operation in the header's order (numpy never fuses two of them)."""
import numpy as np

import ensem3a_openclraytracer_b200 as rt
from oracle import oracle
from oracle_denoise import denoise

f32 = np.float32
SMOOTH = rt.SAMPLING_SMOOTH_NORMALS


def _dot(a, b):
    return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]


def smooth_normal(scene, tri, x):
    """(n, 3) float32: the shading normal of hits on triangles tri (n,) at points x (n, 3), by the header's rule"""
    face = scene["faceData"].reshape(-1, 10)[np.asarray(tri)]
    vp, vn = scene["V_p"].reshape(-1, 3), scene["V_n"].reshape(-1, 3)
    x = np.asarray(x, f32).reshape(-1, 3)
    n0, n1, n2 = (vn[face[:, j]].astype(f32) for j in (4, 5, 6))
    A, B, C = (vp[face[:, j]].astype(f32) for j in (7, 8, 9))
    e1, e2 = B - A, C - A
    p = x - A
    with np.errstate(all="ignore"):
        d00, d01, d11 = _dot(e1, e1), _dot(e1, e2), _dot(e2, e2)
        d20, d21 = _dot(p, e1), _dot(p, e2)
        den = d00 * d11 - d01 * d01
        b1 = (d11 * d20 - d01 * d21) / den
        b2 = (d00 * d21 - d01 * d20) / den
        b0 = (f32(1) - b1) - b2
        m = (n0 * b0[:, None] + n1 * b1[:, None]) + n2 * b2[:, None]
        n = m / np.sqrt(_dot(m, m))[:, None]
        usable = np.isfinite(n).all(axis=1) & (_dot(n, n) > f32(0))
    flat = (n0.view(np.uint32) == n1.view(np.uint32)).all(axis=1) & (n0.view(np.uint32) == n2.view(np.uint32)).all(axis=1)
    return np.where((~flat & usable)[:, None], n, n0).astype(f32)


def curved(scene):
    """bool per triangle: its three vertex normals are not all equal bit for bit"""
    face = scene["faceData"].reshape(-1, 10)
    vn = scene["V_n"].reshape(-1, 3).view(np.uint32)
    n0, n1, n2 = vn[face[:, 4]], vn[face[:, 5]], vn[face[:, 6]]
    return ~((n0 == n1).all(axis=1) & (n0 == n2).all(axis=1))


def gbuffer(scene, cam, width, height, stack_cap=20):
    """denoise.gbuffer with the G-buffer normal of a smooth-shaded frame: the normalised shading normal at the render's
    point cam_pos + unit(d) * k"""
    g = denoise.gbuffer(scene, cam, width, height, stack_cap=stack_cap)
    p = oracle.primary(scene, cam, width * height, stack_cap=stack_cap)
    tri, d, k = p["tri"], p["dir"].astype(f32), p["k"]
    hit = tri >= 0
    with np.errstate(all="ignore"):
        ud = d / np.sqrt(_dot(d, d))[:, None]
        x = np.asarray(cam[:3], f32)[None, :] + ud * k[:, None]
        n = smooth_normal(scene, np.maximum(tri, 0), x)
        un = n / np.sqrt(_dot(n, n))[:, None]
    un = np.where(np.isfinite(un).all(axis=1)[:, None], un, f32(0))
    normal = g["normal"].reshape(-1, 3).copy()
    normal[hit] = un[hit]
    g["normal"] = normal.reshape(height, width, 3)
    return g


# ---- the quality scene ----------------------------------------------------------------------------------------------
CENTRE = np.array([0.0, 3.0, 0.0])   # in front of an unrotated camera at the origin, which looks along +y
RADIUS = 1.0


def sphere(n_lon, n_lat):
    """UV sphere of RADIUS around CENTRE: n_lon x n_lat quads (the poles' rows as triangles), vertex normals exact
    (the unit radial direction of each vertex), one diffuse material"""
    pos, nrm = [], []
    for j in range(n_lat + 1):
        th = np.pi * j / n_lat
        for i in range(n_lon):
            ph = 2.0 * np.pi * i / n_lon
            r = np.array([np.sin(th) * np.cos(ph), np.sin(th) * np.sin(ph), np.cos(th)])
            pos.append(CENTRE + RADIUS * r)
            nrm.append(r)

    def v(j, i):
        return j * n_lon + i % n_lon

    faces = []
    for j in range(n_lat):
        for i in range(n_lon):
            a, b, c, d = v(j, i), v(j, i + 1), v(j + 1, i), v(j + 1, i + 1)
            if j > 0:
                faces.append((a, c, b))
            if j < n_lat - 1:
                faces.append((b, c, d))
    fd = np.zeros((len(faces), 10), np.int32)
    for t, (a, b, c) in enumerate(faces):
        fd[t] = [0, a, b, c, a, b, c, a, b, c]
    sc = {"V_p": np.asarray(pos, f32).reshape(-1), "V_n": np.asarray(nrm, f32).reshape(-1),
          "V_uv": np.zeros(2, f32), "faceData": fd.reshape(-1),
          "materialData": np.array([1, 0.8, 0.8, 0.8, 0.5, 1], f32), "lightData": np.zeros(0, np.int32)}
    sc["BVH"] = rt.BVH(sc["faceData"], sc["V_p"]).exportArray
    return sc


def sphere_view(width):
    """cam, env (no sun, environment power 1) and a vertically graded environment map (bright rows on top)"""
    cam = np.array([0, 0, 0, 0, 0, 0, width, width, 1, 60.0 * (3.14 / 180)], f32)
    env = np.array([0, 0, 0, 0, 1], f32)
    rows = np.linspace(255, 0, 64).round().astype(np.uint8)
    ibl = np.zeros((64, 128, 4), np.uint8)
    ibl[..., 0] = ibl[..., 1] = ibl[..., 2] = rows[:, None]
    ibl[..., 3] = 255
    return cam, env, ibl
