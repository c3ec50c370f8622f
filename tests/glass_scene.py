"""Refractive glass (include/b200rt.h, B200RT_SAMPLING_DIELECTRIC_GLASS) for the tests: a numpy float32 restatement of
the interface rule, scene variants with glass, and a glass sphere under the uniform grey map or a vertically graded
one.  Every step of the restatement is one elementwise binary32 operation in the header's order (numpy never fuses two
of them)."""
import numpy as np

import ensem3a_openclraytracer_b200 as rt
from tests import fixtures, smooth_scene

f32 = np.float32
GLASS = rt.SAMPLING_DIELECTRIC_GLASS


def _dot(a, b):
    return (a[:, 0] * b[:, 0] + a[:, 1] * b[:, 1]) + a[:, 2] * b[:, 2]


def dielectric(d, n, v, u):
    """the header's rule for m cases: d (m, 3) incoming directions, n (m, 3) unit normals, v (m,) ior slots (not 1),
    u (m,) uniforms -> (directions (m, 3), reflected (m,) bool, F (m,), 1 on total internal reflection)"""
    d, n = np.asarray(d, f32).reshape(-1, 3), np.asarray(n, f32).reshape(-1, 3)
    v, u = np.asarray(v, f32).reshape(-1), np.asarray(u, f32).reshape(-1)
    with np.errstate(all="ignore"):
        w = d / np.sqrt(_dot(d, d))[:, None]
        c = _dot(w, n)
        enter = c < f32(0)
        ior = np.where(v == f32(0), f32(1.5), v).astype(f32)
        eta = np.where(enter, f32(1) / ior, ior).astype(f32)
        ci = np.where(enter, -c, c).astype(f32)
        m = np.where(enter[:, None], n, -n).astype(f32)
        k = f32(1) - (eta * eta) * (f32(1) - ci * ci)
        ok = k >= f32(0)
        ct = np.sqrt(np.where(ok, k, f32(0))).astype(f32)
        rs = (eta * ci - ct) / (eta * ci + ct)
        rp = (ci - eta * ct) / (ci + eta * ct)
        F = np.where(ok, f32(0.5) * (rs * rs + rp * rp), f32(1)).astype(f32)
        refl = ~ok | ~(u >= F)
        dr = w + m * (f32(2) * ci)[:, None]
        dt = w * eta[:, None] + m * (eta * ci - ct)[:, None]
    return np.where(refl[:, None], dr, dt).astype(f32), refl, F


def with_materials(sc, fn):
    """a copy of scene sc whose (n_mat, 6) material table is fn(table copy)"""
    out = dict(sc)
    mat = sc["materialData"].reshape(-1, 6).copy()
    out["materialData"] = np.ascontiguousarray(fn(mat), f32).reshape(-1)
    return out


def glass_ior(sc, v):
    """sc with every glass material's ior slot set to v"""
    def f(m):
        m[m[:, 0] == 3, 5] = v
        return m
    return with_materials(sc, f)


def glass_monkey():
    """config 2 with the monkey's material (4, a closed 15 744-triangle mesh) turned into glass"""
    def f(m):
        m[4] = [3, 1, 1, 1, 0, 0]
        return m
    return with_materials(fixtures.load_scene("monkey_cfg2"), f)


def load(name):
    """a fixture scene, or "monkey_glass" for glass_monkey()"""
    return glass_monkey() if name == "monkey_glass" else fixtures.load_scene(name)


def glass_sphere(colour=(1.0, 1.0, 1.0), ior=0.0, n_lon=48, n_lat=24):
    """smooth_scene's UV sphere (outward vertex normals) as one glass material"""
    sc = smooth_scene.sphere(n_lon, n_lat)
    sc["materialData"] = np.array([3, *colour, 0.0, ior], f32)
    return sc


def grey_view(width):
    """cam, env (no sun, environment power 1) for the sphere, and the uniform grey map"""
    cam, env, _ = smooth_scene.sphere_view(width)
    return cam, env, fixtures.load_ibl("grey")
