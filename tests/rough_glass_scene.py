"""Rough glass (include/b200rt.h, B200RT_SAMPLING_ROUGH_GLASS) for the tests: a numpy float32 restatement of the rough
interface rule, scene variants with rough glass, and a glass slab in front of a checker environment.  Every step of the
restatement is one elementwise binary32 operation in the header's order (numpy never fuses two of them); the sine and
cosine are float64's rounded to binary32, which is the correctly rounded value unless the float64 result lies within
2^-29 relative of a binary32 rounding boundary."""
import numpy as np

import ensem3a_openclraytracer_b200 as rt
from tests import fixtures, glass_scene as gs

f32 = np.float32
GLASS = rt.SAMPLING_DIELECTRIC_GLASS
ROUGH = rt.SAMPLING_ROUGH_GLASS
_dot = gs._dot


def _cross(a, b):
    return np.stack([a[:, 1] * b[:, 2] - a[:, 2] * b[:, 1], a[:, 2] * b[:, 0] - a[:, 0] * b[:, 2],
                     a[:, 0] * b[:, 1] - a[:, 1] * b[:, 0]], axis=1).astype(f32)


def _unit(a):
    return (a / np.sqrt(_dot(a, a))[:, None]).astype(f32)


def visible_normal(al, N, Vw, u1, u2):
    """(m, 3): the header's GGX visible normal of roughness al (m,) around unit N (m, 3) seen from unit Vw (m, 3)"""
    one = f32(1)
    sg = np.copysign(one, N[:, 2]).astype(f32)
    a = -one / (sg + N[:, 2])
    b = (N[:, 0] * N[:, 1]) * a
    T = np.stack([one + ((sg * N[:, 0]) * N[:, 0]) * a, sg * b, -sg * N[:, 0]], axis=1).astype(f32)
    B = np.stack([b, sg + (N[:, 1] * N[:, 1]) * a, -N[:, 1]], axis=1).astype(f32)
    Vh = _unit(np.stack([al * _dot(Vw, T), al * _dot(Vw, B), _dot(N, Vw)], axis=1).astype(f32))
    lensq = Vh[:, 0] * Vh[:, 0] + Vh[:, 1] * Vh[:, 1]
    inv = one / np.sqrt(np.where(lensq > 0, lensq, one))
    T1 = np.where((lensq > 0)[:, None], np.stack([-Vh[:, 1] * inv, Vh[:, 0] * inv, np.zeros_like(inv)], axis=1),
                  np.array([[1, 0, 0]], f32)).astype(f32)
    T2 = _cross(Vh, T1)
    phi = f32(6.2831853) * u2
    sp, cp = np.sin(phi.astype(np.float64)).astype(f32), np.cos(phi.astype(np.float64)).astype(f32)
    r = np.sqrt(u1)
    t1 = r * cp
    t2 = r * sp
    s = f32(0.5) * (one + Vh[:, 2])
    t2 = (one - s) * np.sqrt(np.fmax(f32(0), one - t1 * t1)) + s * t2
    t3 = np.sqrt(np.fmax(f32(0), (one - t1 * t1) - t2 * t2))
    Nh = (T1 * t1[:, None] + T2 * t2[:, None]) + Vh * t3[:, None]
    hl = _unit(np.stack([al * Nh[:, 0], al * Nh[:, 1], np.fmax(f32(0), Nh[:, 2])], axis=1).astype(f32))
    return ((T * hl[:, :1] + B * hl[:, 1:2]) + N * hl[:, 2:3]).astype(f32)


def rough_dielectric(d, n, v, r, uf, u1, u2):
    """the header's rule for m cases: d (m, 3) incoming directions, n (m, 3) unit normals, v (m,) ior slots (not 1),
    r (m,) roughness > 0, uf u1 u2 (m,) uniforms -> (directions (m, 3), reflected (m,) bool, weight (m,))"""
    d, n = np.asarray(d, f32).reshape(-1, 3), np.asarray(n, f32).reshape(-1, 3)
    v, r, uf, u1, u2 = (np.asarray(x, f32).reshape(-1) for x in (v, r, uf, u1, u2))
    one = f32(1)
    with np.errstate(all="ignore"):
        w = _unit(d)
        c = _dot(w, n)
        enter = c < f32(0)
        ior = np.where(v == f32(0), f32(1.5), v).astype(f32)
        eta = np.where(enter, one / ior, ior).astype(f32)
        m = np.where(enter[:, None], n, -n).astype(f32)
        Vw = -w
        h = visible_normal(r, m, Vw, u1, u2)
        fallback = (c == f32(0)) | ~np.isfinite(c) | ~np.isfinite(h).all(axis=1)
        ch = _dot(Vw, h)
        k = one - (eta * eta) * (one - ch * ch)
        ok = k >= f32(0)
        ct = np.sqrt(np.where(ok, k, f32(0))).astype(f32)
        rs = (eta * ch - ct) / (eta * ch + ct)
        rp = (ch - eta * ct) / (ch + eta * ct)
        F = f32(0.5) * (rs * rs + rp * rp)
        refl = ~ok | ~(uf >= F)
        nd = np.where(refl[:, None], w + h * (f32(2) * ch)[:, None], w * eta[:, None] + h * (eta * ch - ct)[:, None])
        co = _dot(nd, m)
        a = np.abs(co)
        a2 = r * r
        g1 = (f32(2) * a) / (a + np.sqrt(a2 + ((one - a2) * a) * a))
        wt = np.where(np.where(refl, co > 0, co < 0), g1, f32(0)).astype(f32)
        d0, r0, _ = gs.dielectric(d, n, v, uf)
    nd = np.where(fallback[:, None], d0, nd).astype(f32)
    return nd, np.where(fallback, r0, refl), np.where(fallback, one, wt).astype(f32)


def glass_roughness(sc, r):
    """sc with every glass material's roughness slot set to r"""
    def f(m):
        m[m[:, 0] == 3, 4] = r
        return m
    return gs.with_materials(sc, f)


def bench_rough(r=0.2):
    """config 2 (the benchmark's scene) with its glass wall (material 1) at roughness r"""
    return glass_roughness(fixtures.load_scene("monkey_cfg2"), r)


def mixed():
    """config 2 with a rough glass wall (material 1, roughness 0.2) and a smooth glass monkey (material 4, roughness 0):
    one frame runs both branches of the rough kernels"""
    def f(m):
        m[1, 4] = 0.2
        m[4] = [3, 1, 1, 1, 0, 0]
        return m
    return gs.with_materials(fixtures.load_scene("monkey_cfg2"), f)


def load(name):
    """"bench_rough", "mixed", or a fixture scene ("proto" ships glass of roughness 0.1)"""
    if name == "bench_rough":
        return bench_rough()
    if name == "mixed":
        return mixed()
    return fixtures.load_scene(name)


def view(name, w, h=None):
    """cam, env of a scene given to load()"""
    return fixtures.cam_env(fixtures.load_scene("proto" if name == "proto" else "monkey_cfg2")["params"], w, h)


def slab(r, colour=(1.0, 1.0, 1.0), ior=0.0):
    """a closed glass box 6 wide, 0.3 deep, 6 high around y = 2.15, in front of an unrotated camera at the origin that
    looks along +y; flat outward normals, one glass material of roughness r"""
    lo, hi = np.array([-3.0, 2.0, -3.0]), np.array([3.0, 2.3, 3.0])
    pos, nrm, faces = [], [], []
    for axis in range(3):
        for side in (0, 1):
            nv = np.zeros(3)
            nv[axis] = 1.0 if side else -1.0
            u, v = [a for a in range(3) if a != axis]
            quad = []
            for cu, cv in ((0, 0), (1, 0), (1, 1), (0, 1)):
                p = np.where(np.arange(3) == axis, (hi if side else lo)[axis], 0.0)
                p[u] = (lo, hi)[cu][u]
                p[v] = (lo, hi)[cv][v]
                quad.append(len(pos))
                pos.append(p)
                nrm.append(nv)
            a, b, c, d = quad
            for tri in ((a, b, c), (a, c, d)):
                e = np.cross(pos[tri[1]] - pos[tri[0]], pos[tri[2]] - pos[tri[0]])
                faces.append(tri if np.dot(e, nv) > 0 else (tri[0], tri[2], tri[1]))
    fd = np.array([[0, a, b, c, a, b, c, a, b, c] for a, b, c in faces], np.int32)
    sc = {"V_p": np.asarray(pos, f32).reshape(-1), "V_n": np.asarray(nrm, f32).reshape(-1),
          "V_uv": np.zeros(2, f32), "faceData": fd.reshape(-1),
          "materialData": np.array([3, *colour, r, ior], f32), "lightData": np.zeros(0, np.int32)}
    sc["BVH"] = rt.BVH(sc["faceData"], sc["V_p"]).exportArray
    return sc


def checker_view(width, tile=8):
    """cam, env (no sun, environment power 1) for the slab, and a black-and-white checker environment map"""
    cam = np.array([0, 0, 0, 0, 0, 0, width, width, 1, 60.0 * (3.14 / 180)], f32)
    env = np.array([0, 0, 0, 0, 1], f32)
    yy, xx = np.mgrid[0:64, 0:128]
    on = ((yy // tile + xx // tile) % 2).astype(np.uint8) * 255
    ibl = np.stack([on, on, on, np.full_like(on, 255)], axis=2)
    return cam, env, np.ascontiguousarray(ibl)
