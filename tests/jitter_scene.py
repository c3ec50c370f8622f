"""A scene whose pixel-area image is known exactly: one emissive triangle of power 1 in the plane y = Y0 in front of an
unrotated camera at the origin, with no sun and no environment light, whose edge crosses the frame obliquely.  A camera
ray through image-plane point (px, pz) (include/b200rt.h, B200RT_SAMPLING_PIXEL_JITTER) meets that plane at
(px, f, pz) * Y0 / f, so the lit part of the image plane is the half-plane px * cos(t) + pz * sin(t) > D, and a pixel's
box-filtered value is the fraction of its footprint inside it."""
import numpy as np

import ensem3a_openclraytracer_b200 as rt

FOV_DEG = 60.0
Y0 = 2.0
THETA = np.deg2rad(33.0)   # the edge's normal in the image plane
D = 0.07                   # its distance from the image centre


def _cam_env(width, height):
    cam = np.array([0, 0, 0, 0, 0, 0, width, height, 1, FOV_DEG * (3.14 / 180)], np.float32)
    env = np.array([0, 0, 0, 0, 0], np.float32)
    return cam, env


def scene(width, height):
    """(scene dict in the reference's layouts, cam, env, ibl)"""
    cam, env = _cam_env(width, height)
    f = 1.0 / (2.0 * np.tan(np.float64(cam[9]) / 2.0))
    n = np.array([np.cos(THETA), np.sin(THETA)])
    u = np.array([-np.sin(THETA), np.cos(THETA)])
    pts = [D * n - 10.0 * u, D * n + 10.0 * u, D * n + 10.0 * n]      # image-plane (px, pz); lit side along +n
    vp = np.array([[p[0] * Y0 / f, Y0, p[1] * Y0 / f] for p in pts], np.float32).reshape(-1)
    sc = {"V_p": vp, "V_n": np.array([0, -1, 0], np.float32), "V_uv": np.zeros(2, np.float32),
          "faceData": np.array([0, 0, 0, 0, 0, 0, 0, 0, 1, 2], np.int32),
          "materialData": np.array([0, 1, 1, 1, 1.0, 1], np.float32), "lightData": np.array([0], np.int32)}
    sc["BVH"] = rt.BVH(sc["faceData"], sc["V_p"]).exportArray
    ibl = np.zeros((2, 4, 4), np.uint8)
    return sc, cam, env, ibl


def coverage(width, height, grid=256):
    """float64 (height, width): the fraction of every pixel's footprint [col - 0.5, col + 0.5) x [row - 0.5, row + 0.5)
    (col = (i + 1) % width, row = (i - col) / width, the reference's mapping) on the lit side, from a grid x grid
    midpoint sub-grid; pixels whose footprint the edge does not cross are exactly 0 or 1"""
    step = 1.0 / width
    i = np.arange(width * height)
    col = (i + 1) % width
    row = np.trunc((i - col) / width).astype(np.int64)   # C's truncating division: row 0 holds i - col = -1
    sub = (np.arange(grid) + 0.5) / grid - 0.5
    c, s = np.cos(THETA), np.sin(THETA)

    def side(fx, fz):
        return (fx * step - 0.5) * c + (0.5 - fz * step) * s - D

    # the signed distance of the centre against the footprint's half-diagonal decides the uncut pixels
    centre = side(col.astype(np.float64), row.astype(np.float64))
    half = 0.5 * step * (abs(c) + abs(s))
    f = (centre > 0).astype(np.float64)
    cut = np.nonzero(np.abs(centre) <= half)[0]
    for k in cut:
        fx = col[k] + sub[None, :]
        fz = row[k] + sub[:, None]
        f[k] = np.mean(side(fx, fz) > 0)
    return f.reshape(height, width)
