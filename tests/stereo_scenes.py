"""Seeded rectified stereo pairs with a known per-pixel disparity, built to reach every branch of searchByStereo.

A scene is a list of textured, planar layers drawn far to near.  Each layer's disparity is affine in the left image's
(rectified) coordinates, d = a + b*x + c*y, which is exactly what a 3-D plane gives, and a pixel of the right view at
(xr, y) shows the layer point at xl = (xr + a + c*y) / (1 - b).  Both views sample the layer textures bilinearly, so
fractional disparities show up in the pixels, and a nearer layer overwrites a farther one in each view on its own, so
occlusions are consistent between the views.  The layers:
  * a far background with disparity in [-0.4, 0.6] px (a slightly negative disparity models a rectification error);
  * a slanted ground plane below the horizon whose disparity grows to about 80 px at the bottom row;
  * a strip whose right view is also shifted down by a fraction of a pixel (rows of the right keypoints then differ from
    the left ones, which exercises the row band of createRowIndexDB);
  * a noise-free patch whose texture repeats every few pixels horizontally (Hamming and SAD ties);
  * a few fronto-parallel occluders with constant fractional disparity in (20, 120), each with its own texture.
The right view gets +-2 grey levels of noise everywhere except on the periodic patch, as synth.synth_stereo_pair does.

`dist` renders the left view through a Brown-Conrady lens (k1, k2, p1, p2, k3) at the camera (fx, fy, cx, cy): a left
pixel shows the scene at its undistorted position, which is where the matcher looks for it after undistorting the left
keypoints.  With barrel distortion (k1 < 0) the left view sees past the right view's border, so undistorted keypoints
land outside the image: their rows leave the row index, or their SAD windows leave the level image.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from orb_slam2_ros2_b200 import synth


@dataclass
class Layer:
    tex: np.ndarray  # float32 texture, indexed at (y + oy, x + ox) of the left view's rectified coordinates
    a: float = 0.0  # disparity d = a + b*x + c*y
    b: float = 0.0
    c: float = 0.0
    rect: tuple = (-1e9, -1e9, 1e9, 1e9)  # (x0, y0, x1, y1): the layer covers x0 <= x < x1, y0 <= y < y1 of the left view
    dy: float = 0.0  # the right view shows the left row y + dy at its row y
    noise: bool = True
    ox: float = 0.0
    oy: float = 0.0


@dataclass
class Scene:
    name: str
    h: int
    w: int
    layers: list = field(default_factory=list)
    seed: int = 0


def _bilinear(tex: np.ndarray, x: np.ndarray, y: np.ndarray) -> np.ndarray:
    th, tw = tex.shape
    x = np.clip(x, 0, tw - 1.001)
    y = np.clip(y, 0, th - 1.001)
    x0, y0 = np.floor(x).astype(np.int64), np.floor(y).astype(np.int64)
    fx, fy = (x - x0).astype(np.float32), (y - y0).astype(np.float32)
    t00, t01 = tex[y0, x0], tex[y0, x0 + 1]
    t10, t11 = tex[y0 + 1, x0], tex[y0 + 1, x0 + 1]
    return (t00 * (1 - fx) + t01 * fx) * (1 - fy) + (t10 * (1 - fx) + t11 * fx) * fy


def _texture(h: int, w: int, seed: int, margin: int = 256) -> np.ndarray:
    """synth's blocky multi-scale texture, large enough for every shifted or undistorted lookup"""
    return synth.synth_image(h + 2 * margin, w + 2 * margin, seed).astype(np.float32)


def _periodic_texture(h: int, period: int, seed: int, margin: int = 256) -> np.ndarray:
    """columns repeat every `period` px; each period is two bars whose grey levels change every 4 rows"""
    rng = np.random.default_rng(seed)
    rows = h + 2 * margin
    cells = rng.integers(20, 236, ((rows + 3) // 4, 2)).astype(np.float32)
    col = (np.arange(period) >= period // 2).astype(np.int64)
    one = cells[np.arange(rows) // 4][:, col]  # (rows, period)
    return np.tile(one, (1, (2 * margin + 4096) // period + 1))


def make_scene(name: str, h: int, w: int, seed: int, period: int = 6) -> Scene:
    """the layer set above, placed relative to the image size; the seed moves the occluders and draws the textures"""
    rng = np.random.default_rng(seed)
    s = Scene(name, h, w, seed=seed)
    m = 256
    # far background: disparity from -0.4 at the left border to 0.6 at the right border, rising 0.1 px over the rows too
    s.layers.append(Layer(_texture(h, w, seed * 10 + 1), a=-0.45, b=0.9 / w, c=0.1 / h, ox=m, oy=m))
    # ground plane: 0 at the horizon, about 80 px at the bottom row
    yh = 0.55 * h
    c = 80.0 / (h - 1 - yh)
    s.layers.append(Layer(_texture(h, w, seed * 10 + 2), a=-c * yh, c=c, rect=(-1e9, yh, 1e9, 1e9), ox=m, oy=m))
    # a strip whose right view is shifted vertically by a fraction of a pixel
    y0 = float(int(0.30 * h))
    s.layers.append(Layer(_texture(h, w, seed * 10 + 3), a=float(rng.uniform(6, 14)), rect=(0.05 * w, y0, 0.45 * w, y0 + 0.12 * h),
                          dy=float(rng.uniform(0.3, 0.7)), ox=m, oy=m))
    # noise-free periodic patch
    px0 = float(int(rng.uniform(0.5, 0.6) * w))
    s.layers.append(Layer(_periodic_texture(h, period, seed * 10 + 4), a=float(rng.uniform(8, 16)), rect=(px0, 0.08 * h, px0 + 0.22 * w, 0.40 * h),
                          noise=False, ox=m, oy=m))
    # fronto-parallel occluders; the last one sits at the right border and reaches past it
    for k in range(2):
        d = float(rng.uniform(20, 120))
        ww, hh = rng.uniform(0.10, 0.18) * w, rng.uniform(0.18, 0.35) * h
        x0, y0 = float(rng.uniform(0.15, 0.75) * w), float(rng.uniform(0.1, 0.9) * h - hh / 2)
        s.layers.append(Layer(_texture(h, w, seed * 10 + 5 + k), a=d, rect=(x0, y0, x0 + ww, y0 + hh), ox=m, oy=m))
    # the nearest occluder covers the right border and continues past it, where only an undistorted left view reaches;
    # its disparity brings that part into the right view
    d = float(rng.uniform(80, 120))
    s.layers.append(Layer(_texture(h, w, seed * 10 + 7), a=d, rect=(w - 0.12 * w, 0.2 * h, 1.25 * w, 0.8 * h), ox=m, oy=m))
    return s


def undistort_grid(h: int, w: int, fx: float, fy: float, cx: float, cy: float, dist) -> tuple[np.ndarray, np.ndarray]:
    """undistorted position of every left pixel (cv::undistortPoints' fixed-point iteration, in double)"""
    k1, k2, p1, p2, k3 = (list(dist) + [0.0] * 5)[:5]
    yd, xd = np.mgrid[0:h, 0:w].astype(np.float64)
    x0, y0 = (xd - cx) / fx, (yd - cy) / fy
    x, y = x0.copy(), y0.copy()
    for _ in range(20):
        r2 = x * x + y * y
        icd = 1.0 / (1.0 + ((k3 * r2 + k2) * r2 + k1) * r2)
        ddx = 2 * p1 * x * y + p2 * (r2 + 2 * x * x)
        ddy = p1 * (r2 + 2 * y * y) + 2 * p2 * x * y
        x, y = (x0 - ddx) * icd, (y0 - ddy) * icd
    return x * fx + cx, y * fy + cy


def render(s: Scene, cam: dict | None = None, dist=None):
    """-> (left, right, disparity) with disparity[y, x] the true disparity of the left pixel (of its undistorted position
    when `dist` is given)"""
    h, w = s.h, s.w
    if dist is not None and any(dist):
        xl, yl = undistort_grid(h, w, cam["fx"], cam["fy"], cam["cx"], cam["cy"], dist)
    else:
        yl, xl = np.mgrid[0:h, 0:w].astype(np.float64)
    left = np.zeros((h, w), np.float32)
    disp = np.zeros((h, w), np.float32)
    for L in s.layers:
        x0, y0, x1, y1 = L.rect
        cov = (xl >= x0) & (xl < x1) & (yl >= y0) & (yl < y1)
        left[cov] = _bilinear(L.tex, xl[cov] + L.ox, yl[cov] + L.oy)
        disp[cov] = (L.a + L.b * xl[cov] + L.c * yl[cov]).astype(np.float32)
    yr, xr = np.mgrid[0:h, 0:w].astype(np.float64)
    right = np.zeros((h, w), np.float32)
    noisy = np.ones((h, w), bool)
    for L in s.layers:
        x0, y0, x1, y1 = L.rect
        ys = yr + L.dy
        xs = (xr + L.a + L.c * ys) / (1.0 - L.b)
        cov = (xs >= x0) & (xs < x1) & (ys >= y0) & (ys < y1)
        right[cov] = _bilinear(L.tex, xs[cov] + L.ox, ys[cov] + L.oy)
        noisy[cov] = L.noise
    noise = np.random.default_rng(s.seed + 100).integers(-2, 3, (h, w)).astype(np.float32)
    right = right + np.where(noisy, noise, 0.0)
    to_u8 = lambda a: np.clip(np.rint(a), 0, 255).astype(np.uint8)
    return to_u8(left), to_u8(right), disp
