"""Synthetic two-view scenes for the bench and the parity tests (SURVEY.md §8(d)).

Random 3-D points in front of two known cameras, Gaussian pixel noise, and a stated
fraction of outliers (image-2 coordinates replaced by uniform pixels).  numpy only.
"""
from __future__ import annotations

import numpy as np


def euler_xyz_intrinsic(deg_x: float, deg_y: float, deg_z: float) -> np.ndarray:
    """Rotation matrix of intrinsic X-Y-Z Euler angles (degrees): R = Rx @ Ry @ Rz."""
    ax, ay, az = np.radians([deg_x, deg_y, deg_z])
    cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    rx = np.array([[1.0, 0.0, 0.0], [0.0, cx, -sx], [0.0, sx, cx]])
    ry = np.array([[cy, 0.0, sy], [0.0, 1.0, 0.0], [-sy, 0.0, cy]])
    rz = np.array([[cz, -sz, 0.0], [sz, cz, 0.0], [0.0, 0.0, 1.0]])
    return rx @ ry @ rz


def make_scene(n: int, outlier_frac: float, seed: int, noise_px: float = 0.5,
               f: float = 800.0, w: int = 1280, h: int = 960):
    """Return (K, x1[n,2], x2[n,2], R, t, outlier_idx) in pixel coordinates.

    cam1 = [I|0]; cam2 = [R|t] with R = euler XYZ (2, -8, 1) deg, t = (-1, 0.05, 0.1).
    """
    rng = np.random.default_rng(seed)
    K = np.array([[f, 0.0, w / 2], [0.0, f, h / 2], [0.0, 0.0, 1.0]])
    X = np.column_stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(4, 8, n)])
    R = euler_xyz_intrinsic(2.0, -8.0, 1.0)
    t = np.array([-1.0, 0.05, 0.1])
    x1 = (K @ X.T).T
    x1 = x1[:, :2] / x1[:, 2:]
    X2 = (R @ X.T).T + t
    x2 = (K @ X2.T).T
    x2 = x2[:, :2] / x2[:, 2:]
    x1 += rng.normal(0, noise_px, x1.shape)
    x2 += rng.normal(0, noise_px, x2.shape)
    n_out = int(round(outlier_frac * n))
    idx = rng.choice(n, n_out, replace=False)
    x2[idx] = np.column_stack([rng.uniform(0, w, n_out), rng.uniform(0, h, n_out)])
    return K, np.ascontiguousarray(x1), np.ascontiguousarray(x2), R, t, idx


def make_image_pair(seed: int = 0, h: int = 480, w: int = 640, f: float = 520.0, noise: float = 1.5,
                    planar: bool = False):
    """A synthetic grayscale image pair for the whole pipeline (detector -> matcher -> two-view geometry).

    The scene is three textured fronto-parallel layers at depths 8, 6 and 4.5 in front of camera 1 (so the
    correspondences are not coplanar); camera 2 = [R|t] with R = euler XYZ (1, -4, 0.5) deg, t = (-0.5, 0.02,
    0.05).  Image 1 is the texture; image 2 is rendered by inverse mapping through the plane-induced homographies
    ``H_d = K (R + t n^T / d) K^-1`` (front layer first), bilinear sampling, plus Gaussian noise.  ``planar`` renders the
    back layer (depth 8) over the whole image: every correspondence then lies on one plane.
    Returns (image_1 uint8[h,w], image_2 uint8[h,w], K, R, t).  numpy only."""
    rng = np.random.default_rng(seed)
    tex = np.full((h, w), 110.0)
    for _ in range(260):  # random rectangles: plenty of corners
        y0, x0 = int(rng.integers(0, h - 8)), int(rng.integers(0, w - 8))
        dy, dx = int(rng.integers(8, 60)), int(rng.integers(8, 60))
        tex[y0:y0 + dy, x0:x0 + dx] = rng.integers(10, 246)
    tex += rng.normal(0, 4.0, tex.shape)
    pad = np.pad(tex, 1, mode="edge")
    tex = sum(pad[i:i + h, j:j + w] for i in range(3) for j in range(3)) / 9.0  # a light blur
    K = np.array([[f, 0.0, w / 2], [0.0, f, h / 2], [0.0, 0.0, 1.0]])
    R = euler_xyz_intrinsic(1.0, -4.0, 0.5)
    t = np.array([-0.5, 0.02, 0.05])
    # (depth, region in image-1 pixels [y0, y1, x0, x1]), front to back
    layers = [(4.5, (250, 440, 330, 600)), (6.0, (60, 300, 60, 320)), (8.0, (-10 ** 6, 10 ** 6, -10 ** 6, 10 ** 6))]
    if planar:
        layers = layers[-1:]
    ys, xs = np.mgrid[0:h, 0:w]
    p2 = np.stack([xs.ravel(), ys.ravel(), np.ones(h * w)]).astype(np.float64)
    out = np.zeros(h * w)
    done = np.zeros(h * w, dtype=bool)
    Kinv = np.linalg.inv(K)
    for depth, (y0, y1, x0, x1) in layers:
        H = K @ (R + np.outer(t, [0.0, 0.0, 1.0]) / depth) @ Kinv
        p1 = np.linalg.solve(H, p2)
        u, v = p1[0] / p1[2], p1[1] / p1[2]
        inside = (~done) & (u >= max(x0, 0)) & (u < min(x1, w - 1)) & (v >= max(y0, 0)) & (v < min(y1, h - 1))
        ui, vi = np.floor(u[inside]).astype(int), np.floor(v[inside]).astype(int)
        fu, fv = u[inside] - ui, v[inside] - vi
        out[inside] = ((1 - fv) * ((1 - fu) * tex[vi, ui] + fu * tex[vi, ui + 1])
                       + fv * ((1 - fu) * tex[vi + 1, ui] + fu * tex[vi + 1, ui + 1]))
        done |= inside
    out[~done] = 110.0
    img2 = out.reshape(h, w) + rng.normal(0, noise, (h, w))
    img1 = tex + rng.normal(0, noise, (h, w))
    to_u8 = lambda a: np.clip(np.round(a), 0, 255).astype(np.uint8)  # noqa: E731
    return to_u8(img1), to_u8(img2), K, R, t


def make_planar_scene(n: int, outlier_frac: float, seed: int, noise_px: float = 0.5, rotation_only: bool = False,
                      f: float = 800.0, w: int = 1280, h: int = 960):
    """Return (K, x1[n,2], x2[n,2], H_true, outlier_idx) in pixel coordinates for points on one plane.

    The cameras are those of ``make_scene`` (cam1 = [I|0], cam2 = [R|t]; t = 0 when ``rotation_only``).  The points lie
    on the plane n^T X = d with n = unit(0.15, -0.1, 1), d = 6, tilted against both image planes and in front of both
    cameras; H_true = K (R + t n^T / d) K^-1 maps image-1 pixels to image-2 pixels (the construction of
    ``make_image_pair``), divided by its [2,2] entry.  Noise and outliers as in ``make_scene``."""
    rng = np.random.default_rng(seed)
    K = np.array([[f, 0.0, w / 2], [0.0, f, h / 2], [0.0, 0.0, 1.0]])
    nrm = np.array([0.15, -0.1, 1.0])
    nrm /= np.linalg.norm(nrm)
    d = 6.0
    R = euler_xyz_intrinsic(2.0, -8.0, 1.0)
    t = np.zeros(3) if rotation_only else np.array([-1.0, 0.05, 0.1])
    # rays through uniform image-1 pixels, cut with the plane
    u = np.column_stack([rng.uniform(0, w, n), rng.uniform(0, h, n), np.ones(n)])
    rays = (np.linalg.inv(K) @ u.T).T
    X = rays * (d / (rays @ nrm))[:, None]
    x1 = u[:, :2].copy()
    X2 = (R @ X.T).T + t
    x2 = (K @ X2.T).T
    x2 = x2[:, :2] / x2[:, 2:]
    x1 += rng.normal(0, noise_px, x1.shape)
    x2 += rng.normal(0, noise_px, x2.shape)
    n_out = int(round(outlier_frac * n))
    idx = rng.choice(n, n_out, replace=False)
    x2[idx] = np.column_stack([rng.uniform(0, w, n_out), rng.uniform(0, h, n_out)])
    H_true = K @ (R + np.outer(t, nrm) / d) @ np.linalg.inv(K)
    return K, np.ascontiguousarray(x1), np.ascontiguousarray(x2), H_true / H_true[2, 2], idx
