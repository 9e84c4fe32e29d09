"""Synthetic two-view scenes for the bench and the parity tests (SURVEY.md §8(d)).

Random 3-D points in front of two known cameras, Gaussian pixel noise, and a stated
fraction of outliers (image-2 coordinates replaced by uniform pixels).  numpy only.
"""
from __future__ import annotations

import dataclasses

import numpy as np


def euler_xyz_intrinsic(deg_x: float, deg_y: float, deg_z: float) -> np.ndarray:
    """Rotation matrix of intrinsic X-Y-Z Euler angles (degrees): R = Rx @ Ry @ Rz."""
    ax, ay, az = np.radians([deg_x, deg_y, deg_z])
    cx, sx, cy, sy, cz, sz = np.cos(ax), np.sin(ax), np.cos(ay), np.sin(ay), np.cos(az), np.sin(az)
    rx = np.array([[1.0, 0.0, 0.0], [0.0, cx, -sx], [0.0, sx, cx]])
    ry = np.array([[cy, 0.0, sy], [0.0, 1.0, 0.0], [-sy, 0.0, cy]])
    rz = np.array([[cz, -sz, 0.0], [sz, cz, 0.0], [0.0, 0.0, 1.0]])
    return rx @ ry @ rz


def _camera(K, f, w, h):
    if K is None:
        return np.array([[f, 0.0, w / 2], [0.0, f, h / 2], [0.0, 0.0, 1.0]])
    return np.asarray(K, dtype=np.float64).reshape(3, 3).copy()


def make_scene(n: int, outlier_frac: float, seed: int, noise_px: float = 0.5,
               f: float = 800.0, w: int = 1280, h: int = 960, K=None):
    """Return (K, x1[n,2], x2[n,2], R, t, outlier_idx) in pixel coordinates.

    cam1 = K[I|0]; cam2 = K[R|t] with R = euler XYZ (2, -8, 1) deg, t = (-1, 0.05, 0.1).  K defaults to
    [[f, 0, w/2], [0, f, h/2], [0, 0, 1]]; any other (skewed, fx != fy) may be given.
    """
    rng = np.random.default_rng(seed)
    K = _camera(K, f, w, h)
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
                      f: float = 800.0, w: int = 1280, h: int = 960, K=None):
    """Return (K, x1[n,2], x2[n,2], H_true, outlier_idx) in pixel coordinates for points on one plane.

    The cameras are those of ``make_scene`` (cam1 = [I|0], cam2 = [R|t]; t = 0 when ``rotation_only``).  The points lie
    on the plane n^T X = d with n = unit(0.15, -0.1, 1), d = 6, tilted against both image planes and in front of both
    cameras; H_true = K (R + t n^T / d) K^-1 maps image-1 pixels to image-2 pixels (the construction of
    ``make_image_pair``), divided by its [2,2] entry.  Noise, outliers and K as in ``make_scene``."""
    rng = np.random.default_rng(seed)
    K = _camera(K, f, w, h)
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


def make_pnp_scene(n: int, outlier_frac: float, seed: int, noise_px: float = 0.5,
                   f: float = 800.0, w: int = 1280, h: int = 960, K=None):
    """Return (K, X[n,3], x[n,2], R, t, outlier_idx) for the absolute pose of one camera.

    The world points are those of ``make_scene`` (in front of the world camera [I|0]); the new camera is K[R|t] with
    R = euler XYZ (-3, 12, 2) deg, t = (0.8, -0.1, 0.3), so every point is in front of it too.  x = the projection plus
    Gaussian noise; a fraction ``outlier_frac`` of the pixels is replaced by uniform pixels.  K as in ``make_scene``."""
    rng = np.random.default_rng(seed)
    K = _camera(K, f, w, h)
    X = np.column_stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(4, 8, n)])
    R = euler_xyz_intrinsic(-3.0, 12.0, 2.0)
    t = np.array([0.8, -0.1, 0.3])
    p = (K @ ((R @ X.T).T + t).T).T
    x = p[:, :2] / p[:, 2:]
    x += rng.normal(0, noise_px, x.shape)
    n_out = int(round(outlier_frac * n))
    idx = rng.choice(n, n_out, replace=False)
    x[idx] = np.column_stack([rng.uniform(0, w, n_out), rng.uniform(0, h, n_out)])
    return K, np.ascontiguousarray(X), np.ascontiguousarray(x), R, t, idx


def make_three_view_scene(n: int, outlier_frac: float, seed: int, noise_px: float = 0.5,
                          f: float = 800.0, w: int = 1280, h: int = 960, K=None):
    """Return (K, x1, x2, x3 [n,2] each, (R2, t2), (R3, t3), X[n,3]) for one point set seen by three cameras.

    Cameras 1 and 2 and the points are those of ``make_scene`` (cam1 = K[I|0], cam2 = K[R2|t2]); camera 3 is the new
    view of ``make_pnp_scene`` (K[R3|t3], R3 = euler XYZ (-3, 12, 2) deg, t3 = (0.8, -0.1, 0.3)), all in camera-1
    coordinates.  Noise on every image; outliers (uniform pixels) in image 2 and, independently drawn, in image 3."""
    rng = np.random.default_rng(seed)
    K = _camera(K, f, w, h)
    X = np.column_stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(4, 8, n)])
    R2, t2 = euler_xyz_intrinsic(2.0, -8.0, 1.0), np.array([-1.0, 0.05, 0.1])
    R3, t3 = euler_xyz_intrinsic(-3.0, 12.0, 2.0), np.array([0.8, -0.1, 0.3])

    def project(R, t):
        p = (K @ ((R @ X.T).T + t).T).T
        return p[:, :2] / p[:, 2:] + rng.normal(0, noise_px, (n, 2))

    x1, x2, x3 = project(np.eye(3), np.zeros(3)), project(R2, t2), project(R3, t3)
    n_out = int(round(outlier_frac * n))
    for x in (x2, x3):
        idx = rng.choice(n, n_out, replace=False)
        x[idx] = np.column_stack([rng.uniform(0, w, n_out), rng.uniform(0, h, n_out)])
    return (K, np.ascontiguousarray(x1), np.ascontiguousarray(x2), np.ascontiguousarray(x3), (R2, t2), (R3, t3),
            np.ascontiguousarray(X))


def random_rotation(rng) -> np.ndarray:
    """A rotation drawn uniformly over SO(3) (a normalised Gaussian quaternion)."""
    q = rng.normal(size=4)
    w, x, y, z = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y)],
                     [2 * (x * y + w * z), 1 - 2 * (x * x + z * z), 2 * (y * z - w * x)],
                     [2 * (x * z - w * y), 2 * (y * z + w * x), 1 - 2 * (x * x + y * y)]])


def _axis_rotations():
    """Rotations whose optical axis (third row) is each of +-x, +-y, +-z, and three rotations by 180 deg - 1e-6."""
    out = []
    for k in range(3):
        for s in (1.0, -1.0):
            z = np.zeros(3)
            z[k] = s
            x = np.zeros(3)
            x[(k + 1) % 3] = 1.0
            out.append(np.stack([x, np.cross(z, x), z]))
    for axis in np.eye(3):
        a = np.pi - 1e-6
        Kx = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
        out.append(np.eye(3) + np.sin(a) * Kx + (1 - np.cos(a)) * Kx @ Kx)
    return out


def make_pnp_samples(m: int, seed: int, noise_px: float = 0.0, K=None, w: int = 1280, h: int = 960):
    """m random 4-point PnP samples, each (K, X[4,3], x[4,2], R, t) with x_cam = R X + t.

    Pose: R uniform over SO(3) (the first nine samples: optical axis along each of +-x, +-y, +-z, and rotations by
    180 deg - 1e-6 about each axis), the camera centre uniform in a cube of side 2 D around the origin.  Points: pixels
    uniform in a disc of radius rho f around a random image point, wrapped into the image (so up to ~75 deg off axis for
    f = 150), at depths D exp(U(-1, 1) min(rho, 1)); D is log-uniform in [0.5, 100] and the spread rho log-uniform in
    [1e-3, 10] times the depth.  K: f log-uniform in [150, 20 000], principal point at the image centre, unless given.
    x is the projection plus Gaussian noise of noise_px."""
    rng = np.random.default_rng(seed)
    special = _axis_rotations()
    out = []
    for i in range(m):
        if K is None:
            f = float(np.exp(rng.uniform(np.log(150.0), np.log(20_000.0))))
            Ki = np.array([[f, 0.0, w / 2], [0.0, f, h / 2], [0.0, 0.0, 1.0]])
        else:
            Ki = np.asarray(K, dtype=np.float64)
        f = Ki[0, 0]
        R = special[i] if i < len(special) else random_rotation(rng)
        D = float(np.exp(rng.uniform(np.log(0.5), np.log(100.0))))
        rho = float(10.0 ** rng.uniform(-3.0, 1.0))
        ctr = np.array([rng.uniform(0, w), rng.uniform(0, h)])
        r = rho * f * np.sqrt(rng.uniform(0, 1, 4))
        phi = rng.uniform(0, 2 * np.pi, 4)
        pix = np.mod(ctr + np.column_stack([r * np.cos(phi), r * np.sin(phi)]), [w, h])  # wrapped into the image
        dep = D * np.exp(rng.uniform(-1.0, 1.0, 4) * min(rho, 1.0))
        cam = (np.linalg.solve(Ki, np.column_stack([pix, np.ones(4)]).T) * dep).T
        C = rng.uniform(-D, D, 3)
        t = -R @ C
        X = (R.T @ (cam - t).T).T
        p = (Ki @ ((R @ X.T).T + t).T).T
        x = p[:, :2] / p[:, 2:] + rng.normal(0, noise_px, (4, 2))
        out.append((Ki, np.ascontiguousarray(X), np.ascontiguousarray(x), R, t))
    return out


def make_multi_view_scene(n_points: int, n_views: int, seed: int, noise_px: float = 0.5, outlier_frac: float = 0.0,
                          f: float = 800.0, w: int = 1280, h: int = 960, K=None, arc_deg: float = 60.0,
                          min_len: int = 2, max_len: int = 8):
    """Return (K, R[V,3,3], t[V,3], X[N,3], offsets int64[N+1], view int32[M], x[M,2], outlier bool[M]): tracks of
    the ``make_scene`` point cloud seen by V cameras on an arc.

    The cameras lie on a horizontal circular arc of ``arc_deg`` degrees and radius 6 about the cloud's centre (0, 0, 6),
    view 0 at one end, each looking at the centre; x_cam = R X + t.  Point i is seen in a contiguous window of views
    whose length is uniform in [min_len, max_len] (at most V) and whose start is uniform among the windows that fit;
    its observations are in view order.  x = the projection plus Gaussian noise of ``noise_px``; a fraction
    ``outlier_frac`` of all observations is replaced by uniform pixels (``outlier`` marks them).  K as in
    ``make_scene``."""
    rng = np.random.default_rng(seed)
    K = _camera(K, f, w, h)
    N, V = int(n_points), int(n_views)
    X = np.column_stack([rng.uniform(-2, 2, N), rng.uniform(-1.5, 1.5, N), rng.uniform(4, 8, N)])
    centre = np.array([0.0, 0.0, 6.0])
    R = np.empty((V, 3, 3))
    t = np.empty((V, 3))
    for c, th in enumerate(np.radians(np.linspace(-arc_deg / 2, arc_deg / 2, V))):
        C = centre + 6.0 * np.array([np.sin(th), 0.0, -np.cos(th)])
        z = (centre - C) / np.linalg.norm(centre - C)
        xa = np.cross([0.0, 1.0, 0.0], z)
        xa /= np.linalg.norm(xa)
        R[c] = np.stack([xa, np.cross(z, xa), z])
        t[c] = -R[c] @ C
    hi = min(max_len, V)
    length = rng.integers(min(min_len, hi), hi + 1, N)
    start = (rng.uniform(0, 1, N) * (V - length + 1)).astype(np.int64)
    offsets = np.zeros(N + 1, dtype=np.int64)
    np.cumsum(length, out=offsets[1:])
    M = int(offsets[-1])
    pt = np.repeat(np.arange(N), length)
    view = (start[pt] + np.arange(M) - offsets[pt]).astype(np.int32)
    cam = np.einsum("mij,mj->mi", R[view], X[pt]) + t[view]
    p = cam @ K.T
    x = p[:, :2] / p[:, 2:] + rng.normal(0, noise_px, (M, 2))
    outlier = np.zeros(M, dtype=bool)
    outlier[rng.choice(M, int(round(outlier_frac * M)), replace=False)] = True
    n_out = int(outlier.sum())
    x[outlier] = np.column_stack([rng.uniform(0, w, n_out), rng.uniform(0, h, n_out)])
    return K, R, t, X, offsets, view, np.ascontiguousarray(x), outlier


@dataclasses.dataclass
class MatchGraph:
    K: np.ndarray                 # (3,3)
    R: np.ndarray                 # float64[V,3,3] world to camera, x_cam = R X + t
    t: np.ndarray                 # float64[V,3]
    X: np.ndarray                 # float64[n_points,3]
    features: list                # V arrays float64[n_v,2]: the pixels of view v's features, in shuffled order
    point: list                   # V arrays int64[n_v]: the point of each feature, -1 for a distractor
    pairs: np.ndarray             # int32[P,2] (a, b), a < b, b - a <= span
    matches: list                 # P arrays int32[E_p,2]: (local index in a, local index in b)
    wrong: list                   # P arrays bool[E_p]: the match was redirected to a random feature of b


def make_match_graph(n_points: int, n_views: int, seed: int, span: int = 2, wrong_frac: float = 0.0,
                     distractor_frac: float = 0.0, **scene_kw) -> MatchGraph:
    """Per-view features and pairwise matches over the tracks of ``make_multi_view_scene(n_points, n_views, seed,
    **scene_kw)``.

    View v's features are its observations plus round(distractor_frac x their number) uniform pixels, in a random
    order.  For every two views a < b with b - a <= span, the pair holds one match per point observed in both (in
    point order), and a fraction ``wrong_frac`` of all matches has its b index replaced by a uniform random feature of
    b.  A point's observations lie in a contiguous window of views, so with span >= 1 the true matches connect all of
    them, and no view holds two of them."""
    K, R, t, X, off, view, x, _ = make_multi_view_scene(n_points, n_views, seed, **scene_kw)
    rng = np.random.default_rng([seed, 1])
    V = int(n_views)
    w, h = float(2 * K[0, 2]), float(2 * K[1, 2])
    pt = np.repeat(np.arange(len(off) - 1), np.diff(off))
    local = np.empty(len(view), dtype=np.int64)
    features, point = [], []
    for v in range(V):
        obs = np.flatnonzero(view == v)
        nd = int(round(distractor_frac * len(obs)))
        n = len(obs) + nd
        perm = rng.permutation(n)  # feature perm[k] of the view is entry k of (observations, distractors)
        local[obs] = perm[:len(obs)]
        f = np.empty((n, 2))
        f[perm[:len(obs)]] = x[obs]
        f[perm[len(obs):]] = np.column_stack([rng.uniform(0, w, nd), rng.uniform(0, h, nd)])
        p = np.full(n, -1, dtype=np.int64)
        p[perm[:len(obs)]] = pt[obs]
        features.append(f)
        point.append(p)
    # observation m and m + d belong to one point when the point's window holds both; their views are then d apart
    ia, ib = [], []
    for d in range(1, int(span) + 1):
        m = np.arange(len(view) - d)
        same = pt[m] == pt[m + d] if len(m) else np.zeros(0, dtype=bool)
        ia.append(m[same])
        ib.append(m[same] + d)
    ia = np.concatenate(ia) if ia else np.zeros(0, dtype=np.int64)
    ib = np.concatenate(ib) if ib else np.zeros(0, dtype=np.int64)
    key = view[ia].astype(np.int64) * V + view[ib]
    order = np.lexsort((pt[ia], key))
    ia, ib, key = ia[order], ib[order], key[order]
    mj = local[ib].copy()
    wrong = np.zeros(len(mj), dtype=bool)
    wrong[rng.choice(len(mj), int(round(wrong_frac * len(mj))), replace=False)] = True
    nb = np.array([len(f) for f in features])[view[ib[wrong]]]
    mj[wrong] = (rng.uniform(0, 1, int(wrong.sum())) * nb).astype(np.int64)
    pairs = [(a, b) for a in range(V) for b in range(a + 1, min(a + int(span), V - 1) + 1)]
    lo = np.searchsorted(key, [a * V + b for a, b in pairs])
    hi = np.searchsorted(key, [a * V + b for a, b in pairs], side="right")
    matches = [np.column_stack([local[ia[s:e]], mj[s:e]]).astype(np.int32) for s, e in zip(lo, hi)]
    return MatchGraph(K=K, R=R, t=t, X=X, features=features, point=point,
                      pairs=np.array(pairs, dtype=np.int32).reshape(-1, 2), matches=matches,
                      wrong=[wrong[s:e] for s, e in zip(lo, hi)])
