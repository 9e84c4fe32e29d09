"""TEST INFRASTRUCTURE ONLY — numpy restatement of the homography pose tail (no reference counterpart).

H (pixel coordinates, image A -> image B) -> Hn = K^-1 H K scaled to sigma_2 = 1 with det(Hn) > 0 -> the four
(R, t, n, d) candidates of the SVD construction of Ma, Soatto, Kosecka & Sastry, "An Invitation to 3-D Vision",
Algorithm 5.2 -> cheirality vote of the RANSAC inliers (oracle.restatement.cheirality_check on K^-1 x, every passing
inlier counts) -> DLT triangulation of the inliers that pass the voted candidate, in pixel coordinates.  All three
steps use the same camera K, which must be upper triangular with K[2,2] = 1 (the library refuses any other).  A pair
whose sigma_1 - sigma_3 is below the rotation tolerance is rotation-only: R is the rotation nearest to Hn, t = 0, no
vote.

Never imported by the product path.
"""
from __future__ import annotations

import numpy as np

from oracle.restatement import DEFAULT_DISTANCE_THRESHOLD, cheirality_check, triangulate_one

ROTATION_TOLERANCE = 1e-2


def normalised_homography(H, K):
    """Hn = K^-1 H K / sigma_2, negated when its determinant is negative."""
    K = np.asarray(K, dtype=np.float64).reshape(3, 3)
    Hn = np.linalg.inv(K) @ np.asarray(H, dtype=np.float64).reshape(3, 3) @ K
    s = np.linalg.svd(Hn, compute_uv=False)
    Hn = Hn / s[1]
    if np.linalg.det(Hn) < 0:
        Hn = -Hn
    return Hn


def decompose_homography(H, K, rotation_tolerance=ROTATION_TOLERANCE):
    """dict(candidates=[(R, t, n, d)], sv, rotation_only); sv = the singular values of Hn (sv[1] == 1).

    Four candidates (R+, T+, N+), (R+, -T+, -N+), (R-, T-, N-), (R-, -T-, -N-) with t = T / |T| (unit), n = N (unit),
    d = 1 / |T|: the plane n^T X = d in camera-1 coordinates, in units of the baseline.  Rotation-only
    (sigma_1 - sigma_3 < rotation_tolerance): one candidate (nearest rotation, t = 0, n = NaN, d = inf)."""
    Hn = normalised_homography(H, K)
    U, s, Vt = np.linalg.svd(Hn)
    if not (s[0] - s[2] >= rotation_tolerance) or not s[0] > s[2]:
        R = U @ np.diag([1.0, 1.0, np.linalg.det(U @ Vt)]) @ Vt
        return dict(candidates=[(R, np.zeros(3), np.full(3, np.nan), np.inf)], sv=s, rotation_only=True)
    v1, v2, v3 = Vt[0], Vt[1], Vt[2]  # eigenvectors of Hn^T Hn, eigenvalues s^2 descending
    s1, s3 = s[0] ** 2, s[2] ** 2
    a, b = np.sqrt(max(1.0 - s3, 0.0)), np.sqrt(max(s1 - 1.0, 0.0))
    cands = []
    for sign in (1.0, -1.0):
        u = (a * v1 + sign * b * v3) / np.sqrt(s1 - s3)
        Um = np.column_stack([v2, u, np.cross(v2, u)])
        Wm = np.column_stack([Hn @ v2, Hn @ u, np.cross(Hn @ v2, Hn @ u)])
        R = Wm @ Um.T
        N = np.cross(v2, u)
        T = (Hn - R) @ N
        nt = np.linalg.norm(T)
        cands.append((R, T / nt, N, 1.0 / nt))
        cands.append((R, -T / nt, -N, 1.0 / nt))
    return dict(candidates=cands, sv=s, rotation_only=False)


def k_inverse(x, y, K):
    """K^-1 (x, y, 1) of an upper-triangular K with K[2,2] = 1, in the kernel's order: yn = (y - cy) / fy, then
    xn = (x - cx - s yn) / fx with the skew s = K[0,1].  With s = 0 this is k_normalise, bit for bit."""
    K = np.asarray(K, dtype=np.float64).reshape(3, 3)
    fx, s, cx, fy, cy = K[0, 0], K[0, 1], K[0, 2], K[1, 1], K[1, 2]
    yn = (np.asarray(y, dtype=np.float64) - cy) / fy
    return ((np.asarray(x, dtype=np.float64) - cx) - s * yn) / fx, yn


def vote(candidates, K, xa, ya, xb, yb, distance_threshold=None):
    """(pass bits uint8[m], counts[4], best) of the inliers (pixel coordinates) under the candidates: bit p = inlier
    passes candidate p (oracle.restatement.cheirality_check on the rays K^-1 x, k_inverse); every passing inlier
    counts; best = first maximum."""
    if distance_threshold is None:
        distance_threshold = DEFAULT_DISTANCE_THRESHOLD
    nxa, nya = k_inverse(xa, ya, K)
    nxb, nyb = k_inverse(xb, yb, K)
    bits = np.zeros(len(nxa), dtype=np.uint8)
    for p, (R, t, _, _) in enumerate(candidates):
        for i in range(len(nxa)):
            if cheirality_check(nxa[i], nya[i], nxb[i], nyb[i], R, t, distance_threshold):
                bits[i] |= 1 << p
    counts = np.array([int(np.count_nonzero((bits >> p) & 1)) for p in range(len(candidates))], dtype=np.int64)
    return bits, counts, int(np.argmax(counts))


def triangulate(K, R, t, xa, ya, xb, yb, passing):
    """DLT in pixel coordinates with P1 = K[I|0], P2 = K[R|t] of the passing inliers; NaN rows elsewhere."""
    K = np.asarray(K, dtype=np.float64)
    P1 = np.hstack([K, np.zeros((3, 1))])
    P2 = K @ np.hstack([R, np.asarray(t, dtype=np.float64).reshape(3, 1)])
    X = np.full((len(xa), 3), np.nan)
    for i in np.flatnonzero(passing):
        X[i] = triangulate_one(xa[i], ya[i], xb[i], yb[i], P1, P2)
    return X
