"""TEST INFRASTRUCTURE ONLY — plain numpy restatement of the essential-matrix / homography choice.

ORB-SLAM's score ratio (Mur-Artal, Montiel & Tardos, 2015, section IV) with the E winner as the pixel fundamental
matrix F = Kd^-T E Kd^-1 (Kd: K without skew, bottom row (0, 0, 1)), written the way the formulas read, with no
attention to evaluation order.  oracle/select_exact.c is the bit-exact checker of the kernel; this file checks that one
against the formulas.
"""
from __future__ import annotations

import numpy as np

GAMMA, T_E, T_H = 5.99, 3.84, 5.99


def essential_camera(K):
    """Kd = [[fx, 0, cx], [0, fy, cy], [0, 0, 1]] of K: the camera of the E path, whose normalisation (x - cx) / fx,
    (y - cy) / fy ignores the skew and the bottom row of K."""
    K = np.asarray(K, dtype=np.float64).reshape(3, 3)
    return np.array([[K[0, 0], 0.0, K[0, 2]], [0.0, K[1, 1], K[1, 2]], [0.0, 0.0, 1.0]])


def fundamental(E, K):
    """F = Kd^-T E Kd^-1 with Kd = essential_camera(K)."""
    Ki = np.linalg.inv(essential_camera(K))
    return Ki.T @ np.asarray(E, dtype=np.float64) @ Ki


def essential_terms(E, K, pts_a, pts_b):
    """(d2_A, d2_B) in px^2: squared distances of a to the line F^T b and of b to the line F a (b^T E a = 0)."""
    F = fundamental(E, K)
    a = np.column_stack([pts_a, np.ones(len(pts_a))])
    b = np.column_stack([pts_b, np.ones(len(pts_b))])
    la = a @ F.T   # F a, one row per correspondence
    lb = b @ F     # F^T b
    r = np.sum(b * la, axis=1)
    with np.errstate(divide="ignore", invalid="ignore"):
        return r ** 2 / (lb[:, 0] ** 2 + lb[:, 1] ** 2), r ** 2 / (la[:, 0] ** 2 + la[:, 1] ** 2)


def homography_terms(H, pts_a, pts_b):
    """(d2_A, d2_B) in px^2: |a - pi(H^-1 b)|^2 and |b - pi(H a)|^2."""
    H = np.asarray(H, dtype=np.float64)
    a = np.column_stack([pts_a, np.ones(len(pts_a))])
    b = np.column_stack([pts_b, np.ones(len(pts_b))])
    p = a @ H.T
    q = b @ np.linalg.inv(H).T
    with np.errstate(divide="ignore", invalid="ignore"):
        db = np.sum((p[:, :2] / p[:, 2:] - pts_b) ** 2, axis=1)
        da = np.sum((q[:, :2] / q[:, 2:] - pts_a) ** 2, axis=1)
    return da, db


def rho(d2, sigma, T):
    x = np.asarray(d2) / sigma ** 2
    with np.errstate(invalid="ignore"):
        ok = x < T
    return np.where(ok, GAMMA - x, 0.0), ok


def score_models(K, pts_a, pts_b, E=None, H=None, sigma=1.0, ratio=0.45):
    """dict(per_point [n,4], score_e, score_h, count_e, count_h, ratio_h, model) with plain float sums."""
    pts_a = np.asarray(pts_a, dtype=np.float64).reshape(-1, 2)
    pts_b = np.asarray(pts_b, dtype=np.float64).reshape(-1, 2)
    n = len(pts_a)
    pp = np.full((n, 4), np.nan)
    out = dict(score_e=0.0, score_h=0.0, count_e=0, count_h=0)
    for key, M, terms, T, cols in (("e", E, lambda M: essential_terms(M, K, pts_a, pts_b), T_E, (0, 1)),
                                   ("h", H, lambda M: homography_terms(M, pts_a, pts_b), T_H, (2, 3))):
        if M is None:
            continue
        da, db = terms(M)
        ra, oka = rho(da, sigma, T)
        rb, okb = rho(db, sigma, T)
        pp[:, cols[0]], pp[:, cols[1]] = da, db
        out["score_" + key] = float(np.sum(ra) + np.sum(rb))
        out["count_" + key] = int(np.count_nonzero(oka & okb))
    tot = out["score_h"] + out["score_e"]
    out["ratio_h"] = out["score_h"] / tot if tot > 0 else 0.0
    out["model"] = 1 if E is None else (0 if H is None else int(out["ratio_h"] > ratio))
    out["per_point"] = pp
    return out
