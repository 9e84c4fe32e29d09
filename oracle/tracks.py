"""TEST INFRASTRUCTURE ONLY — restatement of the multi-view track triangulation (csrc/sfm_tracks.cuh).

- ``pair_table`` / ``pair_search``: the pair search in numpy float64 (SVD DLT of each pair), the decisions and values
  from ``creproj.reproj_exact_many`` (the device's pinned evaluation), and a flag on every (pair, observation) whose
  value lies within ``band`` relative of the threshold (where a DLT that differs in the last bits may decide otherwise).
- ``dlt_exact``: the N-view DLT at 50 digits (mpmath): the null vector of A^T A for the rows of dlt_triangulate.
- ``refine_replay``: the refinement replayed with scipy's MINPACK Levenberg-Marquardt from the same start on the same
  list; the cost is the sum of squared residuals p0 / p2 - u, p1 / p2 - v (not scipy's half of it).
- ``ray_angle``: the largest angle between the lines of sight from the camera centres -R^T t to X over pairs of
  observations.
- ``frame_exponent`` / ``in_frame``: the call's frame - P's fourth column scaled by 2^-s, s the binary exponent of the
  largest |t| entry - in which the device solves every DLT (the algebraic minimum depends on the frame).
"""
from __future__ import annotations

import mpmath
import numpy as np
from scipy.optimize import least_squares

from . import creproj

DPS = 50


def frame_exponent(Rt):
    """s: the binary exponent of the largest |t| entry over all views (0 when every t is 0)."""
    big = float(np.max(np.abs(np.asarray(Rt, dtype=np.float64)[..., 3])))
    return int(np.frexp(big)[1]) - 1 if big > 0 else 0


def in_frame(P, s):
    """P (3x4) with its fourth column scaled by 2^-s (exact)."""
    P = np.array(P, dtype=np.float64).reshape(3, 4)
    P[:, 3] = np.ldexp(P[:, 3], -s)
    return P


def dlt_rows(P, u, v):
    """The two rows dlt_triangulate forms for one observation: v P[2,:] - P[1,:] and P[0,:] - u P[2,:]."""
    P = np.asarray(P, dtype=np.float64).reshape(3, 4)
    return np.stack([v * P[2] - P[1], P[0] - u * P[2]])


def dlt_svd(Ps, xs):
    """float64 N-view DLT by SVD: Ps [n,3,4], xs [n,2] -> X[3]."""
    A = np.concatenate([dlt_rows(P, u, v) for P, (u, v) in zip(Ps, xs)])
    Xh = np.linalg.svd(A)[2][-1]
    return Xh[:3] / Xh[3]


def pair_table(K, Rt, view, x, thr, band=1e-6, frame=0):
    """One track: for every pair (i < j) in lexicographic order, (i, j, X[3], cand, count, sum, mask bool[n], flagged).

    K [V,3,3], Rt [V,3,4]; view int[n], x [n,2] the track's observations; each pair's DLT is solved in the frame
    ``frame`` (``in_frame``).  flagged: some observation's value under the pair's point lies within ``band`` relative of
    thr."""
    n = len(view)
    Ps = [in_frame(creproj.projection(K[c], Rt[c]), frame) for c in view]
    pairs = [(i, j) for i in range(n) for j in range(i + 1, n)]
    if not pairs:
        return []
    Xs = np.ldexp(np.array([dlt_svd([Ps[i], Ps[j]], [x[i], x[j]]) for i, j in pairs]), frame)
    masks = np.empty((len(pairs), n), dtype=bool)
    vals = np.empty((len(pairs), n))
    for o in range(n):
        m, val = creproj.reproj_exact_many(Rt[view[o]], K[view[o]], Xs, np.tile(x[o], (len(pairs), 1)), thr)
        masks[:, o], vals[:, o] = m, val
    out = []
    for k, (i, j) in enumerate(pairs):
        s = 0.0
        for o in range(n):  # in observation order, as the device sums
            if masks[k, o]:
                s += vals[k, o]
        flagged = bool(np.any(np.abs(vals[k] - thr) <= band * abs(thr)))
        out.append((i, j, Xs[k], bool(masks[k, i] and masks[k, j]), int(masks[k].sum()), s, masks[k].copy(), flagged))
    return out


def pair_search(table):
    """The winner of a pair table: the candidate with the most passing observations, then the smallest sum, then the
    lowest pair index.  Returns its index into the table, or -1 without a candidate."""
    best = -1
    for k, (_, _, _, cand, count, s, _, _) in enumerate(table):
        if cand and (best < 0 or count > table[best][4] or (count == table[best][4] and s < table[best][5])):
            best = k
    return best


def dlt_exact(Ps, xs, dps=DPS):
    """N-view DLT at ``dps`` digits: Ps [n] of 3x4 (float64 or mpf entries), xs [n] of (u, v).  Returns mpf X[3]."""
    with mpmath.workdps(dps):
        rows = []
        for P, (u, v) in zip(Ps, xs):
            P = [[mpmath.mpf(P[r][c]) for c in range(4)] for r in range(3)]
            u, v = mpmath.mpf(u), mpmath.mpf(v)
            rows.append([v * P[2][c] - P[1][c] for c in range(4)])
            rows.append([P[0][c] - u * P[2][c] for c in range(4)])
        A = mpmath.matrix(rows)
        E, Q = mpmath.eigsy(A.T * A)
        k = min(range(4), key=lambda i: E[i])
        return [Q[r, k] / Q[3, k] for r in range(3)]


def residuals(X, Ps, xs):
    out = []
    for P, (u, v) in zip(Ps, xs):
        p = P[:, :3] @ X + P[:, 3]
        out += [p[0] / p[2] - u, p[1] / p[2] - v]
    return np.array(out)


def jacobian(X, Ps, xs):
    J = []
    for P in Ps:
        p = P[:, :3] @ X + P[:, 3]
        J.append((P[0, :3] - p[0] / p[2] * P[2, :3]) / p[2])
        J.append((P[1, :3] - p[1] / p[2] * P[2, :3]) / p[2])
    return np.array(J)


def cost(X, Ps, xs):
    r = residuals(np.asarray(X, dtype=np.float64), Ps, xs)
    return float(r @ r)


def refine_replay(X0, Ps, xs):
    """MINPACK LM from X0 over the list (Ps [n] 3x4 float64, xs [n,2]).  Returns (X, cost)."""
    Ps = [np.asarray(P, dtype=np.float64).reshape(3, 4) for P in Ps]
    res = least_squares(residuals, np.asarray(X0, dtype=np.float64), jac=jacobian, args=(Ps, xs), method="lm",
                        xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=2000)
    return res.x, cost(res.x, Ps, xs)


def ray_angle(X, Rt, views):
    """Largest atan2(|a x b|, |a . b|) over pairs of the rays X - C_c, C_c = -R_c^T t_c, for c in views."""
    Rt = np.asarray(Rt, dtype=np.float64)
    rays = [np.asarray(X) + Rt[c][:, :3].T @ Rt[c][:, 3] for c in views]
    best = 0.0
    for i in range(len(rays)):
        for j in range(i + 1, len(rays)):
            best = max(best, float(np.arctan2(np.linalg.norm(np.cross(rays[i], rays[j])), abs(rays[i] @ rays[j]))))
    return best
