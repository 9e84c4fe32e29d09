"""TEST INFRASTRUCTURE ONLY — numpy / mpmath restatement of the absolute-pose (PnP) model (no reference counterpart).

* ``reproj``: the reprojection error and decision of csrc/sfm_pnp.cuh in plain numpy (oracle/reproj_exact.c evaluates
  the device's pinned order bit for bit; this restatement is the readable one the C is checked against).
* ``p3p_exact``: an independent exact P3P - Grunert's distance system, reduced to a quartic by elimination and solved
  with mpmath at 50 digits - so that the device's Lambda Twist is never compared with itself.
* ``select_fourth``: the 4-point rule (positive depths at the three points, smallest reprojection error at the fourth,
  the first on a tie).
* ``ransac_pnp``: fit_with_ransac (lib/ransac/ransac.py:19-93) at model_fit_data_count = 4, as
  oracle/homography.ransac_homography applies it.

Never imported by the product path.
"""
from __future__ import annotations

import random
from math import inf

import mpmath
import numpy as np

from oracle import creproj
from oracle.restatement import AGG_RMS, aggregate_error

COLLINEAR = 1e-6  # csrc/sfm_pnp.cuh kPnpCollinear: sine of the angle at X0
MIN_DEPTH = 2.0 ** -537  # csrc/sfm_pnp.cuh kPnpMinDepthHi: the smallest p2 of an inlier (its square is not 0)
_DPS = 50


def reproj(Rt, K, X, x, thr):
    """(decision bool[n], value [n]) of every record: p = K [R|t] (X, 1), F = (p0 - u p2)^2 + (p1 - v p2)^2,
    inlier iff p2 >= 2^-537 (W = p2^2 > 0), F < inf and F <= thr p2^2, value F / p2^2."""
    Rt = np.asarray(Rt, dtype=np.float64).reshape(3, 4)
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    P = np.asarray(K, dtype=np.float64).reshape(3, 3) @ Rt
    p = X @ P[:, :3].T + P[:, 3]
    with np.errstate(all="ignore"):
        d0 = p[:, 0] - x[:, 0] * p[:, 2]
        d1 = p[:, 1] - x[:, 1] * p[:, 2]
        F = d0 * d0 + d1 * d1
        W = p[:, 2] * p[:, 2]
        return (p[:, 2] >= MIN_DEPTH) & (F < inf) & (F <= thr * W), F / W


def bearings(K, x):
    """Unit bearings of pixels through K^-1 in the order of the device (y first, then x minus the skew's share)."""
    K = np.asarray(K, dtype=np.float64)
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    with np.errstate(all="ignore"):
        yn = (x[:, 1] - K[1, 2]) / K[1, 1]
        xn = ((x[:, 0] - K[0, 2]) - K[0, 1] * yn) / K[0, 0]
        b = np.stack([xn, yn, np.ones_like(xn)], axis=1)
        nrm = np.linalg.norm(b, axis=1, keepdims=True)
        # np.linalg.norm squares: beyond ~1e154 it overflows, so such rows are divided by their largest entry first
        big = ~np.isfinite(nrm[:, 0]) & np.isfinite(b).all(axis=1)
        b[big] /= np.abs(b[big]).max(axis=1, keepdims=True)
        nrm[big] = np.linalg.norm(b[big], axis=1, keepdims=True)
        return b / nrm


def collinear_ratio(X3):
    """|w1 x w2| / (|w1| |w2|) with w1 = X0 - X1, w2 = X0 - X2: the sine the collinearity test compares with
    COLLINEAR (NaN for coincident points)."""
    X3 = np.asarray(X3, dtype=np.float64)
    w1, w2 = X3[0] - X3[1], X3[0] - X3[2]
    with np.errstate(all="ignore"):
        return float(np.linalg.norm(np.cross(w1, w2)) / (np.linalg.norm(w1) * np.linalg.norm(w2)))


def _polymul(a, b):
    out = [mpmath.mpf(0)] * (len(a) + len(b) - 1)
    for i, u in enumerate(a):
        for j, v in enumerate(b):
            out[i + j] += u * v
    return out


def _polyadd(*ps):
    m = max(len(p) for p in ps)
    out = [mpmath.mpf(0)] * m
    for p in ps:
        for i, v in enumerate(p):
            out[i] += v
    return out


def _scale(p, s):
    return [s * v for v in p]


def p3p_exact(y, X):
    """Every real solution (R, t) with three positive depths of the unit bearings y[3,3] of world points X[3,3], at
    50 digits.  Grunert: with s1, s2 = u s1, s3 = v s1 the depths, cos_a = y1.y2, cos_b = y0.y2, cos_c = y0.y1 and
    a = |X1 - X2|, b = |X0 - X2|, c = |X0 - X1|:
        s1^2 (u^2 + v^2 - 2 u v cos_a) = a^2,  s1^2 (1 + v^2 - 2 v cos_b) = b^2,  s1^2 (1 + u^2 - 2 u cos_c) = c^2.
    Eliminating s1 leaves two conics in (u, v), both quadratic in u with the same u^2 coefficient; their difference is
    linear in u, u = N(v) / D(v), and substituting it into the second gives a quartic in v.  Polynomial coefficients
    are formed in mpmath and the quartic is solved with mpmath.polyroots.  Returns a list of (R [3,3], t [3]) as
    float64 (rounded from 50 digits) in no particular order."""
    with mpmath.workdps(_DPS):
        yv = [[mpmath.mpf(float(v)) for v in row] for row in np.asarray(y, dtype=np.float64)]
        Xv = [[mpmath.mpf(float(v)) for v in row] for row in np.asarray(X, dtype=np.float64)]
        dot = lambda p, q: sum(p[k] * q[k] for k in range(3))  # noqa: E731
        sub = lambda p, q: [p[k] - q[k] for k in range(3)]  # noqa: E731
        ca, cb, cc = dot(yv[1], yv[2]), dot(yv[0], yv[2]), dot(yv[0], yv[1])
        a2 = dot(sub(Xv[1], Xv[2]), sub(Xv[1], Xv[2]))
        b2 = dot(sub(Xv[0], Xv[2]), sub(Xv[0], Xv[2]))
        c2 = dot(sub(Xv[0], Xv[1]), sub(Xv[0], Xv[1]))
        one = mpmath.mpf(1)
        Q = [one, -2 * cb, one]  # 1 + v^2 - 2 v cos_b, ascending powers of v
        # (I)  b2 u^2 - 2 b2 cos_a v u + b2 v^2 - a2 Q = 0
        # (II) b2 u^2 - 2 b2 cos_c u + b2 - c2 Q = 0
        # (I) - (II): 2 b2 (cos_c - cos_a v) u + b2 v^2 - b2 - a2 Q + c2 Q = 0  =>  u = N / D
        N = _polyadd([-b2, 0, b2], _scale(Q, c2 - a2))
        N = _scale(N, -1)
        D = [2 * b2 * cc, -2 * b2 * ca]
        # (II) * D^2: b2 N^2 - 2 b2 cos_c N D + (b2 - c2 Q) D^2 = 0
        quart = _polyadd(_scale(_polymul(N, N), b2), _scale(_polymul(N, D), -2 * b2 * cc),
                         _polymul(_polyadd([b2], _scale(Q, -c2)), _polymul(D, D)))
        while len(quart) > 1 and quart[-1] == 0:
            quart.pop()
        coeffs = list(reversed(quart))  # descending for polyroots
        roots = mpmath.polyroots(coeffs, maxsteps=400, extraprec=200)
        out = []
        for r in roots:
            if abs(mpmath.im(r)) > mpmath.mpf(10) ** (-20) * (1 + abs(r)):
                continue
            v = mpmath.re(r)
            d = D[0] + D[1] * v
            if d == 0:
                continue
            u = (N[0] + N[1] * v + N[2] * v * v) / d
            den = 1 + u * u - 2 * u * cc
            if den <= 0:
                continue
            s1 = mpmath.sqrt(c2 / den)
            s = [s1, u * s1, v * s1]
            if not all(si > 0 for si in s):
                continue
            C = [[s[i] * yv[i][k] for k in range(3)] for i in range(3)]
            d1, d2 = sub(C[0], C[1]), sub(C[0], C[2])
            w1, w2 = sub(Xv[0], Xv[1]), sub(Xv[0], Xv[2])
            cr = lambda p, q: [p[1] * q[2] - p[2] * q[1], p[2] * q[0] - p[0] * q[2], p[0] * q[1] - p[1] * q[0]]  # noqa: E731
            Y = mpmath.matrix([[d1[k], d2[k], cr(d1, d2)[k]] for k in range(3)])
            W = mpmath.matrix([[w1[k], w2[k], cr(w1, w2)[k]] for k in range(3)])
            R = Y * mpmath.inverse(W)
            t = [C[0][k] - sum(R[k, j] * Xv[0][j] for j in range(3)) for k in range(3)]
            out.append((np.array([[float(R[i, j]) for j in range(3)] for i in range(3)]),
                        np.array([float(v) for v in t])))
        return out


def select_fourth(K, cands, X4, x4):
    """(index, errors) of the candidate with the smallest reprojection error of point 3 (value F / p2^2 in px^2),
    the first on a tie; NaN errors are never chosen.  index -1 when none qualifies."""
    errs = []
    best = -1
    for i, (R, t) in enumerate(cands):
        _, v = reproj(np.column_stack([R, t]), K, X4[None], x4[None], inf)
        e = float(v[0])
        errs.append(e)
        if e == e and (best < 0 or e < errs[best]):
            best = i
    return best, errs


def fit_pnp_exact(K, X, x):
    """The exact 4-point fit: (Rt [3,4] or None, info).  info: collinear = the sine of collinear_ratio, gap = the
    relative gap between the smallest and the second-smallest point-3 error (inf with fewer than two candidates),
    ncand = the number of candidates.  None when a coordinate is not finite, the world points are collinear
    (sine <= COLLINEAR) or no candidate remains."""
    X = np.asarray(X, dtype=np.float64).reshape(4, 3)
    x = np.asarray(x, dtype=np.float64).reshape(4, 2)
    # the sine and the solve are scale-free: they run on the world points scaled by a power of two (exact), so that
    # float64 norms and mpmath's singularity test see coordinates of order 1 at any world scale; t is scaled back
    with np.errstate(all="ignore"):
        spread = np.abs(X[:3, None, :] - X[None, :3, :]).max()
    e = int(np.frexp(spread)[1]) if np.isfinite(spread) and spread > 0 else 0
    Xs = np.ldexp(X[:3], -e)
    info = dict(collinear=collinear_ratio(Xs), gap=inf, ncand=0)
    if not (np.isfinite(X).all() and np.isfinite(x).all()):
        return None, info
    if not info["collinear"] > COLLINEAR:
        return None, info
    cands = [(R, np.ldexp(t, e)) for R, t in p3p_exact(bearings(K, x[:3]), Xs)]
    info["ncand"] = len(cands)
    best, errs = select_fourth(K, cands, X[3], x[3])
    if best < 0:
        return None, info
    fin = sorted(e for e in errs if e == e)
    if len(fin) >= 2:
        info["gap"] = (fin[1] - fin[0]) / max(fin[1], 1e-300)
    R, t = cands[best]
    Rt = np.column_stack([R, t])
    return (Rt if np.isfinite(Rt).all() else None), info


def ransac_pnp(K, X, x, threshold, min_num_extra_inliers=0, method=AGG_RMS, max_iterations=100, table=None,
               models=None):
    """fit_with_ransac(data, 4, ...) for PnP on the process-global random state (or a table [H,8]).  models =
    (Rt [H,3,4], valid [H]) replaces the fits (to test the loop against a device fit).  Decisions and values come
    from oracle/reproj_exact.c.  Returns dict(best_index, Rt, error, inlier_indices, num_invalid, first_invalid)."""
    X = np.asarray(X, dtype=np.float64)
    x = np.asarray(x, dtype=np.float64)
    n = X.shape[0]
    own_sampling = table is None
    perm = list(range(n))
    best = dict(best_index=-1, Rt=None, error=inf, inlier_indices=None, num_invalid=0, first_invalid=-1)
    for it in range(max_iterations):
        if own_sampling:
            random.shuffle(perm)  # ransac.py:62
            sample = np.asarray(perm[:4], dtype=np.int64)
        else:
            sample = np.asarray(table[it][:4], dtype=np.int64)
        if models is None:
            Rt, _ = fit_pnp_exact(K, X[sample], x[sample])
            ok = Rt is not None
        else:
            Rt, ok = models[0][it], bool(models[1][it])
        if not ok:
            if best["num_invalid"] == 0:
                best["first_invalid"] = it
            best["num_invalid"] += 1
            continue
        inl, val = creproj.reproj_exact_many(Rt, K, X, x, threshold)
        is_sample = np.zeros(n, dtype=bool)
        is_sample[sample] = True
        extra_mask = inl & ~is_sample
        count_extra = int(extra_mask.sum())
        if min_num_extra_inliers <= count_extra:
            if own_sampling:
                rest = np.asarray(perm[4:], dtype=np.int64)
                extra = rest[extra_mask[rest]]
            else:
                extra = np.nonzero(extra_mask)[0]
            inliers = np.concatenate([sample, extra])
            err = aggregate_error([float(v) for v in val[inliers]], method)
            if err < best["error"]:
                best.update(best_index=it, Rt=Rt, error=err, inlier_indices=inliers)
    if best["Rt"] is None:
        raise ValueError(f"No model could be found with at least {min_num_extra_inliers + 4} inliers.")
    return best


def expected_selection(models, valid, K, X, x, threshold, table, aggregation, selection, min_extra=0.0):
    """What the GPU estimate must report for the given poses (Rt [h,3,4], valid [h]) and table: dict of count_extra[h],
    S1[h], S2[h] (creproj.reproj_score_batch: samples never counted, always summed), err[h] (the aggregated error, the
    MSAC cost for selection "msac", inf for a non-candidate) and winners: every index whose err (or count for
    "max_inliers") is the best one or within 1e-12 of it.  The rule of oracle.homography.expected_selection."""
    valid = np.asarray(valid, dtype=bool)
    cnt, s1, s2 = creproj.reproj_score_batch(models, K, X, x, threshold, table, valid.astype(np.uint8), nthreads=8)
    n4 = 4.0 + cnt
    with np.errstate(all="ignore"):
        err = {"sum": s1, "square": s2, "mean": s1 / n4, "rms": np.sqrt(s2 / n4)}[aggregation].copy()
    if selection == "msac":
        for i in np.flatnonzero(valid):
            m, v = creproj.reproj_exact_many(models[i], K, X, x, threshold)
            err[i] = np.sum(np.where(m, v, threshold))
    cand = valid & (min_extra <= cnt) & ~np.isnan(err)
    err = np.where(cand, err, inf)
    if not cand.any():
        winners = np.array([-1])
    elif selection == "max_inliers":
        best = np.max(cnt[cand])
        winners = np.array([int(np.flatnonzero(cand & (cnt == best))[0])])
    else:
        best = np.min(err)
        winners = np.flatnonzero(cand & (np.abs(err - best) <= 1e-12 * np.abs(best)))
        if not len(winners):
            winners = np.flatnonzero(cand & (err == best))
    return dict(count_extra=cnt, S1=s1, S2=s2, err=err, winners=winners)


def cubic_branch(y, X):
    """1 or 3: the number of real roots cubic_roots (csrc/sfm_pnp.cuh) takes for the Lambda Twist cubic
    det(D1 + g D2) of unit bearings y[3,3] and world points X[3,3], restated in float64 (the sign of the depressed
    cubic's discriminant; a sample within rounding of disc = 0 may fall on either side on the device).  0 when the
    leading coefficient is 0 or a coefficient is not finite."""
    y = np.asarray(y, dtype=np.float64)
    X = np.asarray(X, dtype=np.float64)
    w1, w2, w12 = X[0] - X[1], X[0] - X[2], X[1] - X[2]
    a01, a02, a12 = w1 @ w1, w2 @ w2, w12 @ w12
    b01, b02, b12 = y[0] @ y[1], y[0] @ y[2], y[1] @ y[2]
    D1 = np.array([[a12, -a12 * b01, 0.0], [-a12 * b01, a12 - a01, a01 * b12], [0.0, a01 * b12, -a01]])
    D2 = np.array([[a12, 0.0, -a12 * b02], [0.0, -a02, a02 * b12], [-a12 * b02, a02 * b12, a12 - a02]])
    det = lambda a, b, c: float(np.dot(a, np.cross(b, c)))  # noqa: E731  (columns = rows: both are symmetric)
    A, B = D1, D2
    k3 = det(B[0], B[1], B[2])
    k2 = det(A[0], B[1], B[2]) + det(B[0], A[1], B[2]) + det(B[0], B[1], A[2])
    k1 = det(A[0], A[1], B[2]) + det(A[0], B[1], A[2]) + det(B[0], A[1], A[2])
    k0 = det(A[0], A[1], A[2])
    if not (k3 != 0 and np.isfinite([k3, k2, k1, k0]).all()):
        return 0
    p, q, r = k2 / k3, k1 / k3, k0 / k3
    P = q - p * p / 3.0
    Q = 2.0 * p * p * p / 27.0 - p * q / 3.0 + r
    return 1 if 0.25 * Q * Q + P * P * P / 27.0 > 0.0 else 3


def bearing_angles(y):
    """The smallest angle (radians) between two of the unit bearings y[3,3]: the conditioning of a P3P sample."""
    y = np.asarray(y, dtype=np.float64)
    ang = [np.arctan2(np.linalg.norm(np.cross(y[i], y[j])), y[i] @ y[j]) for i, j in ((0, 1), (0, 2), (1, 2))]
    return float(min(ang))
