"""TEST INFRASTRUCTURE ONLY — numpy restatement of the homography model (no reference counterpart).

The RANSAC loop is the one of oracle/restatement.py's ransac_essential — fit_with_ransac (lib/ransac/ransac.py:19-93)
at model_fit_data_count = 4 — with the exact 4-point homography fit and the symmetric transfer error.  Decisions and
values come from oracle/transfer_exact.c, which evaluates the device kernels' pinned order.

Never imported by the product path.
"""
from __future__ import annotations

import random
from math import inf

import numpy as np

from oracle import ctransfer
from oracle.restatement import AGG_RMS, aggregate_error, hartley_normalise

# --------------------------------------------------------------------------------------
# Homography  (no reference counterpart: the model of structure_from_motion_b200/homography.py,
# with fit_with_ransac's loop, ransac.py:19-93, at model_fit_data_count = 4)
# --------------------------------------------------------------------------------------
COLLINEAR = 1e-8  # |2 x triangle area| in Hartley-normalised coordinates (csrc/sfm_homography.cuh kCollinear)


def _collinear(normalised):
    for o in range(4):
        i, j, k = [q for q in range(4) if q != o]
        a = normalised[j] - normalised[i]
        b = normalised[k] - normalised[i]
        if not abs(a[0] * b[1] - a[1] * b[0]) > COLLINEAR:
            return True
    return False


def homography_4pt(a, b):
    """Exact homography through 4 correspondences ([4,2] pixel arrays): Hartley normalisation of each image, the 8x9
    DLT, its null vector from numpy.linalg.svd, denormalised and divided by H[2,2].  Returns (H, valid); valid is False
    when three points are collinear in either image or H[2,2] is 0 / not finite."""
    a = np.asarray(a, dtype=np.float64).reshape(4, 2)
    b = np.asarray(b, dtype=np.float64).reshape(4, 2)
    with np.errstate(all="ignore"):
        na, Ta = hartley_normalise(a)
        nb, Tb = hartley_normalise(b)
        ok = not (_collinear(na) or _collinear(nb))
        A = np.zeros((8, 9))
        for k in range(4):
            x, y = na[k]
            u, v = nb[k]
            A[2 * k] = [-x, -y, -1.0, 0.0, 0.0, 0.0, u * x, u * y, u]
            A[2 * k + 1] = [0.0, 0.0, 0.0, -x, -y, -1.0, v * x, v * y, v]
        if not np.all(np.isfinite(A)):
            return np.full((3, 3), np.nan), False
        _, _, vh = np.linalg.svd(A)
        H = np.linalg.inv(Tb) @ vh[-1].reshape(3, 3) @ Ta
        h22 = H[2, 2]
        ok = ok and h22 != 0.0 and np.isfinite(h22)
        H = H / h22
    return H, bool(ok and np.all(np.isfinite(H)))


def transfer_error_vectorised(H, xa, ya, xb, yb):
    """Symmetric transfer error |x_b - pi(H x_a)|^2 + |x_a - pi(adj(H) x_b)|^2 (px^2) for arrays and one H, numpy's
    own rounding (the device order is pinned in oracle/transfer_exact.c: use ctransfer.transfer_exact_many when bits matter)."""
    H = np.asarray(H, dtype=np.float64).reshape(3, 3)
    adj = np.array([np.cross(H[1], H[2]), np.cross(H[2], H[0]), np.cross(H[0], H[1])]).T  # cofactors, transposed
    pa = np.stack([xa, ya, np.ones_like(xa)])
    pb = np.stack([xb, yb, np.ones_like(xb)])
    p = H @ pa
    q = adj @ pb
    return (xb - p[0] / p[2]) ** 2 + (yb - p[1] / p[2]) ** 2 + (xa - q[0] / q[2]) ** 2 + (ya - q[1] / q[2]) ** 2


def ransac_homography(xa, ya, xb, yb, threshold, min_num_extra_inliers=None, method=None, max_iterations=None,
                      table=None, return_all=False, models=None):
    """The loop of ransac_essential with 4-point samples and the homography model: own sampling (cumulative
    random.shuffle of the data list, sample = first 4, inliers in permutation order) when table is None, else the
    given table (columns 0-3; inliers ascending).  Degenerate samples are skipped and counted.  Decisions and values
    come from the C scorer in the pinned order (ctransfer.transfer_exact_many).  models = (H[h,3,3], valid[h]): take these
    per-iteration models instead of fitting — the selection on given models, for data whose errors are at the rounding
    level of the fit (noise-free scenes, thresholds <= 0), where two correct solvers pick different winners."""
    if max_iterations is None:
        max_iterations = 100 if table is None else len(table)
    if method is None:
        method = AGG_RMS
    if min_num_extra_inliers is None:
        min_num_extra_inliers = 0
    xa, ya, xb, yb = (np.asarray(v, dtype=np.float64) for v in (xa, ya, xb, yb))
    n = len(xa)
    own_sampling = table is None
    perm = list(range(n))
    best = dict(best_index=-1, H=None, error=inf, inlier_indices=None, num_invalid=0, first_invalid=-1)
    if return_all:
        all_H = np.full((max_iterations, 3, 3), np.nan)
        all_valid = np.zeros(max_iterations, dtype=bool)
        all_count = np.full(max_iterations, -1, dtype=np.int64)
        all_err = np.full(max_iterations, inf)
    for it in range(max_iterations):
        if own_sampling:
            random.shuffle(perm)  # ransac.py:62
            sample = np.asarray(perm[:4], dtype=np.int64)
        else:
            sample = np.asarray(table[it][:4], dtype=np.int64)
        if models is None:
            H, ok = homography_4pt(np.stack([xa[sample], ya[sample]], 1), np.stack([xb[sample], yb[sample]], 1))
        else:
            H, ok = models[0][it], bool(models[1][it])
        if not ok:
            if best["num_invalid"] == 0:
                best["first_invalid"] = it
            best["num_invalid"] += 1
            continue
        inl, val = ctransfer.transfer_exact_many(H, xa, ya, xb, yb, threshold)
        is_sample = np.zeros(n, dtype=bool)
        is_sample[sample] = True
        extra_mask = inl & ~is_sample
        count_extra = int(extra_mask.sum())
        if return_all:
            all_H[it], all_valid[it], all_count[it] = H, True, count_extra
        if min_num_extra_inliers <= count_extra:
            if own_sampling:
                rest = np.asarray(perm[4:], dtype=np.int64)
                extra = rest[extra_mask[rest]]
            else:
                extra = np.nonzero(extra_mask)[0]
            inliers = np.concatenate([sample, extra])
            err = aggregate_error([float(v) for v in val[inliers]], method)
            if return_all:
                all_err[it] = err
            if err < best["error"]:
                best.update(best_index=it, H=H, error=err, inlier_indices=inliers)
    if best["H"] is None:
        raise ValueError(f"No model could be found with at least {min_num_extra_inliers + 4} inliers.")
    if return_all:
        best.update(all_H=all_H, all_valid=all_valid, all_count=all_count, all_err=all_err)
    return best


def expected_selection(models, valid, xa, ya, xb, yb, threshold, table, aggregation, selection, min_extra=0.0):
    """What the GPU estimate must report for the given per-hypothesis models (H[h,3,3], valid[h]) and table: dict of
    count_extra[h], S1[h], S2[h] (ctransfer.transfer_score_batch: samples never counted, always summed), err[h] (the
    aggregated error, the MSAC cost sum_i min(value_i, thr) for selection "msac", inf for a non-candidate) and
    winners: every index whose err (or count for "max_inliers") is the best one or within 1e-12 of it."""
    valid = np.asarray(valid, dtype=bool)
    cnt, s1, s2 = ctransfer.transfer_score_batch(models, xa, ya, xb, yb, threshold, table, valid.astype(np.uint8),
                                                 nthreads=8)
    n4 = 4.0 + cnt
    with np.errstate(all="ignore"):
        err = {"sum": s1, "square": s2, "mean": s1 / n4, "rms": np.sqrt(s2 / n4)}[aggregation].copy()
    if selection == "msac":
        for i in np.flatnonzero(valid):
            m, v = ctransfer.transfer_exact_many(models[i], xa, ya, xb, yb, threshold)
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
        if not len(winners):  # an infinite minimum
            winners = np.flatnonzero(cand & (err == best))
    return dict(count_extra=cnt, S1=s1, S2=s2, err=err, winners=winners)
