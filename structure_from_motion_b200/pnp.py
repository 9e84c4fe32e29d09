"""Absolute pose of a new view (PnP) on arrays: RANSAC over 2-D-3-D correspondences, numpy in, numpy out.

Registers a further image against triangulated points: given world points X (for points from ``two_view_arrays`` the
frame of camera 1, with the baseline |t| = 1) and their pixels x in the new image, find [R | t] with x_cam = R X + t.
K must be upper triangular with K[2,2] = 1.  The error is the squared reprojection error in px^2, F / p2^2 with
p = K [R | t] (X, 1) and F = (p0 - u p2)^2 + (p1 - v p2)^2, and a record is an inlier iff p2 >= 2^-537, F < inf and
F <= thr p2^2 (division-free; csrc/sfm_pnp.cuh pins the evaluation order).  The minimal solver is P3P (Lambda Twist) on the first
three points of a sample, the fourth choosing among its solutions.  The RANSAC loop is the reference's
``fit_with_ransac(data, 4, ...)`` (lib/ransac/ransac.py:19-93) as ``ransac_homography_arrays`` applies it.  Everything
numeric runs in libsfm_b200.so; there is no CPU fallback.
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import numpy as np

from . import _native
from .two_view import _agg_name, _inlier_order, _load_samples, _replay_near_ties, _restore_random_state

_SAMPLE = 4  # points per minimal sample


@dataclasses.dataclass
class PnpRefinement:
    R: np.ndarray                 # (3,3) refined rotation (the start pose's R when not refined)
    t: np.ndarray                 # (3,)
    cost_ransac: float            # the start pose's summed squared reprojection error over the list (px^2)
    cost_start: float             # the same at the start point (R projected onto the rotations)
    cost_final: float             # at the reported pose, <= cost_start
    num: int                      # records in the list
    iterations: int               # proposals evaluated
    status: str                   # converged, max_iterations, stalled or nonfinite
    rejected: int                 # of those, proposals rejected
    mask: np.ndarray              # bool[n]: inlier decision under the reported pose (no forced samples)
    err: np.ndarray               # float64[n]: squared reprojection error under the reported pose (px^2)


def _refinement(rep, mask, err) -> PnpRefinement:
    Rt = np.array(rep.Rt[:], dtype=np.float64).reshape(3, 4)
    return PnpRefinement(R=Rt[:, :3].copy(), t=Rt[:, 3].copy(), cost_ransac=float(rep.cost_ransac),
                         cost_start=float(rep.cost_start), cost_final=float(rep.cost_final), num=int(rep.num),
                         iterations=int(rep.iterations), status=_native.REFINE_STATUS[int(rep.status)],
                         rejected=int(rep.rejected), mask=mask, err=err)


@dataclasses.dataclass
class PnpResult:
    R: np.ndarray                 # (3,3) rotation, world -> camera
    t: np.ndarray                 # (3,) translation: x_cam = R X + t
    best_index: int               # winning iteration (global hypothesis index)
    error: float                  # aggregated error of the winner
    count_extra: int              # inliers beyond the 4 samples
    inlier_indices: np.ndarray    # int64; samples, then the rest in that iteration's permutation order (reference
                                  # sampler) or ascending (table / device sampler)
    mask: np.ndarray              # bool[n]: inlier decision under the winner
    err: np.ndarray               # float64[n]: squared reprojection error under the winner (px^2)
    sample: np.ndarray            # int32[4] the winner's minimal sample
    num_invalid: int              # degenerate samples (skipped)
    first_invalid: int            # earliest such iteration, -1 if none
    refinement: Optional[PnpRefinement] = None  # refine_iterations > 0: the winner refined over its inliers


def _camera(camera_matrix) -> np.ndarray:
    K = np.asarray(camera_matrix, dtype=np.float64)
    if K.shape != (3, 3):
        raise ValueError(f"Camera intrinsic matrix is not 3x3, actual shape: {K.shape}")
    return K


def _records(points_3d, pts):
    X = np.ascontiguousarray(points_3d, dtype=np.float64)
    x = np.ascontiguousarray(pts, dtype=np.float64)
    if X.ndim != 2 or X.shape[1] != 3 or x.ndim != 2 or x.shape[1] != 2 or X.shape[0] != x.shape[0]:
        raise ValueError(f"expected points_3d [n,3] and pts [n,2], got {X.shape} and {x.shape}")
    return X, x


def ransac_pnp_arrays(
    camera_matrix,
    points_3d,
    pts,
    threshold: float,
    min_num_extra_inliers=None,
    error_aggregation_method=None,
    max_iterations: Optional[int] = None,
    *,
    sampler: str = "reference",
    seed: int = 0,
    hyp_offset: int = 0,
    selection: str = "min_error",
    engine: Optional[_native.Engine] = None,
    table: Optional[np.ndarray] = None,
    refine_iterations: int = 0,
) -> PnpResult:
    """RANSAC absolute pose from world points [n,3] and their pixels [n,2] in the new view (n >= 8).

    sampler: "reference" — ``random.shuffle`` of the data list per iteration on the process-global state, sample =
             the first 4 entries; the state advances exactly as ``fit_with_ransac(data, 4, ...)`` would advance it;
             "device" — Philox sampler on the GPU (``seed``, ``hyp_offset`` for split runs); "table" — the given int
             table, [H,4] or [H,8] (columns 0-3 are the sample).
    threshold: on the squared reprojection error in px^2, finite.  Defaults: 100 iterations, RMS, 0 extra inliers.
    refine_iterations > 0: the final winner (after the near-tie replay) is refined over its inliers plus its sample by
             Levenberg-Marquardt on the reprojection error (``refine_pnp_arrays``) into ``refinement``; R, t and
             everything else stay the RANSAC result.  0 (the default) makes no refinement call.
    """
    refine_iterations = int(refine_iterations)
    if refine_iterations < 0:
        raise ValueError(f"refine_iterations must be >= 0, got {refine_iterations}")
    if max_iterations is None:
        max_iterations = 100  # ransac.py:48-49
    if min_num_extra_inliers is None:
        min_num_extra_inliers = 0  # ransac.py:52-53
    agg = _agg_name(error_aggregation_method)
    K = _camera(camera_matrix)
    X, x = _records(points_3d, pts)
    if not np.isfinite(threshold):
        raise ValueError(f"the threshold must be finite, got {threshold}")
    n = X.shape[0]
    H = int(max_iterations)

    def no_model():
        return ValueError(f"No model could be found with at least {min_num_extra_inliers + _SAMPLE} inliers.")

    if sampler not in ("reference", "device", "table"):
        raise ValueError(f"unknown sampler {sampler!r}")
    if H <= 0 and sampler != "table":
        raise no_model()  # ransac.py:88-91 (loop never ran)
    if n < 8:
        raise ValueError(f"RANSAC PnP needs at least 8 correspondences, got {n}")
    eng = engine or _native.get_engine()
    if sampler == "table":
        table = np.ascontiguousarray(table, dtype=np.int32)
        if table.ndim != 2 or table.shape[1] not in (_SAMPLE, 8) or table.shape[0] == 0:
            raise ValueError(f"expected a [H,4] or [H,8] sample table, got shape {table.shape}")
        if table.shape[1] == _SAMPLE:
            table = np.ascontiguousarray(np.concatenate([table, table], axis=1))  # columns 4-7 are never read
        H = table.shape[0]

    eng.upload_pnp(X, x, K)
    table, ref = _load_samples(eng, sampler, n, H, table, seed, hyp_offset)
    best, Rt, mask, err, _, _ = eng.ransac_pnp(threshold, float(min_num_extra_inliers), agg, selection)
    _restore_random_state(ref)  # no exception aborts the loop: every shuffle happened
    if best.index < 0:
        raise no_model()

    def score(t):
        Rt_t, _ = eng.get_pnp_models(t, 1)
        return eng.pnp_mask(Rt_t[0], threshold)

    # near-ties are settled in the reference's list order and summation (SURVEY.md H1), as on the E and H paths
    t, e = _replay_near_ties(eng, sampler, selection, table, ref, n, _SAMPLE, threshold, agg, score) or (None, None)
    if t is not None and t != int(best.index):
        Rt_t, _ = eng.get_pnp_models(t, 1)
        best.index = t
        Rt = Rt_t[0]
        mask, err = score(t)
        best.count_extra = int(mask.sum() - mask[table[t][:_SAMPLE]].sum())
        best.err = e

    mask = np.asarray(mask).astype(bool)
    sample, inliers = _inlier_order(best, sampler, table, ref, mask, _SAMPLE)
    Rt = np.array(Rt, dtype=np.float64).reshape(3, 4)
    refinement = None
    if refine_iterations > 0:  # the winner as settled above, with its own sample: the reference's tie rule holds
        refinement = _refinement(*eng.refine_pnp(threshold, refine_iterations, Rt=Rt, sample=sample))
    return PnpResult(
        R=Rt[:, :3].copy(),
        t=Rt[:, 3].copy(),
        best_index=int(best.index) + (hyp_offset if sampler == "device" else 0),
        error=float(best.err),
        count_extra=int(best.count_extra),
        inlier_indices=inliers,
        mask=mask,
        err=err,
        sample=sample,
        num_invalid=int(best.num_invalid),
        first_invalid=int(best.first_invalid),
        refinement=refinement,
    )


def fit_pnp_arrays(camera_matrix, points_3d, pts, engine: Optional[_native.Engine] = None):
    """The P3P pose (R, t) through 4 correspondences (points_3d [4,3], pts [4,2]): the solution of the first three
    with positive depths whose reprojection error at the fourth is smallest.  Raises ValueError on an invalid sample
    (a non-finite coordinate, collinear world points, no solution with positive depths)."""
    K = _camera(camera_matrix)
    X, x = _records(points_3d, pts)
    if X.shape[0] != _SAMPLE:
        raise ValueError("Exactly four correspondences are needed")
    eng = engine or _native.get_engine()
    eng.upload_pnp(X, x, K)
    eng.set_table(np.array([[0, 1, 2, 3, 0, 1, 2, 3]], dtype=np.int32))
    Rt, valid = eng.fit_pnp()
    if not valid[0]:
        raise ValueError("Degenerate sample: no P3P pose with positive depths through these points")
    return Rt[0][:, :3].copy(), Rt[0][:, 3].copy()


def reprojection_error_arrays(R, t, camera_matrix, points_3d, pts, threshold: float = np.inf,
                              engine: Optional[_native.Engine] = None):
    """(inlier decision bool[n], squared reprojection error float64[n] in px^2) of every record under [R | t]."""
    K = _camera(camera_matrix)
    X, x = _records(points_3d, pts)
    Rt = np.concatenate([np.asarray(R, dtype=np.float64).reshape(3, 3),
                         np.asarray(t, dtype=np.float64).reshape(3, 1)], axis=1)
    eng = engine or _native.get_engine()
    eng.upload_pnp(X, x, K)
    return eng.pnp_mask(Rt, threshold)


def refine_pnp_arrays(R, t, camera_matrix, points_3d, pts, threshold: float, max_iterations: int = 20, sample=None,
                      engine: Optional[_native.Engine] = None) -> PnpRefinement:
    """Refine a caller's pose [R | t] over its inlier list by Levenberg-Marquardt on the squared reprojection error.

    The list is the records whose decision passes under [R | t] at ``threshold`` (px^2), plus the optional forced
    indices ``sample`` (4 ints), in ascending order; it stays fixed while the refinement runs.  The start is the
    rotation nearest to R (a reflection is projected onto a rotation) and t.  A start under which a list record lies
    behind the camera, or with a non-finite entry, reports ``nonfinite`` and keeps the pose."""
    K = _camera(camera_matrix)
    X, x = _records(points_3d, pts)
    if not np.isfinite(threshold):
        raise ValueError(f"the threshold must be finite, got {threshold}")
    if int(max_iterations) < 1:
        raise ValueError(f"max_iterations must be >= 1, got {max_iterations}")
    Rt = np.concatenate([np.asarray(R, dtype=np.float64).reshape(3, 3),
                         np.asarray(t, dtype=np.float64).reshape(3, 1)], axis=1)
    eng = engine or _native.get_engine()
    eng.upload_pnp(X, x, K)
    return _refinement(*eng.refine_pnp(threshold, int(max_iterations), Rt=Rt, sample=sample))
