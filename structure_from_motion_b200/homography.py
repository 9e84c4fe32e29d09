"""RANSAC homography estimation on arrays (numpy in, numpy out) — the model for planar scenes and rotation-only pairs,
where the essential matrix is not determined by the data (coplanar points) or vanishes (t = 0).

H maps image-A pixels to image-B pixels (x_b ~ H x_a) and is returned divided by H[2,2].  The error is the symmetric
transfer error in px^2, ``|x_b - pi(H x_a)|^2 + |x_a - pi(adj(H) x_b)|^2``, and a correspondence is an inlier iff the
division-free form of ``error <= threshold`` holds (csrc/sfm_homography.cuh pins the evaluation order).  The RANSAC
loop is the reference's ``fit_with_ransac(data, 4, ...)`` (lib/ransac/ransac.py:19-93): 4-point samples, never counted
as extra inliers and always part of the error, the same aggregation methods, defaults and strict-< selection as
``two_view.ransac_essential_arrays``.  A sample with three collinear points (in either image) is skipped and counted
in ``num_invalid`` / ``first_invalid``.  Everything numeric runs in libsfm_b200.so; there is no CPU fallback.

``two_view_homography_arrays`` continues from the winner to a camera pose and 3-D points, as ``two_view_arrays`` does
from E: the decomposition of K^-1 H K into four (R, t, n, d) candidates (csrc/sfm_hpose.cuh), the cheirality vote of
the winner's inliers and the triangulation of the inliers that pass the voted candidate.  t is a unit vector, the plane
is n^T X = d in camera-1 coordinates in units of the baseline.  A rotation-only pair (sigma_1 - sigma_3 of the
normalised homography below ``rotation_tolerance``) gets R, t = 0, no vote and no points.
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import numpy as np

from . import _native
from .errors import EightPointCalculationError
from .two_view import (Refinement, _agg_name, _inlier_order, _load_samples, _ransac_list, _refine_count, _refinement,
                       _replay_near_ties, _restore_random_state, _tail_inliers)

_SAMPLE = 4  # points per minimal sample


@dataclasses.dataclass
class HomographyResult:
    H: np.ndarray                 # (3,3), H[2,2] == 1, image A -> image B
    best_index: int               # winning iteration (global hypothesis index)
    error: float                  # aggregated error of the winner
    count_extra: int              # inliers beyond the 4 samples
    inlier_indices: np.ndarray    # int64; samples, then the rest in that iteration's permutation order (reference
                                  # sampler) or ascending (table / device sampler)
    mask: np.ndarray              # bool[n]: inlier decision under the winner
    err: np.ndarray               # float64[n]: transfer error under the winner (px^2)
    sample: np.ndarray            # int32[4] the winner's minimal sample
    num_invalid: int              # degenerate samples (skipped)
    first_invalid: int            # earliest such iteration, -1 if none


def ransac_homography_arrays(
    pts_a,
    pts_b,
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
) -> HomographyResult:
    """RANSAC homography from [n,2] arrays of matched pixel coordinates (n >= 8).

    sampler: "reference" — ``random.shuffle`` of the data list per iteration on the process-global state, sample =
             the first 4 entries; the state advances exactly as ``fit_with_ransac(data, 4, ...)`` would advance it;
             "device" — Philox sampler on the GPU (``seed``, ``hyp_offset`` for split runs); "table" — the given int
             table, [H,4] or [H,8] (columns 0-3 are the sample).
    threshold: on the symmetric transfer error in px^2.  Defaults: 100 iterations, RMS, 0 extra inliers.
    """
    if max_iterations is None:
        max_iterations = 100  # ransac.py:48-49
    if min_num_extra_inliers is None:
        min_num_extra_inliers = 0  # ransac.py:52-53
    agg = _agg_name(error_aggregation_method)
    pts_a = np.ascontiguousarray(pts_a, dtype=np.float64).reshape(-1, 2)
    pts_b = np.ascontiguousarray(pts_b, dtype=np.float64).reshape(-1, 2)
    if pts_a.shape != pts_b.shape:
        raise ValueError("pts_a and pts_b must have the same shape")
    n = pts_a.shape[0]
    H = int(max_iterations)

    def no_model():
        return ValueError(f"No model could be found with at least {min_num_extra_inliers + _SAMPLE} inliers.")

    if sampler not in ("reference", "device", "table"):
        raise ValueError(f"unknown sampler {sampler!r}")
    if H <= 0 and sampler != "table":
        raise no_model()  # ransac.py:88-91 (loop never ran)
    if n < 8:
        raise ValueError(f"RANSAC homography needs at least 8 correspondences, got {n}")
    eng = engine or _native.get_engine()
    if sampler == "table":
        table = np.ascontiguousarray(table, dtype=np.int32)
        if table.ndim != 2 or table.shape[1] not in (_SAMPLE, 8) or table.shape[0] == 0:
            raise ValueError(f"expected a [H,4] or [H,8] sample table, got shape {table.shape}")
        if table.shape[1] == _SAMPLE:
            table = np.ascontiguousarray(np.concatenate([table, table], axis=1))  # columns 4-7 are never read
        H = table.shape[0]

    eng.upload_pairs(pts_a, pts_b, np.eye(3))  # K = I: the records hold pixel coordinates
    # reference sampler: columns 0-3 = perm[:4], the shuffle is size-independent
    table, ref = _load_samples(eng, sampler, n, H, table, seed, hyp_offset)
    best, mask, err, _, _ = eng.ransac_homography(threshold, float(min_num_extra_inliers), agg, selection)
    _restore_random_state(ref)  # no exception aborts the loop: every shuffle happened
    if best.index < 0:
        raise no_model()

    def score(t):
        H_t, _ = eng.get_models(t, 1)
        return eng.homography_mask(H_t[0], threshold)

    # near-ties are settled in the reference's list order and summation (SURVEY.md H1), as on the E path
    t, e = _replay_near_ties(eng, sampler, selection, table, ref, n, _SAMPLE, threshold, agg, score) or (None, None)
    if t is not None and t != int(best.index):
        H_t, _ = eng.get_models(t, 1)
        best.index = t
        best.E[:] = tuple(H_t.reshape(9))
        mask, err = score(t)
        best.count_extra = int(mask.sum() - mask[table[t][:_SAMPLE]].sum())
        best.err = e

    mask = np.asarray(mask).astype(bool)
    sample, inliers = _inlier_order(best, sampler, table, ref, mask, _SAMPLE)
    return HomographyResult(
        H=np.array(best.E, dtype=np.float64).reshape(3, 3),
        best_index=int(best.index) + (hyp_offset if sampler == "device" else 0),
        error=float(best.err),
        count_extra=int(best.count_extra),
        inlier_indices=inliers,
        mask=mask,
        err=err,
        sample=sample,
        num_invalid=int(best.num_invalid),
        first_invalid=int(best.first_invalid),
    )


def fit_homography_arrays(pts_a, pts_b, engine: Optional[_native.Engine] = None) -> np.ndarray:
    """The exact homography through 4 correspondences ([4,2] pixel arrays), H[2,2] == 1.  Raises ValueError when three
    of the points are collinear in either image (no unique solution)."""
    pts_a = np.ascontiguousarray(pts_a, dtype=np.float64).reshape(-1, 2)
    pts_b = np.ascontiguousarray(pts_b, dtype=np.float64).reshape(-1, 2)
    if pts_a.shape[0] != _SAMPLE or pts_b.shape[0] != _SAMPLE:
        raise ValueError("Exactly four matches are needed")
    eng = engine or _native.get_engine()
    eng.upload_pairs(pts_a, pts_b, np.eye(3))
    eng.set_table(np.array([[0, 1, 2, 3, 0, 1, 2, 3]], dtype=np.int32))
    H, valid = eng.fit_homography()
    if not valid[0]:
        raise ValueError("Degenerate sample: three of the four points are collinear")
    return H[0]


def transfer_error_arrays(H, pts_a, pts_b, threshold: float = np.inf, engine: Optional[_native.Engine] = None):
    """(inlier decision bool[n], symmetric transfer error float64[n] in px^2) of every correspondence under H."""
    pts_a = np.ascontiguousarray(pts_a, dtype=np.float64).reshape(-1, 2)
    pts_b = np.ascontiguousarray(pts_b, dtype=np.float64).reshape(-1, 2)
    eng = engine or _native.get_engine()
    eng.upload_pairs(pts_a, pts_b, np.eye(3))
    return eng.homography_mask(np.asarray(H, dtype=np.float64).reshape(3, 3), threshold)


@dataclasses.dataclass
class HomographyDecomposition:
    candidates: list              # [(R, t, n, d)]: four, or one (R, 0, NaN, inf) when rotation_only
    singular_values: np.ndarray   # of K^-1 H K, scaled so that the middle one is 1
    rotation_only: bool


def _candidates(p) -> list:
    R = np.array(p.R, dtype=np.float64).reshape(4, 3, 3)
    t = np.array(p.t, dtype=np.float64).reshape(4, 3)
    n = np.array(p.n, dtype=np.float64).reshape(4, 3)
    d = np.array(p.d, dtype=np.float64)
    return [(R[i], t[i], n[i], float(d[i])) for i in range(1 if p.rotation_only else 4)]


def decompose_homography_arrays(H, camera_matrix, rotation_tolerance: float = 1e-2,
                                engine: Optional[_native.Engine] = None) -> HomographyDecomposition:
    """Relative pose and plane candidates of a homography H (3x3, image-A pixels -> image-B pixels) for cameras with
    intrinsics ``camera_matrix``.  The order of the four candidates depends on eigenvector signs; compare them as a
    set."""
    eng = engine or _native.get_engine()
    p = eng.decompose_homography(H, camera_matrix, rotation_tolerance)
    return HomographyDecomposition(candidates=_candidates(p), singular_values=np.array(p.sv, dtype=np.float64),
                                   rotation_only=bool(p.rotation_only))


@dataclasses.dataclass
class HomographyTwoViewResult:
    ransac: HomographyResult
    R: np.ndarray                 # (3,3) voted rotation (the nearest rotation to K^-1 H K when rotation_only)
    t: np.ndarray                 # (3,) unit translation; 0 when rotation_only
    n: np.ndarray                 # (3,) plane normal, camera-1 frame; NaN when rotation_only
    d: float                      # plane distance in units of the baseline; inf when rotation_only
    rotation_only: bool
    candidates: list              # [(R, t, n, d)] as decompose_homography_arrays returns them
    counts: np.ndarray            # cheirality votes per candidate (zeros when rotation_only)
    inlier_indices: np.ndarray    # ascending indices of the winner's inliers (samples included)
    passing: np.ndarray           # bool per inlier: passes the voted candidate (all False when rotation_only)
    points: np.ndarray            # [m,3] triangulated points (NaN where not passing)
    refinement: Optional[Refinement] = None  # with refine_iterations > 0: everything above but ``ransac`` describes
                                             # the refined H


def two_view_homography_arrays(
    camera_matrix,
    pts_a,
    pts_b,
    threshold: float,
    min_num_extra_inliers=None,
    error_aggregation_method=None,
    max_iterations: Optional[int] = None,
    distance_threshold=None,
    *,
    rotation_tolerance: float = 1e-2,
    sampler: str = "reference",
    seed: int = 0,
    selection: str = "min_error",
    engine: Optional[_native.Engine] = None,
    table: Optional[np.ndarray] = None,
    refine_iterations: int = 0,
) -> HomographyTwoViewResult:
    """RANSAC homography -> pose and plane candidates -> cheirality vote -> triangulation, for [n,2] pixel arrays.

    The RANSAC part (``ransac``) is ``ransac_homography_arrays`` on the same arguments, random state included.  Every
    inlier of the winner is triangulated under each candidate (K-normalised coordinates, P1 = [I|0], P2 = [R|t]); it
    passes when both depths are >= -1e-8 and |X| <= ``distance_threshold`` (default 50), every passing inlier counts,
    and the first maximum wins.  The passing inliers are triangulated in pixel coordinates (P1 = K[I|0], P2 = K[R|t]).
    Raises EightPointCalculationError when no inlier passes any candidate.  With ``sampler="device"`` the estimate and
    the tail are one library call.  refine_iterations > 0 refines the winning H over its inliers (Levenberg-Marquardt
    on the symmetric transfer error, at most that many iterations, on the device) before the decomposition; the pose,
    inliers and points then describe the refined H and ``refinement`` reports it."""
    refine_iterations = _refine_count(refine_iterations)
    if distance_threshold is None:
        distance_threshold = 50.0
    K = np.asarray(camera_matrix, dtype=np.float64)
    if K.shape != (3, 3):
        raise ValueError(f"Camera intrinsic matrix is not 3x3, actual shape: {K.shape}")
    eng = engine or _native.get_engine()
    pa = np.ascontiguousarray(pts_a, dtype=np.float64).reshape(-1, 2)
    pb = np.ascontiguousarray(pts_b, dtype=np.float64).reshape(-1, 2)
    iterations = 100 if max_iterations is None else int(max_iterations)
    if sampler == "device" and pa.shape == pb.shape and pa.shape[0] >= 8 and iterations > 0:
        # nothing on the host depends on the winner (no near-tie replay): estimate and tail in one call
        min_extra = 0 if min_num_extra_inliers is None else min_num_extra_inliers
        eng.upload_pairs(pa, pb, np.eye(3))  # K = I: the records hold pixel coordinates
        eng.sample_device(seed, iterations)
        best, mask, err, p, _, idx, ok, X = eng.two_view_homography(
            K, threshold, float(min_extra), _agg_name(error_aggregation_method), selection, distance_threshold,
            rotation_tolerance, refine_iterations=refine_iterations)
        if best.index < 0:
            raise ValueError(f"No model could be found with at least {min_extra + _SAMPLE} inliers.")
        sample, inliers = _tail_inliers(best, _ransac_list(best, mask, _SAMPLE) if refine_iterations else idx, _SAMPLE)
        res = HomographyResult(H=np.array(best.E, dtype=np.float64).reshape(3, 3), best_index=int(best.index),
                               error=float(best.err), count_extra=int(best.count_extra),
                               inlier_indices=inliers, mask=mask.astype(bool),
                               err=err, sample=sample, num_invalid=int(best.num_invalid),
                               first_invalid=int(best.first_invalid))
    else:
        res = ransac_homography_arrays(pa, pb, threshold, min_num_extra_inliers, error_aggregation_method, max_iterations,
                                       sampler=sampler, seed=seed, selection=selection, engine=eng, table=table)
        eng.set_winner(res.best_index)  # the host's winner (a near-tie replay may have moved it)
        p, _, idx, ok, X = eng.homography_pose_and_triangulate(K, threshold, distance_threshold, rotation_tolerance,
                                                               refine_iterations=refine_iterations)
    cands = _candidates(p)
    counts = np.array(p.counts, dtype=np.int64)
    if p.rotation_only:
        R, t, n, d = cands[0]
        passing = np.zeros(len(idx), dtype=bool)
    else:
        if 0 == np.count_nonzero(counts):
            raise EightPointCalculationError("None of the transformations pass the cheirality check.")
        R, t, n, d = cands[int(p.best)]
        passing = ((ok >> int(p.best)) & 1).astype(bool)
    return HomographyTwoViewResult(ransac=res, R=R.copy(), t=t.copy(), n=n.copy(), d=d,
                                   rotation_only=bool(p.rotation_only), candidates=cands, counts=counts,
                                   inlier_indices=idx, passing=passing, points=X,
                                   refinement=_refinement(eng) if refine_iterations else None)
