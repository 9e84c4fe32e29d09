"""Essential matrix or homography for one image pair (numpy in, numpy out).

On a planar scene E is not determined by the data, on a rotation-only pair it vanishes, and on a general scene a
homography fits one depth layer at best: a two-view initialiser estimates both models and keeps one.  The rule is
ORB-SLAM's score ratio (Mur-Artal, Montiel & Tardos, 2015, section IV), with E turned into the pixel fundamental matrix
F = K^-T E K^-1 and both models scored on the same correspondences, one-way in each image:

    rho_M(d2) = 5.99 - d2 / sigma^2  when d2 / sigma^2 < T_M (T_E = 3.84, T_H = 5.99), else 0
    S_M = sum_i rho_M(d2_A,i) + rho_M(d2_B,i)
    R_H = S_H / (S_H + S_E);  H is chosen iff R_H > homography_ratio (default 0.45)

d2 for E is the squared distance in px to the epipolar line, for H the one-way transfer error in px^2.  sigma is the
correspondence noise in px.  The sums are exact (every term rounded to a multiple of 2^-32, csrc/sfm_select.cuh), so the
scores and the choice are bit-reproducible.  Everything numeric runs in libsfm_b200.so; there is no CPU fallback.
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import numpy as np

from . import _native
from .errors import EightPointCalculationError
from .homography import HomographyTwoViewResult, two_view_homography_arrays
from .two_view import TwoViewResult, two_view_arrays

_MODEL = {0: "essential", 1: "homography"}


@dataclasses.dataclass
class ModelScores:
    model: str                    # "essential" or "homography"
    score_e: float                # S_E (0 when E was not given)
    score_h: float                # S_H (0 when H was not given)
    ratio_h: float                # S_H / (S_H + S_E), 0 when both are 0
    fixed_e: int                  # S_E * 2^32, the exact integer sum
    fixed_h: int
    count_e: int                  # correspondences whose two one-way errors both pass T_E (a diagnostic)
    count_h: int
    per_point: Optional[np.ndarray]  # [n,4] (d2_A,E, d2_B,E, d2_A,H, d2_B,H) in px^2, NaN for a model not given


def _scores(eng, E, H, K, sigma, homography_ratio, per_point) -> ModelScores:
    s, pp = eng.model_scores(E, H, K, sigma, homography_ratio, per_point)
    return ModelScores(model=_MODEL[int(s.model)], score_e=float(s.score_e), score_h=float(s.score_h),
                       ratio_h=float(s.ratio_h), fixed_e=int(s.fixed_e), fixed_h=int(s.fixed_h),
                       count_e=int(s.count_e), count_h=int(s.count_h), per_point=pp)


def model_scores_arrays(camera_matrix, pts_a, pts_b, E=None, H=None, *, sigma: float = 1.0,
                        homography_ratio: float = 0.45, per_point: bool = False,
                        engine: Optional[_native.Engine] = None) -> ModelScores:
    """Scores of E (3x3, b^T E a = 0 in K-normalised coordinates) and / or H (3x3, image-A pixels -> image-B pixels) on
    [n,2] arrays of matched pixel coordinates, and the model the ratio rule picks.  When only one model is given it is
    the one picked."""
    K = np.asarray(camera_matrix, dtype=np.float64)
    if K.shape != (3, 3):
        raise ValueError(f"Camera intrinsic matrix is not 3x3, actual shape: {K.shape}")
    pa = np.ascontiguousarray(pts_a, dtype=np.float64).reshape(-1, 2)
    pb = np.ascontiguousarray(pts_b, dtype=np.float64).reshape(-1, 2)
    if pa.shape != pb.shape:
        raise ValueError("pts_a and pts_b must have the same shape")
    eng = engine or _native.get_engine()
    eng.upload_pairs(pa, pb, np.eye(3))  # the scores read the pixel coordinates
    return _scores(eng, E, H, K, sigma, homography_ratio, per_point)


@dataclasses.dataclass
class TwoViewSelection:
    model: str                                      # "essential" or "homography"
    scores: ModelScores
    essential: Optional[TwoViewResult]              # two_view_arrays' result, None when it failed
    homography: Optional[HomographyTwoViewResult]   # two_view_homography_arrays' result, None when it failed
    essential_failure: Optional[str]                # the message of the failed call
    homography_failure: Optional[str]
    # the chosen model's pose and points
    R: np.ndarray
    t: np.ndarray                 # unit; 0 for a rotation-only pair
    inlier_indices: np.ndarray
    passing: np.ndarray
    points: np.ndarray
    rotation_only: bool


def two_view_select_arrays(
    camera_matrix,
    pts_a,
    pts_b,
    essential_threshold: float,
    homography_threshold: float,
    min_num_extra_inliers=None,
    error_aggregation_method=None,
    max_iterations: Optional[int] = None,
    distance_threshold=None,
    *,
    sigma: float = 1.0,
    homography_ratio: float = 0.45,
    rotation_tolerance: float = 1e-2,
    sampler: str = "reference",
    seed: int = 0,
    selection: str = "min_error",
    engine: Optional[_native.Engine] = None,
) -> TwoViewSelection:
    """Both two-view paths on one pair, then the ratio rule on their winners.

    Runs ``two_view_arrays(..., on_degenerate="skip")`` with ``essential_threshold`` (SED, K-normalised units) and
    ``two_view_homography_arrays`` with ``homography_threshold`` (symmetric transfer error, px^2), on the same engine
    and with the same remaining arguments: each sub-result equals the standalone call, and with the reference sampler
    the global ``random`` state ends where the E call followed by the H call leaves it.  A call that raises ValueError
    or EightPointCalculationError leaves its model out (its message is kept) and the other one is chosen; when both
    fail, ValueError carries both messages."""
    eng = engine or _native.get_engine()
    K = np.asarray(camera_matrix, dtype=np.float64)
    common = dict(sampler=sampler, seed=seed, selection=selection, engine=eng)
    ess = hom = None
    ess_fail = hom_fail = None
    try:
        ess = two_view_arrays(K, pts_a, pts_b, essential_threshold, min_num_extra_inliers, error_aggregation_method,
                              max_iterations, distance_threshold, on_degenerate="skip", **common)
    except (ValueError, EightPointCalculationError) as exc:
        ess_fail = str(exc)
    try:
        hom = two_view_homography_arrays(K, pts_a, pts_b, homography_threshold, min_num_extra_inliers,
                                         error_aggregation_method, max_iterations, distance_threshold,
                                         rotation_tolerance=rotation_tolerance, **common)
    except (ValueError, EightPointCalculationError) as exc:
        hom_fail = str(exc)
    if ess is None and hom is None:
        raise ValueError(f"neither model could be estimated: essential matrix: {ess_fail}; homography: {hom_fail}")
    # both calls uploaded these correspondences: the context's pixel coordinates are this pair's
    scores = _scores(eng, None if ess is None else ess.ransac.E, None if hom is None else hom.ransac.H, K, sigma,
                     homography_ratio, False)
    win = hom if scores.model == "homography" else ess
    return TwoViewSelection(model=scores.model, scores=scores, essential=ess, homography=hom,
                            essential_failure=ess_fail, homography_failure=hom_fail, R=win.R, t=win.t,
                            inlier_indices=win.inlier_indices, passing=win.passing, points=win.points,
                            rotation_only=bool(scores.model == "homography" and hom.rotation_only))
