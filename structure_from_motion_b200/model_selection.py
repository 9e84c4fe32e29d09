"""Essential matrix or homography for one image pair or a batch of pairs (numpy in, numpy out).

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
    refine_iterations: int = 0,
) -> TwoViewSelection:
    """Both two-view paths on one pair, then the ratio rule on their winners.

    Runs ``two_view_arrays(..., on_degenerate="skip")`` with ``essential_threshold`` (SED, K-normalised units) and
    ``two_view_homography_arrays`` with ``homography_threshold`` (symmetric transfer error, px^2), on the same engine
    and with the same remaining arguments: each sub-result equals the standalone call, and with the reference sampler
    the global ``random`` state ends where the E call followed by the H call leaves it.  A call that raises ValueError
    or EightPointCalculationError leaves its model out (its message is kept) and the other one is chosen; when both
    fail, ValueError carries both messages.  With refine_iterations > 0 both winners are refined over their inliers
    before their poses, and the ratio rule scores the refined models."""
    eng = engine or _native.get_engine()
    K = np.asarray(camera_matrix, dtype=np.float64)
    common = dict(sampler=sampler, seed=seed, selection=selection, engine=eng, refine_iterations=refine_iterations)
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
    E = None if ess is None else (ess.refinement.model if ess.refinement else ess.ransac.E)
    H = None if hom is None else (hom.refinement.model if hom.refinement else hom.ransac.H)
    scores = _scores(eng, E, H, K, sigma, homography_ratio, False)
    win = hom if scores.model == "homography" else ess
    return TwoViewSelection(model=scores.model, scores=scores, essential=ess, homography=hom,
                            essential_failure=ess_fail, homography_failure=hom_fail, R=win.R, t=win.t,
                            inlier_indices=win.inlier_indices, passing=win.passing, points=win.points,
                            rotation_only=bool(scores.model == "homography" and hom.rotation_only))


_SCORE_FIELDS = ("score_e", "score_h", "ratio_h", "fixed_e", "fixed_h", "count_e", "count_h")


def _essential_status(r, sv2) -> np.ndarray:
    """Per pair, why two_view_arrays would fail on it (None when it would not): no model (a pair of fewer than 8
    correspondences has none), an E whose smallest singular value is not ~0, or no inlier passing any pose."""
    st = np.full(len(r["best_index"]), None, dtype=object)
    for p in range(len(st)):
        if r["best_index"][p] < 0:
            st[p] = "no model"
        elif not np.isclose(0.0, sv2[p]):
            st[p] = "degenerate essential matrix"
        elif np.count_nonzero(r["counts"][p]) == 0:
            st[p] = "no passing inlier"
    return st


def _homography_status(r) -> np.ndarray:
    """Per pair, why two_view_homography_arrays would fail on it (None when it would not).  A rotation-only pair is
    kept: it has no vote."""
    st = np.full(len(r["best_index"]), None, dtype=object)
    for p in range(len(st)):
        if r["best_index"][p] < 0:
            st[p] = "no model"
        elif not r["rotation_only"][p] and np.count_nonzero(r["counts"][p]) == 0:
            st[p] = "no passing inlier"
    return st


def batch_two_view_select_arrays(
    pts_a,
    pts_b,
    offsets,
    Ks,
    essential_threshold: float,
    homography_threshold: float,
    h: int,
    seed: int,
    *,
    min_extra: float = 0.0,
    aggregation: str = "rms",
    selection: str = "min_error",
    distance_threshold: float = 50.0,
    sigma: float = 1.0,
    homography_ratio: float = 0.45,
    rotation_tolerance: float = 1e-2,
    pair_id0: int = 0,
    engine: Optional[_native.Engine] = None,
    refine_iterations: int = 0,
) -> dict:
    """``two_view_select_arrays(sampler="device")`` for every pair of a batch: pair p owns rows
    [offsets[p], offsets[p+1]) of the [n,2] pixel arrays and the camera Ks[p] (upper triangular, K[2,2] = 1).

    Runs ``Engine.batch_two_view`` (E, ``essential_threshold``) and ``Engine.batch_two_view_homography`` (H,
    ``homography_threshold`` in px^2) with the same h, seed and pair_id0, then ``Engine.batch_score_models`` on the
    homography call's upload.  A side is given to the scorer for pair p exactly when the single-pair rule keeps it: it
    has a winner and its vote has a passing inlier (an essential matrix also needs a smallest singular value ~0); a
    rotation-only homography is kept.  Returns a dict:
      essential, homography   the two batch dicts, each equal to its standalone call
      essential_status, homography_status   object[P]: None where the side is kept, else why it is left out
      model                   object[P]: "essential", "homography" or None (neither side kept)
      score_e ... count_h     the scores of batch_score_models [P] (zero for a side left out)
      R [P,3,3], t [P,3], rotation_only [P]   the chosen side's pose (NaN without a model)
      inlier_offsets [P+1], inlier_idx, passing, points   the chosen side's inlier segments (empty without a model)
    With refine_iterations > 0 both batch calls refine their winners (refined_E / refined_H and the refine_* keys in
    their dicts) and the scorer reads the refined models.
    """
    eng = engine or _native.get_engine()
    offsets = np.ascontiguousarray(offsets, dtype=np.int64)
    P = len(offsets) - 1
    Ks = np.asarray(Ks, dtype=np.float64).reshape(P, 3, 3)
    ess, sv2 = eng._batch_two_view(pts_a, pts_b, offsets, Ks, h, seed, essential_threshold, min_extra, aggregation,
                                   selection, distance_threshold, pair_id0, refine_iterations)
    hom = eng.batch_two_view_homography(pts_a, pts_b, offsets, Ks, h, seed, homography_threshold, min_extra, aggregation,
                                        selection, distance_threshold, rotation_tolerance, pair_id0, refine_iterations)
    e_st, h_st = _essential_status(ess, sv2), _homography_status(hom)
    keep_e, keep_h = np.equal(e_st, None), np.equal(h_st, None)
    s, _ = eng.batch_score_models(ess.get("refined_E", ess["E"]), hom.get("refined_H", hom["H"]), keep_e, keep_h, sigma,
                                  homography_ratio)
    out = dict(essential=ess, homography=hom, essential_status=e_st, homography_status=h_st)
    for f in _SCORE_FIELDS:
        out[f] = np.array([getattr(x, f) for x in s[:P]], dtype=np.float64 if f[:5] in ("score", "ratio") else np.int64)
    code = np.array([x.model for x in s[:P]], dtype=np.int64)
    out["model"] = np.array([_MODEL.get(int(m)) for m in code], dtype=object)
    R = np.full((P, 3, 3), np.nan)
    t = np.full((P, 3), np.nan)
    rot = np.zeros(P, dtype=bool)
    ioff, idx, passing, pts = [0], [], [], []
    for p in range(P):
        side = hom if code[p] == 1 else ess if code[p] == 0 else None
        if side is None:
            ioff.append(ioff[-1])
            continue
        lo, hi = side["inlier_offsets"][p], side["inlier_offsets"][p + 1]
        b = int(side["pose_index"][p])
        R[p], t[p] = side["R"][p], side["t"][p]
        rot[p] = bool(code[p] == 1 and hom["rotation_only"][p])
        idx.append(side["inlier_idx"][lo:hi])
        passing.append(np.zeros(hi - lo, dtype=bool) if b < 0 else ((side["pass_bits"][lo:hi] >> b) & 1).astype(bool))
        pts.append(side["points"][lo:hi])
        ioff.append(ioff[-1] + (hi - lo))
    out.update(R=R, t=t, rotation_only=rot, inlier_offsets=np.array(ioff, dtype=np.int64),
               inlier_idx=np.concatenate(idx) if idx else np.zeros(0, dtype=np.int32),
               passing=np.concatenate(passing) if passing else np.zeros(0, dtype=bool),
               points=np.concatenate(pts) if pts else np.zeros((0, 3)))
    return out
