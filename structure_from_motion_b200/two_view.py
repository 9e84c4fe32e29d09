"""Array-native entry points of the two-view hot path (numpy in, numpy out).

These are the twins of the reference's list-of-dataclass callables (SURVEY.md fact 2):
marshalling 10^5..10^6 ``Feature`` objects costs more than the GPU work, so the
list-based mirrors in ``ransac/`` and ``epipolar/`` convert once and call these.
Everything numeric happens in libsfm_b200.so (CUDA, sm_100a); there is no CPU fallback.
"""
from __future__ import annotations

import dataclasses
import random
from math import inf
from typing import Optional

import numpy as np

from . import _native
from .errors import EIGHT_POINT_ERROR_MESSAGE, EightPointCalculationError
from .ransac.ransac import ErrorAggregationMethod


@dataclasses.dataclass
class RansacResult:
    E: np.ndarray                 # (3,3), E[2,2] == 1
    best_index: int               # winning iteration (global hypothesis index)
    error: float                  # aggregated error of the winner
    count_extra: int              # inliers beyond the 8 samples
    inlier_indices: np.ndarray    # int64; reference order (samples, then permuted rest) with the
                                  # reference sampler, else samples then ascending
    mask: np.ndarray              # bool[n]: sed <= threshold under the winner
    sed: np.ndarray               # float64[n]
    sample: np.ndarray            # int32[8] the winner's minimal sample
    num_invalid: int
    first_invalid: int


@dataclasses.dataclass
class Refinement:
    """The least-squares refinement of a winner over its inliers (include/sfm_b200.h, sfm_set_refinement)."""
    model: np.ndarray     # (3,3) refined E or H, [2,2] == 1; the RANSAC model when status is no_model / nonfinite
    cost_ransac: float    # sum of the RANSAC model's errors over the inlier list
    cost_start: float     # at the start point (E: the RANSAC E projected onto the essential manifold)
    cost_final: float     # at the refined model, <= cost_start
    num: int              # correspondences in the inlier list
    iterations: int       # proposals evaluated
    status: str           # converged | max_iterations | stalled | no_model | nonfinite
    rejected: int = 0     # of those, proposals rejected (cost not strictly lower)


def _refinement(eng) -> Refinement:
    """The report of the last single-pair tail call that refined."""
    r = eng.get_refinement(1)[0]
    return Refinement(model=np.array(r.model, dtype=np.float64).reshape(3, 3), cost_ransac=float(r.cost_ransac),
                      cost_start=float(r.cost_start), cost_final=float(r.cost_final), num=int(r.num),
                      iterations=int(r.iterations), status=_native.REFINE_STATUS[int(r.status)],
                      rejected=int(r.rejected))


def _refine_count(refine_iterations) -> int:
    n = int(refine_iterations)
    if n < 0:
        raise ValueError(f"refine_iterations must be >= 0, got {n}")
    return n


def _agg_name(method) -> str:
    if method is None:
        return "rms"  # ransac.py:50-51
    # the reference compares ``.value`` (ransac.py:99-105), so any Enum with the same values is accepted
    return str(getattr(method, "value", method))


def _reference_error(errors, agg: str) -> float:
    """_aggregate_error (lib/ransac/ransac.py:96-108) on a python list in [samples..., extra inliers...] order:
    the reference's own summation order (python ``sum`` / numpy pairwise) — used only to settle near-ties."""
    if agg == "sum":
        return sum(errors)
    if agg == "square":
        return np.sum(np.square(errors)).item()
    if agg == "mean":
        return np.mean(errors).item()
    return np.sqrt(np.mean(np.square(errors))).item()


def _resolve_near_ties(eng, ties, threshold, agg, rows, order_after, score=None):
    """SURVEY.md H1.  The GPU selects on exactly rounded sums; the reference keeps ``model_error < best_model_error``
    (ransac.py:83) on errors summed in list order.  For the hypotheses whose errors agree to 1e-12 the list-order error
    is recomputed here from the device's exact per-correspondence scores and the strict ``<`` is replayed in iteration
    order.  rows(t) -> the sample indices of hypothesis t; order_after(t) -> the correspondences that follow the
    samples in that iteration's list (the permutation tail for the reference sampler); score(t) -> (inlier decision
    bool[n], per-correspondence error [n]) under hypothesis t, by default the SED of ``eng``'s essential matrix t
    against ``threshold``.  Returns the local index."""
    if score is None:
        def score(t):
            eng.set_winner(t)
            _, sed = eng.inlier_mask(threshold)
            return sed <= threshold, sed

    best_t, best_err = None, float("inf")
    for t in ties:  # ascending = iteration order
        inl, sed = score(int(t))
        rest = order_after(int(t))
        errs = [float(v) for v in sed[rows(int(t))]] + [float(v) for v in sed[rest][inl[rest]]]
        e = _reference_error(errs, agg)
        if e < best_err:
            best_t, best_err = int(t), e
    return best_t, best_err


def _get_state_words():
    version, words, gauss = random.getstate()
    return version, np.array(words, dtype=np.uint32), gauss


def _set_state_words(version, words, gauss):
    random.setstate((version, tuple(int(w) for w in words), gauss))


def _load_samples(eng, sampler, n, h, table, seed, hyp_offset):
    """The minimal samples of ``h`` hypotheses onto ``eng``, after its upload.  "reference" draws the table with
    CPython's random.shuffle semantics from the process-global state but leaves that state alone (_restore_random_state
    advances it once the caller knows how far the reference's loop ran); "device" draws on the GPU; "table" loads
    ``table`` ([h,8]).  Returns (table, ref): ref = (ReferenceSampler, state version, gauss) or None."""
    ref = None
    if sampler == "reference":
        version, words, gauss = _get_state_words()
        ref = (_native.ReferenceSampler(words, n, h), version, gauss)
        table = ref[0].table
    if sampler == "device":
        eng.sample_device(seed, h, hyp_offset=hyp_offset)
    else:
        eng.set_table(table)
    return table, ref


def _degenerate_sample_error(pts_a, pts_b, K) -> Exception:
    """The exception the reference raises for one degenerate 8-point sample (pixel coordinates [8,2]).  When the
    Hartley-normalised coordinates are not finite (a coordinate is NaN or infinite, or all eight points of one image
    coincide and their mean rounds back to the point, so that the scale is sqrt(2)/0), np.linalg.eig refuses Y^T Y
    (eight_point.py:410) with numpy's LinAlgError; otherwise the validity test raises EightPointCalculationError
    (:414-421).  The normalisation repeats the reference's numpy calls (:127-133, :319-326), so both decide alike."""
    K = np.asarray(K, dtype=np.float64)
    with np.errstate(all="ignore"):
        for pts in (pts_a, pts_b):
            pts = np.asarray(pts, dtype=np.float64)
            coords = np.stack([(pts[:, 0] - K[0][2]) / K[0][0], (pts[:, 1] - K[1][2]) / K[1][1]], axis=1)
            centered = coords - np.mean(coords, axis=0)
            scale = np.sqrt(2.0) / np.mean(np.linalg.norm(centered, axis=1))
            if not np.isfinite(centered * scale).all():
                return np.linalg.LinAlgError("Array must not contain infs or NaNs")
    return EightPointCalculationError(EIGHT_POINT_ERROR_MESSAGE)


def _restore_random_state(ref, iteration=None):
    """Leave the global random state where the reference's loop does: after every shuffle, or after the shuffle of
    ``iteration`` when the loop stops there."""
    if ref is not None:
        sampler, version, gauss = ref
        words = sampler.final_state if iteration is None else sampler.after(iteration)[0]
        _set_state_words(version, words, gauss)


def _replay_near_ties(eng, sampler, selection, table, ref, n, k, threshold, agg, score=None):
    """The near-tie replay of ``_resolve_near_ties`` for a k-point sample, where the reference's list order is known:
    the sample, then the rest of that iteration's permutation (reference sampler) or ascending (table).  Returns its
    (local index, error), or None when it does not run: device sampler, other selections, or no 2..64 near-ties."""
    if sampler == "device" or selection != "min_error":
        return None
    ties, total = eng.near_ties(1e-12, 64)
    if not 1 < total <= 64:
        return None

    def rows(t):
        return np.asarray(table[t][:k], dtype=np.int64)

    def order_after(t):
        if ref is not None:
            return ref[0].after(t)[1][k:].astype(np.int64)
        keep = np.ones(n, dtype=bool)
        keep[table[t][:k]] = False
        return np.nonzero(keep)[0]

    return _resolve_near_ties(eng, ties, threshold, agg, rows, order_after, score)


def _inlier_order(best, sampler, table, ref, mask, k):
    """(sample int32[k], inlier indices int64) of the winner: the sample, then the other inliers in the reference's
    order — the rest of the winning iteration's permutation (reference sampler) or ascending (table, device)."""
    local = int(best.index)
    if sampler == "device":
        sample = np.array(best.sample[:k], dtype=np.int32)
    else:
        sample = np.asarray(table[local][:k], dtype=np.int32)
    if ref is not None:
        rest = ref[0].after(local)[1][k:].astype(np.int64)  # replayed from the nearest snapshot
        extra = rest[mask[rest]]
    else:
        is_sample = np.zeros(mask.shape[0], dtype=bool)
        is_sample[sample] = True
        extra = np.nonzero(mask & ~is_sample)[0]
    return sample, np.concatenate([sample.astype(np.int64), extra])


def _ransac_list(best, mask, k):
    """The list T1 compacts for the RANSAC winner (decision or sample, ascending), rebuilt from its mask."""
    keep = np.asarray(mask).astype(bool).copy()
    keep[np.array(best.sample[:k], dtype=np.int64)] = True
    return np.flatnonzero(keep)


def _tail_inliers(best, idx, k):
    """(sample int32[k], inlier indices int64) of a winner selected on the device: the sample, then the rest of the
    tail's compacted list (decision | sample, ascending)."""
    sample = np.array(best.sample[:k], dtype=np.int32)
    return sample, np.concatenate([sample.astype(np.int64), idx[~np.isin(idx, sample)]])


def ransac_essential_arrays(
    camera_matrix,
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
    on_degenerate: str = "raise",
    selection: str = "min_error",
    engine: Optional[_native.Engine] = None,
    table: Optional[np.ndarray] = None,
    _tail: Optional[dict] = None,
) -> RansacResult:
    """estimate_essential_mat_with_ransac (lib/epipolar/epipolar_ransac.py:45-70) on arrays.

    pts_a, pts_b: [n,2] matched pixel coordinates (row i of each is one correspondence).
    sampler: "reference" — CPython random.shuffle semantics on the process-global state
             (lib/ransac/ransac.py:62), the state advances exactly as in the reference;
             "device" — Philox sampler on the GPU (seed), for sizes where the reference's
             O(N) shuffle per iteration is infeasible; "table" — use the given table.
    """
    if max_iterations is None:
        max_iterations = 100  # ransac.py:48-49
    if min_num_extra_inliers is None:
        min_num_extra_inliers = 0  # ransac.py:52-53
    agg = _agg_name(error_aggregation_method)
    pts_a = np.ascontiguousarray(pts_a, dtype=np.float64).reshape(-1, 2)
    pts_b = np.ascontiguousarray(pts_b, dtype=np.float64).reshape(-1, 2)
    n = pts_a.shape[0]
    H = int(max_iterations)

    def no_model():
        return ValueError(f"No model could be found with at least {min_num_extra_inliers + 8} inliers.")

    if H <= 0:
        raise no_model()  # ransac.py:88-91 (loop never ran)
    if n < 8:
        if sampler == "reference":
            random.shuffle(list(range(n)))  # the reference shuffles once before the fitter raises
        raise ValueError("Eight feature pairs are expected.")  # epipolar_ransac.py:31-32
    eng = engine or _native.get_engine()
    if sampler == "table":
        table = np.ascontiguousarray(table, dtype=np.int32).reshape(-1, 8)
        H = table.shape[0]

    eng.upload_pairs(pts_a, pts_b, camera_matrix)
    table, ref = _load_samples(eng, sampler, n, H, table, seed, hyp_offset)
    if _tail is None:
        best, mask, sed = eng.ransac_essential(threshold, float(min_num_extra_inliers), agg, selection)
    else:  # two_view_arrays: selection, inlier mask, pose vote and triangulation in one C call
        best, mask, sed, *rest = eng.two_view(threshold, float(min_num_extra_inliers), agg, selection,
                                              _tail["distance_threshold"], refine_iterations=_tail["refine_iterations"])
        _tail["out"] = rest

    if best.num_invalid > 0 and on_degenerate == "raise":
        # the reference aborts inside iteration first_invalid: only that many shuffles happened
        first = int(best.first_invalid)
        row = eng.get_table(1, first)[0] if sampler == "device" else np.asarray(table[first], dtype=np.int64)
        _restore_random_state(ref, first)
        raise _degenerate_sample_error(pts_a[row], pts_b[row], camera_matrix)
    _restore_random_state(ref)
    if best.index < 0:
        raise no_model()

    # H1: near-ties are settled in the reference's own list order and summation
    tie = _replay_near_ties(eng, sampler, selection, table, ref, n, 8, threshold, agg)
    if tie is not None:
        t, e = tie
        if t is not None and t != int(best.index):
            E_t, _ = eng.get_models(t, 1)
            best.index = t
            best.E[:] = tuple(E_t.reshape(9))
            eng.set_winner(t)
            m2, sed = eng.inlier_mask(threshold)
            mask = m2.astype(np.uint8)
            best.count_extra = int(m2.sum() - m2[table[t]].sum())
            best.err = e
            if _tail is not None:  # the tail (and the refinement) of the replayed winner
                _tail["out"] = list(eng.pose_and_triangulate(threshold, _tail["distance_threshold"],
                                                             refine_iterations=_tail["refine_iterations"]))
        else:
            eng.set_winner(int(best.index))

    mask = mask.astype(bool)
    sample, inliers = _inlier_order(best, sampler, table, ref, mask, 8)
    return RansacResult(
        E=np.array(best.E, dtype=np.float64).reshape(3, 3),
        best_index=int(best.index) + (hyp_offset if sampler == "device" else 0),
        error=float(best.err),
        count_extra=int(best.count_extra),
        inlier_indices=inliers,
        mask=mask,
        sed=sed,
        sample=sample,
        num_invalid=int(best.num_invalid),
        first_invalid=int(best.first_invalid),
    )


def ransac_essential_adaptive(camera_matrix, pts_a, pts_b, threshold, min_num_extra_inliers=None,
                              error_aggregation_method=None, max_iterations: int = 65536, *, confidence: float = 0.99,
                              chunk: int = 4096, seed: int = 0, selection: str = "max_inliers",
                              engine: Optional[_native.Engine] = None):
    """Early termination (SURVEY.md §8(f) N4; the reference always runs ``max_iterations``): hypotheses are drawn
    by the device sampler and evaluated ``chunk`` at a time; after each chunk the standard RANSAC bound
    ``log(1 - confidence) / log(1 - w^8)`` is recomputed from the inlier ratio ``w`` of the best model so far and the
    run stops once that many hypotheses have been evaluated.  Because the sampler is keyed by the global hypothesis
    index, the result equals ``ransac_essential_arrays(..., sampler="device")`` over the same number of hypotheses.
    Returns (RansacResult, hypotheses evaluated)."""
    from .distributed import merge_best, pack_local_best

    eng = engine or _native.get_engine()
    n = np.asarray(pts_a).reshape(-1, 2).shape[0]
    best_row, best_res, done = None, None, 0
    needed = float(max_iterations)
    while done < max_iterations and done < needed:
        h = int(min(chunk, max_iterations - done))
        try:
            res = ransac_essential_arrays(camera_matrix, pts_a, pts_b, threshold, min_num_extra_inliers,
                                          error_aggregation_method, h, sampler="device", seed=seed, hyp_offset=done,
                                          on_degenerate="skip", selection=selection, engine=eng)
            row = pack_local_best(res.error, res.best_index, res.count_extra, res.E)
            rows = row[None] if best_row is None else np.stack([best_row, row])
            owner, *_ = merge_best(rows, selection)
            if best_row is None or owner == 1:
                best_row, best_res = row, res
        except ValueError:
            pass  # no candidate in this chunk
        done += h
        if best_res is not None:
            w = min(1.0, (8 + best_res.count_extra) / max(n, 1))
            miss = 1.0 - w ** 8
            needed = 0.0 if miss <= 0.0 else (np.log(1.0 - confidence) / np.log(miss) if miss < 1.0 else float(max_iterations))
    if best_res is None:
        raise ValueError(f"No model could be found with at least {(min_num_extra_inliers or 0) + 8} inliers.")
    return best_res, done


def eight_point_arrays(pts_a, pts_b, camera_matrix=None, engine=None) -> np.ndarray:
    """estimate_essential_mat / estimate_fundamental_mat on 8 gathered pairs ([8,2] arrays).

    lib/epipolar/eight_point.py:99-170; camera_matrix None = fundamental matrix (pixel coords).
    """
    pts_a = np.ascontiguousarray(pts_a, dtype=np.float64).reshape(-1, 2)
    pts_b = np.ascontiguousarray(pts_b, dtype=np.float64).reshape(-1, 2)
    if pts_a.shape[0] != 8 or pts_b.shape[0] != 8:
        raise ValueError("Exactly eight matches are needed")  # eight_point.py:151-152
    eng = engine or _native.get_engine()
    K = np.eye(3) if camera_matrix is None else camera_matrix
    eng.upload_pairs(pts_a, pts_b, K)
    eng.set_table(np.arange(8, dtype=np.int32).reshape(1, 8))
    E, valid, _ = eng.fit()
    if not valid[0]:
        raise _degenerate_sample_error(pts_a, pts_b, K)
    return E[0]


def sed_arrays(e, norm_a, norm_b, engine=None) -> np.ndarray:
    """calculate_symmetric_epipolar_distance (lib/epipolar/sed.py:7-30) for [n,2] arrays of
    K-normalised coordinates and one E."""
    eng = engine or _native.get_engine()
    na = np.ascontiguousarray(norm_a, dtype=np.float64).reshape(-1, 2)
    nb = np.ascontiguousarray(norm_b, dtype=np.float64).reshape(-1, 2)
    eng.upload_pairs(na, nb, np.eye(3))
    eng.set_models(np.asarray(e, dtype=np.float64).reshape(1, 9))
    eng.set_winner(0)
    _, sed = eng.inlier_mask(inf)
    return sed


@dataclasses.dataclass
class PoseResult:
    R: np.ndarray
    t: np.ndarray
    passing_indices: np.ndarray  # int64 indices of correspondences passing the chosen pose
    counts: np.ndarray           # votes per candidate (with the reference's index-0 quirk)
    candidates: list             # [(R, t)] * 4 in the reference's enumeration order
    singular_values: np.ndarray


def _check_decomposition(p):
    # lib/epipolar/eight_point.py:268-271 — np.isclose(0.0, s[-1]) with default tolerances
    if not np.isclose(0.0, p.sv[2]):
        raise EightPointCalculationError(
            "The smallest singular value of the Essential matrix is expected to be ~0")


def _svd_refuses(*arrays):
    """np.linalg.svd raises LinAlgError ("SVD did not converge") on a matrix with a NaN, which the device's SVDs would
    turn into NaN results instead.  A NaN anywhere in E, in P1 / P2 or in a coordinate reaches the reference's SVD input
    (eight_point.py:254, triangulation.py:34).  So does an infinite coordinate wherever the camera's third row has a
    zero entry (inf * 0 = NaN in the DLT row): P1 = [I|0] of the cheirality test and K[I|0] of triangulate_points always
    have one.  Against a third row without zeros the DLT row is infinite but NaN-free, and what numpy's SVD does with it
    depends on the LAPACK build (tests/golden/pose_nonfinite_fixture.json records one such case); an infinite coordinate
    is refused with LinAlgError there too, the reference's answer wherever it gives one.  An infinite entry of E or of a
    camera gives no NaN: the reference goes on (E: EightPointCalculationError from the check of U; a camera: non-finite
    points), and so does the device."""
    for a, coords in arrays:
        a = np.asarray(a, dtype=np.float64)
        if np.isnan(a).any() or (coords and not np.isfinite(a).all()):
            return np.linalg.LinAlgError("SVD did not converge")
    return None


def recover_all_r_t_arrays(e, engine=None):
    """_recover_all_r_t (lib/epipolar/eight_point.py:245-280) -> (R1, R2, t1)."""
    eng = engine or _native.get_engine()
    exc = _svd_refuses((e, False))
    if exc is not None:
        raise exc
    p = eng.decompose_essential(e)
    _check_decomposition(p)
    R = np.array(p.R, dtype=np.float64).reshape(4, 3, 3)
    t = np.array(p.t, dtype=np.float64).reshape(4, 3)
    return R[0], R[2], t[0]


def recover_pose_arrays(e, pts_a, pts_b, distance_threshold=None, engine=None, camera_matrix=None) -> PoseResult:
    """_recover_r_t (lib/epipolar/eight_point.py:181-242) on [m,2] arrays of K-normalised coordinates; with
    ``camera_matrix`` the arrays hold pixel coordinates and to_normalized_image_coords (eight_point.py:127-133) runs
    on the device first — recover_r_t_from_e (eight_point.py:65-96)."""
    if distance_threshold is None:
        distance_threshold = 50.0  # eight_point.py:469-470
    eng = engine or _native.get_engine()
    na = np.ascontiguousarray(pts_a, dtype=np.float64).reshape(-1, 2)
    nb = np.ascontiguousarray(pts_b, dtype=np.float64).reshape(-1, 2)
    exc = _svd_refuses((e, False), (na, True), (nb, True))
    if exc is not None:
        # the reference decomposes E before it triangulates a point (eight_point.py:207): its errors come first
        recover_all_r_t_arrays(e, engine=eng)
        raise exc
    p, pass4 = eng.recover_pose(e, na, nb, distance_threshold, camera_matrix=camera_matrix)
    _check_decomposition(p)
    counts = np.array(p.counts, dtype=np.int64)
    if 0 == np.count_nonzero(counts):
        raise EightPointCalculationError("None of the transformations pass the cheirality check.")
    R = np.array(p.R, dtype=np.float64).reshape(4, 3, 3)
    t = np.array(p.t, dtype=np.float64).reshape(4, 3)
    b = int(p.best)
    idx = np.nonzero((pass4 >> b) & 1)[0].astype(np.int64)
    return PoseResult(R=R[b].copy(), t=t[b].copy(), passing_indices=idx, counts=counts,
                      candidates=[(R[i], t[i]) for i in range(4)], singular_values=np.array(p.sv))


def triangulate_arrays(pts_a, pts_b, P1, P2, engine=None) -> np.ndarray:
    """triangulate_point_correspondence over arrays (lib/epipolar/triangulation.py:9-39)."""
    eng = engine or _native.get_engine()
    exc = _svd_refuses((np.asarray(P1)[:3], False), (np.asarray(P2)[:3], False), (pts_a, True), (pts_b, True))
    if exc is not None:
        raise exc
    return eng.triangulate(P1, P2, pts_a, pts_b)


def camera_matrices(intrinsic_camera_matrix, cam2_T_cam1_Tmat):
    """P1 = K[I|0], P2 = K[R|t] as lib/epipolar/triangulation.py:52-56 builds them."""
    K = np.asarray(intrinsic_camera_matrix, dtype=np.float64)
    if (3, 3) != K.shape:
        raise ValueError(f"Camera intrinsic matrix is not 3x3, actual shape: {K.shape}")
    K_ext = np.hstack((K, np.zeros((3, 1))))
    P1 = K_ext @ np.eye(4)
    P2 = K_ext @ (np.asarray(cam2_T_cam1_Tmat, dtype=np.float64) @ np.eye(4))
    return P1, P2


@dataclasses.dataclass
class TwoViewResult:
    ransac: RansacResult
    R: np.ndarray
    t: np.ndarray
    inlier_indices: np.ndarray   # ascending indices of the winner's inliers (samples included)
    passing: np.ndarray          # bool per inlier: passed the cheirality vote
    points: np.ndarray           # [m,3] triangulated points (NaN where not passing)
    counts: np.ndarray
    refinement: Optional[Refinement] = None  # with refine_iterations > 0: R, t and the inlier arrays are those of the
                                             # refined E; ``ransac`` is the RANSAC result, unchanged


def two_view_arrays(camera_matrix, pts_a, pts_b, threshold, min_num_extra_inliers=None,
                    error_aggregation_method=None, max_iterations=None, distance_threshold=None,
                    refine_iterations: int = 0, **kw) -> TwoViewResult:
    """The whole hot path of apps/sfm.py:110-186 in one call: RANSAC E -> cheirality vote ->
    triangulation of the passing inliers.  Correspondences are uploaded once; only results
    come back.  refine_iterations > 0 refines the winning E over its inliers (Levenberg-Marquardt on the essential
    manifold, at most that many iterations, on the device) before the vote; the pose, inliers and points then describe
    the refined E and ``refinement`` reports it."""
    refine_iterations = _refine_count(refine_iterations)
    if distance_threshold is None:
        distance_threshold = 50.0
    eng = kw.get("engine") or _native.get_engine()
    kw["engine"] = eng
    if (kw.get("sampler") == "device" and kw.get("on_degenerate", "raise") == "skip" and kw.get("hyp_offset", 0) == 0
            and np.asarray(pts_a).reshape(-1, 2).shape[0] >= 8 and (max_iterations or 100) > 0):
        # device sampler, degenerate samples skipped: nothing on the host depends on intermediate results, so the
        # whole estimate is enqueued in one go (un-synchronised upload included) and fetched once
        return _two_view_device(eng, camera_matrix, pts_a, pts_b, threshold, min_num_extra_inliers or 0,
                                _agg_name(error_aggregation_method), int(max_iterations or 100), float(distance_threshold),
                                int(kw.get("seed", 0)), kw.get("selection", "min_error"), refine_iterations)
    tail = {"distance_threshold": float(distance_threshold), "refine_iterations": refine_iterations}
    res = ransac_essential_arrays(camera_matrix, pts_a, pts_b, threshold, min_num_extra_inliers,
                                  error_aggregation_method, max_iterations, _tail=tail, **kw)
    p, num, idx, ok, X = tail["out"]
    _check_decomposition(p)
    counts = np.array(p.counts, dtype=np.int64)
    if 0 == np.count_nonzero(counts):
        raise EightPointCalculationError("None of the transformations pass the cheirality check.")
    b = int(p.best)
    R = np.array(p.R, dtype=np.float64).reshape(4, 3, 3)[b].copy()
    t = np.array(p.t, dtype=np.float64).reshape(4, 3)[b].copy()
    return TwoViewResult(ransac=res, R=R, t=t, inlier_indices=idx, passing=((ok >> b) & 1).astype(bool),
                         points=X, counts=counts, refinement=_refinement(eng) if refine_iterations else None)


@dataclasses.dataclass
class ImagePairResult:
    corners_a: np.ndarray        # [na,2] (x, y), descending cornerness
    corners_b: np.ndarray
    match_a: np.ndarray          # int64 indices into corners_a of the matches handed to RANSAC
    match_b: np.ndarray
    match_score: np.ndarray
    two_view: TwoViewResult      # indices inside it refer to the match arrays


def image_pair_arrays(image_a, image_b, camera_matrix, *, num_harris_corners: int = 600, ncc_window_size: int = 9,
                      ratio_test_threshold: float = 0.7, match_score_threshold: float = 0.3,
                      sed_inlier_threshold: float = 1.5e-6, min_num_extra_inliers=10, max_iterations: int = 2000,
                      error_aggregation_method="rms", sampler: str = "reference", seed: int = 0,
                      engine: Optional[_native.Engine] = None) -> ImagePairResult:
    """The whole of apps/sfm.py:64-186 on arrays, with the defaults of apps/config/config.yaml: Harris corners on
    both images -> brute-force NCC matching with ratio test + cross-check -> score filter (apps/sfm.py:280-296) ->
    RANSAC essential matrix -> cheirality vote -> triangulation.  No ``Feature`` / ``Match`` objects are built; with
    ``sampler="reference"`` the results equal those of the list-based pipeline (same global ``random`` stream)."""
    eng = engine or _native.get_engine()
    ca, _, _ = eng.harris_corners(image_a, num_harris_corners)
    cb, _, _ = eng.harris_corners(image_b, num_harris_corners)
    if len(ca) == 0 or len(cb) == 0:
        raise ValueError("Eight feature pairs are expected.")
    best_b, best_s, keep, _ = eng.match_brute_force(image_a, image_b, ca, cb, kind="ncc", window=ncc_window_size,
                                                    ratio_test=True, crosscheck=True, ratio_threshold=ratio_test_threshold)
    keep &= ~(best_s > match_score_threshold)
    ia = np.flatnonzero(keep)
    ib = best_b[ia].astype(np.int64)
    tv = two_view_arrays(camera_matrix, ca[ia], cb[ib], sed_inlier_threshold, min_num_extra_inliers,
                         error_aggregation_method, max_iterations, sampler=sampler, seed=seed, engine=eng)
    return ImagePairResult(corners_a=ca, corners_b=cb, match_a=ia, match_b=ib, match_score=best_s[ia], two_view=tv)


def _device_submit(eng, out, camera_matrix, pts_a, pts_b, threshold, min_extra, agg, max_iterations, distance_threshold,
                   seed, selection, refine_iterations=0):
    eng.upload_pairs(pts_a, pts_b, camera_matrix, sync=False)
    eng.sample_device(seed, max_iterations)
    return eng.two_view_async(threshold, float(min_extra), agg, selection, distance_threshold, out=out,
                              refine_iterations=refine_iterations)


def _device_result(eng, mask, sed, min_extra, copy: bool, refine_iterations=0) -> "TwoViewResult":
    best, p, num, idx, ok, X = eng.two_view_fetch()
    if best.index < 0:
        raise ValueError(f"No model could be found with at least {min_extra + 8} inliers.")
    _check_decomposition(p)
    counts = np.array(p.counts, dtype=np.int64)
    if 0 == np.count_nonzero(counts):
        raise EightPointCalculationError("None of the transformations pass the cheirality check.")
    # with refinement the tail's list is the refined model's: the RANSAC list is the mask plus the sample
    sample, inliers = _tail_inliers(best, _ransac_list(best, mask, 8) if refine_iterations else idx, 8)
    b = int(p.best)
    res = RansacResult(E=np.array(best.E, dtype=np.float64).reshape(3, 3), best_index=int(best.index),
                       error=float(best.err), count_extra=int(best.count_extra),
                       inlier_indices=inliers, mask=mask.astype(bool),
                       sed=sed.copy() if copy else sed, sample=sample, num_invalid=int(best.num_invalid),
                       first_invalid=int(best.first_invalid))
    R = np.array(p.R, dtype=np.float64).reshape(4, 3, 3)[b].copy()
    t = np.array(p.t, dtype=np.float64).reshape(4, 3)[b].copy()
    return TwoViewResult(ransac=res, R=R, t=t, inlier_indices=idx, passing=((ok >> b) & 1).astype(bool), points=X,
                         counts=counts, refinement=_refinement(eng) if refine_iterations else None)


def _two_view_device(eng, camera_matrix, pts_a, pts_b, threshold, min_extra, agg, max_iterations, distance_threshold, seed,
                     selection, refine_iterations=0):
    n = np.asarray(pts_a).reshape(-1, 2).shape[0]
    out = eng.pinned_out(n)  # engine-owned pinned landing buffers: page-locking per call would dominate the transfers
    mask, sed = _device_submit(eng, out, camera_matrix, pts_a, pts_b, threshold, min_extra, agg, max_iterations,
                               distance_threshold, seed, selection, refine_iterations)
    return _device_result(eng, mask, sed, min_extra, copy=True, refine_iterations=refine_iterations)


class TwoViewStream:
    """Back-to-back estimates from HOST buffers with the transfers of one estimate hidden behind the kernels of
    another: ``depth`` contexts on the same GPU (each its own stream); ``submit`` only ENQUEUES the upload of the
    correspondences, the device sampler, fit, score, selection and tail on the next context and returns a ticket;
    ``result`` synchronises that context and builds the ``TwoViewResult``.  While context A scores estimate s, the copy
    engine moves the correspondences of estimate s+1 and the host unpacks estimate s-1.  Device sampler only (the
    reference sampler is a sequential host computation); results are identical to ``two_view_arrays(...,
    sampler="device")``."""

    def __init__(self, depth: int = 2, device: Optional[int] = None):
        dev = _native.default_device() if device is None else int(device)
        self.engines = [_native.Engine(dev) for _ in range(depth)]
        self._next = 0
        self._pending = {}

    def set_score_variant(self, *a, **k):
        for e in self.engines:
            e.set_score_variant(*a, **k)

    def submit(self, camera_matrix, pts_a, pts_b, threshold, min_num_extra_inliers=0, error_aggregation_method="rms",
               max_iterations: int = 100, distance_threshold: float = 50.0, seed: int = 0, selection: str = "min_error"):
        k = self._next
        eng = self.engines[k % len(self.engines)]
        if any(t % len(self.engines) == k % len(self.engines) for t in self._pending):
            raise RuntimeError("fetch the estimate submitted to this context before submitting another one")
        self._next += 1
        n = np.asarray(pts_a).reshape(-1, 2).shape[0]
        mask, sed = _device_submit(eng, eng.pinned_out(n), camera_matrix, pts_a, pts_b, threshold, min_num_extra_inliers or 0,
                                   _agg_name(error_aggregation_method), int(max_iterations), float(distance_threshold),
                                   seed, selection)
        self._pending[k] = (eng, mask, sed, min_num_extra_inliers or 0)
        return k

    def result(self, ticket) -> TwoViewResult:
        eng, mask, sed, min_extra = self._pending.pop(ticket)
        return _device_result(eng, mask, sed, min_extra, copy=True)

    def close(self):
        for e in self.engines:
            e.close()
