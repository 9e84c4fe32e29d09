"""Multi-view triangulation of tracks on arrays: one 3-D point per track from its observations in registered views.

A track is one 3-D point observed in some subset of the registered views: observations (view index, pixel) in CSR form,
``offsets`` int64[T+1], ``view`` int32[M] and ``x`` float64[M,2].  Per track, every pair of observations is
triangulated (two-view DLT) and scored by the PnP reprojection decision over the whole track; the best pair's passing
observations give the N-view DLT point, optionally refined by Levenberg-Marquardt on the reprojection error.  A track
is usable when its status is "ok": at least ``min_views`` inliers and rays that meet at ``min_angle_deg`` or more.
``bundle_adjust_arrays`` then refines the free poses and the points jointly (Levenberg-Marquardt on the reprojection
error, the points eliminated by a Schur complement).  ``build_tracks_arrays`` makes the tracks from pairwise feature
matches (the connected components of the match graph).  The semantics are pinned in include/sfm_b200.h
(sfm_build_tracks, sfm_triangulate_tracks, sfm_bundle_adjust), csrc/sfm_track_build.cuh, csrc/sfm_tracks.cuh and
csrc/sfm_bundle.cuh.  Everything numeric runs in libsfm_b200.so; there is no CPU fallback.
"""
from __future__ import annotations

import dataclasses
from typing import Optional

import numpy as np

from . import _native


@dataclasses.dataclass
class TrackRefinement:
    cost_start: np.ndarray        # float64[T] summed squared reprojection error (px^2) at the linear point, over the list
    cost_final: np.ndarray        # float64[T] the same at the reported point, <= cost_start
    num: np.ndarray               # int32[T] observations in the list (those passing under the linear point)
    iterations: np.ndarray        # int32[T] proposals evaluated
    status: np.ndarray            # str[T] converged, max_iterations, stalled, no_model (short / no_pair) or nonfinite
    rejected: np.ndarray          # int32[T] of those, proposals rejected


@dataclasses.dataclass
class TracksResult:
    points: np.ndarray            # float64[T,3] world points; NaN for "short" and "no_pair" tracks
    status: np.ndarray            # str[T] ok, short, no_pair, few_inliers or small_angle
    num_inliers: np.ndarray       # int32[T] passing observations under the reported point
    angle: np.ndarray             # float64[T] largest angle (radians) between the rays of two passing observations
    mask: np.ndarray              # bool[M] decision of every observation under its track's point
    err: np.ndarray               # float64[M] squared reprojection error (px^2) under its track's point
    refinement: Optional[TrackRefinement] = None  # refine_iterations > 0


def tracks_from_dense(visible, pixels):
    """CSR tracks for the layout "point i seen in the views where visible[i, c]": visible bool[N,V], pixels
    float64[N,V,2] (read where visible).  Observations are in view order.  Returns (offsets int64[N+1], view int32[M],
    x float64[M,2])."""
    visible = np.asarray(visible, dtype=bool)
    pixels = np.asarray(pixels, dtype=np.float64)
    if visible.ndim != 2 or pixels.shape != visible.shape + (2,):
        raise ValueError(f"expected visible [N,V] and pixels [N,V,2], got {visible.shape} and {pixels.shape}")
    pt, view = np.nonzero(visible)  # row-major: by point, then by view
    offsets = np.zeros(visible.shape[0] + 1, dtype=np.int64)
    np.cumsum(visible.sum(axis=1), out=offsets[1:])
    return offsets, view.astype(np.int32), np.ascontiguousarray(pixels[pt, view])


@dataclasses.dataclass
class TrackSet:
    feature_offsets: np.ndarray   # int64[V+1]: view v owns the global feature ids [feature_offsets[v], feature_offsets[v+1])
    offsets: np.ndarray           # int64[T+1] track CSR
    view: np.ndarray              # int32[M] view of every observation
    feature: np.ndarray           # int32[M] its global feature id; the local index is feature - feature_offsets[view]
    x: np.ndarray                 # float64[M,2] its pixel
    status: np.ndarray            # str[T] ok, conflict (a view holds two of its features) or long (more than 64)
    track: np.ndarray             # int32[N] the track of every feature, -1 for a feature in no track

    def ok(self) -> "TrackSet":
        """The "ok" tracks only, renumbered in order; ``track`` maps the features of every other track to -1."""
        keep = self.status == "ok"
        n = np.diff(self.offsets)
        obs = np.repeat(keep, n)
        offsets = np.zeros(int(keep.sum()) + 1, dtype=np.int64)
        np.cumsum(n[keep], out=offsets[1:])
        renum = (np.cumsum(keep) - 1).astype(np.int32)
        tr = self.track
        inside = tr >= 0
        track = np.full_like(tr, -1)
        track[inside] = np.where(keep[tr[inside]], renum[tr[inside]], -1)
        return TrackSet(feature_offsets=self.feature_offsets, offsets=offsets, view=self.view[obs],
                        feature=self.feature[obs], x=self.x[obs], status=self.status[keep], track=track)


def build_tracks_arrays(features, pairs, matches, engine: Optional[_native.Engine] = None) -> TrackSet:
    """Tracks from pairwise feature matches: the connected components of the match graph with two or more features.

    features: a list of V float64[n_v,2] pixel arrays (only their lengths and, for ``x``, their pixels are used).
    pairs: int[P,2] view pairs (a, b), a != b.  matches: a list of P int[E_p,2] arrays of local indices (i in a, j in b).
    A pair may repeat, in either order, and so may matches.  For one pair matched by ``sfm_match_brute_force``
    (``Engine.match_brute_force``), optionally filtered by a RANSAC inlier mask ``inl`` over the kept matches::

        i = np.flatnonzero(keep)
        m = np.column_stack([i, best_b[keep]])      # or m[inl]

    Tracks are ordered by their smallest global feature id, and observations run by view, then by local index.  A
    track whose features include two of one view is "conflict" (reported whole); otherwise one of more than 64
    observations is "long"; the rest are "ok".  ``TrackSet.ok()`` keeps the ok tracks, ready for
    ``triangulate_tracks_arrays`` and ``bundle_adjust_arrays``.
    """
    feats = [np.asarray(f, dtype=np.float64).reshape(-1, 2) for f in features]
    if not feats:
        raise ValueError("at least one view is needed")
    fo = np.zeros(len(feats) + 1, dtype=np.int64)
    np.cumsum([len(f) for f in feats], out=fo[1:])
    pv = np.asarray(pairs, dtype=np.int64).reshape(-1, 2)
    if len(matches) != len(pv):
        raise ValueError(f"{len(pv)} pairs but {len(matches)} match arrays")
    ms = [np.asarray(m, dtype=np.int64).reshape(-1, 2) for m in matches]
    mo = np.zeros(len(ms) + 1, dtype=np.int64)
    np.cumsum([len(m) for m in ms], out=mo[1:])
    for name, a in (("pairs", pv), ("matches", np.concatenate(ms) if ms else pv)):
        if a.size and (a.min() < np.iinfo(np.int32).min or a.max() > np.iinfo(np.int32).max):
            raise ValueError(f"{name} do not fit int32")
    m = np.concatenate(ms).astype(np.int32) if ms else np.zeros((0, 2), dtype=np.int32)
    eng = engine or _native.get_engine()
    offsets, status, view, feature, track = eng.build_tracks(fo, pv.astype(np.int32), mo, m)
    allx = np.concatenate(feats) if fo[-1] else np.zeros((0, 2))
    names = np.array([_native.BUILT_TRACK_STATUS[s] for s in range(len(_native.BUILT_TRACK_STATUS))])
    return TrackSet(feature_offsets=fo, offsets=offsets, view=view, feature=feature,
                    x=np.ascontiguousarray(allx[feature]), status=names[status], track=track)


def triangulate_tracks_arrays(K, R, t, offsets, view, x, threshold: float, min_angle_deg: float = 1.5,
                              min_views: int = 2, refine_iterations: int = 0,
                              engine: Optional[_native.Engine] = None) -> TracksResult:
    """Triangulate T tracks seen in V registered views.

    K: one (3,3) camera for every view or (V,3,3), upper triangular with K[2,2] = 1.  R (V,3,3), t (V,3): world to
    camera, x_cam = R X + t (the ``ransac_pnp_arrays`` convention).  offsets int64[T+1], view int32[M], x float64[M,2]
    pixels.  threshold: on the squared reprojection error in px^2, finite.  A track has at most 64 observations.
    refine_iterations > 0 refines each point over the observations passing under its linear point.
    """
    R = np.asarray(R, dtype=np.float64)
    t = np.asarray(t, dtype=np.float64)
    if R.ndim != 3 or R.shape[1:] != (3, 3) or t.shape != (R.shape[0], 3):
        raise ValueError(f"expected R (V,3,3) and t (V,3), got {R.shape} and {t.shape}")
    V = R.shape[0]
    K = np.asarray(K, dtype=np.float64)
    if K.shape == (3, 3):
        K = np.broadcast_to(K, (V, 3, 3))
    if K.shape != (V, 3, 3):
        raise ValueError(f"expected K (3,3) or ({V},3,3), got {K.shape}")
    refine_iterations = int(refine_iterations)
    if refine_iterations < 0:
        raise ValueError(f"refine_iterations must be >= 0, got {refine_iterations}")
    Rt = np.concatenate([R, t[:, :, None]], axis=2)
    eng = engine or _native.get_engine()
    X, status, num, angle, mask, err, rep = eng.triangulate_tracks(K, Rt, offsets, view, x, threshold, min_angle_deg,
                                                                  min_views, refine_iterations)
    names = np.array([_native.TRACK_STATUS[s] for s in range(len(_native.TRACK_STATUS))])
    result = TracksResult(points=X, status=names[status], num_inliers=num, angle=angle, mask=mask, err=err)
    if rep is not None:
        r = np.ctypeslib.as_array(rep)
        rnames = np.array([_native.REFINE_STATUS[s] for s in range(len(_native.REFINE_STATUS))])
        result.refinement = TrackRefinement(
            cost_start=r["cost_start"].copy(), cost_final=r["cost_final"].copy(), num=r["num"].copy(),
            iterations=r["iterations"].copy(), status=rnames[r["status"]], rejected=r["rejected"].copy())
    return result


@dataclasses.dataclass
class BundleReport:
    cost_start: float             # summed squared reprojection error (px^2) over the list at the (projected) start
    cost_final: float             # the same at the reported parameters, <= cost_start
    num_observations: int         # observations in the list
    num_points: int               # parameter points (finite start, at least 2 list observations)
    num_free_views: int
    iterations: int               # proposals evaluated
    status: str                   # converged, max_iterations, stalled or nonfinite
    rejected: int                 # of those, proposals rejected


@dataclasses.dataclass
class BundleResult:
    R: np.ndarray                 # float64[V,3,3] world to camera
    t: np.ndarray                 # float64[V,3]
    points: np.ndarray            # float64[T,3]; non-parameter tracks exactly as given
    mask: np.ndarray              # bool[M] decision of every observation under the reported parameters
    err: np.ndarray               # float64[M] squared reprojection error (px^2) under them
    report: BundleReport


def bundle_adjust_arrays(K, R, t, X, offsets, view, x, threshold: float, fixed=(0,), scale_view=None,
                         max_iterations: int = 50, engine: Optional[_native.Engine] = None) -> BundleResult:
    """Refine V registered views and the points of T tracks jointly.

    K: one (3,3) camera or (V,3,3), upper triangular with K[2,2] = 1.  R (V,3,3), t (V,3): the start, x_cam = R X + t.
    X (T,3): the start points; a track with a non-finite X (a non-ok track of ``triangulate_tracks_arrays`` set to
    NaN) is left as it is.  offsets, view, x: the tracks as for ``triangulate_tracks_arrays``.  The observations
    passing the reprojection rule at ``threshold`` (px^2) under the start form the fixed list.  ``fixed``: the indices
    of the views held constant (at least one).  ``scale_view``: a free view whose largest translation component is
    held constant; None picks the lowest-index free view when exactly one view is fixed, and none otherwise.
    """
    R = np.asarray(R, dtype=np.float64)
    t = np.asarray(t, dtype=np.float64)
    if R.ndim != 3 or R.shape[1:] != (3, 3) or t.shape != (R.shape[0], 3):
        raise ValueError(f"expected R (V,3,3) and t (V,3), got {R.shape} and {t.shape}")
    V = R.shape[0]
    K = np.asarray(K, dtype=np.float64)
    if K.shape == (3, 3):
        K = np.broadcast_to(K, (V, 3, 3))
    if K.shape != (V, 3, 3):
        raise ValueError(f"expected K (3,3) or ({V},3,3), got {K.shape}")
    fixed_mask = np.zeros(V, dtype=bool)
    idx = np.asarray(fixed, dtype=np.int64).reshape(-1)
    if idx.size and (idx.min() < 0 or idx.max() >= V):
        raise ValueError(f"fixed view index outside [0, {V})")
    fixed_mask[idx] = True
    if scale_view is None:
        free = np.flatnonzero(~fixed_mask)
        scale_view = int(free[0]) if fixed_mask.sum() == 1 and free.size else -1
    Rt = np.concatenate([R, t[:, :, None]], axis=2)
    eng = engine or _native.get_engine()
    Rt_out, X_out, rep, mask, err = eng.bundle_adjust(K, Rt, fixed_mask, int(scale_view), offsets, view, x, X,
                                                      threshold, int(max_iterations))
    report = BundleReport(cost_start=rep.cost_start, cost_final=rep.cost_final, num_observations=rep.num_observations,
                          num_points=rep.num_points, num_free_views=rep.num_free_views, iterations=rep.iterations,
                          status=_native.REFINE_STATUS[rep.status], rejected=rep.rejected)
    return BundleResult(R=np.ascontiguousarray(Rt_out[:, :, :3]), t=np.ascontiguousarray(Rt_out[:, :, 3]), points=X_out,
                        mask=mask, err=err, report=report)
