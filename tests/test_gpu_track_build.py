"""sfm_build_tracks on the GPU: every output bit-equal to the oracle (oracle/track_build.py, scipy's connected
components) on random graphs, match graphs, empty cases, a 10^6-feature chain, a 10^5-edge star and the 64 / 65-view
limit; invariance under edge order, direction, duplication and grouping; the refusals; the truth; and the incremental
loop from matches to bundle adjustment."""
from __future__ import annotations

import ctypes as C
import random

import numpy as np
import pytest

from oracle import track_build as otb
from structure_from_motion_b200 import _native
from structure_from_motion_b200.multiview import build_tracks_arrays, bundle_adjust_arrays, triangulate_tracks_arrays
from structure_from_motion_b200.pnp import ransac_pnp_arrays
from structure_from_motion_b200.scenes import make_match_graph
from structure_from_motion_b200.two_view import two_view_arrays

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]

KEYS = ("offsets", "status", "view", "feature", "track")


@pytest.fixture(scope="module")
def eng():
    return _native.get_engine(0)


def _csr(features_n, pairs, matches):
    fo = np.zeros(len(features_n) + 1, dtype=np.int64)
    np.cumsum(features_n, out=fo[1:])
    mo = np.zeros(len(matches) + 1, dtype=np.int64)
    np.cumsum([len(m) for m in matches], out=mo[1:])
    pv = np.asarray(pairs, dtype=np.int32).reshape(-1, 2)
    m = np.concatenate([np.asarray(x).reshape(-1, 2) for x in matches]).astype(np.int32) if matches else \
        np.zeros((0, 2), dtype=np.int32)
    return fo, pv, mo, m


def _check(eng, fo, pv, mo, m):
    got = dict(zip(KEYS, eng.build_tracks(fo, pv, mo, m)))
    ref = otb.build_tracks(fo, pv, mo, m)
    for k in KEYS:
        assert got[k].dtype == ref[k].dtype, k
        assert np.array_equal(got[k], ref[k]), k
    return got


def _random_case(seed):
    rng = np.random.default_rng(seed)
    V = int(rng.choice([1, 2, 3, 5, 16, 70, 300]))
    nmax = int(rng.choice([0, 1, 3, 40, 2000]))
    n = rng.integers(0, nmax + 1, V)
    nz = np.flatnonzero(n > 0)
    pairs, matches = [], []
    if len(nz) >= 2:
        for _ in range(int(rng.integers(0, 3 * V + 2))):
            a, b = rng.choice(nz, 2, replace=False)
            k = int(rng.choice([0, 1, 5, 100, 3000]))
            pairs.append((a, b))
            matches.append(np.column_stack([rng.integers(0, n[a], k), rng.integers(0, n[b], k)]))
    return _csr(n, pairs, matches)


# ---- against the oracle ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(40))
def test_random_graphs(eng, seed):
    _check(eng, *_random_case(seed))


@pytest.mark.parametrize("wrong", [0.0, 0.02])
def test_match_graph(eng, wrong):
    g = make_match_graph(30000, 16, 3, span=3, wrong_frac=wrong, distractor_frac=0.25)
    got = _check(eng, *_csr([len(f) for f in g.features], g.pairs, g.matches))
    if wrong:
        assert (got["status"] == otb.CONFLICT).any()


def test_empty_cases(eng):
    # no pairs
    got = _check(eng, *_csr([5, 3], [], []))
    assert len(got["offsets"]) == 1 and (got["track"] == -1).all()
    # pairs without matches
    _check(eng, *_csr([5, 3, 4], [(0, 1), (2, 1)], [np.zeros((0, 2)), np.zeros((0, 2))]))
    # views without features, between and around matched ones
    _check(eng, *_csr([0, 4, 0, 0, 3, 0], [(1, 4), (4, 1)], [[(0, 0), (3, 2)], [(1, 1)]]))
    # no features at all
    got = _check(eng, *_csr([0, 0, 0], [], []))
    assert len(got["track"]) == 0
    # a single view with features and nothing else
    _check(eng, *_csr([7], [], []))


def _chain(n, order, rng):
    k = np.arange(n - 1)
    i = np.where(k % 2 == 0, k // 2, (k + 1) // 2)  # feature k is local k // 2 of view k % 2
    j = np.where(k % 2 == 0, k // 2, (k - 1) // 2)
    m = np.column_stack([i, j])
    if order == "reverse":
        m = m[::-1]
    elif order == "random":
        m = m[rng.permutation(len(m))]
    return _csr([(n + 1) // 2, n // 2], [(0, 1)], [m])


@pytest.mark.parametrize("order", ["forward", "reverse", "random"])
def test_chain_of_a_million(eng, order):
    got = _check(eng, *_chain(1_000_000, order, np.random.default_rng(0)))
    assert list(got["offsets"]) == [0, 1_000_000] and list(got["status"]) == [otb.CONFLICT]


@pytest.mark.parametrize("centre", ["lowest id", "highest id"])
def test_star(eng, centre):
    n = 100_000
    if centre == "lowest id":  # view 0's single feature against every feature of view 1
        case = _csr([1, n], [(0, 1)], [np.column_stack([np.zeros(n, dtype=int), np.arange(n)])])
    else:  # every feature of view 0 against view 1's single feature, the largest id: every hook CASes one root
        case = _csr([n, 1], [(1, 0)], [np.column_stack([np.zeros(n, dtype=int), np.arange(n)])])
    got = _check(eng, *case)
    assert list(got["offsets"]) == [0, n + 1]


@pytest.mark.parametrize("views,status", [(64, otb.OK), (65, otb.LONG)])
def test_track_length_limit(eng, views, status):
    rng = np.random.default_rng(views)
    n = rng.integers(1, 6, views)
    loc = [int(rng.integers(0, k)) for k in n]
    pairs = [(v + 1, v) for v in range(views - 1)]
    got = _check(eng, *_csr(n, pairs, [[(loc[v + 1], loc[v])] for v in range(views - 1)]))
    assert list(got["status"]) == [status] and got["offsets"][-1] == views


# ---- independence ----------------------------------------------------------------------------------------------------
def test_independence(eng):
    g = make_match_graph(20000, 12, 8, span=2, wrong_frac=0.03, distractor_frac=0.25)
    n = [len(f) for f in g.features]
    base = eng.build_tracks(*_csr(n, g.pairs, g.matches))
    rng = np.random.default_rng(2)
    pairs = [tuple(p) for p in g.pairs]
    # every match of all pairs in one random order, each its own pair entry, half of them reversed, some twice
    entries = [(a, b, m) for (a, b), ms in zip(pairs, g.matches) for m in ms]
    variants = {}
    perm = rng.permutation(len(entries))
    variants["permuted singletons"] = ([entries[i][:2] for i in perm], [[entries[i][2]] for i in perm])
    flip = rng.uniform(size=len(entries)) < 0.5
    variants["directions swapped"] = ([(b, a) if f else (a, b) for (a, b, _), f in zip(entries, flip)],
                                      [[m[::-1]] if f else [m] for (_, _, m), f in zip(entries, flip)])
    dup = [ms[np.sort(np.concatenate([np.arange(len(ms)), rng.integers(0, max(len(ms), 1), len(ms) // 3)]))]
           if len(ms) else ms for ms in g.matches]
    variants["duplicated"] = (pairs, dup)
    regroup_p, regroup_m = [], []
    for p, ms in zip(pairs, g.matches):  # each pair split into up to three entries, in reverse order
        for part in np.array_split(ms[rng.permutation(len(ms))], 3)[::-1]:
            regroup_p.append(p)
            regroup_m.append(part)
    variants["regrouped"] = (regroup_p, regroup_m)
    for name, (pp, mm) in variants.items():
        got = eng.build_tracks(*_csr(n, pp, mm))
        for a, b, k in zip(base, got, KEYS):
            assert np.array_equal(a, b), (name, k)
    again = eng.build_tracks(*_csr(n, g.pairs, g.matches))
    fresh = _native.Engine(0)
    try:
        other = fresh.build_tracks(*_csr(n, g.pairs, g.matches))
    finally:
        fresh.close()
    for a, b, c, k in zip(base, again, other, KEYS):
        assert np.array_equal(a, b) and np.array_equal(a, c), k


# ---- refusals --------------------------------------------------------------------------------------------------------
def _raw(eng, V, fo, P, pv, mo, m):
    p = lambda a: None if a is None else np.ascontiguousarray(a).ctypes.data_as(C.c_void_p)  # noqa: E731
    keep = [None if a is None else np.ascontiguousarray(a) for a in (fo, pv, mo, m)]
    fo, pv, mo, m = keep
    return eng.lib.sfm_build_tracks(eng.h, int(V), p(fo), int(P), p(pv), p(mo), p(m), None, None, None, None, None, None,
                                    None)


def test_refusals(eng):
    fo = np.array([0, 3, 5], dtype=np.int64)
    pv = np.array([[0, 1]], dtype=np.int32)
    mo = np.array([0, 2], dtype=np.int64)
    m = np.array([[0, 0], [2, 1]], dtype=np.int32)
    assert _raw(eng, 2, fo, 1, pv, mo, m) == 0
    bad = {
        "V < 1": (0, fo, 1, pv, mo, m),
        "feature_offsets[0] != 0": (2, np.array([1, 3, 5]), 1, pv, mo, m),
        "feature_offsets decrease": (2, np.array([0, 3, 2]), 1, pv, mo, m),
        "N > INT32_MAX": (2, np.array([0, 1, 2 ** 31]), 1, pv, mo, m),
        "match_offsets[0] != 0": (2, fo, 1, pv, np.array([1, 2]), m),
        "match_offsets decrease": (2, fo, 2, np.array([[0, 1], [1, 0]], dtype=np.int32), np.array([0, 2, 1]), m),
        "a == b": (2, fo, 1, np.array([[1, 1]], dtype=np.int32), mo, m),
        "view < 0": (2, fo, 1, np.array([[-1, 1]], dtype=np.int32), mo, m),
        "view >= V": (2, fo, 1, np.array([[0, 2]], dtype=np.int32), mo, m),
        "local index >= n_a": (2, fo, 1, pv, mo, np.array([[3, 0], [0, 0]], dtype=np.int32)),
        "local index >= n_b": (2, fo, 1, pv, mo, np.array([[0, 0], [0, 2]], dtype=np.int32)),
        "local index < 0": (2, fo, 1, pv, mo, np.array([[0, -1], [0, 0]], dtype=np.int32)),
        "P < 0": (2, fo, -1, pv, mo, m),
        "null feature_offsets": (2, None, 1, pv, mo, m),
        "null pair_views": (2, fo, 1, None, mo, m),
        "null match_offsets": (2, fo, 1, pv, None, m),
        "null matches": (2, fo, 1, pv, mo, None),
    }
    for name, args in bad.items():
        assert _raw(eng, *args) == -1, name
    # after the refusals the context still works
    _check(eng, fo, pv, mo, m)


# ---- the truth -------------------------------------------------------------------------------------------------------
def test_ok_tracks_are_the_truth(eng):
    g = make_match_graph(50000, 20, 4, span=2, wrong_frac=0.0, distractor_frac=0.25)
    ts = build_tracks_arrays(g.features, g.pairs, g.matches, engine=eng)
    assert (ts.status == "ok").all()
    ok = ts.ok()
    local = ok.feature - ok.feature_offsets[ok.view]
    got = {frozenset(zip(ok.view[s:e].tolist(), local[s:e].tolist())) for s, e in zip(ok.offsets[:-1], ok.offsets[1:])}
    truth = {}
    for v, p in enumerate(g.point):
        for i in np.flatnonzero(p >= 0):
            truth.setdefault(int(p[i]), set()).add((v, int(i)))
    assert got == {frozenset(s) for s in truth.values() if len(s) >= 2}
    pix = np.concatenate(g.features)[ok.feature]
    assert np.array_equal(ok.x, pix)


# ---- end to end ------------------------------------------------------------------------------------------------------
def test_incremental_loop_from_matches(eng):
    """Eight views of make_match_graph with 2 % wrong matches: the ok tracks; two_view_arrays on views 0-1; each further
    view registered by ransac_pnp_arrays against the points of its tracks, and the tracks re-triangulated over the
    registered views; then every view and point bundle-adjusted (view 0 fixed, view 1 anchored).  Rotation errors
    against the truth in camera-0 coordinates.  First run on one B200: 3116 ok tracks, 3114 points; the largest R error
    over views 1-7 is 2.17e-3 before the bundle adjustment and 7.1e-4 after (6 iterations, converged); the bounds are
    about 3x those."""
    V = 8
    g = make_match_graph(4000, V, 21, span=2, wrong_frac=0.02, distractor_frac=0.25)
    ok = build_tracks_arrays(g.features, g.pairs, g.matches, engine=eng).ok()
    T = len(ok.offsets) - 1
    tix = np.repeat(np.arange(T), np.diff(ok.offsets))
    dense = np.full((T, V, 2), np.nan)
    seen = np.zeros((T, V), dtype=bool)
    dense[tix, ok.view] = ok.x
    seen[tix, ok.view] = True
    K = g.K
    Rr = np.array([g.R[c] @ g.R[0].T for c in range(V)])
    both = np.flatnonzero(seen[:, 0] & seen[:, 1])
    random.seed(1)
    tv = two_view_arrays(K, dense[both, 0], dense[both, 1], 1e-5, 100, "rms", 300, engine=eng, refine_iterations=20)
    X = np.full((T, 3), np.nan)
    X[both[tv.inlier_indices[tv.passing]]] = tv.points[tv.passing]
    Rs, ts = [np.eye(3), tv.R], [np.zeros(3), tv.t]
    for c in range(2, V):
        have = np.flatnonzero(np.isfinite(X[:, 0]) & seen[:, c])
        random.seed(c)
        p = ransac_pnp_arrays(K, X[have], dense[have, c], 4.0, 10, "rms", 300, engine=eng, refine_iterations=20)
        Rs.append(p.refinement.R)
        ts.append(p.refinement.t)
        reg = seen[:, :c + 1]
        sel = np.flatnonzero(reg.sum(axis=1) >= 2)
        off = np.zeros(len(sel) + 1, dtype=np.int64)
        np.cumsum(reg[sel].sum(axis=1), out=off[1:])
        rows, cols = np.nonzero(reg[sel])
        res = triangulate_tracks_arrays(K, np.stack(Rs), np.stack(ts), off, cols.astype(np.int32),
                                        dense[sel[rows], cols], 4.0, refine_iterations=10, engine=eng)
        X = np.full((T, 3), np.nan)
        X[sel[res.status == "ok"]] = res.points[res.status == "ok"]
    Ra, ta = np.stack(Rs), np.stack(ts)
    ba = bundle_adjust_arrays(K, Ra, ta, X, ok.offsets, ok.view, ok.x, 4.0, fixed=(0,), scale_view=1, max_iterations=50,
                              engine=eng)
    before = max(np.abs(Ra[c] - Rr[c]).max() for c in range(1, V))
    after = max(np.abs(ba.R[c] - Rr[c]).max() for c in range(1, V))
    print(f"eight views from matches: {T} ok tracks, {int(np.isfinite(X[:, 0]).sum())} points; bundle "
          f"{ba.report.num_points} points, {ba.report.num_observations} observations, {ba.report.iterations} iterations "
          f"({ba.report.status}); largest R error over views 1-7 {before:.3g} -> {after:.3g}; cost "
          f"{ba.report.cost_start:.6g} -> {ba.report.cost_final:.6g}")
    assert ba.report.cost_final < ba.report.cost_start
    assert before < 6.5e-3
    assert after < 2.1e-3
