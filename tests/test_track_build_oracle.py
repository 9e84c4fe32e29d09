"""The track-building oracle (oracle/track_build.py, scipy's connected components) against a pure-Python union-find
and a hand-worked example; the host build of the kernels' union-find (tools/track_build_check.cu) against the oracle;
the invariants of scenes.make_match_graph; TrackSet.ok() on hand-made data.  No GPU."""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import track_build as tb
from structure_from_motion_b200.multiview import TrackSet
from structure_from_motion_b200.scenes import make_match_graph

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _random_graph(rng, V, nmax, E):
    n = rng.integers(0, nmax + 1, V)
    fo = np.zeros(V + 1, dtype=np.int64)
    np.cumsum(n, out=fo[1:])
    pairs, matches = [], []
    nonempty = np.flatnonzero(n > 0)
    for _ in range(int(rng.integers(0, 2 * V + 1))):
        if len(nonempty) < 2:
            break
        a, b = rng.choice(nonempty, 2, replace=False)
        k = int(rng.integers(0, E + 1))
        pairs.append((a, b))
        matches.append(np.column_stack([rng.integers(0, n[a], k), rng.integers(0, n[b], k)]))
    mo = np.zeros(len(pairs) + 1, dtype=np.int64)
    np.cumsum([len(m) for m in matches], out=mo[1:])
    pv = np.array(pairs, dtype=np.int32).reshape(-1, 2)
    m = np.concatenate(matches).astype(np.int32) if matches else np.zeros((0, 2), dtype=np.int32)
    return fo, pv, mo, m


def _python_union_find(fo, pv, mo, m):
    N = int(fo[-1])
    parent = list(range(N))

    def find(x):
        while parent[x] != x:
            x = parent[x]
        return x

    for u, v in tb.global_edges(fo, pv, mo, m):
        ru, rv = find(int(u)), find(int(v))
        if ru != rv:
            parent[max(ru, rv)] = min(ru, rv)
    comps = {}
    for g in range(N):
        comps.setdefault(find(g), []).append(g)
    tracks = sorted((sorted(c) for c in comps.values() if len(c) >= 2), key=lambda c: c[0])
    view_of = lambda g: int(np.searchsorted(fo, g, side="right") - 1)  # noqa: E731
    status = []
    for c in tracks:
        views = [view_of(g) for g in c]
        status.append(tb.CONFLICT if len(set(views)) < len(views) else tb.LONG if len(c) > 64 else tb.OK)
    return tracks, status


@pytest.mark.parametrize("seed", range(40))
def test_oracle_against_python_union_find(seed):
    rng = np.random.default_rng(seed)
    fo, pv, mo, m = _random_graph(rng, int(rng.integers(1, 9)), int(rng.integers(0, 30)), int(rng.integers(0, 25)))
    got = tb.build_tracks(fo, pv, mo, m)
    tracks, status = _python_union_find(fo, pv, mo, m)
    assert [list(got["feature"][s:e]) for s, e in zip(got["offsets"][:-1], got["offsets"][1:])] == tracks
    assert list(got["status"]) == status
    assert np.array_equal(got["view"], np.searchsorted(fo, got["feature"], side="right") - 1)
    for t, c in enumerate(tracks):
        assert (got["track"][c] == t).all()
    assert (got["track"] >= 0).sum() == sum(len(c) for c in tracks)


def test_hand_worked_example():
    """Views 0-2 with 3, 2, 2 features (global ids 0-2 | 3-4 | 5-6), and a 65-view chain after them.  Edges {0, 3},
    {3, 5}: a clean track.  {1, 4}, {4, 2}: features 1 and 2 of view 0 in one component, a conflict.  Feature 6 and 0..
    nothing: 6 is alone and in no track.  The chain joins one feature of each of 65 more views: long."""
    fo = np.array([0, 3, 5, 7] + [7 + k + 1 for k in range(65)], dtype=np.int64)
    pv = [(0, 1), (2, 1), (1, 0)] + [(3 + k, 4 + k) for k in range(64)]
    ms = [[(0, 0)], [(0, 0)], [(1, 1), (1, 2)]] + [[(0, 0)]] * 64
    mo = np.zeros(len(ms) + 1, dtype=np.int64)
    np.cumsum([len(x) for x in ms], out=mo[1:])
    got = tb.build_tracks(fo, np.array(pv, dtype=np.int32), mo, np.concatenate([np.array(x) for x in ms]))
    assert list(got["offsets"]) == [0, 3, 6, 71]
    assert list(got["feature"][:6]) == [0, 3, 5, 1, 2, 4]
    assert list(got["view"][:6]) == [0, 1, 2, 0, 0, 1]
    assert list(got["feature"][6:]) == list(range(7, 72))
    assert list(got["status"]) == [tb.OK, tb.CONFLICT, tb.LONG]
    assert list(got["track"][:7]) == [0, 1, 1, 0, 1, 0, -1]
    # one view fewer on the chain: exactly 64 observations is ok
    got64 = tb.build_tracks(fo[:-1], np.array(pv[:-1], dtype=np.int32), mo[:-1], np.concatenate([np.array(x) for x in ms[:-1]]))
    assert list(got64["status"]) == [tb.OK, tb.CONFLICT, tb.OK]


# ---- the host build of the union-find of csrc/sfm_track_build.cuh -------------------------------------------------------
@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    from structure_from_motion_b200 import build as b

    try:
        nvcc = b._nvcc()
    except RuntimeError:
        pytest.skip("no nvcc: the host build of sfm_track_build.cuh cannot be made")
    out = str(tmp_path_factory.mktemp("track_build") / "libtbcheck.so")
    subprocess.check_call([nvcc, "-O2", "-shared", "-Xcompiler", "-fPIC", *b.ARCH, "-o", out,
                           os.path.join(ROOT, "tools", "track_build_check.cu")])
    return ctypes.CDLL(out)


def _labels(lib, N, edges, threads):
    e = np.ascontiguousarray(edges, dtype=np.int32).reshape(-1, 2)
    out = np.empty(N, dtype=np.int32)
    lib.tb_components(ctypes.c_int(N), ctypes.c_longlong(len(e)), e.ctypes.data_as(ctypes.c_void_p),
                      ctypes.c_int(threads), out.ctypes.data_as(ctypes.c_void_p))
    return out


def _oracle_labels(N, edges):
    """Each feature's label, its component's smallest id, by the oracle: view 0 holds the N features, view 1 a copy of
    them, pair entry 0 carries the edges (into the copy) and entry 1 joins every feature to its copy, so each component
    is a track whose first observation is its smallest id."""
    e = np.asarray(edges, dtype=np.int64).reshape(-1, 2)
    fo = np.array([0, N, 2 * N], dtype=np.int64)
    pv = np.array([[0, 1], [0, 1]], dtype=np.int32)
    m = np.concatenate([e, np.column_stack([np.arange(N), np.arange(N)])])
    res = tb.build_tracks(fo, pv, np.array([0, len(e), len(m)]), m)
    first = res["feature"][res["offsets"][:-1]]
    return first[res["track"][:N]]


@pytest.mark.parametrize("case", ["random", "chain forward", "chain reverse", "chain shuffled", "star high", "star low"])
@pytest.mark.parametrize("threads", [1, 8])
def test_host_union_find_against_the_oracle(lib, case, threads):
    rng = np.random.default_rng(7)
    if case == "random":
        N = 5000
        edges = rng.integers(0, N, (4000, 2))
    elif case.startswith("chain"):
        N = 20000
        edges = np.column_stack([np.arange(N - 1), np.arange(1, N)])
        if case.endswith("reverse"):
            edges = edges[::-1, ::-1]
        elif case.endswith("shuffled"):
            edges = edges[rng.permutation(N - 1)]
    else:
        N = 20000
        centre = N - 1 if case.endswith("high") else 0
        edges = np.column_stack([np.full(N - 1, centre), np.setdiff1d(np.arange(N), [centre])])
    assert np.array_equal(_labels(lib, N, edges, threads), _oracle_labels(N, edges))


def test_host_view_of(lib):
    off = np.array([0, 0, 3, 3, 3, 7, 8], dtype=np.int64)
    f = lib.tb_view_of
    f.restype = ctypes.c_int
    got = [f(off.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(6), ctypes.c_longlong(g)) for g in range(8)]
    assert got == list(np.searchsorted(off, np.arange(8), side="right") - 1) == [1, 1, 1, 4, 4, 4, 4, 5]


# ---- scenes.make_match_graph --------------------------------------------------------------------------------------------
@pytest.mark.parametrize("span,wrong,distract", [(1, 0.0, 0.0), (2, 0.0, 0.25), (3, 0.05, 0.5)])
def test_match_graph_invariants(span, wrong, distract):
    g = make_match_graph(3000, 7, 5, span=span, wrong_frac=wrong, distractor_frac=distract, max_len=5)
    V = 7
    assert len(g.features) == len(g.point) == V
    n_obs = [int((p >= 0).sum()) for p in g.point]
    for v in range(V):
        assert len(g.features[v]) == n_obs[v] + int(round(distract * n_obs[v]))
        seen = g.point[v][g.point[v] >= 0]
        assert len(np.unique(seen)) == len(seen)  # a point at most once per view
    assert [tuple(p) for p in g.pairs] == [(a, b) for a in range(V) for b in range(a + 1, min(a + span, V - 1) + 1)]
    total = sum(len(m) for m in g.matches)
    assert sum(int(w.sum()) for w in g.wrong) == int(round(wrong * total))
    for (a, b), m, w in zip(g.pairs, g.matches, g.wrong):
        assert (m[:, 0] < len(g.features[a])).all() and (m[:, 1] < len(g.features[b])).all() and (m >= 0).all()
        pa = g.point[a][m[:, 0]]
        assert (pa >= 0).all()
        assert (g.point[b][m[~w, 1]] == pa[~w]).all()  # true matches join one point's observations
        # every point seen in both views has exactly one match
        both = np.intersect1d(g.point[a][g.point[a] >= 0], g.point[b][g.point[b] >= 0])
        assert np.array_equal(np.sort(pa), both)
    # the pixels are the points' projections (plus noise) in the right view
    v = 3
    i = np.flatnonzero(g.point[v] >= 0)
    cam = g.X[g.point[v][i]] @ g.R[v].T + g.t[v]
    p = cam @ g.K.T
    assert np.median(np.abs(p[:, :2] / p[:, 2:] - g.features[v][i])) < 2.0


def test_match_graph_truth_is_the_tracks():
    """No wrong matches: the oracle's tracks are exactly the points seen in two or more views, all ok."""
    g = make_match_graph(2000, 6, 9, span=2, distractor_frac=0.3)
    fo = np.zeros(7, dtype=np.int64)
    np.cumsum([len(f) for f in g.features], out=fo[1:])
    mo = np.zeros(len(g.matches) + 1, dtype=np.int64)
    np.cumsum([len(m) for m in g.matches], out=mo[1:])
    got = tb.build_tracks(fo, g.pairs, mo, np.concatenate(g.matches))
    pt = np.concatenate(g.point)
    assert (got["status"] == tb.OK).all()
    tracks = {frozenset(got["feature"][s:e]) for s, e in zip(got["offsets"][:-1], got["offsets"][1:])}
    cnt = np.bincount(pt[pt >= 0])
    truth = {frozenset(np.flatnonzero(pt == k)) for k in np.flatnonzero(cnt >= 2)}
    assert tracks == truth


# ---- TrackSet.ok() ------------------------------------------------------------------------------------------------------
def test_trackset_ok():
    """Views 0 (features 0-3) and 1 (4-7): tracks {0, 4} ok, {1, 2, 5} conflict, {3, 6} ok; 7 is in no track."""
    ts = TrackSet(feature_offsets=np.array([0, 4, 8], dtype=np.int64), offsets=np.array([0, 2, 5, 7], dtype=np.int64),
                  view=np.array([0, 1, 0, 0, 1, 0, 1], dtype=np.int32),
                  feature=np.array([0, 4, 1, 2, 5, 3, 6], dtype=np.int32), x=np.arange(14.0).reshape(7, 2),
                  status=np.array(["ok", "conflict", "ok"]), track=np.array([0, 1, 1, 2, 0, 1, 2, -1], dtype=np.int32))
    ok = ts.ok()
    assert list(ok.offsets) == [0, 2, 4]
    assert list(ok.view) == [0, 1, 0, 1]
    assert list(ok.feature) == [0, 4, 3, 6]
    assert np.array_equal(ok.x, np.array([[0, 1], [2, 3], [10, 11], [12, 13]], dtype=float))
    assert list(ok.status) == ["ok", "ok"]
    assert list(ok.track) == [0, -1, -1, 1, 0, -1, 1, -1]
    again = ok.ok()
    assert np.array_equal(again.offsets, ok.offsets) and np.array_equal(again.track, ok.track)
