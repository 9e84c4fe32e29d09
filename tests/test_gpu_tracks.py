"""Multi-view triangulation of tracks (sfm_triangulate_tracks, csrc/sfm_tracks.cuh) on the GPU: noise-free recovery,
bit-exact self-consistency with the C reprojection checker, the pair search and the linear point against the oracle,
the refinement against MINPACK, independence of the batch, world and pixel scales, the edges and refusals, the engine
state, and the four-view incremental loop."""
import ctypes as C
import random

import numpy as np
import pytest

from oracle import creproj
from oracle import tracks as otr
from structure_from_motion_b200 import _native
from structure_from_motion_b200.multiview import triangulate_tracks_arrays
from structure_from_motion_b200.homography import two_view_homography_arrays
from structure_from_motion_b200.pnp import ransac_pnp_arrays
from structure_from_motion_b200.scenes import (make_multi_view_scene, make_planar_scene, make_pnp_scene, make_scene)
from structure_from_motion_b200.two_view import two_view_arrays

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]

THR = 4.0


@pytest.fixture(scope="module")
def eng():
    return _native.Engine(0)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _scene(n, V, seed, **kw):
    K, R, t, X, off, view, x, out = make_multi_view_scene(n, V, seed, **kw)
    return K, R, t, X, off, view, x, out


def _Rt(R, t):
    return np.concatenate([R, t[:, :, None]], axis=2)


def _run(eng, K, R, t, off, view, x, thr=THR, **kw):
    return triangulate_tracks_arrays(K, R, t, off, view, x, thr, engine=eng, **kw)


def _sub(off, view, x, idx):
    """The tracks idx (in that order) as a CSR batch of their own."""
    n = np.diff(off)[idx]
    o = np.zeros(len(idx) + 1, dtype=np.int64)
    np.cumsum(n, out=o[1:])
    rows = np.concatenate([np.arange(off[i], off[i + 1]) for i in idx]) if len(idx) else np.zeros(0, dtype=np.int64)
    return o, view[rows], x[rows], rows


def _track_tuple(res, i, off):
    s = slice(off[i], off[i + 1])
    return (_bits(res.points[i]).tobytes(), res.status[i], int(res.num_inliers[i]), _bits(res.angle[i]).tobytes(),
            res.mask[s].tobytes(), _bits(res.err[s]).tobytes())


@pytest.fixture(scope="module")
def noisy(eng):
    """8 views, 20 000 points, 0.5 px noise, 20 % outlier observations."""
    K, R, t, X, off, view, x, out = _scene(20_000, 8, 21, noise_px=0.5, outlier_frac=0.2)
    lin = _run(eng, K, R, t, off, view, x)
    ref = _run(eng, K, R, t, off, view, x, refine_iterations=50)
    return K, R, t, X, off, view, x, out, lin, ref


# ---- 1. noise-free ----------------------------------------------------------------------------------------------------
def test_noise_free_scene(eng):
    K, R, t, X, off, view, x, _ = _scene(20_000, 8, 1, noise_px=0.0)
    res = _run(eng, K, R, t, off, view, x, thr=1.0)
    assert (res.status == "ok").all() and res.mask.all()
    pt = np.repeat(np.arange(len(X)), np.diff(off))
    depth = np.einsum("mij,mj->mi", R[view], X[pt])[:, 2] + t[view][:, 2]
    dmin = np.minimum.reduceat(depth, off[:-1])
    rel = np.linalg.norm(res.points - X, axis=1) / dmin
    print("noise-free: worst |X - X_true| / depth", rel.max())
    assert rel.max() <= 1e-9


# ---- 2. bit-exact self-consistency ------------------------------------------------------------------------------------
def test_self_consistency(noisy):
    K, R, t, X, off, view, x, out, lin, ref = noisy
    Rt = _Rt(R, t)
    pt = np.repeat(np.arange(len(off) - 1), np.diff(off))
    for res in (lin, ref):
        fin = np.isfinite(res.points).all(axis=1)
        assert set(res.status[~fin]) <= {"short", "no_pair"} and not ({"short", "no_pair"} & set(res.status[fin]))
        assert not res.mask[~fin[pt]].any()
        for c in range(len(R)):
            sel = (view == c) & fin[pt]
            m, val = creproj.reproj_exact_many(Rt[c], K, res.points[pt[sel]], x[sel], THR)
            assert np.array_equal(m, res.mask[sel]) and _same(val, res.err[sel]), c
        cnt = np.add.reduceat(res.mask.astype(np.int64), off[:-1])
        assert np.array_equal(cnt, res.num_inliers)
        rng = np.random.default_rng(0)
        worst = 0.0
        for i in rng.choice(np.flatnonzero(fin), 3000, replace=False):
            s = slice(off[i], off[i + 1])
            a = otr.ray_angle(res.points[i], Rt, view[s][res.mask[s]])
            worst = max(worst, abs(a - res.angle[i]))
        print("angle: worst |device - oracle| (rad)", worst)
        assert worst <= 1e-12
        min_angle = 1.5 * (np.pi / 180.0)
        want = np.where(res.num_inliers < 2, "few_inliers", np.where(res.angle >= min_angle, "ok", "small_angle"))
        assert np.array_equal(res.status[fin], want[fin])
        assert (res.status == "ok").mean() > 0.9


# ---- 3. and 4. pair search and linear point against the oracle ---------------------------------------------------------
def test_pair_search_and_linear_point(eng, noisy):
    """The winner's passing set is the oracle's (most inliers; the linear point then agrees with the 50-digit N-view DLT
    over that set, both in the call's frame) for every track without band flags and without a near tie on the sum.
    Tolerance: 1e-9 relative times cond / 1e6 when the condition number cond = s1 / s3 of the DLT matrix (rows of
    dlt_triangulate) exceeds 1e6."""
    K, R, t, X, off, view, x, out, lin, _ = noisy
    Rt = _Rt(R, t)
    Ks = np.broadcast_to(K, (len(R), 3, 3))
    fs = otr.frame_exponent(Rt)
    rng = np.random.default_rng(1)
    checked, worst, two = 0, 0.0, 0
    for i in rng.choice(len(off) - 1, 1500, replace=False):
        s = slice(off[i], off[i + 1])
        vs, xs = view[s], x[s]
        table = otr.pair_table(Ks, Rt, vs, xs, THR, frame=fs)
        w = otr.pair_search(table)
        if w < 0:
            assert lin.status[i] == "no_pair"
            continue
        if any(r[7] for r in table):
            continue
        best = table[w]
        rivals = [r for r in table if r[3] and r[4] == best[4] and not np.array_equal(r[6], best[6])]
        if any(abs(r[5] - best[5]) <= 1e-9 * best[5] for r in rivals):
            continue
        S = np.flatnonzero(best[6])
        Ps = [otr.in_frame(creproj.projection(K, Rt[c]), fs) for c in vs[S]]
        if len(S) == 2:
            tri = np.ldexp(eng.triangulate(Ps[0], Ps[1], xs[S[:1]], xs[S[1:]])[0], fs)
            assert np.linalg.norm(lin.points[i] - tri) <= 1e-12 * np.linalg.norm(tri)
            two += 1
        want = np.ldexp(np.array([float(v) for v in otr.dlt_exact(Ps, xs[S])]), fs)
        A = np.concatenate([otr.dlt_rows(P, u, v) for P, (u, v) in zip(Ps, xs[S])])
        sv = np.linalg.svd(A, compute_uv=False)
        tol = 1e-9 * max(1.0, sv[0] / sv[2] / 1e6)
        rel = np.linalg.norm(lin.points[i] - want) / np.linalg.norm(want)
        worst = max(worst, rel / tol)
        assert rel <= tol, (i, rel, tol)
        checked += 1
    print(f"linear point vs 50-digit DLT: {checked} tracks ({two} of two observations), worst error / tolerance {worst:.3g}")
    assert checked >= 1000
    # planted outliers far off under the true point are rejected in tracks with at least 3 other observations (with
    # fewer, a uniform pixel near the epipolar line of the only other one is a consistent pair of its own)
    pt = np.repeat(np.arange(len(off) - 1), np.diff(off))
    clean = np.add.reduceat((~out).astype(np.int64), off[:-1]) >= 3
    far = np.zeros(len(view), dtype=bool)
    for c in range(len(R)):
        sel = (view == c) & out
        _, val = creproj.reproj_exact_many(Rt[c], K, X[pt[sel]], x[sel], THR)
        far[np.flatnonzero(sel)[val > 100 * THR]] = True
    far &= clean[pt]
    assert far.sum() > 1000 and not lin.mask[far].any()


# ---- 5. refinement ----------------------------------------------------------------------------------------------------
def test_refinement_reports(noisy):
    K, R, t, X, off, view, x, out, lin, ref = noisy
    r = ref.refinement
    have = r.status != "no_model"
    assert np.array_equal(have, np.isfinite(lin.points).all(axis=1))
    assert (r.cost_final[have] <= r.cost_start[have]).all()
    assert set(r.status[have]) <= {"converged", "max_iterations", "stalled"}
    ok = (lin.status == "ok") & (ref.status == "ok")
    e_lin = np.median(np.linalg.norm(lin.points[ok] - X[ok], axis=1))
    e_ref = np.median(np.linalg.norm(ref.points[ok] - X[ok], axis=1))
    print("median |X - X_true| linear / refined:", e_lin, e_ref)
    assert e_ref <= e_lin
    # the refinement starts at the reported linear point: its start cost is the cost of that point over the list
    Rt = _Rt(R, t)
    for i in np.flatnonzero(have)[:300]:
        s = slice(off[i], off[i + 1])
        lst = lin.mask[s]
        assert r.num[i] == lst.sum()
        Ps = [creproj.projection(K, Rt[c]) for c in view[s][lst]]
        c0 = otr.cost(lin.points[i], Ps, x[s][lst]) if lst.any() else 0.0
        assert abs(c0 - r.cost_start[i]) <= 1e-9 * c0 + 1e-300


def test_refinement_off_writes_no_report(eng):
    K, R, t, X, off, view, x, _ = _scene(500, 8, 3, noise_px=0.5)
    a = _run(eng, K, R, t, off, view, x)
    assert a.refinement is None
    T, M = len(off) - 1, len(view)
    sentinel = (_native.TrackRefinement * T)()
    C.memset(sentinel, 0x5a, C.sizeof(sentinel))
    before = bytes(sentinel)
    Xo = np.empty((T, 3))
    Kv = np.ascontiguousarray(np.broadcast_to(K, (len(R), 3, 3)))
    Rt = np.ascontiguousarray(_Rt(R, t))
    rc = eng.lib.sfm_triangulate_tracks(eng.h, Kv.ctypes.data, Rt.ctypes.data, len(R), off.ctypes.data, T,
                                        view.ctypes.data, x.ctypes.data, THR, 1.5, 2, 0, Xo.ctypes.data, None, None,
                                        None, None, None, C.cast(sentinel, C.c_void_p))
    assert rc == 0 and bytes(sentinel) == before and _same(Xo, a.points)


def _long_track(V, seed, noise=1.0):
    """One point seen by V cameras on an arc, pixel noise only."""
    K, R, t, X, off, view, x, _ = make_multi_view_scene(1, V, seed, noise_px=noise, min_len=V, max_len=V, arc_deg=90.0)
    return K, R, t, X, off, view, x


@pytest.mark.parametrize("n", [2, 3, 8, 64])
def test_refinement_matches_minpack(eng, n):
    Rt_all, worst = None, 0.0
    for seed in range(5):
        K, R, t, X, off, view, x = _long_track(n, 100 + seed)
        lin = _run(eng, K, R, t, off, view, x, thr=1e4)
        ref = _run(eng, K, R, t, off, view, x, thr=1e4, refine_iterations=100)
        rep = ref.refinement
        assert rep.num[0] == n and lin.mask.all()
        Rt_all = _Rt(R, t)
        Ps = [creproj.projection(K, Rt_all[c]) for c in view]
        _, c_mp = otr.refine_replay(lin.points[0], Ps, x)
        rel = abs(rep.cost_final[0] - c_mp) / c_mp
        worst = max(worst, rel)
        assert rep.cost_final[0] <= rep.cost_start[0]
        assert rel <= 1e-9, (seed, rep.cost_final[0], c_mp, rep.status[0])
        assert abs(otr.cost(ref.points[0], Ps, x) - rep.cost_final[0]) <= 1e-9 * rep.cost_final[0]
    print(f"{n} observations: worst |cost - MINPACK| / MINPACK {worst:.3g}")


# ---- 6. independence --------------------------------------------------------------------------------------------------
def test_independence(eng):
    K, R, t, X, off, view, x, _ = _scene(1_000_000, 16, 5, noise_px=0.5, outlier_frac=0.1)
    T = len(off) - 1
    full = _run(eng, K, R, t, off, view, x, refine_iterations=5)
    rng = np.random.default_rng(2)
    probe = rng.choice(T, 200, replace=False)
    perm = rng.permutation(T)
    po, pv, px, _ = _sub(off, view, x, perm)
    permuted = _run(eng, K, R, t, po, pv, px, refine_iterations=5)
    where = np.empty(T, dtype=np.int64)
    where[perm] = np.arange(T)
    half = T // 3
    ao, av, ax, _ = _sub(off, view, x, np.arange(half))
    bo, bv, bx, _ = _sub(off, view, x, np.arange(half, T))
    first = _run(eng, K, R, t, ao, av, ax, refine_iterations=5)
    second = _run(eng, K, R, t, bo, bv, bx, refine_iterations=5)
    for i in probe:
        want = _track_tuple(full, i, off)
        assert _track_tuple(permuted, where[i], po) == want
        part, j, o = (first, i, ao) if i < half else (second, i - half, bo)
        assert _track_tuple(part, j, o) == want
        so, sv, sx, _ = _sub(off, view, x, np.array([i]))
        alone = _run(eng, K, R, t, so, sv, sx, refine_iterations=5)
        assert _track_tuple(alone, 0, so) == want
        assert _same(alone.refinement.cost_final, full.refinement.cost_final[i:i + 1])


# ---- 7. scale ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [-300, -120, -7, 7, 120, 300])
def test_world_scale_is_bit_exact(eng, k):
    K, R, t, X, off, view, x, _ = _scene(3000, 8, 7, noise_px=0.5, outlier_frac=0.2)
    for it in (0, 10):
        a = _run(eng, K, R, t, off, view, x, refine_iterations=it)
        b = _run(eng, K, R, np.ldexp(t, k), off, view, x, refine_iterations=it)
        assert _same(np.ldexp(a.points, k), b.points)
        assert np.array_equal(a.status, b.status) and np.array_equal(a.num_inliers, b.num_inliers)
        assert np.array_equal(a.mask, b.mask) and _same(a.err, b.err) and _same(a.angle, b.angle)
        if it:
            assert _same(a.refinement.cost_final, b.refinement.cost_final)
            assert np.array_equal(a.refinement.iterations, b.refinement.iterations)


@pytest.mark.parametrize("k", [-200, -50, 50, 200])
def test_pixel_scale(eng, k):
    """Pixels and K's first two rows x 2^k, threshold x 4^k: the same masks and statuses, and (measured on the B200,
    refinement off and on) the points bit for bit - the frame depends on t alone."""
    K, R, t, X, off, view, x, _ = _scene(3000, 8, 8, noise_px=0.5, outlier_frac=0.2)
    Ks = K.copy()
    Ks[:2] = np.ldexp(Ks[:2], k)
    for it in (0, 10):
        a = _run(eng, K, R, t, off, view, x, refine_iterations=it)
        b = _run(eng, Ks, R, t, off, view, np.ldexp(x, k), thr=np.ldexp(THR, 2 * k), refine_iterations=it)
        assert np.array_equal(a.status, b.status) and np.array_equal(a.mask, b.mask)
        fin = np.isfinite(a.points).all(axis=1)
        rel = np.linalg.norm(a.points[fin] - b.points[fin], axis=1) / np.linalg.norm(a.points[fin], axis=1)
        print(f"pixels x 2^{k}, refine {it}: points bit-identical {_same(a.points, b.points)}, worst rel {rel.max():.3g}")
        assert rel.max() <= 1e-12 and _same(a.points, b.points)


# ---- 8. edges and refusals --------------------------------------------------------------------------------------------
def test_edges(eng):
    K, R, t, X, off, view, x, _ = _scene(50, 8, 9, noise_px=0.0, min_len=5, max_len=5)
    Rt = _Rt(R, t)
    P = [creproj.projection(K, Rt[c]) for c in range(8)]

    def proj(c, Xw):
        p = P[c] @ np.append(Xw, 1.0)
        return p[:2] / p[2]

    C0 = -R[0].T @ t[0]
    C1 = -R[1].T @ t[1]
    tracks = [
        [],                                                     # 0: empty
        [(0, proj(0, X[0]))],                                   # 1: one observation
        [(2, proj(2, X[1])), (2, proj(2, X[1]) + 0.1)],         # 2: two observations in the same view
        [(0, proj(0, C0 + 2.0 * (C1 - C0))), (1, proj(1, C0 + 2.0 * (C1 - C0)))],   # 3: on the baseline
        [(0, proj(0, C0 + 0.5 * (C1 - C0) + 1e-9)), (1, proj(1, C0 + 0.5 * (C1 - C0) + 1e-9))],
        [(c, proj(c, np.array([0.3, -0.2, -30.0]))) for c in range(4)],  # 5: behind every camera
        [(c, proj(c, X[2])) for c in range(5)],                 # 6: a NaN pixel
        [(c, proj(c, X[3])) for c in range(5)],                 # 7: an infinite pixel
    ]
    tracks[6][2] = (2, np.array([np.nan, 100.0]))
    tracks[7][1] = (1, np.array([np.inf, -np.inf]))
    off2 = np.zeros(len(tracks) + 1, dtype=np.int64)
    np.cumsum([len(tr) for tr in tracks], out=off2[1:])
    v2 = np.array([c for tr in tracks for c, _ in tr], dtype=np.int32)
    x2 = np.array([p for tr in tracks for _, p in tr], dtype=np.float64)
    res = _run(eng, K, R, t, off2, v2, x2, thr=1.0)
    assert res.status[0] == "short" and res.status[1] == "short"
    assert np.isnan(res.points[:2]).all()
    for i in (2, 3, 4):
        assert res.status[i] != "ok", (i, res.status[i])
    assert res.status[5] == "no_pair" and np.isnan(res.points[5]).all()
    for i, bad, Xt in ((6, 2, X[2]), (7, 1, X[3])):
        s = slice(off2[i], off2[i + 1])
        m = res.mask[s]
        assert res.status[i] == "ok" and not m[bad] and m.sum() == 4
        assert np.linalg.norm(res.points[i] - Xt) <= 1e-9 * np.linalg.norm(Xt)
    # 64 observations are accepted, 65 refused
    K64, R64, t64, X64, o64, v64, x64 = _long_track(64, 3)
    assert _run(eng, K64, R64, t64, o64, v64, x64).status[0] == "ok"
    v65 = np.append(v64, v64[:1])
    x65 = np.vstack([x64, x64[:1]])
    with pytest.raises(_native.NativeError):
        _run(eng, K64, R64, t64, np.array([0, 65]), v65, x65)


def test_refusals(eng):
    K, R, t, X, off, view, x, _ = _scene(20, 4, 10)
    bad = lambda **kw: pytest.raises(_native.NativeError)  # noqa: E731
    for v in (-1, 4):
        vv = view.copy()
        vv[3] = v
        with bad():
            _run(eng, K, R, t, off, vv, x)
    o = off.copy()
    o[2], o[3] = o[3], o[2]  # decreasing
    with bad():
        _run(eng, K, R, t, o, view, x)
    with bad():
        eng.triangulate_tracks(np.broadcast_to(K, (4, 3, 3)), _Rt(R, t), off + 1, np.append(view, 0),
                               np.vstack([x, x[:1]]), THR)  # offsets[0] != 0
    tn = t.copy()
    tn[1, 2] = np.nan
    with bad():
        _run(eng, K, R, tn, off, view, x)
    for Kb in (np.diag([800.0, 800.0, 0.0]), np.array([[800.0, 0, 640], [0, 800, 480], [0.1, 0, 1]]),
               np.array([[800.0, 0, 640], [0, 800, 480], [0, 0, 2]]), np.full((3, 3), np.inf)):
        with bad():
            _run(eng, Kb, R, t, off, view, x)
    with bad():
        _run(eng, K, R, t, off, view, x, thr=np.nan)
    with bad():
        _run(eng, K, R, t, off, view, x, min_views=1)
    with bad():
        eng.triangulate_tracks(np.broadcast_to(K, (4, 3, 3)), _Rt(R, t), off, view, x, THR, refine_iterations=-1)
    with pytest.raises(ValueError):
        _run(eng, K, R, t, off, view, x, refine_iterations=-1)


# ---- 9. engine state --------------------------------------------------------------------------------------------------
def test_engine_state(eng):
    e2 = _native.Engine(0)
    Kp, Xp, xp, _, _, _ = make_pnp_scene(700, 0.3, seed=12)
    random.seed(3)
    p0 = ransac_pnp_arrays(Kp, Xp, xp, 4.0, 100, "rms", 300, engine=e2, refine_iterations=10)
    K, x1, x2, _, _, _ = make_scene(600, 0.3, seed=3)
    random.seed(5)
    two_view_arrays(K, x1, x2, 1.5e-6, 10, "rms", 64, engine=e2, refine_iterations=10)
    before_ref = bytes(e2.get_refinement(1))
    e2.upload_pnp(Xp, xp, Kp)
    random.seed(3)
    ransac_pnp_arrays(Kp, Xp, xp, 4.0, 100, "rms", 300, engine=e2)
    ties0 = e2.near_ties(1e-3, 64)
    m0, v0 = e2.pnp_mask(None, 4.0)
    Kt, Rt_, tt, _, off, view, x, _ = _scene(2000, 8, 11, outlier_frac=0.2)
    _run(e2, Kt, Rt_, tt, off, view, x, refine_iterations=10)
    ties1 = e2.near_ties(1e-3, 64)
    m1, v1 = e2.pnp_mask(None, 4.0)
    assert np.array_equal(ties0[0], ties1[0]) and ties0[1] == ties1[1]
    assert np.array_equal(m0, m1) and _same(v0, v1)
    assert bytes(e2.get_refinement(1)) == before_ref
    fresh = _native.Engine(0)
    random.seed(6)
    a = two_view_arrays(K, x1, x2, 1.5e-6, 10, "rms", 64, engine=e2)
    random.seed(6)
    b = two_view_arrays(K, x1, x2, 1.5e-6, 10, "rms", 64, engine=fresh)
    for u, w in ((a.R, b.R), (a.t, b.t), (a.points, b.points), (a.ransac.E, b.ransac.E)):
        assert _same(u, w)
    Kh, y1, y2, _, _ = make_planar_scene(600, 0.3, seed=4)
    _run(e2, Kt, Rt_, tt, off, view, x)
    random.seed(7)
    a = two_view_homography_arrays(Kh, y1, y2, 4.0, 10, "rms", 64, engine=e2)
    random.seed(7)
    b = two_view_homography_arrays(Kh, y1, y2, 4.0, 10, "rms", 64, engine=fresh)
    assert _same(a.ransac.H, b.ransac.H) and _same(a.R, b.R) and _same(a.points, b.points)
    _run(e2, Kt, Rt_, tt, off, view, x)
    random.seed(3)
    a = ransac_pnp_arrays(Kp, Xp, xp, 4.0, 100, "rms", 300, engine=e2, refine_iterations=10)
    random.seed(3)
    b = ransac_pnp_arrays(Kp, Xp, xp, 4.0, 100, "rms", 300, engine=fresh, refine_iterations=10)
    assert _same(a.R, b.R) and _same(a.t, b.t) and _same(a.refinement.R, b.refinement.R)
    assert _same(a.R, p0.R) and _same(a.err, p0.err)


# ---- 10. four-view composition ----------------------------------------------------------------------------------------
def test_four_view_composition(eng):
    """Views 1-2 by two_view_arrays, view 3 by ransac_pnp_arrays against the pair's points, the tracks over views 1-3
    triangulated (points the pair did not reconstruct included), view 4 by ransac_pnp_arrays against only those new
    points.  Every estimate is refined.  On the B200 (1000 W): 1150 new points, R4 off the truth by 3.2e-3 (max entry),
    t4 by 1.6e-3 (unit baseline 1-2), R3 by 1.8e-3; the bounds are about 3x that."""
    K, R, t, X, off, view, x, out = make_multi_view_scene(6000, 4, 42, noise_px=0.5, outlier_frac=0.1, arc_deg=40.0,
                                                          min_len=2, max_len=4)
    T = len(off) - 1
    dense = np.full((T, 4, 2), np.nan)
    seen = np.zeros((T, 4), dtype=bool)
    pt = np.repeat(np.arange(T), np.diff(off))
    dense[pt, view] = x
    seen[pt, view] = True
    # truth in camera-1 coordinates, scaled to a unit baseline 1-2
    Rr = np.array([R[c] @ R[0].T for c in range(4)])
    tr = np.array([t[c] - Rr[c] @ t[0] for c in range(4)])
    tr /= np.linalg.norm(tr[1])
    both = np.flatnonzero(seen[:, 0] & seen[:, 1])
    random.seed(1)
    tv = two_view_arrays(K, dense[both, 0], dense[both, 1], 1e-5, 100, "rms", 300, engine=eng, refine_iterations=20)
    idx = tv.inlier_indices[tv.passing]
    done = np.zeros(T, dtype=bool)
    done[both[idx]] = True
    have3 = seen[both[idx], 2]
    random.seed(2)
    p3 = ransac_pnp_arrays(K, tv.points[tv.passing][have3], dense[both[idx][have3], 2], 4.0, 10, "rms", 300,
                           engine=eng, refine_iterations=20)
    Rs = np.stack([np.eye(3), tv.R, p3.refinement.R])
    ts = np.stack([np.zeros(3), tv.t, p3.refinement.t])
    sel = np.flatnonzero(seen[:, :3].sum(axis=1) >= 2)
    o3 = np.zeros(len(sel) + 1, dtype=np.int64)
    np.cumsum(seen[sel, :3].sum(axis=1), out=o3[1:])
    rows, cols = np.nonzero(seen[sel, :3])
    res = triangulate_tracks_arrays(K, Rs, ts, o3, cols.astype(np.int32), dense[sel[rows], cols], 4.0,
                                    refine_iterations=10, engine=eng)
    new = (res.status == "ok") & ~done[sel] & seen[sel, 3]
    assert new.sum() >= 500
    random.seed(3)
    p4 = ransac_pnp_arrays(K, res.points[new], dense[sel[new], 3], 4.0, 10, "rms", 300, engine=eng,
                           refine_iterations=20)
    eR, et = np.abs(p4.refinement.R - Rr[3]).max(), np.abs(p4.refinement.t - tr[3]).max()
    print(f"four views: {new.sum()} new points; R4 error {eR:.3g}, t4 error {et:.3g}; R3 error "
          f"{np.abs(p3.refinement.R - Rr[2]).max():.3g}")
    assert eR <= 1e-2 and et <= 5e-3
