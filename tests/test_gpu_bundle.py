"""Bundle adjustment (sfm_bundle_adjust, csrc/sfm_bundle.cuh) on the GPU: noise-free recovery, the refined cost against
MINPACK, the first step against the dense solve, exact decisions, the gauge and the non-parameters, world and pixel
scales, determinism and the view limit, edges and refusals, the engine state, and the four-view incremental loop."""
import random

import numpy as np
import pytest

from oracle import bundle as oba
from oracle import creproj
from oracle.refine import rodrigues
from structure_from_motion_b200 import _native
from structure_from_motion_b200.multiview import bundle_adjust_arrays, triangulate_tracks_arrays
from structure_from_motion_b200.pnp import ransac_pnp_arrays
from structure_from_motion_b200.scenes import make_multi_view_scene, make_pnp_scene, make_scene
from structure_from_motion_b200.two_view import two_view_arrays

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]


@pytest.fixture(scope="module")
def eng():
    return _native.Engine(0)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _Rt(R, t):
    return np.concatenate([R, t[:, :, None]], axis=2)


def _perturb(R, t, X, seed, deg=1.0, tfrac=0.01, xfrac=0.01, anchor=1):
    """Every pose but view 0 rotated by about `deg` and its t moved by about `tfrac` of |t| (the anchor's largest
    component kept), every point moved by about `xfrac` of its depth."""
    rng = np.random.default_rng(seed)
    R0, t0 = R.copy(), t.copy()
    for c in range(1, len(R)):
        w = rng.normal(size=3)
        R0[c] = R[c] @ rodrigues(w / np.linalg.norm(w) * np.radians(deg))
        t0[c] = t[c] + rng.normal(size=3) * tfrac * np.linalg.norm(t[c]) / np.sqrt(3)
    if anchor is not None:
        k = int(np.argmax(np.abs(t[anchor])))
        t0[anchor, k] = t[anchor, k]
    X0 = X + rng.normal(size=X.shape) * xfrac * X[:, 2:] / np.sqrt(3)
    return R0, t0, X0


def _run(eng, K, R, t, X, off, view, x, thr, **kw):
    return bundle_adjust_arrays(K, R, t, X, off, view, x, thr, engine=eng, **kw)


# ---- 1. noise-free ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [1, 2])
def test_noise_free_recovers_the_truth(eng, seed):
    K, R, t, X, off, view, x, _ = make_multi_view_scene(2000, 8, seed, noise_px=0.0)
    R0, t0, X0 = _perturb(R, t, X, seed + 10)
    res = _run(eng, K, R0, t0, X0, off, view, x, 1e4, max_iterations=100)
    rep = res.report
    assert rep.status == "converged" and rep.num_observations == len(view) and rep.num_points == len(X)
    assert rep.num_free_views == 7 and rep.cost_final < 1e-12 * rep.cost_start
    assert np.abs(res.R - R).max() <= 1e-9
    assert np.abs(res.t - t).max() <= 1e-9 * np.abs(t).max()
    assert (np.linalg.norm(res.points - X, axis=1) <= 1e-9 * np.linalg.norm(X, axis=1)).all()


@pytest.fixture(scope="module")
def noisy(eng):
    """V views (8 by default), 0.5 px noise, 10 % outlier observations; the start from noisy poses and
    triangulate_tracks_arrays."""
    def make(n, seed, V=8):
        K, R, t, X, off, view, x, out = make_multi_view_scene(n, V, seed, noise_px=0.5, outlier_frac=0.1)
        R0, t0, _ = _perturb(R, t, X, seed + 1, deg=0.05, tfrac=0.002)
        tr = triangulate_tracks_arrays(K, R0, t0, off, view, x, 16.0, engine=eng)
        X0 = np.where((tr.status == "ok")[:, None], tr.points, np.nan)
        return K, R0, t0, X0, off, view, x
    return make


# ---- 2. against MINPACK -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,seed", [(150, 3), (300, 4)])
def test_cost_matches_minpack(eng, noisy, n, seed):
    """MINPACK works on the dense Jacobian, so the problems are a few hundred points (about 1000 parameters)."""
    K, R0, t0, X0, off, view, x = noisy(n, seed)
    res = _run(eng, K, R0, t0, X0, off, view, x, 16.0, max_iterations=200)
    prob = oba.problem(K, _Rt(R0, t0), X0, off, view, x, 16.0, np.arange(8) == 0, 1)
    assert res.report.num_observations == len(prob.obs_track) and res.report.num_points == len(prob.points)
    _, _, _, cm = oba.minpack_replay(prob)
    print(f"n {n}: device {res.report.cost_final!r} ({res.report.iterations} it, {res.report.status}), minpack {cm!r}")
    assert res.report.status == "converged"
    assert abs(res.report.cost_final - cm) <= 1e-9 * cm


# ---- 3. the step is the stated system ---------------------------------------------------------------------------------
@pytest.mark.parametrize("V,anchor,fixed", [(8, 1, (0,)), (8, -1, (0, 4)), (8, -1, (0, 4, 5, 6, 7)), (17, 1, (0,)),
                                            (23, -1, (0, 11)), (64, 1, (0,))])
def test_first_step_matches_dense_solve(eng, noisy, V, anchor, fixed):
    """7, 6, 3, 16, 21 and 63 free views: S padded to 64, 32, 96, 128 and 384 rows - 1 to 12 tile columns of the Cholesky, so
    that its left-looking updates and the right-hand side row run over several earlier panels (and S's entries do not
    always fill whole warps)."""
    K, R0, t0, X0, off, view, x = noisy({8: 300, 17: 600, 23: 600, 64: 1500}[V], 5, V)
    res = _run(eng, K, R0, t0, X0, off, view, x, 16.0, max_iterations=1, fixed=fixed, scale_view=anchor)
    assert res.report.iterations == 1 and res.report.rejected == 0
    assert res.report.num_free_views == V - len(fixed)
    fmask = np.zeros(V, dtype=bool)
    fmask[list(fixed)] = True
    prob = oba.problem(K, _Rt(R0, t0), X0, off, view, x, 16.0, fmask, anchor)
    R1, t1, X1, _ = oba.dense_step(prob, 1e-3)
    assert np.abs(res.R - R1).max() <= 1e-9
    assert np.abs(res.t - t1).max() <= 1e-9 * np.abs(t1).max()
    fin = np.isfinite(X1).all(axis=1)
    assert (np.linalg.norm(res.points[fin] - X1[fin], axis=1) <= 1e-9 * np.linalg.norm(X1[fin], axis=1)).all()
    assert abs(res.report.cost_final - oba.cost(prob, R1, t1, X1)) <= 1e-9 * res.report.cost_final


# ---- 4. exact decisions -----------------------------------------------------------------------------------------------
def test_mask_and_err_are_the_checkers(eng, noisy):
    K, R0, t0, X0, off, view, x = noisy(2000, 6)
    res = _run(eng, K, R0, t0, X0, off, view, x, 16.0, max_iterations=20)
    pt = np.repeat(np.arange(len(off) - 1), np.diff(off))
    for c in range(8):
        sel = np.flatnonzero(view == c)
        m, v = creproj.reproj_exact_many(_Rt(res.R, res.t)[c], K, res.points[pt[sel]], x[sel], 16.0)
        assert np.array_equal(m, res.mask[sel]) and _same(v, res.err[sel])
    assert res.report.cost_final <= res.report.cost_start


# ---- 5. gauge and non-parameters --------------------------------------------------------------------------------------
def test_gauge_and_non_parameters(eng, noisy):
    K, R0, t0, X0, off, view, x = noisy(1000, 7)
    T = len(off) - 1
    # view 8: free, with no observation at all; track 0: a NaN point; track 1: one observation left passing
    R0 = np.concatenate([R0, (R0[3] * 1.001)[None]])
    t0 = np.concatenate([t0, t0[3:4] + 0.1])
    X0 = X0.copy()
    X0[0] = [np.nan, 1.0, 2.0]
    i1 = np.flatnonzero(np.isfinite(X0).all(axis=1) & (np.diff(off) >= 3))[1]
    x = x.copy()
    x[off[i1] + 1:off[i1 + 1]] += 300.0
    res = _run(eng, K, R0, t0, X0, off, view, x, 16.0, max_iterations=20, fixed=(0, 2))
    assert res.report.num_free_views == 7
    for c in (0, 2):
        assert _same(res.R[c], R0[c]) and _same(res.t[c], t0[c])
    assert _same(res.points[0], X0[0]) and _same(res.points[i1], X0[i1])
    nonpar = ~np.isfinite(X0).all(axis=1)
    assert _same(res.points[nonpar], X0[nonpar])
    assert _same(res.t[8], t0[8])
    assert np.abs(res.R[8] - oba.nearest_rotation(R0[8])).max() <= 1e-14
    # the anchor: one fixed view plus the lowest free view's largest t component
    res = _run(eng, K, R0[:8], t0[:8], X0, off, view, x, 16.0, max_iterations=20)
    k = int(np.argmax(np.abs(t0[1])))
    assert _same(res.t[1, k], t0[1, k]) and not _same(res.t[1], t0[1])
    assert np.isfinite(res.points[1:T]).any()


# ---- 6. scale ---------------------------------------------------------------------------------------------------------
def _report_tuple(rep):
    return (rep.num_observations, rep.num_points, rep.iterations, rep.status, rep.rejected)


@pytest.mark.parametrize("k", [-300, -37, 41, 300])
def test_world_scale_is_bit_exact(eng, noisy, k):
    K, R0, t0, X0, off, view, x = noisy(1000, 8)
    a = _run(eng, K, R0, t0, X0, off, view, x, 16.0, max_iterations=15)
    b = _run(eng, K, R0, np.ldexp(t0, k), np.ldexp(X0, k), off, view, x, 16.0, max_iterations=15)
    assert _same(a.R, b.R) and _same(np.ldexp(a.t, k), b.t) and _same(np.ldexp(a.points, k), b.points)
    assert _same(a.report.cost_final, b.report.cost_final) and _same(a.report.cost_start, b.report.cost_start)
    assert _report_tuple(a.report) == _report_tuple(b.report)
    assert np.array_equal(a.mask, b.mask) and _same(a.err, b.err)


@pytest.mark.parametrize("k", [-200, -50, 50, 200])
def test_pixel_scale_is_bit_exact(eng, noisy, k):
    K, R0, t0, X0, off, view, x = noisy(1000, 9)
    Ks = K.copy()
    Ks[:2] = np.ldexp(Ks[:2], k)
    a = _run(eng, K, R0, t0, X0, off, view, x, 16.0, max_iterations=15)
    b = _run(eng, Ks, R0, t0, X0, off, view, np.ldexp(x, k), np.ldexp(16.0, 2 * k), max_iterations=15)
    assert _same(a.R, b.R) and _same(a.t, b.t) and _same(a.points, b.points)
    assert _same(np.ldexp(a.report.cost_final, 2 * k), b.report.cost_final)
    assert _report_tuple(a.report) == _report_tuple(b.report)
    assert np.array_equal(a.mask, b.mask) and _same(np.ldexp(a.err, 2 * k), b.err)


# ---- 7. determinism and the view limit --------------------------------------------------------------------------------
def test_determinism(eng, noisy):
    K, R0, t0, X0, off, view, x = noisy(3000, 10)
    a = _run(eng, K, R0, t0, X0, off, view, x, 16.0, max_iterations=10)
    b = _run(eng, K, R0, t0, X0, off, view, x, 16.0, max_iterations=10)
    c = _run(_native.Engine(0), K, R0, t0, X0, off, view, x, 16.0, max_iterations=10)
    for r in (b, c):
        assert _same(a.R, r.R) and _same(a.t, r.t) and _same(a.points, r.points) and _same(a.err, r.err)
        assert _same(a.report.cost_final, r.report.cost_final) and _report_tuple(a.report) == _report_tuple(r.report)


def test_view_limit(eng):
    K, R, t, X, off, view, x, _ = make_multi_view_scene(4000, 256, 11, noise_px=0.5, outlier_frac=0.1, arc_deg=120.0)
    R0, t0, X0 = _perturb(R, t, X, 12, deg=0.02, tfrac=0.001, xfrac=0.001)
    res = _run(eng, K, R0, t0, X0, off, view, x, 16.0, max_iterations=4)
    assert res.report.num_free_views == 255 and res.report.iterations >= 1
    assert res.report.cost_final <= res.report.cost_start and res.report.status in ("converged", "max_iterations")
    with pytest.raises(_native.NativeError):
        _run(eng, K, np.concatenate([R0, R0[:1]]), np.concatenate([t0, t0[:1]]), X0, off, view, x, 16.0)


# ---- 8. edges and refusals --------------------------------------------------------------------------------------------
def test_empty_list(eng):
    K, R, t, X, off, view, x, _ = make_multi_view_scene(50, 4, 13)
    R0 = R * 1.01
    res = _run(eng, K, R0, t, np.full_like(X, np.nan), off, view, x, 16.0)
    rep = res.report
    assert rep.status == "converged" and rep.iterations == 0 and rep.cost_final == 0.0 and rep.num_observations == 0
    assert _same(res.t, t) and _same(res.R[0], R0[0]) and np.abs(res.R[1:] - R[1:]).max() <= 1e-14
    assert not res.mask.any()
    e = _native.Engine(0)  # no tracks at all
    r2 = bundle_adjust_arrays(K, R, t, np.zeros((0, 3)), np.zeros(1, np.int64), np.zeros(0, np.int32),
                              np.zeros((0, 2)), 16.0, engine=e)
    assert r2.report.status == "converged" and r2.report.iterations == 0 and r2.points.shape == (0, 3)


def test_nonfinite_start(eng):
    """The list is formed under the given R = 2 I of view 1, in front of which the point lies; the start rotation
    (its projection, I) puts the point behind view 1: the start cost is +inf and the input is reported."""
    K = np.array([[800.0, 0, 640], [0, 800, 480], [0, 0, 1]])
    R = np.stack([np.eye(3), 2 * np.eye(3)])
    t = np.array([[0.0, 0, 0], [0.1, 0, -1.5]])
    X = np.array([[0.05, -0.02, 1.0]])
    x = np.array([creproj.projection(K, _Rt(R, t)[c]) @ np.append(X[0], 1.0) for c in range(2)])
    x = x[:, :2] / x[:, 2:]
    res = _run(eng, K, R, t, X, np.array([0, 2]), np.array([0, 1], np.int32), x, 1.0, scale_view=-1)
    assert res.report.status == "nonfinite" and res.report.num_observations == 2
    assert not np.isfinite(res.report.cost_start) and _same(res.R, R) and _same(res.t, t) and _same(res.points, X)


def test_refusals(eng):
    K, R, t, X, off, view, x, _ = make_multi_view_scene(30, 4, 14)
    Kv = np.broadcast_to(K, (4, 3, 3))
    Rt = _Rt(R, t)
    fixed = np.array([1, 0, 0, 0], bool)

    def call(K_=Kv, Rt_=Rt, fixed_=fixed, sv=1, off_=off, view_=view, x_=x, X_=X, thr=16.0, it=5):
        return eng.bundle_adjust(K_, Rt_, fixed_, sv, off_, view_, x_, X_, thr, it)

    call()
    bad = lambda: pytest.raises(_native.NativeError)  # noqa: E731
    with bad():
        eng.bundle_adjust(np.zeros((0, 3, 3)), np.zeros((0, 3, 4)), np.zeros(0, bool), -1, off, view, x, X, 16.0)
    for Kb in (np.diag([800.0, 800.0, 0.0]), np.array([[800.0, 0, 640], [0, 800, 480], [0.1, 0, 1]]),
               np.full((3, 3), np.inf)):
        with bad():
            call(K_=np.broadcast_to(Kb, (4, 3, 3)))
    Rn = Rt.copy()
    Rn[2, 1, 3] = np.inf
    with bad():
        call(Rt_=Rn)
    with bad():
        call(fixed_=np.zeros(4, bool))
    for sv in (0, 4, -2):
        with bad():
            call(sv=sv)
    o = off.copy()
    o[2], o[3] = o[3], o[2]
    with bad():
        call(off_=o)
    with bad():
        call(off_=off + 1, view_=np.append(view, 0), x_=np.vstack([x, x[:1]]))
    for v in (-1, 4):
        vv = view.copy()
        vv[3] = v
        with bad():
            call(view_=vv)
    v65 = np.arange(65, dtype=np.int32) % 4
    with bad():
        call(off_=np.array([0, 65]), view_=v65, x_=np.zeros((65, 2)), X_=np.zeros((1, 3)))
    with bad():
        call(thr=np.nan)
    with bad():
        call(it=0)


# ---- 9. engine state --------------------------------------------------------------------------------------------------
def test_engine_state(eng):
    e2, fresh = _native.Engine(0), _native.Engine(0)
    K, R, t, X, off, view, x, _ = make_multi_view_scene(2000, 8, 15, outlier_frac=0.1)
    R0, t0, X0 = _perturb(R, t, X, 16, deg=0.05, tfrac=0.002, xfrac=0.002)
    Kp, Xp, xp, _, _, _ = make_pnp_scene(700, 0.3, seed=12)
    Kt, x1, x2, _, _, _ = make_scene(600, 0.3, seed=3)

    def flow(e, with_ba):
        out = []
        random.seed(3)
        p = ransac_pnp_arrays(Kp, Xp, xp, 4.0, 100, "rms", 300, engine=e, refine_iterations=10)
        out += [p.R, p.t, p.refinement.R, p.err]
        if with_ba:
            _run(e, K, R0, t0, X0, off, view, x, 16.0, max_iterations=5)
        random.seed(6)
        a = two_view_arrays(Kt, x1, x2, 1.5e-6, 10, "rms", 64, engine=e, refine_iterations=10)
        out += [a.R, a.t, a.points, a.ransac.E]
        if with_ba:
            _run(e, K, R0, t0, X0, off, view, x, 16.0, max_iterations=5)
        tr = triangulate_tracks_arrays(K, R0, t0, off, view, x, 16.0, refine_iterations=5, engine=e)
        out += [tr.points, tr.err]
        return out

    for u, w in zip(flow(e2, True), flow(fresh, False)):
        assert _same(u, w)


# ---- 10. the loop -----------------------------------------------------------------------------------------------------
def test_four_view_loop_then_bundle(eng):
    """The flow of test_four_view_composition (both stages refined), then all four views and the ok tracks bundle-
    adjusted with view 1 fixed and view 2 anchored.  Rotation errors against the truth in camera-1 coordinates."""
    K, R, t, X, off, view, x, out = make_multi_view_scene(6000, 4, 42, noise_px=0.5, outlier_frac=0.1, arc_deg=40.0,
                                                          min_len=2, max_len=4)
    T = len(off) - 1
    dense = np.full((T, 4, 2), np.nan)
    seen = np.zeros((T, 4), dtype=bool)
    pt = np.repeat(np.arange(T), np.diff(off))
    dense[pt, view] = x
    seen[pt, view] = True
    Rr = np.array([R[c] @ R[0].T for c in range(4)])
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
    random.seed(3)
    p4 = ransac_pnp_arrays(K, res.points[new], dense[sel[new], 3], 4.0, 10, "rms", 300, engine=eng,
                           refine_iterations=20)
    Ra = np.concatenate([Rs, p4.refinement.R[None]])
    ta = np.concatenate([ts, p4.refinement.t[None]])
    # every track over the four views, triangulated under the four registered poses
    tr = triangulate_tracks_arrays(K, Ra, ta, off, view, x, 4.0, refine_iterations=10, engine=eng)
    X0 = np.where((tr.status == "ok")[:, None], tr.points, np.nan)
    ba = bundle_adjust_arrays(K, Ra, ta, X0, off, view, x, 4.0, fixed=(0,), scale_view=1, max_iterations=50,
                              engine=eng)
    before = max(np.abs(Ra[c] - Rr[c]).max() for c in (1, 2, 3))
    after = max(np.abs(ba.R[c] - Rr[c]).max() for c in (1, 2, 3))
    print(f"four views + bundle: {ba.report.num_points} points, {ba.report.num_observations} observations, "
          f"{ba.report.iterations} iterations ({ba.report.status}); largest R error over views 2-4 {before:.3g} -> "
          f"{after:.3g} ({before / after:.3g}x); cost {ba.report.cost_start:.6g} -> {ba.report.cost_final:.6g}")
    assert ba.report.cost_final < ba.report.cost_start
    assert after * 2 <= before
