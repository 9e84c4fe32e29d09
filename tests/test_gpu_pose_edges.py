"""The essential-matrix pose tail — decompose_essential (svd3_rank2_frames, Jacobi fallback), the cheirality test and
vote, dlt_triangulate (null_vector4_fast, Jacobi fallback) — against the exact references of oracle/pose_exact.py,
through the stand-alone calls (k_decompose, k_cheirality, k_vote, k_triangulate) and the fused tail (T1, T2, T3).

Bounds (u = 2^-53; s0 >= s1 >= s2 the exact singular values of E, sigma_1..4 those of a 4x4 DLT system A):
- null vector: the residual excess |A xh| - sigma_4 of the returned point (xh = [X, 1] / |[X, 1]|) is at most
  C_RES u sigma_1 (backward stability); its direction is within C_FWD u / gap + STOP(q) of the exact one, where
  gap = (sigma_3 - sigma_4) / sigma_1 (the perturbation bound of a singular subspace) and STOP(q) = 8e-13 q / (1 - q),
  q = (sigma_4 / sigma_3)^4, is what null_vector4_fast's absolute stopping rule (two steps within 1e-13, each step
  contracting the error by (sigma_4 / sigma_3)^2) leaves behind (0 when the Jacobi SVD answered); X is within that
  direction bound times 2 |[X*, 1]|^2 (the dehomogenisation divides by x4 = 1 / |[X*, 1]|);
- decomposition: the candidate set (R1, R2, +-t) is within C_FRAME u cond of the exact set, cond = s0 / (s1 - s2) (the
  separation of the null vectors; the closed form's cross products err by u s0 / s1 in direction); R1, R2 are proper
  and orthonormal to C_ORTH u and |t| = 1 to C_ORTH u; the reported s2 is within C_SV u s0 cond of the exact s2 (the
  closed form reports the component of E v3 along u2, whose v3 and u2 carry the frame error); the np.isclose(0, s2)
  decision equals the exact one wherever the exact s2 is further than that from the limit, and numpy's wherever numpy's
  s[-1] is too - the sweep includes E with s0 = 4 and s2 just below the limit, which the closed form takes;
- scale: E 2^k and (P1, P2) 2^k give bit-identical candidates and points, for every k in [-1000, 1000] that keeps
  the input exact;
- cheirality: a pass bit equals the exact decision (depths >= -1e-8, |X| <= distance threshold, at the exact X of
  the device's candidate pose) wherever each quantity is further from its limit than the X bound above moves it, and
  numpy's decision there too; the vote is the first maximum of the counts; no votes raise EightPointCalculationError;
- fused tail: pose, counts and pass bits equal recover_pose_arrays(camera_matrix=K) on the same list; the points are
  within the X bound of the exact DLT in pixel coordinates, and T2 (<= 512 inliers) and T3 give the same bits;
- non-finite input: what tests/golden/pose_nonfinite_fixture.json recorded from the unmodified reference.
"""
import json
import os

import numpy as np
import pytest

from oracle import pose_exact as px
from oracle import restatement as o
from structure_from_motion_b200 import two_view
from structure_from_motion_b200.errors import EightPointCalculationError

pytestmark = pytest.mark.gpu
U = px.U
C_RES, C_FWD, C_FRAME, C_ORTH, C_SV = 16, 64, 64, 16, 64
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
Z4 = np.zeros((1, 2))
WORST = {}


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same(a, b):
    return np.array_equal(bits(a), bits(b))


def note(key, ratio):
    WORST[key] = max(WORST.get(key, 0.0), float(ratio))


def stop_term(s):
    q = (s[3] / s[2]) ** 4 if s[2] > 0 else 1.0
    return 8e-13 * q / (1.0 - q) if q < 1.0 else np.inf


def dir_bound(ex, fast=True):
    return C_FWD * U / max(ex.gap, 1e-300) + (stop_term(ex.s) if fast else 0.0)


def x_bound(ex, db):
    return 2.0 * db * (1.0 + float(np.dot(ex.X, ex.X)))


def tri(P1, P2, a=Z4, b=Z4):
    return two_view.triangulate_arrays(a, b, P1, P2)


def check_point(X, A, key, fast=True):
    ex = px.null_exact(A)
    res = px.residual_excess(A, X)
    note(f"{key} residual / (u sigma_1)", res / (U * ex.s[0]))
    assert res <= C_RES * U * ex.s[0], (key, res, ex.s)
    if ex.gap > 1e-6:
        db = dir_bound(ex, fast)
        d = px.direction_error(X, ex)
        note(f"{key} direction / bound", d / db)
        assert d <= db, (key, d, db, ex.s)
        if np.isfinite(ex.X).all():
            xb = x_bound(ex, db)
            e = float(np.abs(np.asarray(X) - ex.X).max())
            note(f"{key} X / bound", e / xb)
            assert e <= xb, (key, e, xb)
    return ex


@pytest.fixture(scope="module", autouse=True)
def report():
    yield
    for k in sorted(WORST):
        print(f"worst {k}: {WORST[k]:.3g}")


# ---------------------------------------------------------------------------------------------------------------------
# null vector
# ---------------------------------------------------------------------------------------------------------------------
def test_null_vector_on_constructed_systems_across_the_fallback_switch(engine):
    for fam, r, A in px.null_sweep():
        P1, P2 = px.cameras_for(A)
        X = tri(P1, P2)[0]
        # the route: <= NULL_FAST_MAX the fast one (test_pose_oracle confirms it on the host build), >= the switch the
        # Jacobi SVD; in between no stopping-rule term is granted to either
        fast = r <= px.NULL_FAST_MAX
        check_point(X, A, f"null {fam} {'fast' if fast else 'jacobi'}", fast=fast)


def test_null_vector_on_real_dlt_systems(engine):
    rng = np.random.default_rng(8)
    K = np.array([[800.0, 0.0, 640.0], [0.0, 800.0, 480.0], [0.0, 0.0, 1.0]])
    for parallax in (1e-1, 1e-3, 1e-5, 1e-7):
        R, t, na, nb = px.scene(40, rng, parallax=parallax, noise=1e-5)
        P2n = np.hstack([R, t[:, None]])
        Xn = tri(np.eye(4)[:3], P2n, na, nb)
        pa = na * 800.0 + [640.0, 480.0]
        pb = nb * 800.0 + [640.0, 480.0]
        P1p, P2p = two_view.camera_matrices(K, o.tmat(R, t))
        Xp = tri(P1p, P2p, pa, pb)
        for i in range(len(na)):
            check_point(Xn[i], px.dlt_system(*na[i], *nb[i], np.eye(4)[:3], P2n), "dlt normalised")
            check_point(Xp[i], px.dlt_system(*pa[i], *pb[i], P1p[:3], P2p[:3]), "dlt pixel")


def test_null_vector_noise_free_clamp_and_points_on_the_baseline(engine):
    # an exactly consistent system: X = (1, 2, 4), camera 2 = [I | (1, 0, 0)] -> sigma_4 = 0, R's last pivot clamped
    P2 = np.hstack([np.eye(3), [[1.0], [0.0], [0.0]]])
    X = tri(np.eye(4)[:3], P2, np.array([[0.25, 0.5]]), np.array([[0.5, 0.5]]))[0]
    assert np.abs(X - [1.0, 2.0, 4.0]).max() <= 64 * U * 4, X
    # a point on the baseline: both rays lie along t and the null space is two-dimensional, spanned by the first
    # camera's centre (0, 0, 0, 1) and the point at infinity (t, 0).  Which vector of that plane comes back is
    # arbitrary: numpy's SVD returns the centre (X = 0), the device's QR and inverse iteration the point at infinity.
    # Both are exact null vectors and neither passes the cheirality test (the centre lies at depth -t[2] = -1 in the
    # second camera, the point at infinity beyond any distance threshold), so the vote does not depend on the choice.
    t = np.array([0.3, 0.1, 1.0])
    P2 = np.hstack([np.eye(3), -t[:, None]])
    a = np.array([[0.3, 0.1]])
    X = tri(np.eye(4)[:3], P2, a, a)[0]
    A = px.dlt_system(0.3, 0.1, 0.3, 0.1, np.eye(4)[:3], P2)
    ex = px.null_exact(A)
    assert ex.s[2] <= 4 * U * ex.s[0] and ex.s[3] <= 4 * U * ex.s[0], ex.s
    if np.isfinite(X).all():
        assert np.abs(A @ np.append(X, 1.0)).max() <= 64 * U * ex.s[0] * (1 + np.abs(X).max())
    else:
        assert np.isinf(X).all(), X


def test_null_vector_is_bit_identical_under_power_of_two_scaling(engine):
    cases = px.null_sweep(trials=1)[::3]
    rng = np.random.default_rng(9)
    R, t, na, nb = px.scene(4, rng, parallax=0.05, noise=1e-4)
    P2n = np.hstack([R, t[:, None]])
    for k in (-1000, -700, -300, -101, -100, -60, -1, 1, 60, 100, 101, 300, 700, 1000):
        for fam, r, A in cases:
            P1, P2 = px.cameras_for(A)
            S1, S2 = np.ldexp(P1, k), np.ldexp(P2, k)
            if not (np.array_equal(np.ldexp(S1, -k), P1) and np.array_equal(np.ldexp(S2, -k), P2)):
                continue
            assert same(tri(S1, S2), tri(P1, P2)), (fam, r, k)
        S1, S2 = np.ldexp(np.eye(4)[:3], k), np.ldexp(P2n, k)
        if np.array_equal(np.ldexp(S2, -k), P2n):
            assert same(tri(S1, S2, na, nb), tri(np.eye(4)[:3], P2n, na, nb)), k


# ---------------------------------------------------------------------------------------------------------------------
# decomposition
# ---------------------------------------------------------------------------------------------------------------------
def candidates(p):
    R = np.array(p.R, dtype=np.float64).reshape(4, 3, 3)
    t = np.array(p.t, dtype=np.float64).reshape(4, 3)
    return R, t


def test_decomposition_against_the_exact_candidates(engine):
    decided = {"exact": 0, "numpy": 0, "band": 0}
    for name, E in px.decomposition_sweep():
        ex = px.decompose_exact(E)
        p = engine.decompose_essential(E)
        R, t = candidates(p)
        assert same(R[0], R[1]) and same(R[2], R[3]) and same(t[0], -t[1]) and same(t[0], t[2]) and same(t[1], t[3])
        er, et = px.candidate_error(R[0], R[2], t[0], ex)
        # a rank-3 E: the closed form's cross products are null vectors of its rank-2 part, s2 / (s1 - s2) away
        fb = C_FRAME * U * ex.cond + 2.0 * ex.s[2] / (ex.s[1] - ex.s[2])
        note("decomposition candidates / bound", max(er, et) / fb)
        assert er <= fb and et <= fb, (name, er, et, ex.cond)
        for Rk in (R[0], R[2]):
            assert np.abs(Rk.T @ Rk - np.eye(3)).max() <= C_ORTH * U, name
            assert abs(np.linalg.det(Rk) - 1.0) <= C_ORTH * U, name
        assert abs(np.linalg.norm(t[0]) - 1.0) <= C_ORTH * U, name
        sb = C_SV * U * ex.s[0] * ex.cond
        note("decomposition s2 / bound", abs(p.sv[2] - ex.s[2]) / sb)
        assert abs(p.sv[2] - ex.s[2]) <= sb, (name, p.sv[2], ex.s[2], sb)
        try:
            two_view.recover_all_r_t_arrays(E, engine=engine)
            accepted = True
        except EightPointCalculationError:
            accepted = False
        if abs(ex.s[2] - px.SV_LIMIT) > sb:
            decided["exact"] += 1
            decided["band"] += name.startswith("s2_band_")
            assert accepted == ex.accepted, (name, ex.s, p.sv[2])
        s_np = np.linalg.svd(E, compute_uv=False)[-1]
        if abs(s_np - px.SV_LIMIT) > sb + 8 * U * ex.s[0]:
            decided["numpy"] += 1
            assert accepted == bool(np.isclose(0.0, s_np)), (name, s_np, p.sv[2])
    assert decided["exact"] > 40 and decided["numpy"] > 40 and decided["band"] >= 50, decided


def test_decomposition_is_bit_identical_under_power_of_two_scaling(engine):
    for name, E in px.decomposition_sweep(trials=1):
        p0 = engine.decompose_essential(E)
        R0, t0 = candidates(p0)
        for k in (-1000, -800, -500, -300, -101, -100, -50, -1, 1, 50, 100, 101, 300, 500, 800, 1000):
            Ek = np.ldexp(E, k)
            if not np.array_equal(np.ldexp(Ek, -k), E):
                continue
            p = engine.decompose_essential(Ek)
            R, t = candidates(p)
            assert same(R, R0) and same(t, t0), (name, k)
            assert same(np.array(p.sv), np.ldexp(np.array(p0.sv), k)), (name, k)


# ---------------------------------------------------------------------------------------------------------------------
# cheirality and vote
# ---------------------------------------------------------------------------------------------------------------------
def edge_points(rng, R, t):
    """Normalised correspondences of points near the limits: depth about -1e-8 in camera 1 or 2, |X| about 50, and
    points far away (near infinity)."""
    pts = []
    for z in (-1e-8 * 0.5, -1e-8 * 2.0, 1e-3):
        pts.append(np.array([0.1 * z, -0.05 * z, z]))
    # depth about -1e-8 in camera 2: X = R^T (Xc2 - t)
    for z in (-1e-8 * 0.5, -1e-8 * 2.0):
        Xc2 = np.array([0.2 * 0.5, 0.1 * 0.5, z])
        pts.append(R.T @ (Xc2 - t))
    for f in (1 - 1e-3, 1 + 1e-3, 1 - 1e-10, 1 + 1e-10):
        d = np.array([0.1, -0.2, 1.0])
        pts.append(d / np.linalg.norm(d) * 50.0 * f)
    for zf in (1e3, 1e6, 1e9):
        pts.append(np.array([0.3 * zf, 0.1 * zf, zf]))
    X = np.array(pts)
    Xb = X @ R.T + t
    return X[:, :2] / X[:, 2:3], Xb[:, :2] / Xb[:, 2:3]


def check_pose(engine, E, na, nb, dist_thr=50.0, K=None, clear_count=None):
    if K is None:
        res = two_view.recover_pose_arrays(E, na, nb, dist_thr, engine=engine)
        ca, cb = na, nb
    else:
        res = two_view.recover_pose_arrays(E, na, nb, dist_thr, engine=engine, camera_matrix=K)
        ca = np.stack(o.k_normalise(na[:, 0], na[:, 1], K), 1)
        cb = np.stack(o.k_normalise(nb[:, 0], nb[:, 1], K), 1)
    p, pass4 = engine.recover_pose(E, ca, cb, dist_thr)
    counts = np.array(p.counts)
    assert np.array_equal(counts, res.counts)
    assert int(p.best) == int(np.argmax(counts))
    for q, (Rq, tq) in enumerate(res.candidates):
        for i in range(len(ca)):
            c = px.cheirality_exact(*ca[i], *cb[i], Rq, tq, lambda ex: x_bound(ex, dir_bound(ex)))
            bit = bool((pass4[i] >> q) & 1)
            if c.clear(dist_thr):
                if clear_count is not None:
                    clear_count[c.passes(dist_thr)] += 1
                assert bit == c.passes(dist_thr), (i, q, c)
                assert bit == o.cheirality_check(*ca[i], *cb[i], Rq, tq, dist_thr), (i, q)
    want = np.array([np.count_nonzero(np.nonzero((pass4 >> q) & 1)[0]) for q in range(4)])
    assert np.array_equal(counts, want)
    return res, pass4


def test_cheirality_decisions_at_their_edges(engine):
    rng = np.random.default_rng(12)
    tally = {True: 0, False: 0}
    K = np.array([[700.0, 0.0, 320.0], [0.0, 710.0, 240.0], [0.0, 0.0, 1.0]])
    for parallax in (1e-1, 1e-3, 1e-5, 1e-7):
        R, t, na, nb = px.scene(24, rng, parallax=parallax, noise=1e-6, depth=(2.0, 60.0))
        ea, eb = edge_points(rng, R, t)
        na, nb = np.vstack([na, ea]), np.vstack([nb, eb])
        E = px.essential_of(R, t)
        check_pose(engine, E, na, nb, clear_count=tally)
        pa = np.stack([na[:, 0] * 700.0 + 320.0, na[:, 1] * 710.0 + 240.0], 1)
        pb = np.stack([nb[:, 0] * 700.0 + 320.0, nb[:, 1] * 710.0 + 240.0], 1)
        check_pose(engine, E, pa, pb, K=K, clear_count=tally)
    assert tally[True] > 50 and tally[False] > 500, tally


def test_vote_ties_pick_the_first_maximum_and_no_votes_raise(engine):
    R = px.rotation([0.0, 1.0, 0.0], 0.05)
    t = np.array([1.0, 0.1, 0.05])
    E = px.essential_of(R, t)
    front = np.array([0.2, -0.1, 5.0])
    behind = -front  # behind both cameras: passes the candidate with -t, as the front point passes the true one
    X = np.array([[0.1, 0.1, 4.0], front, behind])
    Xb = X @ R.T + t
    na, nb = X[:, :2] / X[:, 2:3], Xb[:, :2] / Xb[:, 2:3]
    res, _ = check_pose(engine, E, na, nb)
    c = res.counts
    assert sorted(c.tolist()) == [0, 0, 1, 1], c
    assert int(np.argmax(c)) == int(np.flatnonzero(c == 1)[0])
    Rr, tr, _, cr = o.recover_r_t(na[:, 0], na[:, 1], nb[:, 0], nb[:, 1], E)
    assert np.array_equal(np.sort(c), np.sort(cr))
    # one correspondence: index 0 never counts -> no votes
    with pytest.raises(EightPointCalculationError):
        two_view.recover_pose_arrays(E, na[:1], nb[:1], engine=engine)
    with pytest.raises(o.OracleEightPointError):
        o.recover_r_t(na[:1, 0], na[:1, 1], nb[:1, 0], nb[:1, 1], E)


# ---------------------------------------------------------------------------------------------------------------------
# fused tail against the stand-alone calls
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def fused_scene():
    rng = np.random.default_rng(21)
    K = np.array([[800.0, 0.0, 640.0], [0.0, 800.0, 480.0], [0.0, 0.0, 1.0]])
    R, t, na, nb = px.scene(5000, rng, parallax=0.05, noise=2e-4, depth=(2.0, 40.0))
    pa = na * 800.0 + [640.0, 480.0]
    pb = nb * 800.0 + [640.0, 480.0]
    return K, px.essential_of(R, t), pa, pb


@pytest.mark.parametrize("m", [511, 512, 513, 1023, 1024, 1025, 5000])
def test_fused_tail_equals_the_stand_alone_calls(engine, fused_scene, m):
    K, E, pa, pb = fused_scene
    a, b = pa[:m], pb[:m]
    engine.upload_pairs(a, b, K)
    engine.set_winner(-1, E)
    p, num, idx, ok, X = engine.pose_and_triangulate(1e100, 50.0)
    assert num == m and np.array_equal(idx, np.arange(m))
    res = two_view.recover_pose_arrays(E, a, b, 50.0, engine=engine, camera_matrix=K)
    ps, pass4 = engine.recover_pose(E, np.stack(o.k_normalise(a[:, 0], a[:, 1], K), 1),
                                    np.stack(o.k_normalise(b[:, 0], b[:, 1], K), 1), 50.0)
    assert np.array_equal(np.array(p.counts), res.counts)
    assert np.array_equal(ok, pass4)
    bst = int(p.best)
    R, t = candidates(p)
    assert same(R[bst], res.R) and same(t[bst], res.t)
    passing = ((ok >> bst) & 1).astype(bool)
    assert np.isnan(X[~passing]).all() and np.isfinite(X[passing]).all()
    P1, P2 = two_view.camera_matrices(K, o.tmat(R[bst], t[bst]))
    rng = np.random.default_rng(m)
    pick = np.unique(np.concatenate([rng.choice(np.flatnonzero(passing), 60, replace=False),
                                     np.flatnonzero(passing)[-4:]]))
    for i in pick:
        check_point(X[i], px.dlt_system(*a[i], *b[i], P1[:3], P2[:3]), "fused tail pixel")
    Xs = tri(P1, P2, a, b)
    assert np.abs(Xs[passing] - X[passing]).max() <= 1e-9 * max(1.0, np.abs(X[passing]).max())
    if m == 513:
        engine.upload_pairs(pa[:512], pb[:512], K)
        engine.set_winner(-1, E)
        p2, num2, _, ok2, X2 = engine.pose_and_triangulate(1e100, 50.0)
        assert num2 == 512 and int(p2.best) == bst and np.array_equal(ok2, ok[:512])
        assert same(X2, X[:512])  # T2 triangulated these, T3 the 513 above


# ---------------------------------------------------------------------------------------------------------------------
# non-finite input
# ---------------------------------------------------------------------------------------------------------------------
def test_non_finite_input_follows_the_reference(engine):
    """tests/golden/pose_nonfinite_fixture.json, from the unmodified reference: numpy's LinAlgError where a NaN reaches
    its SVD (or an infinite coordinate does, through the DLT rows), EightPointCalculationError for an infinite E (the
    check of U) and for a rank-3 E ahead of a NaN coordinate, and non-finite points for an infinite camera entry.
    For those points only finiteness is compared, not NaN against inf: numpy's SVD of a system with an infinite (and
    no NaN) entry is not defined by LAPACK, and its output pattern is the build's - the reference returned all NaN
    for an infinite entry of P1 and [NaN, inf, NaN] for the same entry of P2, where the device's QR gives NaN."""
    with open(os.path.join(GOLDEN, "pose_nonfinite_fixture.json")) as fh:
        cases = json.load(fh)["cases"]
    kinds = {"numpy.linalg.LinAlgError": np.linalg.LinAlgError,
             "lib.epipolar.eight_point.EightPointCalculationError": EightPointCalculationError}
    for c in cases:
        arr = {k: np.array(v, dtype=np.float64) for k, v in c.items() if k in ("E", "pts_a", "pts_b", "P1", "P2")}
        if c["call"] == "recover_all_r_t":
            run = lambda: two_view.recover_all_r_t_arrays(arr["E"], engine=engine)  # noqa: E731
        elif c["call"] == "recover_r_t":
            run = lambda: two_view.recover_pose_arrays(arr["E"], arr["pts_a"], arr["pts_b"], engine=engine)  # noqa: E731
        else:
            run = lambda: two_view.triangulate_arrays(arr["pts_a"], arr["pts_b"], arr["P1"], arr["P2"], engine=engine)  # noqa: E731
        if c["raises"]:
            with pytest.raises(kinds[c["raises"]]):
                run()
        else:
            got = run()
            want = np.array(c["result"], dtype=np.float64)
            assert np.array_equal(np.isfinite(got), np.isfinite(want)), (c["name"], got, want)
