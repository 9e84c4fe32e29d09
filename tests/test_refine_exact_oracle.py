"""CPU checks of oracle/refine_exact.py — the exact replay of the least-squares refinement — and of the kernel's own
formulas: the replay's analytic Jacobians against mpmath's numerical derivatives, its optimum against scipy's MINPACK
LM (oracle/refine.py), and a host build of the __host__ __device__ helpers of csrc/sfm_refine.cuh (tools/refine_check.cu)
against the replay at the edges — records near the epipole, H records near the line H sends to infinity, H[2,2] down to
1e-12 of the largest entry, |w| on both sides of refine_rotate's Taylor switch, tied and axis-aligned t.  Each residual
and Jacobian entry is bounded by C u times the sum of the magnitudes of the terms it is made of, times the condition of
its cancelling sums (|s|abs / |s|, na_abs / na, p2_abs / |p2| ...)."""
import ctypes
import os
import subprocess

import mpmath as mp
import numpy as np
import pytest

from oracle import refine as O
from oracle import refine_exact as X
from structure_from_motion_b200.scenes import make_planar_scene, make_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = X.U
C_ROW = 64  # rounding steps in one residual / Jacobian entry, with room


def _normalised(K, p):
    q = np.column_stack([p, np.ones(len(p))]) @ np.linalg.inv(K).T
    return q[:, :2]


def _mpx(kind, x):
    return [mp.mpf(float(v)) for v in x]


# ---- the replay's Jacobians against numerical derivatives --------------------------------------------------------
@pytest.mark.parametrize("kind", ["E", "H"])
def test_jacobians_match_numerical_derivatives(kind):
    rng = np.random.default_rng(1)
    if kind == "E":
        K, x1, x2, R, t, _ = make_scene(12, 0.0, 3)
        pts = np.column_stack([_normalised(K, x1), _normalised(K, x2)])
        x0 = list((R @ O.rodrigues(rng.normal(size=3) * 0.05)).reshape(9)) + list(t / np.linalg.norm(t))
    else:
        K, x1, x2, H, _ = make_planar_scene(12, 0.0, 4)
        pts = np.column_stack([x1, x2])
        x0 = list((H * (1 + 1e-3 * rng.normal(size=(3, 3)))).reshape(9)[:8])
    with mp.workdps(X.DPS):
        x = _mpx(kind, x0)
        P = X._pts(pts)
        for row in P[:6]:
            _, J = X.jacobian_rows(kind, x, *row)
            for k in range(X.NP[kind]):
                def f(e, k=k, row=row):
                    d = [mp.mpf(0)] * X.NP[kind]
                    d[k] = e
                    return X.residuals_at(kind, X.retract(kind, x, d), [row])
                num = [mp.diff(lambda e, i=i: f(e)[i], 0) for i in range(len(J))]
                for i in range(len(J)):
                    assert abs(J[i][k] - num[i]) <= mp.mpf(10) ** (-30) * (1 + abs(num[i])), (kind, k, i)


# ---- the replay's optimum against scipy --------------------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1])
def test_essential_replay_optimum_matches_scipy(seed):
    rng = np.random.default_rng(seed)
    K, x1, x2, R, t, _ = make_scene(150, 0.0, 10 + seed)
    na, nb = _normalised(K, x1), _normalised(K, x2)
    E0 = O.e_from_pose(R @ O.rodrigues(rng.normal(size=3) * 0.02), t + 0.02 * rng.normal(size=3))
    tr = X.replay("E", E0, np.column_stack([na, nb]), 50)
    rep = X.report_after(tr, 50)
    R0, t0 = O.pose_start(E0)
    Eo, co, _ = O.refine_e(R0, t0, na, nb)
    assert rep.status == X.CONVERGED
    assert abs(rep.cost_final - co) <= 1e-9 * co
    Mr = rep.model.reshape(3, 3)
    assert min(np.abs(Mr - Eo).max(), np.abs(Mr + Eo).max()) <= 1e-5 * np.abs(Eo).max()


@pytest.mark.parametrize("seed,rot", [(0, False), (1, True)])
def test_homography_replay_optimum_matches_scipy(seed, rot):
    rng = np.random.default_rng(seed)
    K, x1, x2, H, _ = make_planar_scene(60, 0.0, 20 + seed, rotation_only=rot)
    H0 = H * (1 + 1e-3 * rng.normal(size=(3, 3)))
    tr = X.replay("H", H0, np.column_stack([x1, x2]), 50)
    rep = X.report_after(tr, 50)
    Ho, co = O.refine_h(H0, x1, x2)
    assert rep.status == X.CONVERGED
    assert abs(rep.cost_final - co) <= 1e-9 * co
    assert np.abs(rep.model.reshape(3, 3) - Ho).max() <= 1e-5 * np.abs(Ho).max()


def test_report_after_follows_the_cap():
    K, x1, x2, R, t, _ = make_scene(40, 0.0, 5)
    E0 = O.e_from_pose(R @ O.rodrigues([0.05, -0.02, 0.01]), t + np.array([0.05, 0.0, 0.0]))
    tr = X.replay("E", E0, np.column_stack([_normalised(K, x1), _normalised(K, x2)]), 50)
    full = X.report_after(tr, 50)
    assert full.status == X.CONVERGED and full.iterations >= 2
    one = X.report_after(tr, 1)
    assert one.status == X.MAX_ITER and one.iterations == 1 and one.cost_final < one.cost_start
    for k in range(1, full.iterations):
        rk = X.report_after(tr, k)
        assert rk.iterations == k and rk.cost_final >= full.cost_final


# ---- the host build of the kernel's helpers against the replay ------------------------------------------------------
@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    from structure_from_motion_b200 import build as b

    try:
        nvcc = b._nvcc()
    except RuntimeError:
        pytest.skip("no nvcc: the host build of sfm_refine.cuh cannot be made")
    out = str(tmp_path_factory.mktemp("refine") / "librefine.so")
    subprocess.check_call([nvcc, "-O2", "-shared", "-Xcompiler", "-fPIC", "-Wno-deprecated-gpu-targets", "-o", out,
                           os.path.join(ROOT, "tools", "refine_check.cu")])
    L = ctypes.CDLL(out)
    L.e_residual.restype = ctypes.c_double
    return L


def P(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _e_host(lib, E, c):
    g = np.empty(9)
    r = lib.e_residual(P(np.ascontiguousarray(E, dtype=np.float64)), P(np.ascontiguousarray(c, dtype=np.float64)), P(g))
    return r, g


def _e_bound(E, c):
    """(exact r, exact gE, bound on |r|, bound on each |gE|): C u times the absolute terms times the condition."""
    E = np.asarray(E, dtype=np.float64)
    with mp.workdps(X.DPS):
        Em = [mp.mpf(float(v)) for v in E]
        cm = [mp.mpf(float(v)) for v in c]
        r, g = X.e_residual(Em, *cm)
        a, b = [cm[0], cm[1], 1], [cm[2], cm[3], 1]
        la = [sum(Em[3 * j + k] * a[k] for k in range(3)) for j in range(3)]
        lb = [sum(Em[3 * i + j] * b[i] for i in range(3)) for j in range(3)]
        la_abs = [sum(abs(Em[3 * j + k] * a[k]) for k in range(3)) for j in range(3)]
        lb_abs = [sum(abs(Em[3 * i + j] * b[i]) for i in range(3)) for j in range(3)]
        s = sum(lb[j] * a[j] for j in range(3))
        s_abs = sum(lb_abs[j] * abs(a[j]) for j in range(3))
        na, nb = la[0] ** 2 + la[1] ** 2, lb[0] ** 2 + lb[1] ** 2
        na_abs, nb_abs = la_abs[0] ** 2 + la_abs[1] ** 2, lb_abs[0] ** 2 + lb_abs[1] ** 2
        cond = 1 + s_abs / abs(s) + na_abs / na + nb_abs / nb if s != 0 else mp.inf
        w = mp.sqrt(1 / na + 1 / nb)
        ca, cb = abs(s) / w / na ** 2, abs(s) / w / nb ** 2
        gb = [float(C_ROW * U * (1 + na_abs / na + nb_abs / nb)
                    * (w * abs(b[j] * a[k]) + (ca * la_abs[j] * abs(a[k]) if j < 2 else 0)
                       + (cb * lb_abs[k] * abs(b[j]) if k < 2 else 0)))
              for j in range(3) for k in range(3)]
        return float(r), np.array([float(v) for v in g]), float(C_ROW * U * cond * abs(r)), np.array(gb)


def test_e_residual_near_the_epipole(lib):
    """Records a with |(E a)_0,1|^2 from 1 down to 1e-30: residual and gradient within C u cond of the exact ones."""
    rng = np.random.default_rng(7)
    worst = 0.0
    for _ in range(4):
        Rr = O.rodrigues(rng.normal(size=3) * 0.2)
        t = rng.normal(size=3)
        E = O.e_from_pose(Rr, t).reshape(9)
        e = np.linalg.svd(E.reshape(3, 3))[2][-1]
        ea = e[:2] / e[2]   # the epipole in image A: E (ea, 1) = 0
        for d in [1e-0, 1e-3, 1e-6, 1e-9, 1e-12, 1e-15]:
            a = ea + d * rng.normal(size=2)
            b = rng.normal(size=2) * 0.3
            c = np.array([a[0], a[1], b[0], b[1]])
            r, g = _e_host(lib, E, c)
            re, ge, rb, gb = _e_bound(E, c)
            assert abs(r - re) <= rb, (d, r, re, rb)
            assert (np.abs(g - ge) <= gb).all(), (d, g - ge, gb)
            worst = max(worst, abs(r - re) / rb, float((np.abs(g - ge) / gb).max()))
    print(f"near-epipole worst ratio {worst:.3g}")


def test_e_model_against_the_replay(lib):
    """E = [t]x R and its 9 x 5 derivative, for t along each axis, with tied smallest components, and generic: within
    8 u of the exact ones (|R| = |t| = 1), and the same tangent axis as the replay (first on ties)."""
    rng = np.random.default_rng(8)
    ts = [np.eye(3)[k] for k in range(3)] + [-np.eye(3)[k] for k in range(3)]
    ts += [np.array([1.0, 1.0, 1.0]), np.array([0.3, 0.3, 0.9]), np.array([0.2, 0.9, 0.2]), np.array([0.9, -0.1, 0.1]),
           np.array([0.0, 0.6, 0.0]), rng.normal(size=3)]
    for t in ts:
        t = t / np.linalg.norm(t)
        R = O.rodrigues(rng.normal(size=3))
        E, M = np.empty(9), np.empty(45)
        lib.e_model(P(np.ascontiguousarray(R.reshape(9))), P(t), P(E), P(M))
        b1, b2 = np.empty(3), np.empty(3)
        lib.tangent_basis(P(t), P(b1), P(b2))
        with mp.workdps(X.DPS):
            Rm, tm = [mp.mpf(float(v)) for v in R.reshape(9)], [mp.mpf(float(v)) for v in t]
            Ee, cols = X.e_model(Rm, tm)
            e1, e2 = X.tangent_basis(tm)
            assert np.abs(E - np.array([float(v) for v in Ee])).max() <= 8 * U
            Me = np.array([[float(cols[p][j]) for p in range(5)] for j in range(9)]).reshape(45)
            assert np.abs(M - Me).max() <= 8 * U, t
            assert np.abs(b1 - np.array([float(v) for v in e1])).max() <= 8 * U, t
            assert np.abs(b2 - np.array([float(v) for v in e2])).max() <= 8 * U, t


def test_rotate_on_both_sides_of_the_taylor_switch(lib):
    """R exp([w]x) for |w| from 1e-12 to 1, across the 1e-4 switch: within 8 u of the exact rotation."""
    rng = np.random.default_rng(9)
    for th in [0.0, 1e-12, 1e-8, 1e-5, 9.9e-5, 1e-4 * (1 - 1e-15), 1e-4, 1.01e-4, 1e-3, 0.1, 1.0]:
        R = O.rodrigues(rng.normal(size=3))
        w = rng.normal(size=3)
        w = w / np.linalg.norm(w) * th
        out = np.empty(9)
        lib.rotate(P(np.ascontiguousarray(R.reshape(9))), P(w), P(out))
        with mp.workdps(X.DPS):
            ex = X.rotate([mp.mpf(float(v)) for v in R.reshape(9)], [mp.mpf(float(v)) for v in w])
            assert np.abs(out - np.array([float(v) for v in ex])).max() <= 8 * U, th


def _h_bound(h, c):
    with mp.workdps(X.DPS):
        hm = [mp.mpf(float(v)) for v in h]
        cm = [mp.mpf(float(v)) for v in c]
        r, J = X.h_residuals(hm, *cm)
        a, b = [cm[0], cm[1], 1], [cm[2], cm[3], 1]
        ad = X.adj(hm)
        adab = X.adj([abs(v) for v in hm])  # the magnitude of each adjugate entry's terms (2 products)
        p2, q2 = sum(hm[6 + k] * a[k] for k in range(3)), sum(ad[6 + k] * b[k] for k in range(3))
        p_abs = [sum(abs(hm[3 * i + k] * a[k]) for k in range(3)) for i in range(3)]
        q_abs = [sum(abs(adab[3 * i + k]) * abs(b[k]) for k in range(3)) for i in range(3)]
        cp = 1 + p_abs[2] / abs(p2)
        cq = 1 + q_abs[2] / abs(q2)
        rb = [C_ROW * U * cp * (p_abs[0] / abs(p2) + abs(b[0])), C_ROW * U * cp * (p_abs[1] / abs(p2) + abs(b[1])),
              C_ROW * U * cq * (q_abs[0] / abs(q2) + abs(a[0])), C_ROW * U * cq * (q_abs[1] / abs(q2) + abs(a[1]))]
        # each Jacobian entry is (d_num - u d_den) / den with the same cancellations, derivatives of at most 4 terms
        hmax = max(abs(v) for v in hm)
        dq_abs = 2 * hmax * (abs(b[0]) + abs(b[1]) + 1)
        Jb = [[C_ROW * U * cp * (1 + p_abs[0] / abs(p2) + p_abs[1] / abs(p2)) * (abs(a[0]) + abs(a[1]) + 1) / abs(p2)] * 8,
              [C_ROW * U * cp * (1 + p_abs[0] / abs(p2) + p_abs[1] / abs(p2)) * (abs(a[0]) + abs(a[1]) + 1) / abs(p2)] * 8,
              [C_ROW * U * cq * (1 + q_abs[0] / abs(q2) + q_abs[1] / abs(q2)) * dq_abs / abs(q2)] * 8,
              [C_ROW * U * cq * (1 + q_abs[0] / abs(q2) + q_abs[1] / abs(q2)) * dq_abs / abs(q2)] * 8]
        return (np.array([float(v) for v in r]), np.array([[float(v) for v in row] for row in J]),
                np.array([float(v) for v in rb]), np.array([[float(v) for v in row] for row in Jb]))


def _h_host(lib, h, c):
    r, J = np.empty(4), np.empty(32)
    lib.h_residuals(P(np.ascontiguousarray(h, dtype=np.float64)), P(np.ascontiguousarray(c, dtype=np.float64)), P(r), P(J))
    return r, J.reshape(4, 8)


@pytest.mark.parametrize("h22", [1.0, 1e-3, 1e-6, 1e-9, 1e-12])
def test_h_residuals_as_h22_vanishes(lib, h22):
    """H with H[2,2] = h22 times its largest entry, scaled to h8 = 1 (the refinement's gauge): residuals and Jacobian
    rows within C u cond of the exact ones, on records spread over the image."""
    K, x1, x2, H, _ = make_planar_scene(30, 0.0, 5, rotation_only=True)
    Hs = H / np.abs(H).max()
    Hs[2, 2] = h22
    h = (Hs / Hs[2, 2]).reshape(9)
    h[8] = 1.0
    worst = 0.0
    for a, b in zip(x1, x2):
        c = np.array([a[0], a[1], b[0], b[1]])
        r, J = _h_host(lib, h, c)
        re, Je, rb, Jb = _h_bound(h, c)
        assert (np.abs(r - re) <= rb).all(), (h22, r - re, rb)
        assert (np.abs(J - Je) <= Jb).all(), (h22, np.abs(J - Je) / Jb)
        worst = max(worst, float((np.abs(r - re) / rb).max()), float((np.abs(J - Je) / Jb).max()))
    print(f"h22 {h22:g} worst ratio {worst:.3g}")


def test_h_residuals_near_the_line_at_infinity(lib):
    """Records a whose p2 = (H a)_2 is 1e-3 down to 1e-15 of its terms: within C u cond of the exact rows."""
    K, x1, x2, H, _ = make_planar_scene(5, 0.0, 6)
    h = (H / H[2, 2]).reshape(9)
    rng = np.random.default_rng(6)
    worst = 0.0
    for d in [1e-3, 1e-6, 1e-9, 1e-12, 1e-15]:
        xa = rng.uniform(0, 1280)
        ya = -(h[6] * xa + h[8]) / h[7] + d * abs((h[6] * xa + h[8]) / h[7]) * rng.normal()
        b = rng.uniform(0, 1000, 2)
        c = np.array([xa, ya, b[0], b[1]])
        r, J = _h_host(lib, h, c)
        re, Je, rb, Jb = _h_bound(h, c)
        assert (np.abs(r - re) <= rb).all(), (d, r - re, rb)
        assert (np.abs(J - Je) <= Jb).all(), (d, np.abs(J - Je) / Jb)
        worst = max(worst, float((np.abs(r - re) / rb).max()), float((np.abs(J - Je) / Jb).max()))
    print(f"near-infinity worst ratio {worst:.3g}")
