"""CPU checks of the PnP pose refinement's oracle (oracle/pnp_refine.py) and of a host build of the kernel's residual
helper (tools/pnp_refine_check.cu, refine_p_residuals of csrc/sfm_refine.cuh).  No GPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import creproj
from oracle import pnp as opnp
from oracle import pnp_refine as opr
from oracle.refine import rodrigues
from structure_from_motion_b200.scenes import make_pnp_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = 2.0 ** -53


def _scene(n=300, noise=0.5, seed=3, outliers=0.0):
    return make_pnp_scene(n, outliers, seed=seed, noise_px=noise)


def test_jacobian_matches_central_differences():
    K, X, x, R, t, _ = _scene(40)
    rng = np.random.default_rng(1)
    R0 = R @ rodrigues(rng.normal(0, 0.02, 3))
    t0 = t + rng.normal(0, 0.02, 3)
    J = opr.jacobian(R0, t0, K, X, x).reshape(-1, 6)
    h = 1e-6
    for k in range(6):
        z = np.zeros(6)
        z[k] = h
        rp = opr.residuals(R0 @ rodrigues(z[:3]), t0 + z[3:], K, X, x).ravel()
        rm = opr.residuals(R0 @ rodrigues(-z[:3]), t0 - z[3:], K, X, x).ravel()
        num = (rp - rm) / (2 * h)
        assert np.allclose(J[:, k], num, rtol=1e-6, atol=1e-6 * np.abs(J).max()), k


def test_cost_equals_the_scorers_value():
    """r0^2 + r1^2 is the squared reprojection error RANSAC scores: oracle/pnp.reproj and reproj_exact.c agree with
    it to rounding."""
    K, X, x, R, t, _ = _scene(500, outliers=0.2)
    Rt = np.column_stack([R, t])
    r = opr.residuals(R, t, K, X, x)
    per = np.sum(r * r, axis=1)
    _, v_np = opnp.reproj(Rt, K, X, x, np.inf)
    _, v_c = creproj.reproj_exact_many(Rt, K, X, x, np.inf)
    assert np.allclose(per, v_np, rtol=1e-9, atol=1e-12)
    assert np.allclose(per, v_c, rtol=1e-9, atol=1e-12)
    assert abs(per.sum() - v_c.sum()) <= 1e-9 * v_c.sum()


def test_true_pose_is_stationary_on_noise_free_data():
    K, X, x, R, t, _ = _scene(200, noise=0.0)
    r = opr.residuals(R, t, K, X, x).ravel()
    J = opr.jacobian(R, t, K, X, x).reshape(-1, 6)
    assert opr.cost(R, t, K, X, x) < 1e-18
    g = J.T @ r
    assert np.abs(g).max() < 1e-9 * np.abs(J).max()


def test_scipy_from_a_p3p_start_lowers_the_cost_and_approaches_the_truth():
    K, X, x, R, t, out = _scene(1000, noise=0.5, outliers=0.3, seed=5)
    inl = np.setdiff1d(np.arange(len(X)), out)
    rng = np.random.default_rng(2)
    done = 0
    for _ in range(20):
        s = rng.choice(inl, 4, replace=False)
        Rt0, _ = opnp.fit_pnp_exact(K, X[s], x[s])
        if Rt0 is None:
            continue
        lst = opr.inlier_list(Rt0, K, X, x, 4.0, forced=s)
        R0 = opr.nearest_rotation(Rt0[:, :3])
        c0 = opr.cost(R0, Rt0[:, 3], K, X[lst], x[lst])
        R1, t1, c1 = opr.refine(R0, Rt0[:, 3], K, X[lst], x[lst])
        assert c1 <= c0
        e0 = np.linalg.norm(R0 - R) + np.linalg.norm(Rt0[:, 3] - t)
        e1 = np.linalg.norm(R1 - R) + np.linalg.norm(t1 - t)
        assert e1 <= e0 + 1e-12
        done += 1
    assert done >= 10


def test_nearest_rotation_projects_reflections():
    rng = np.random.default_rng(4)
    for _ in range(20):
        Q = rodrigues(rng.normal(0, 1, 3))
        M = Q @ np.diag([1.0, 1.0, -1.0])  # a reflection
        Rn = opr.nearest_rotation(M)
        assert abs(np.linalg.det(Rn) - 1) < 1e-12 and np.allclose(Rn @ Rn.T, np.eye(3), atol=1e-12)
        Rq = opr.nearest_rotation(Q + rng.normal(0, 1e-7, (3, 3)))
        assert np.allclose(Rq, Q, atol=1e-6)


# ---- the host build of the kernel's helper against the oracle -------------------------------------------------------
@pytest.fixture(scope="module")
def lib(tmp_path_factory):
    from structure_from_motion_b200 import build as b

    try:
        nvcc = b._nvcc()
    except RuntimeError:
        pytest.skip("no nvcc: the host build of sfm_refine.cuh cannot be made")
    out = str(tmp_path_factory.mktemp("pnp_refine") / "libpnprefine.so")
    subprocess.check_call([nvcc, "-O2", "-shared", "-Xcompiler", "-fPIC", "-Wno-deprecated-gpu-targets", "-o", out,
                           os.path.join(ROOT, "tools", "pnp_refine_check.cu")])
    L = ctypes.CDLL(out)
    L.p_residuals.restype = ctypes.c_double
    return L


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _host(lib, K, Rt, rec):
    K = np.ascontiguousarray(K, dtype=np.float64).reshape(9)
    P = np.empty(12)
    lib.p_projection(_p(K), _p(np.ascontiguousarray(Rt, dtype=np.float64).reshape(12)), _p(P))
    r, J = np.empty(2), np.empty(12)
    p2 = lib.p_residuals(_p(P), _p(K), _p(np.ascontiguousarray(rec, dtype=np.float64)), _p(r), _p(J))
    return P, p2, r, J.reshape(2, 6)


def test_host_helper_matches_the_oracle(lib):
    """Each residual and Jacobian entry within 16 u times its condition: the sum of the absolute values of the terms
    that form it (the projection, the quotient and the cross products)."""
    rng = np.random.default_rng(7)
    checked = 0
    for seed in range(5):
        K, X, x, R, t, _ = _scene(200, seed=seed, outliers=0.2)
        Rq = R @ rodrigues(rng.normal(0, 0.05, 3))
        tq = t + rng.normal(0, 0.05, 3)
        Rt = np.column_stack([Rq, tq])
        P_c = creproj.projection(K, Rt).reshape(12)
        r_o = opr.residuals(Rq, tq, K, X, x)
        J_o = opr.jacobian(Rq, tq, K, X, x)
        KR, Kt = np.abs(K) @ np.abs(Rq), np.abs(K) @ np.abs(tq)
        for i in range(len(X)):
            P, p2, r, J = _host(lib, K, Rt, [*X[i], *x[i]])
            assert np.array_equal(P, P_c)
            pa = KR @ np.abs(X[i]) + Kt  # |terms| of p
            cond_p = pa / abs(p2)
            u = np.abs(P.reshape(3, 4)[:2] @ np.append(X[i], 1.0)) / abs(p2)
            bound_r = 16 * U * (cond_p[:2] * (1 + u) + cond_p[2] * u + np.abs(x[i]))
            assert np.all(np.abs(r - r_o[i]) <= bound_r + 1e-300), (i, r, r_o[i])
            scale = (pa.max() * np.abs(X[i]).max() + np.abs(K).max()) / abs(p2) * (1 + u.max())
            assert np.all(np.abs(J - J_o[i]) <= 64 * U * scale * (1 + cond_p.max())), i
            checked += 1
    assert checked == 1000
