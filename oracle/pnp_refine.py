"""TEST INFRASTRUCTURE ONLY — numpy/scipy restatement of the PnP pose refinement (csrc/sfm_refine.cuh, MODEL_P).

Cost: over a fixed list of records (X, u, v), two residuals each, r0 = p0 / p2 - u and r1 = p1 / p2 - v with
p = K [R | t] (X, 1), so that r0^2 + r1^2 is the squared reprojection error RANSAC scores (oracle.pnp.reproj).
Parameters: R = R0 exp([w]x), t = t0 + dt.  The analytic Jacobian: dp/dw_k = K R (e_k x X), dp/dt_k = K e_k, then the
quotient rule.  ``nearest_rotation`` is the start the kernel takes (SVD, det fixed to +1); ``refine`` gives an
independent optimum from that start with scipy's MINPACK Levenberg-Marquardt.

Never imported by the product path.
"""
from __future__ import annotations

import numpy as np
from scipy.optimize import least_squares

from oracle import pnp as opnp
from oracle.refine import rodrigues


def nearest_rotation(M):
    """The rotation nearest to M in the Frobenius norm: U diag(1, 1, det(U V^T)) V^T."""
    U, _, Vt = np.linalg.svd(np.asarray(M, dtype=np.float64).reshape(3, 3))
    d = np.sign(np.linalg.det(U @ Vt))
    return U @ np.diag([1.0, 1.0, d if d != 0 else 1.0]) @ Vt


def inlier_list(Rt, K, X, x, thr, forced=None):
    """The list the kernel refines over: the decision under Rt at thr, plus the forced indices, ascending."""
    keep = opnp.reproj(Rt, K, X, x, thr)[0].copy()
    if forced is not None:
        keep[np.asarray(forced, dtype=np.int64)] = True
    return np.flatnonzero(keep)


def residuals(R, t, K, X, x):
    """r [m, 2] of every record under [R | t]."""
    P = np.asarray(K, dtype=np.float64).reshape(3, 3) @ np.column_stack([R, t])
    p = np.asarray(X, dtype=np.float64).reshape(-1, 3) @ P[:, :3].T + P[:, 3]
    return p[:, :2] / p[:, 2:] - np.asarray(x, dtype=np.float64).reshape(-1, 2)


def jacobian(R, t, K, X, x):
    """J [m, 2, 6]: d r / d(w0, w1, w2, t0, t1, t2) at w = 0, dt = 0."""
    K = np.asarray(K, dtype=np.float64).reshape(3, 3)
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    KR = K @ R
    p = X @ KR.T + K @ t
    m = X.shape[0]
    dp = np.empty((m, 3, 6))
    for k in range(3):
        e = np.zeros(3)
        e[k] = 1.0
        dp[:, :, k] = np.cross(e, X) @ KR.T
        dp[:, :, 3 + k] = K[:, k]
    u = p[:, :2] / p[:, 2:]
    return (dp[:, :2, :] - u[:, :, None] * dp[:, 2:3, :]) / p[:, 2, None, None]


def cost(R, t, K, X, x):
    r = residuals(R, t, K, X, x)
    return float(np.sum(r * r))


def refine(R0, t0, K, X, x, max_nfev=2000):
    """scipy LM from (R0, t0) over all records given: (R, t, cost)."""
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    if X.shape[0] == 0:
        return R0, t0, 0.0

    def pose(z):
        return R0 @ rodrigues(z[:3]), t0 + z[3:]

    def fun(z):
        return residuals(*pose(z), K, X, x).ravel()

    def jac(z):
        R, t = pose(z)
        # jacobian() is the derivative in the chart R exp([w]x) at R; the right Jacobian of SO(3) maps it to z
        J = jacobian(R, t, K, X, x).reshape(-1, 6)
        return J @ _chart_derivative(z)

    if X.shape[0] * 2 < 6:
        z = least_squares(fun, np.zeros(6), jac=jac, method="trf", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=max_nfev).x
    else:
        z = least_squares(fun, np.zeros(6), jac=jac, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=max_nfev).x
    R, t = pose(z)
    return R, t, cost(R, t, K, X, x)


def _chart_derivative(z):
    """d(w_local, dt) / dz for R = R0 exp([z0:3]x) (right Jacobian of SO(3)) and t = t0 + z3:6."""
    w = np.asarray(z[:3], dtype=np.float64)
    th = np.linalg.norm(w)
    W = np.array([[0.0, -w[2], w[1]], [w[2], 0.0, -w[0]], [-w[1], w[0], 0.0]])
    if th < 1e-8:
        Jr = np.eye(3) - 0.5 * W
    else:
        Jr = np.eye(3) - (1 - np.cos(th)) / th ** 2 * W + (th - np.sin(th)) / th ** 3 * (W @ W)
    D = np.eye(6)
    D[:3, :3] = Jr
    return D
