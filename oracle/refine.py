"""TEST INFRASTRUCTURE ONLY — numpy/scipy restatement of the least-squares refinement (csrc/sfm_refine.cuh).

Costs (sums over a fixed inlier set):
  E  residual r = (b^T E a) sqrt(1/na + 1/nb) in K-normalised coordinates (a = (xa, ya, 1), na = |(E a)_0,1|^2,
     nb = |(E^T b)_0,1|^2), so that r^2 is the symmetric epipolar distance;
  H  four residuals per correspondence, pi(H a) - b and pi(adj(H) b) - a in pixels, whose squares sum to the symmetric
     transfer error.
Parameterisations: E = [t]x R with R = R0 exp([w]x) and t = normalise(t0 + beta1 b1 + beta2 b2), (b1, b2) the tangent
basis of t0 that the kernel uses; H = h0..h7 with H[2,2] = 1.  The Jacobians are analytic: for E by the product rule
through dE/dtheta, for H with the exact polarisation of the quadratic adjugate, adj(H + D) - adj(H) - adj(D).
``refine_e`` / ``refine_h`` give an independent optimum from the same start with scipy's MINPACK Levenberg-Marquardt.

Never imported by the product path.
"""
from __future__ import annotations

import numpy as np
from scipy.optimize import least_squares


def skew(v):
    return np.array([[0.0, -v[2], v[1]], [v[2], 0.0, -v[0]], [-v[1], v[0], 0.0]])


def rodrigues(w):
    w = np.asarray(w, dtype=np.float64)
    th = np.linalg.norm(w)
    W = skew(w)
    if th < 1e-8:
        return np.eye(3) + W + 0.5 * W @ W
    return np.eye(3) + np.sin(th) / th * W + (1.0 - np.cos(th)) / th ** 2 * W @ W


def tangent_basis(t):
    """(b1, b2): b1 = t x e_k / |t x e_k| with e_k the axis of t's smallest component (first on ties), b2 = t x b1."""
    t = np.asarray(t, dtype=np.float64)
    k = int(np.argmin(np.abs(t)))
    b1 = np.cross(t, np.eye(3)[k])
    b1 /= np.linalg.norm(b1)
    return b1, np.cross(t, b1)


def e_from_pose(R, t):
    """E = [t]x R scaled to E[2,2] = 1."""
    E = skew(t) @ R
    return E / E[2, 2]


def pose_start(E):
    """A pose (R, unit t) on the essential manifold with [t]x R = +-E projected onto it (singular values (1, 1, 0))."""
    U, _, Vt = np.linalg.svd(np.asarray(E, dtype=np.float64).reshape(3, 3))
    if np.linalg.det(U) < 0:
        U = -U
    if np.linalg.det(Vt) < 0:
        Vt = -Vt
    W = np.array([[0.0, -1.0, 0.0], [1.0, 0.0, 0.0], [0.0, 0.0, 1.0]])
    return U @ W.T @ Vt, U[:, 2].copy()


def retract_e(R0, t0, theta):
    b1, b2 = tangent_basis(t0)
    t = t0 + theta[3] * b1 + theta[4] * b2
    return R0 @ rodrigues(theta[:3]), t / np.linalg.norm(t)


def _lines(E, a, b):
    return a @ E.T, b @ E  # rows: E a, E^T b


def e_residuals(E, na_pts, nb_pts):
    """Residuals of [m,2] K-normalised correspondences under E (any scale)."""
    a = np.column_stack([na_pts, np.ones(len(na_pts))])
    b = np.column_stack([nb_pts, np.ones(len(nb_pts))])
    la, lb = _lines(np.asarray(E, dtype=np.float64).reshape(3, 3), a, b)
    s = np.sum(lb * a, axis=1)
    u = 1.0 / (la[:, 0] ** 2 + la[:, 1] ** 2) + 1.0 / (lb[:, 0] ** 2 + lb[:, 1] ** 2)
    return s * np.sqrt(u)


def e_cost(E, na_pts, nb_pts):
    return float(np.sum(e_residuals(E, na_pts, nb_pts) ** 2))


def e_jacobian(R, t, na_pts, nb_pts):
    """d residual / d(w0, w1, w2, beta1, beta2) at theta = 0 of the chart around (R, t): [m,5]."""
    a = np.column_stack([na_pts, np.ones(len(na_pts))])
    b = np.column_stack([nb_pts, np.ones(len(nb_pts))])
    E = skew(t) @ R
    la, lb = _lines(E, a, b)
    s = np.sum(lb * a, axis=1)
    na = la[:, 0] ** 2 + la[:, 1] ** 2
    nb = lb[:, 0] ** 2 + lb[:, 1] ** 2
    w = np.sqrt(1.0 / na + 1.0 / nb)
    # dr/dE[j,k] = w b_j a_k - (s / w) (la_j a_k [j<2] / na^2 + lb_k b_j [k<2] / nb^2)
    la2 = la.copy()
    la2[:, 2] = 0.0
    lb2 = lb.copy()
    lb2[:, 2] = 0.0
    g = (w[:, None, None] * b[:, :, None] * a[:, None, :]
         - (s / w)[:, None, None] * (la2[:, :, None] * a[:, None, :] / na[:, None, None] ** 2
                                     + b[:, :, None] * lb2[:, None, :] / nb[:, None, None] ** 2))
    b1, b2 = tangent_basis(t)
    dE = [E @ skew(np.eye(3)[k]) for k in range(3)] + [skew(b1) @ R, skew(b2) @ R]
    return np.stack([np.einsum("mjk,jk->m", g, D) for D in dE], axis=1)


def adj(H):
    H = np.asarray(H, dtype=np.float64).reshape(3, 3)
    return np.array([
        [H[1, 1] * H[2, 2] - H[1, 2] * H[2, 1], H[0, 2] * H[2, 1] - H[0, 1] * H[2, 2], H[0, 1] * H[1, 2] - H[0, 2] * H[1, 1]],
        [H[1, 2] * H[2, 0] - H[1, 0] * H[2, 2], H[0, 0] * H[2, 2] - H[0, 2] * H[2, 0], H[0, 2] * H[1, 0] - H[0, 0] * H[1, 2]],
        [H[1, 0] * H[2, 1] - H[1, 1] * H[2, 0], H[0, 1] * H[2, 0] - H[0, 0] * H[2, 1], H[0, 0] * H[1, 1] - H[0, 1] * H[1, 0]],
    ])


def h_from_params(h8):
    return np.append(np.asarray(h8, dtype=np.float64), 1.0).reshape(3, 3)


def h_residuals(H, pa, pb):
    """[4m] residuals (per correspondence: forward x, y, backward x, y) of pixel correspondences under H."""
    H = np.asarray(H, dtype=np.float64).reshape(3, 3)
    a = np.column_stack([pa, np.ones(len(pa))])
    b = np.column_stack([pb, np.ones(len(pb))])
    p = a @ H.T
    q = b @ adj(H).T
    r = np.column_stack([p[:, 0] / p[:, 2] - pb[:, 0], p[:, 1] / p[:, 2] - pb[:, 1],
                         q[:, 0] / q[:, 2] - pa[:, 0], q[:, 1] / q[:, 2] - pa[:, 1]])
    return r.reshape(-1)


def h_cost(H, pa, pb):
    return float(np.sum(h_residuals(H, pa, pb) ** 2))


def h_jacobian(H, pa, pb):
    """d residual / d(h0..h7) with H[2,2] fixed: [4m, 8]."""
    H = np.asarray(H, dtype=np.float64).reshape(3, 3)
    a = np.column_stack([pa, np.ones(len(pa))])
    b = np.column_stack([pb, np.ones(len(pb))])
    p = a @ H.T
    q = b @ adj(H).T
    A = adj(H)
    J = np.zeros((len(pa), 4, 8))
    for k in range(8):
        D = np.zeros(9)
        D[k] = 1.0
        D = D.reshape(3, 3)
        dp = a @ D.T
        dq = b @ (adj(H + D) - A - adj(D)).T  # the linear part of the quadratic adjugate
        for c in range(2):
            J[:, c, k] = (dp[:, c] - p[:, c] / p[:, 2] * dp[:, 2]) / p[:, 2]
            J[:, 2 + c, k] = (dq[:, c] - q[:, c] / q[:, 2] * dq[:, 2]) / q[:, 2]
    return J.reshape(-1, 8)


def refine_e(R0, t0, na_pts, nb_pts):
    """scipy's LM from (R0, t0) in the chart around it (finite-difference Jacobian: the analytic one lives in the chart
    of the point it is evaluated at) -> (E with E[2,2] = 1, cost, (R, t))."""
    def f(th):
        R, t = retract_e(R0, t0, th)
        return e_residuals(skew(t) @ R, na_pts, nb_pts)

    sol = least_squares(f, np.zeros(5), jac="3-point", method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=4000)
    R, t = retract_e(R0, t0, sol.x)
    return e_from_pose(R, t), float(np.sum(sol.fun ** 2)), (R, t)


def refine_h(H0, pa, pb):
    """scipy's LM from H0 over h0..h7 -> (H with H[2,2] = 1, cost)."""
    H0 = np.asarray(H0, dtype=np.float64).reshape(3, 3)
    x0 = (H0 / H0[2, 2]).reshape(9)[:8]
    sol = least_squares(lambda x: h_residuals(h_from_params(x), pa, pb), x0,
                        jac=lambda x: h_jacobian(h_from_params(x), pa, pb), method="lm", x_scale="jac",
                        xtol=1e-15, ftol=1e-15, gtol=1e-15, max_nfev=4000)
    return h_from_params(sol.x), float(np.sum(sol.fun ** 2))
