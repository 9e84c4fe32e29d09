"""TEST INFRASTRUCTURE ONLY — numpy/scipy restatement of the bundle adjustment (csrc/sfm_bundle.cuh).

Problem: V views (K fixed, [R | t] world to camera) and T tracks; the list is the observations passing the PnP record
rule under the start, of the tracks with a finite start point and at least 2 such observations (the parameter points).
Parameters, in this order: for each free view in index order (w0, w1, w2, t0, t1, t2) of R <- R exp([w]x), t <- t + dt,
without the anchored t component of ``scale_view``; then dX of each parameter point in track order.  Residuals, two
per list observation in observation order: p0 / p2 - u and p1 / p2 - v, p = K [R | t] (X, 1).  The cost is the plain
sum of squares (not scipy's half).

``dense_step`` is one Levenberg-Marquardt step from the full J^T J in the Marquardt-scaled variables the kernel solves
in, (D^-1 J^T J D^-1 + lambda I) y = -D^-1 J^T r, d = y / D, with no Schur complement.  ``minpack_replay`` runs scipy's
MINPACK Levenberg-Marquardt from the same start, list, gauge and chart.  ``jacobian`` is analytic; the CPU tests check
it against central differences.

Never imported by the product path.
"""
from __future__ import annotations

import dataclasses

import numpy as np
import scipy.sparse as sp
from scipy.optimize import least_squares

from oracle import creproj
from oracle.pnp_refine import _chart_derivative, nearest_rotation
from oracle.refine import rodrigues


@dataclasses.dataclass
class Problem:
    K: np.ndarray            # [V,3,3]
    R: np.ndarray            # [V,3,3] the start: free views projected onto rotations
    t: np.ndarray            # [V,3]
    X: np.ndarray            # [T,3]
    free: np.ndarray         # int[F] free views, ascending
    anchor: tuple            # (view, component) or None
    points: np.ndarray       # int[P] parameter points, ascending
    obs_track: np.ndarray    # int[L] the list, in observation order
    obs_view: np.ndarray     # int[L]
    obs_x: np.ndarray        # [L,2]
    obs_index: np.ndarray    # int[L] observation index in the CSR

    @property
    def n_cam(self):
        return 6 * len(self.free) - (1 if self.anchor is not None else 0)

    @property
    def n(self):
        return self.n_cam + 3 * len(self.points)


def start_list(K, Rt, X, offsets, view, x, thr):
    """The list flags bool[M] and the parameter flags bool[T] under the start, by the C checker (the device's rule)."""
    Rt = np.asarray(Rt, dtype=np.float64).reshape(-1, 3, 4)
    K = np.broadcast_to(np.asarray(K, dtype=np.float64).reshape(-1, 3, 3), (Rt.shape[0], 3, 3))
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    offsets = np.asarray(offsets, dtype=np.int64)
    view = np.asarray(view)
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    T = len(offsets) - 1
    pt = np.repeat(np.arange(T), np.diff(offsets))
    dec = np.zeros(len(view), dtype=bool)
    for c in range(Rt.shape[0]):
        sel = np.flatnonzero(view == c)
        if sel.size:
            dec[sel] = creproj.reproj_exact_many(Rt[c], K[c], X[pt[sel]], x[sel], thr)[0]
    finite = np.isfinite(X).all(axis=1)
    dec &= finite[pt]
    count = np.bincount(pt[dec], minlength=T)
    param = finite & (count >= 2)
    return dec & param[pt], param


def anchor_component(t):
    """The component of t with the largest |value|, lowest index on ties."""
    a = np.abs(np.asarray(t, dtype=np.float64))
    return int(np.flatnonzero(a == a.max())[0])


def problem(K, Rt, X, offsets, view, x, thr, fixed, scale_view=-1, inlist=None):
    """The problem the kernel solves; ``inlist`` (bool[M]) overrides the start list."""
    Rt = np.asarray(Rt, dtype=np.float64).reshape(-1, 3, 4)
    V = Rt.shape[0]
    K = np.broadcast_to(np.asarray(K, dtype=np.float64), (V, 3, 3)) if np.ndim(K) == 2 else np.asarray(K, dtype=np.float64)
    X = np.asarray(X, dtype=np.float64).reshape(-1, 3)
    offsets = np.asarray(offsets, dtype=np.int64)
    view = np.asarray(view, dtype=np.int64)
    x = np.asarray(x, dtype=np.float64).reshape(-1, 2)
    fixed = np.asarray(fixed, dtype=bool)
    if inlist is None:
        inlist, param = start_list(K, Rt, X, offsets, view, x, thr)
    else:
        T = len(offsets) - 1
        pt = np.repeat(np.arange(T), np.diff(offsets))
        param = np.bincount(pt[inlist], minlength=T) >= 2
        inlist = inlist & param[pt]
    T = len(offsets) - 1
    pt = np.repeat(np.arange(T), np.diff(offsets))
    free = np.flatnonzero(~fixed)
    R = Rt[:, :, :3].copy()
    for c in free:
        R[c] = nearest_rotation(R[c])
    t = Rt[:, :, 3].copy()
    anchor = None if scale_view is None or scale_view < 0 else (int(scale_view), anchor_component(t[scale_view]))
    idx = np.flatnonzero(inlist)
    return Problem(K=np.array(K), R=R, t=t, X=X.copy(), free=free, anchor=anchor, points=np.flatnonzero(param),
                   obs_track=pt[idx], obs_view=view[idx], obs_x=x[idx], obs_index=idx)


def _cam_columns(prob):
    """For each free view, the column of each of its 6 parameters in z (-1 for the anchored component)."""
    cols = {}
    q = 0
    for c in prob.free:
        col = []
        for k in range(6):
            if prob.anchor is not None and prob.anchor[0] == c and k == 3 + prob.anchor[1]:
                col.append(-1)
            else:
                col.append(q)
                q += 1
        cols[int(c)] = col
    return cols


def residuals(prob, R, t, X):
    """r [2L] in observation order."""
    P = np.einsum("vij,vjk->vik", prob.K, np.concatenate([R, t[:, :, None]], axis=2))
    Pv = P[prob.obs_view]
    Xh = np.column_stack([X[prob.obs_track], np.ones(len(prob.obs_track))])
    p = np.einsum("mij,mj->mi", Pv, Xh)
    return (p[:, :2] / p[:, 2:] - prob.obs_x).ravel()


def cost(prob, R, t, X):
    r = residuals(prob, R, t, X)
    return float(r @ r)


def jacobian(prob, R, t, X, chart=None):
    """J (scipy.sparse CSR) [2L, n]: d r / dz at z = 0 in the chart R exp([w]x), t + dt, X + dX at (R, t, X).  With
    ``chart`` (the z of each free view's w), the rotation columns are multiplied by the right Jacobian of SO(3)."""
    cols = _cam_columns(prob)
    pcol = {int(p): prob.n_cam + 3 * i for i, p in enumerate(prob.points)}
    rows, cidx, vals = [], [], []
    for m in range(len(prob.obs_track)):
        c, tr = int(prob.obs_view[m]), int(prob.obs_track[m])
        K = prob.K[c]
        KR = K @ R[c]
        Xm = X[tr]
        p = KR @ Xm + K @ t[c]
        dp = np.empty((3, 9))
        for k in range(3):
            e = np.zeros(3)
            e[k] = 1.0
            dp[:, k] = KR @ np.cross(e, Xm)
            dp[:, 3 + k] = K[:, k]
        dp[:, 6:9] = KR
        u = p[:2] / p[2]
        J = (dp[:2] - u[:, None] * dp[2:3]) / p[2]
        if chart is not None and c in cols:
            J[:, :6] = J[:, :6] @ _chart_derivative(chart[c])
        for k in range(2):
            row = 2 * m + k
            if c in cols:
                for j, col in enumerate(cols[c]):
                    if col >= 0:
                        rows.append(row); cidx.append(col); vals.append(J[k, j])
            for j in range(3):
                rows.append(row); cidx.append(pcol[tr] + j); vals.append(J[k, 6 + j])
    return sp.csr_matrix((vals, (rows, cidx)), shape=(2 * len(prob.obs_track), prob.n))


def apply(prob, R, t, X, d):
    """The parameters moved by d (in z order): R exp([w]x), t + dt, X + dX."""
    cols = _cam_columns(prob)
    R2, t2, X2 = R.copy(), t.copy(), X.copy()
    for c, col in cols.items():
        v = np.array([d[q] if q >= 0 else 0.0 for q in col])
        R2[c] = R[c] @ rodrigues(v[:3])
        t2[c] = t[c] + v[3:]
    for i, p in enumerate(prob.points):
        X2[p] = X[p] + d[prob.n_cam + 3 * i: prob.n_cam + 3 * i + 3]
    return R2, t2, X2


def dense_step(prob, lam=1e-3, R=None, t=None, X=None):
    """One damped step from (R, t, X) (default: the start) solved on the full J^T J: (R, t, X, y), y the scaled step."""
    R = prob.R if R is None else R
    t = prob.t if t is None else t
    X = prob.X if X is None else X
    J = jacobian(prob, R, t, X)
    r = residuals(prob, R, t, X)
    A = (J.T @ J).toarray()
    g = J.T @ r
    dg = np.diag(A)
    D = np.where((dg > 0) & np.isfinite(dg), np.sqrt(np.where(dg > 0, dg, 1.0)), 1.0)
    Ah = A / np.outer(D, D) + lam * np.eye(prob.n)
    y = np.linalg.solve(Ah, -g / D)
    return (*apply(prob, R, t, X, y / D), y)


def minpack_replay(prob, max_nfev=None):
    """scipy MINPACK Levenberg-Marquardt from the start over the list: (R, t, X, cost)."""
    if len(prob.obs_track) == 0:
        return prob.R, prob.t, prob.X, 0.0
    cols = _cam_columns(prob)

    def unpack(z):
        return apply(prob, prob.R, prob.t, prob.X, z)

    def chart(z):
        return {c: np.array([z[q] if q >= 0 else 0.0 for q in col[:3]]) for c, col in cols.items()}

    def fun(z):
        return residuals(prob, *unpack(z))

    def jac(z):
        return jacobian(prob, *unpack(z), chart=chart(z)).toarray()

    res = least_squares(fun, np.zeros(prob.n), jac=jac, method="lm", xtol=1e-15, ftol=1e-15, gtol=1e-15,
                        max_nfev=max_nfev or 200 * (prob.n + 1))
    R, t, X = unpack(res.x)
    return R, t, X, cost(prob, R, t, X)
