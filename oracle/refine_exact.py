"""TEST INFRASTRUCTURE ONLY — an exact replay of the least-squares refinement of csrc/sfm_refine.cuh.

Not a generic Levenberg-Marquardt: the iteration stated in the header of sfm_refine.cuh, step for step, in mpmath at
``DPS`` digits (the inputs — the RANSAC model and the correspondences — are doubles and are taken as exact).

- Start.  E: candidate 0 (R1, t) of the exact decomposition of the RANSAC or caller E (pose_exact.decompose_exact, whose
  candidate order the pose-edge tests pin to the device's).  H: H / H[2,2].
- Chart.  E = [t]x R, R <- R exp([w]x) (Rodrigues), t <- normalise(t + beta1 b1 + beta2 b2) with b1 = t x e_k / |t x e_k|,
  e_k the axis of t's smallest component (first on ties), b2 = t x b1.  H: h0..h7, h8 = 1.
- Residuals and Jacobians.  Those of refine_e_residual / refine_e_model and refine_h_residuals, analytic (checked
  against mpmath's numerical derivatives by tests/test_refine_exact_oracle.py).
- Control.  Cholesky of the unit-diagonal Marquardt-scaled damped system (A_hat + lambda I) y = -g_hat; lambda from
  1e-3, /10 on a strictly lower cost, *10 otherwise; the stops of refine_control in its order.

``replay`` returns every evaluation (cost, lambda, accepted, the accepted model) and, for every discrete decision, its
relative margin — how far the compared quantity was from its switch — so that a test can tell a decision rounding could
flip from one it must not.  ``report_after(trace, k)`` is the report the kernel gives with ``max_iter = k``.

Never imported by the product path.
"""
from __future__ import annotations

import dataclasses
import math

import mpmath as mp
import numpy as np

from . import pose_exact as px

DPS = 40
U = 2.0 ** -53
LAMBDA0, LAMBDA_FACTOR, LAMBDA_CAP = 1e-3, 10.0, 1e16
FTOL, XTOL, COST_FLOOR = 1e-12, 1e-9, 1e-24
ROTATE_TAYLOR = 1e-4
CONVERGED, MAX_ITER, STALLED, NO_MODEL, NONFINITE = 0, 1, 2, 3, 4
NP = {"E": 5, "H": 8}


def _f(x):
    return mp.mpf(float(x))


# ---------------------------------------------------------------------------------------------------------------------
# chart, residuals and Jacobians
# ---------------------------------------------------------------------------------------------------------------------
def skew(v):
    return [mp.mpf(0), -v[2], v[1], v[2], mp.mpf(0), -v[0], -v[1], v[0], mp.mpf(0)]


def mul3(A, B):
    return [sum(A[3 * i + k] * B[3 * k + j] for k in range(3)) for i in range(3) for j in range(3)]


def cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def tangent_axis(t):
    """(k, margin): the axis of t's smallest |component| (first on ties) and the relative gap to the runner-up."""
    a = [abs(c) for c in t]
    k = 0
    if a[1] < a[k]:
        k = 1
    if a[2] < a[k]:
        k = 2
    others = [a[j] for j in range(3) if j != k]
    gap = min(others) - a[k]
    return k, float(gap / max(a)) if max(a) > 0 else 0.0


def tangent_basis(t):
    k, _ = tangent_axis(t)
    e = [mp.mpf(1 if j == k else 0) for j in range(3)]
    b1 = cross(t, e)
    n = mp.sqrt(sum(c * c for c in b1))
    b1 = [c / n for c in b1]
    return b1, cross(t, b1)


def e_model(R, t):
    """E = [t]x R and dE/dtheta as 5 lists of 9 (theta = w0, w1, w2, beta1, beta2)."""
    E = mul3(skew(t), R)
    cols = [mul3(E, skew([mp.mpf(1 if j == k else 0) for j in range(3)])) for k in range(3)]
    b1, b2 = tangent_basis(t)
    cols += [mul3(skew(b1), R), mul3(skew(b2), R)]
    return E, cols


def e_residual(E, xa, ya, xb, yb):
    """(r, dr/dE[9]) of one K-normalised correspondence: r = (b^T E a) sqrt(1/na + 1/nb)."""
    a, b = [xa, ya, mp.mpf(1)], [xb, yb, mp.mpf(1)]
    la = [E[3 * j] * xa + E[3 * j + 1] * ya + E[3 * j + 2] for j in range(3)]
    lb = [E[j] * xb + E[3 + j] * yb + E[6 + j] for j in range(3)]
    s = lb[0] * xa + lb[1] * ya + lb[2]
    na, nb = la[0] ** 2 + la[1] ** 2, lb[0] ** 2 + lb[1] ** 2
    w = mp.sqrt(1 / na + 1 / nb)
    ca, cb = s / w / na ** 2, s / w / nb ** 2
    g = []
    for j in range(3):
        for k in range(3):
            v = w * b[j] * a[k]
            if j < 2:
                v -= ca * la[j] * a[k]
            if k < 2:
                v -= cb * lb[k] * b[j]
            g.append(v)
    return s * w, g


def adj(h):
    return [h[4] * h[8] - h[5] * h[7], h[2] * h[7] - h[1] * h[8], h[1] * h[5] - h[2] * h[4],
            h[5] * h[6] - h[3] * h[8], h[0] * h[8] - h[2] * h[6], h[2] * h[3] - h[0] * h[5],
            h[3] * h[7] - h[4] * h[6], h[1] * h[6] - h[0] * h[7], h[0] * h[4] - h[1] * h[3]]


def adj_derivatives(h):
    """d adj(H) / d h_k for k = 0..7: the polarisation adj(H + e_k) - adj(H) (adj(e_k) = 0 for a single entry)."""
    ad = adj(h)
    return [[x - y for x, y in zip(adj([hh + (1 if m == k else 0) for m, hh in enumerate(h)]), ad)] for k in range(8)]


def h_residuals(h, xa, ya, xb, yb, dads=None):
    """(r[4], J[4][8]) of one pixel correspondence under H = (h0..h7, h8), derivatives over h0..h7."""
    p = [h[3 * i] * xa + h[3 * i + 1] * ya + h[3 * i + 2] for i in range(3)]
    ad = adj(h)
    dads = adj_derivatives(h) if dads is None else dads
    q = [ad[3 * i] * xb + ad[3 * i + 1] * yb + ad[3 * i + 2] for i in range(3)]
    u0, u1, v0, v1 = p[0] / p[2], p[1] / p[2], q[0] / q[2], q[1] / q[2]
    r = [u0 - xb, u1 - yb, v0 - xa, v1 - ya]
    a = [xa, ya, mp.mpf(1)]
    J = [[mp.mpf(0)] * 8 for _ in range(4)]
    for k in range(8):
        i, j = divmod(k, 3)
        dp = [mp.mpf(0)] * 3
        dp[i] = a[j]
        dad = dads[k]
        dq = [dad[3 * m] * xb + dad[3 * m + 1] * yb + dad[3 * m + 2] for m in range(3)]
        J[0][k] = (dp[0] - u0 * dp[2]) / p[2]
        J[1][k] = (dp[1] - u1 * dp[2]) / p[2]
        J[2][k] = (dq[0] - v0 * dq[2]) / q[2]
        J[3][k] = (dq[1] - v1 * dq[2]) / q[2]
    return r, J


def rotate(R, w):
    """R exp([w]x) (exact Rodrigues: the kernel's Taylor branch below 1e-4 is its own rounding, not a different map)."""
    th2 = sum(c * c for c in w)
    th = mp.sqrt(th2)
    if th == 0:
        A, B = mp.mpf(1), mp.mpf(0.5)
    else:
        A, B = mp.sin(th) / th, (1 - mp.cos(th)) / th2
    W = skew(w)
    W2 = mul3(W, W)
    X = [A * W[j] + B * W2[j] + (1 if j % 4 == 0 else 0) for j in range(9)]
    return mul3(R, X)


# ---------------------------------------------------------------------------------------------------------------------
# evaluation and replay
# ---------------------------------------------------------------------------------------------------------------------
def _pts(pts):
    pts = np.asarray(pts, dtype=np.float64).reshape(-1, 4)
    return [[_f(v) for v in row] for row in pts]


def evaluate(kind, x, pts):
    """(cost, J^T J [NP][NP], J^T r [NP], sum of squared coordinates) at the point x (E: R[9] + t[3], H: h0..h7)."""
    n = NP[kind]
    A = [[mp.mpf(0)] * n for _ in range(n)]
    g = [mp.mpf(0)] * n
    cost = S = mp.mpf(0)
    rows = []
    if kind == "E":
        E, cols = e_model(x[:9], x[9:12])
        for xa, ya, xb, yb in pts:
            S += xa * xa + ya * ya + xb * xb + yb * yb
            r, gE = e_residual(E, xa, ya, xb, yb)
            rows.append((r, [mp.fdot(gE, c) for c in cols]))
    else:
        h = list(x[:8]) + [mp.mpf(1)]
        dads = adj_derivatives(h)
        for xa, ya, xb, yb in pts:
            S += xa * xa + ya * ya + xb * xb + yb * yb
            r, J = h_residuals(h, xa, ya, xb, yb, dads)
            rows += list(zip(r, J))
    for r, J in rows:
        cost += r * r
        for i in range(n):
            g[i] += J[i] * r
            for j in range(i, n):
                A[i][j] += J[i] * J[j]
    for i in range(n):
        for j in range(i):
            A[i][j] = A[j][i]
    return cost, A, g, S


def jacobian_rows(kind, x, xa, ya, xb, yb):
    """The residual(s) and Jacobian row(s) of one correspondence at x (for the numerical-derivative check)."""
    xa, ya, xb, yb = (mp.mpf(v) for v in (xa, ya, xb, yb))
    if kind == "E":
        E, cols = e_model(x[:9], x[9:12])
        r, gE = e_residual(E, xa, ya, xb, yb)
        return [r], [[mp.fdot(gE, c) for c in cols]]
    return h_residuals(list(x[:8]) + [mp.mpf(1)], xa, ya, xb, yb)


def retract(kind, x, d):
    if kind == "E":
        R = rotate(x[:9], d[:3])
        b1, b2 = tangent_basis(x[9:12])
        t = [x[9 + k] + d[3] * b1[k] + d[4] * b2[k] for k in range(3)]
        n = mp.sqrt(sum(c * c for c in t))
        return R + [c / n for c in t]
    return [x[k] + d[k] for k in range(8)]


def residuals_at(kind, x, pts):
    """All residuals at x (for numerical derivatives of the chart)."""
    out = []
    if kind == "E":
        E = mul3(skew(x[9:12]), x[:9])
        for row in pts:
            out.append(e_residual(E, *row)[0])
    else:
        h = list(x[:8]) + [mp.mpf(1)]
        for row in pts:
            out += h_residuals(h, *row)[0]
    return out


def damped_solve(A, g, D, lam):
    """Cholesky of (A_hat + lam I) y = -g_hat, A_hat = D^-1 A D^-1: (ok, y, smallest pivot^2 / (1 + lam), cond)."""
    n = len(g)
    M = [[A[i][j] / (D[i] * D[j]) + (lam if i == j else 0) for j in range(n)] for i in range(n)]
    L = [[mp.mpf(0)] * n for _ in range(n)]
    piv = mp.inf
    for i in range(n):
        for j in range(i + 1):
            v = M[i][j] - sum(L[i][k] * L[j][k] for k in range(j))
            if i == j:
                piv = min(piv, v / (1 + lam))
                if not v > 0:
                    return False, None, float(piv), math.inf
                L[i][i] = mp.sqrt(v)
            else:
                L[i][j] = v / L[j][j]
    z = [mp.mpf(0)] * n
    for i in range(n):
        z[i] = (-g[i] / D[i] - sum(L[i][k] * z[k] for k in range(i))) / L[i][i]
    y = [mp.mpf(0)] * n
    for i in reversed(range(n)):
        y[i] = (z[i] - sum(L[k][i] * y[k] for k in range(i + 1, n))) / L[i][i]
    ev = np.linalg.eigvalsh(np.array([[float(v) for v in row] for row in M]))
    return True, y, float(piv), float(ev[-1] / ev[0]) if ev[0] > 0 else math.inf


@dataclasses.dataclass
class Step:
    """One evaluation: its cost, whether it was accepted, lambda after the control ran, and the state then."""
    iteration: int            # the kernel's `iter` after this evaluation
    cost: float               # of the evaluated point
    accepted: bool
    lam: float                # lambda after the control
    best_cost: float          # the accepted cost after the control
    rejected: int
    status: int | None        # the stop this evaluation made (None: running)
    x: list                   # the accepted point after the control (mp)
    margins: dict             # decision -> relative margin, for the decisions this evaluation made
    cond: float = 1.0         # condition of the last damped system solved after this evaluation


@dataclasses.dataclass
class Trace:
    kind: str
    steps: list
    cost_start: float
    sum_sq: float
    start_axis_margin: float = math.inf

    def model(self, x=None):
        x = self.steps[-1].x if x is None else x
        return model_of(self.kind, x)


def model_of(kind, x):
    """The reported model (E / E[8] or h0..h7, 1) in double, from the exact point."""
    if kind == "E":
        E = mul3(skew(x[9:12]), x[:9])
        return np.array([float(e / E[8]) for e in E])
    return np.array([float(v) for v in x[:8]] + [1.0])


def start_point(kind, M, pose0=None):
    """E: the exact candidate (R, t) of M nearest the device's candidate 0 ``pose0`` = (R, t) when given, else (R1, t).
    The choice matters: [t]x R1 = -[t]x R2, but the two charts move t against different rotations, so LM's steps from
    them differ.  H: M / M[2,2]."""
    M = np.asarray(M, dtype=np.float64).reshape(9)
    if kind == "E":
        ex = px.decompose_exact(M.reshape(3, 3), dps=DPS + 10)
        R, t = ex.R1, ex.t
        if pose0 is not None:
            R0, t0 = (np.asarray(a, dtype=np.float64) for a in pose0)
            R = min((ex.R1, ex.R2), key=lambda Q: np.abs(Q - R0.reshape(3, 3)).max())
            t = min((ex.t, -ex.t), key=lambda v: np.abs(v - t0.reshape(3)).max())
        return [_f(v) for v in R.reshape(9)] + [_f(v) for v in t]
    return [_f(M[k]) / _f(M[8]) for k in range(8)]


def replay(kind, M0, pts, max_iter=50, dps=DPS, pose0=None, start=None):
    """The refinement of the list ``pts`` ([n, 4]: xa, ya, xb, yb — K-normalised for E, pixels for H) from the RANSAC
    model M0 (E: from the exact candidate nearest ``pose0``, see start_point; or from ``start``, 12 or 8 doubles taken
    as they are), up to ``max_iter`` evaluated proposals."""
    n = NP[kind]
    with mp.workdps(dps):
        P = _pts(pts)
        px_ = start_point(kind, M0, pose0) if start is None else [_f(v) for v in start]
        x = None
        A = g = None
        cost = mp.nan
        lam = mp.mpf(LAMBDA0)
        it = rejected = evals = 0
        steps = []
        cost_start = sum_sq = None
        axis_margin = tangent_axis(px_[9:12])[1] if kind == "E" else math.inf
        while True:
            c, A1, g1, S = evaluate(kind, px_, P)
            margins = {}
            if evals == 0:
                cost_start, sum_sq = c, S
                accept = True
            else:
                it += 1
                accept = c < cost
                margins["accept"] = float(abs(c - cost) / cost) if cost > 0 else math.inf
            evals += 1
            status = None
            if accept:
                before = cost
                x, A, g, cost = px_, A1, g1, c
                if it > 0:
                    lam /= LAMBDA_FACTOR
                    margins["ftol"] = float(abs((before - c) - FTOL * before) / before)
                    if before - c <= FTOL * before:
                        status = CONVERGED
                if status is None:
                    fl = COST_FLOOR * S
                    margins["floor"] = float(abs(c - fl) / fl) if fl > 0 else math.inf
                    if c <= fl:
                        status = CONVERGED
            else:
                lam *= LAMBDA_FACTOR
                rejected += 1
            if status is None and it >= max_iter:
                status = MAX_ITER
            cond = 1.0
            if status is None:
                D = [mp.sqrt(A[i][i]) if A[i][i] > 0 else mp.mpf(1) for i in range(n)]
                while True:
                    margins["lambda_cap"] = min(margins.get("lambda_cap", math.inf), float(abs(lam - LAMBDA_CAP) / LAMBDA_CAP))
                    if not lam <= LAMBDA_CAP:
                        status = STALLED
                        break
                    ok, y, piv, cond = damped_solve(A, g, D, lam)
                    margins["pivot"] = min(margins.get("pivot", math.inf), abs(piv))
                    if ok:
                        break
                    lam *= LAMBDA_FACTOR
                if status is None:
                    ny = mp.sqrt(sum(v * v for v in y))
                    lim = XTOL * mp.sqrt(cost)
                    margins["xtol"] = float(abs(ny - lim) / lim) if lim > 0 else math.inf
                    if ny <= lim:
                        status = CONVERGED
                    else:
                        d = [y[i] / D[i] for i in range(n)]
                        if kind == "E":
                            thn = float(mp.sqrt(sum(v * v for v in d[:3])))
                            margins["taylor"] = abs(thn - ROTATE_TAYLOR) / ROTATE_TAYLOR
                            margins["axis"] = tangent_axis(x[9:12])[1]
                        px_ = retract(kind, x, d)
            steps.append(Step(iteration=it, cost=float(c), accepted=accept, lam=float(lam), best_cost=float(cost),
                              rejected=rejected, status=status, x=list(x), margins=margins, cond=cond))
            if status is not None:
                break
        return Trace(kind=kind, steps=steps, cost_start=float(cost_start), sum_sq=float(sum_sq),
                     start_axis_margin=axis_margin)


@dataclasses.dataclass
class Report:
    status: int
    iterations: int
    rejected: int
    cost_start: float
    cost_final: float
    model: np.ndarray
    min_margin: float         # the smallest decision margin up to and including the last evaluation
    cond: float               # the largest damped-system condition met on the way
    prior_margin: float = math.inf  # the smallest margin of the decisions before the last evaluation


def report_after(trace: Trace, k: int) -> Report:
    """The report of the kernel run with max_iter = k, from a replay run with max_iter >= k."""
    mm, cond = trace.start_axis_margin, 1.0
    for s in trace.steps:
        prior = mm
        stop = s.status if s.status is not None else (MAX_ITER if s.iteration >= k else None)
        ms = dict(s.margins)
        if stop == MAX_ITER and s.status != MAX_ITER:  # the capped run makes none of the later decisions
            for key in ("lambda_cap", "pivot", "xtol", "taylor", "axis"):
                ms.pop(key, None)
        mm = min([mm] + list(ms.values()))
        if stop is None:
            cond = max(cond, s.cond)
        if stop is not None:
            return Report(status=stop, iterations=s.iteration, rejected=s.rejected, cost_start=trace.cost_start,
                          cost_final=s.best_cost, model=trace.model(s.x), min_margin=mm, cond=cond, prior_margin=prior)
    raise ValueError(f"the replay stopped before iteration {k}: replay it with max_iter >= {k}")


def exact_gradient(kind, model, pts, dps=DPS):
    """|D^-1 J^T r| / sqrt(cost) at a reported model (D = sqrt(diag J^T J)): 0 at a stationary point of the cost, the
    cosine of the residual with the worst-aligned scaled Jacobian column otherwise.  E: the chart around candidate 0 of
    the exact decomposition of the model; H: h0..h7 of the model with H[2,2] = 1."""
    with mp.workdps(dps):
        x = start_point(kind, model)
        c, A, g, _ = evaluate(kind, x, _pts(pts))
        n = NP[kind]
        return float(mp.sqrt(sum(g[i] ** 2 / A[i][i] for i in range(n) if A[i][i] > 0)) / mp.sqrt(c)), float(c)


def start_cost(kind, M0, pts, dps=30):
    """The start's cost summed exactly rounded (math.fsum of the terms, each computed at ``dps`` digits)."""
    with mp.workdps(dps):
        x = start_point(kind, M0)
        terms = []
        if kind == "E":
            E = mul3(skew(x[9:12]), x[:9])
            for xa, ya, xb, yb in np.asarray(pts, dtype=np.float64).reshape(-1, 4).tolist():
                la0, la1 = E[0] * xa + E[1] * ya + E[2], E[3] * xa + E[4] * ya + E[5]
                lb = [E[j] * xb + E[3 + j] * yb + E[6 + j] for j in range(3)]
                s = lb[0] * xa + lb[1] * ya + lb[2]
                terms.append(float(s * s * (1 / (la0 * la0 + la1 * la1) + 1 / (lb[0] * lb[0] + lb[1] * lb[1]))))
        else:
            h = list(x) + [mp.mpf(1)]
            for row in np.asarray(pts, dtype=np.float64).reshape(-1, 4):
                terms += [float(v * v) for v in h_residuals(h, *(_f(v) for v in row))[0]]
        return math.fsum(terms)
