"""TEST INFRASTRUCTURE ONLY — a replay of the bundle adjustment's iteration (csrc/sfm_bundle.cuh), step by step.

Not a generic Levenberg-Marquardt: the iteration stated in the header of sfm_bundle.cuh, decision for decision, with
the parameters, projections and residuals in ``np.longdouble`` and every solve refined against the full system.

- Problem.  ``oracle.bundle.problem``: the list formed under the given Rt, the nearest-rotation start of the free views,
  the anchored component, the parameter points.
- Residuals and Jacobians.  Per list observation, vectorised: r = p0 / p2 - u, p1 / p2 - v with p = K [R | t] (X, 1);
  J_c over (w, dt) of R exp([w]x), t + dt (the anchored column zero), J_p over dX.  A proposal under which a list
  observation has p2 < 2^-537 or a non-finite residual costs +inf.
- Cost.  Each term r0^2 + r1^2 in longdouble, the terms added exactly rounded (math.fsum of their double-double
  splits).  The cost floor is 1e-24 sum(u^2 + v^2) over the list.
- Step.  (D^-1 J^T J D^-1 + lambda I) y = -D^-1 J^T r, D = sqrt(diag J^T J) (1 where 0 or not finite), from the double
  sums of the per-observation blocks, as the kernel forms them.  Solved by a double Schur complement (each damped
  V_hat_p inverted, the reduced 6F x 6F system factored), then refined against the full system, with its residual
  formed in longdouble from the per-observation blocks, until the correction is below the longdouble unit.  A damped
  V_hat_p or reduced system with a non-finite entry or a pivot that is not positive is not positive definite.
- Control.  k_ba_views_sum / k_ba_points: lambda from 1e-3, / 10 on a strictly lower cost, x 10 otherwise; the stops in
  the order ftol, cost floor, max_iter, lambda cap; Xtol on |y| against sqrt(cost); a system that is not positive
  definite multiplies lambda by 10 and is solved again without counting an iteration, and lambda reaching 0 or passing
  the cap there is stalled.
- Rotation.  refine_rotate: Rodrigues, with the Taylor coefficients below |w| = 1e-4.

``replay`` returns every evaluation with the relative margin of each decision it made (how far the compared quantity
was from its switch), the smallest pivot margin and the condition of the damped systems solved after it.
``report_after(trace, k)`` is the report the kernel gives with max_iterations = k.

Never imported by the product path.
"""
from __future__ import annotations

import dataclasses
import math

import numpy as np

from oracle import bundle as oba

LD = np.longdouble
U = 2.0 ** -53
LAMBDA0, LAMBDA_FACTOR, LAMBDA_CAP = 1e-3, 10.0, 1e16
FTOL, XTOL, COST_FLOOR = 1e-12, 1e-9, 1e-24
ROTATE_TAYLOR = 1e-4
P2_MIN = 2.0 ** -537
CONVERGED, MAX_ITER, STALLED, NONFINITE = 0, 1, 2, 4


# ---------------------------------------------------------------------------------------------------------------------
# sums and indices
# ---------------------------------------------------------------------------------------------------------------------
def group_sum(keys, vals, n):
    """out[k] = sum of vals[i] over keys[i] == k (any dtype; rows of vals may be arrays)."""
    vals = np.asarray(vals)
    out = np.zeros((n,) + vals.shape[1:], dtype=vals.dtype)
    if len(keys) == 0:
        return out
    order = np.argsort(keys, kind="stable")
    ks = np.asarray(keys)[order]
    starts = np.flatnonzero(np.r_[True, ks[1:] != ks[:-1]])
    out[ks[starts]] = np.add.reduceat(vals[order], starts, axis=0)
    return out


def _fsum_ld(terms):
    """The exactly rounded double of a sum of longdouble terms (+inf on overflow)."""
    terms = np.asarray(terms, dtype=LD).ravel()
    if not np.isfinite(terms).all():
        return math.inf
    hi = terms.astype(np.float64)
    lo = (terms - hi.astype(LD)).astype(np.float64)
    try:
        return math.fsum(np.concatenate([hi, lo]).tolist())
    except OverflowError:
        return math.inf


@dataclasses.dataclass
class Layout:
    """Indices of the list: free index and point index of every list observation, and the observation pairs of one
    track in free views (the reduced system's terms)."""
    F: int
    P: int
    fi: np.ndarray            # int[L] free index of the observation's view, -1 = fixed
    pi: np.ndarray            # int[L] index of its track in prob.points
    anchor: tuple             # (free index, component) or None
    pair_i: np.ndarray        # int[npairs] list positions
    pair_j: np.ndarray


def layout(prob):
    free = np.asarray(prob.free, dtype=np.int64)
    V = prob.K.shape[0]
    fidx = np.full(V, -1, dtype=np.int64)
    fidx[free] = np.arange(len(free))
    fi = fidx[np.asarray(prob.obs_view, dtype=np.int64)]
    pidx = np.full(len(prob.X), -1, dtype=np.int64)
    pidx[prob.points] = np.arange(len(prob.points))
    pi = pidx[np.asarray(prob.obs_track, dtype=np.int64)]
    anchor = None if prob.anchor is None else (int(fidx[prob.anchor[0]]), int(prob.anchor[1]))
    # pairs (i, j) of list observations of one track, both in free views
    sel = np.flatnonzero(fi >= 0)
    order = sel[np.argsort(pi[sel], kind="stable")]
    tr = pi[order]
    n = len(order)
    if n:
        starts = np.flatnonzero(np.r_[True, tr[1:] != tr[:-1]])
        counts = np.diff(np.r_[starts, n])
        grp = np.repeat(np.arange(len(starts)), counts)
        cnt = counts[grp]
        ii = np.repeat(np.arange(n), cnt)
        within = np.arange(cnt.sum()) - np.repeat(np.cumsum(cnt) - cnt, cnt)
        jj = starts[grp[ii]] + within
        pair_i, pair_j = order[ii], order[jj]
    else:
        pair_i = pair_j = np.zeros(0, dtype=np.int64)
    return Layout(F=len(free), P=len(prob.points), fi=fi, pi=pi, anchor=anchor, pair_i=pair_i, pair_j=pair_j)


# ---------------------------------------------------------------------------------------------------------------------
# rotation, residuals, Jacobian blocks
# ---------------------------------------------------------------------------------------------------------------------
def _skew(w):
    z = np.zeros_like(w[..., 0])
    return np.stack([np.stack([z, -w[..., 2], w[..., 1]], -1), np.stack([w[..., 2], z, -w[..., 0]], -1),
                     np.stack([-w[..., 1], w[..., 0], z], -1)], -2)


def rotate(R, w):
    """R exp([w]x) as refine_rotate (Taylor coefficients below |w| = 1e-4), in the precision of the inputs; batched."""
    R, w = np.asarray(R), np.asarray(w)
    th2 = (w * w).sum(-1)
    th = np.sqrt(th2)
    small = th < ROTATE_TAYLOR
    with np.errstate(invalid="ignore", divide="ignore"):
        A = np.where(small, 1 - th2 / 6, np.sin(th) / np.where(small, 1, th))
        B = np.where(small, 0.5 - th2 / 24, (1 - np.cos(th)) / np.where(small, 1, th2))
    W = _skew(w)
    Xm = np.eye(3, dtype=w.dtype) + A[..., None, None] * W + B[..., None, None] * (W @ W)
    return R @ Xm


def projections(K, R, t):
    """P = K [R | t] per view, in the precision of R and t."""
    Kx = np.asarray(K).astype(R.dtype)
    return np.concatenate([Kx @ R, (Kx @ t[:, :, None])], axis=2)


@dataclasses.dataclass
class Eval:
    cost: float               # +inf if a list observation is behind / non-finite
    r: np.ndarray             # [L,2] longdouble
    Jc: np.ndarray            # [L,2,6] longdouble (anchored column zero)
    Jp: np.ndarray            # [L,2,3] longdouble
    p: np.ndarray             # [L,3] longdouble


def evaluate(prob, lay, R, t, X):
    """Residuals and Jacobian blocks of every list observation at (R, t, X) (longdouble)."""
    R, t, X = (np.asarray(a, dtype=LD) for a in (R, t, X))
    P = projections(prob.K, R, t)
    Pv = P[np.asarray(prob.obs_view, dtype=np.int64)]
    Xm = X[np.asarray(prob.obs_track, dtype=np.int64)]
    Xh = np.concatenate([Xm, np.ones((len(Xm), 1), dtype=LD)], axis=1)
    p = np.einsum("mij,mj->mi", Pv, Xh)
    with np.errstate(all="ignore"):
        uv = p[:, :2] / p[:, 2:]
        r = uv - np.asarray(prob.obs_x, dtype=LD)
        KR = Pv[:, :, :3]
        dp = np.empty((len(Xm), 3, 6), dtype=LD)
        # dp/dw_k = K R (e_k x X), dp/dt_k = K e_k
        e = np.eye(3, dtype=LD)
        for k in range(3):
            dp[:, :, k] = np.einsum("mij,mj->mi", KR, np.cross(e[k], Xm))
        dp[:, :, 3:] = np.asarray(prob.K, dtype=LD)[np.asarray(prob.obs_view, dtype=np.int64)]
        Jc = (dp[:, :2, :] - uv[:, :, None] * dp[:, 2:3, :]) / p[:, 2, None, None]
        Jp = (KR[:, :2, :] - uv[:, :, None] * KR[:, 2:3, :]) / p[:, 2, None, None]
        if lay.anchor is not None:
            Jc[lay.fi == lay.anchor[0], :, 3 + lay.anchor[1]] = 0
        ok = (p[:, 2] >= P2_MIN) & np.isfinite(r).all(axis=1)
        cost = _fsum_ld((r * r).sum(axis=1)) if ok.all() else math.inf
    return Eval(cost=cost, r=r, Jc=Jc, Jp=Jp, p=p)


def jacobian_blocks(prob, R=None, t=None, X=None):
    """(Jc [L,2,6], Jp [L,2,3]) in double at (R, t, X) (default: the start), for comparison with oracle.bundle."""
    lay = layout(prob)
    ev = evaluate(prob, lay, prob.R if R is None else R, prob.t if t is None else t, prob.X if X is None else X)
    return ev.Jc.astype(np.float64), ev.Jp.astype(np.float64)


def sparse_jacobian(prob, Jc, Jp):
    """The blocks in oracle.bundle.jacobian's layout (dense [2L, n])."""
    cols = oba._cam_columns(prob)
    L = len(prob.obs_track)
    J = np.zeros((2 * L, prob.n))
    pcol = {int(p): prob.n_cam + 3 * i for i, p in enumerate(prob.points)}
    for m in range(L):
        c, tr = int(prob.obs_view[m]), int(prob.obs_track[m])
        for k in range(2):
            if c in cols:
                for j, col in enumerate(cols[c]):
                    if col >= 0:
                        J[2 * m + k, col] = Jc[m, k, j]
            J[2 * m + k, pcol[tr]:pcol[tr] + 3] = Jp[m, k]
    return J


# ---------------------------------------------------------------------------------------------------------------------
# the damped step
# ---------------------------------------------------------------------------------------------------------------------
def _scale(d):
    with np.errstate(invalid="ignore"):
        return np.where((d > 0) & np.isfinite(d), np.sqrt(np.where((d > 0) & np.isfinite(d), d, 1.0)), 1.0)


@dataclasses.dataclass
class Equations:
    """The double sums the kernel forms at an accepted point, and the longdouble blocks for refinement."""
    U: np.ndarray             # [F,6,6]
    V: np.ndarray             # [P,3,3]
    W: np.ndarray             # [L,6,3] (zero for fixed views)
    gc: np.ndarray            # [F,6] longdouble
    gp: np.ndarray            # [P,3] longdouble
    Dc: np.ndarray            # [F,6]
    Dp: np.ndarray            # [P,3]
    Jc: np.ndarray            # longdouble blocks
    Jp: np.ndarray


def equations(lay, ev):
    free = lay.fi >= 0
    Jc = np.where(free[:, None, None], ev.Jc, 0).astype(LD)
    Jp = ev.Jp
    Jc64, Jp64 = Jc.astype(np.float64), Jp.astype(np.float64)
    with np.errstate(all="ignore"):
        Uo = np.einsum("mki,mkj->mij", Jc64, Jc64)
        Vo = np.einsum("mki,mkj->mij", Jp64, Jp64)
        W = np.einsum("mki,mkj->mij", Jc64, Jp64)
        U = group_sum(np.where(free, lay.fi, lay.F), Uo, lay.F + 1)[:lay.F]
        V = group_sum(lay.pi, Vo, lay.P)
        gc = group_sum(np.where(free, lay.fi, lay.F), np.einsum("mki,mk->mi", Jc, ev.r), lay.F + 1)[:lay.F]
        gp = group_sum(lay.pi, np.einsum("mki,mk->mi", Jp, ev.r), lay.P)
    Dc = _scale(np.diagonal(U, axis1=1, axis2=2))
    Dp = _scale(np.diagonal(V, axis1=1, axis2=2))
    return Equations(U=U, V=V, W=W, gc=gc, gp=gp, Dc=Dc, Dp=Dp, Jc=Jc, Jp=Jp)


@dataclasses.dataclass
class Solve:
    ok: bool
    yc: np.ndarray = None     # [F,6] longdouble
    yp: np.ndarray = None     # [P,3] longdouble
    pivot: float = math.inf   # smallest eigenvalue / (1 + lambda) over every damped V_hat_p and the reduced system
    cond: float = 1.0         # the largest condition of those systems
    refinements: int = 0


def _spd(M):
    """(ok, smallest eigenvalue, condition) of a stack of symmetric matrices."""
    if M.size == 0:
        return True, math.inf, 1.0
    if not np.isfinite(M).all():
        return False, math.inf, math.inf
    ev = np.linalg.eigvalsh(M)
    lo, hi = ev[..., 0], ev[..., -1]
    if (lo <= 0).any():
        return False, float(lo.min()), math.inf
    return True, float(lo.min()), float((hi / lo).max())


class Schur:
    """The damped scaled system at lambda, eliminated by points; ``solve`` takes any right-hand side."""

    def __init__(self, lay, eq, lam):
        self.lay, self.eq, self.lam = lay, eq, lam
        F, P = lay.F, lay.P
        with np.errstate(all="ignore"):
            Vh = eq.V / (eq.Dp[:, :, None] * eq.Dp[:, None, :]) + lam * np.eye(3)
            ok_p, lo_p, cond_p = _spd(Vh)
            self.ok, self.pivot, self.cond = ok_p, lo_p / (1 + lam), cond_p
            if not ok_p:
                return
            self.Vi = np.linalg.inv(Vh)
            Dc = np.vstack([eq.Dc, np.ones((1, 6))])  # row F: the fixed views'
            self.Wh = eq.W / (Dc[np.where(lay.fi >= 0, lay.fi, F)][:, :, None] * eq.Dp[lay.pi][:, None, :])
            self.Wh[lay.fi < 0] = 0
            self.Y = np.einsum("mrs,mst->mrt", self.Wh, self.Vi[lay.pi])
            S4 = np.zeros((F, F, 6, 6))
            S4[np.arange(F), np.arange(F)] = eq.U / (eq.Dc[:, :, None] * eq.Dc[:, None, :]) + lam * np.eye(6)
            i, j = lay.pair_i, lay.pair_j
            if len(i):
                B = np.einsum("nrs,nqs->nrq", self.Y[i], self.Wh[j]).reshape(len(i), 36)
                key = lay.fi[i] * F + lay.fi[j]
                for q in range(36):
                    S4.reshape(F * F, 36)[:, q] -= np.bincount(key, weights=B[:, q], minlength=F * F)
            S = S4.transpose(0, 2, 1, 3).reshape(6 * F, 6 * F)
            self.S = 0.5 * (S + S.T)
            # the rows of zero Jacobian columns (the anchored component, views without list observations) are lambda
            # on the diagonal and 0 elsewhere: solved exactly, they take no part in the condition
            act = np.diagonal(eq.U, axis1=1, axis2=2).reshape(-1) != 0
            ok_s, lo_s, cond_s = _spd(self.S[np.ix_(act, act)])
            if ok_s and not act.all():
                lo_s = min(lo_s, lam)
        self.ok = ok_s
        self.pivot = min(self.pivot, lo_s / (1 + lam))
        self.cond = max(self.cond, cond_s)
        if ok_s and F:
            self.Lc = np.linalg.cholesky(self.S)

    def solve(self, bc, bp):
        """y of the full system with right-hand side (bc [F,6], bp [P,3]) (double)."""
        lay = self.lay
        free = lay.fi >= 0
        dc = np.where(free, lay.fi, lay.F)
        bc2 = bc - group_sum(dc, np.einsum("mrs,ms->mr", self.Y, bp[lay.pi]), lay.F + 1)[:lay.F]
        if lay.F:
            z = np.linalg.solve(self.Lc, bc2.reshape(-1))
            yc = np.linalg.solve(self.Lc.T, z).reshape(lay.F, 6)
        else:
            yc = np.zeros((0, 6))
        yc_i = np.vstack([yc, np.zeros((1, 6))])[dc]
        bp2 = bp - group_sum(lay.pi, np.einsum("mrs,mr->ms", self.Wh, yc_i), lay.P)
        yp = np.einsum("pst,pt->ps", self.Vi, bp2)
        return yc, yp


def apply_full(lay, eq, lam, yc, yp):
    """(A_hat + lambda I) y in longdouble from the per-observation blocks."""
    free = lay.fi >= 0
    dc = (yc / eq.Dc.astype(LD)).astype(LD)
    dp = (yp / eq.Dp.astype(LD)).astype(LD)
    dci = np.vstack([dc, np.zeros((1, 6), dtype=LD)])[np.where(free, lay.fi, lay.F)]
    z = np.einsum("mki,mi->mk", eq.Jc, dci) + np.einsum("mki,mi->mk", eq.Jp, dp[lay.pi])
    oc = group_sum(np.where(free, lay.fi, lay.F), np.einsum("mki,mk->mi", eq.Jc, z), lay.F + 1)[:lay.F]
    op = group_sum(lay.pi, np.einsum("mki,mk->mi", eq.Jp, z), lay.P)
    return oc / eq.Dc.astype(LD) + LD(lam) * yc, op / eq.Dp.astype(LD) + LD(lam) * yp


def damped_step(lay, eq, lam):
    """The scaled step y at lambda, refined against the full system, or ok = False."""
    sch = Schur(lay, eq, lam)
    if not sch.ok:
        return Solve(ok=False, pivot=sch.pivot, cond=sch.cond)
    bc = -eq.gc / eq.Dc.astype(LD)
    bp = -eq.gp / eq.Dp.astype(LD)
    yc0, yp0 = sch.solve(bc.astype(np.float64), bp.astype(np.float64))
    yc, yp = yc0.astype(LD), yp0.astype(LD)
    k = 0
    for k in range(1, 8):
        ac, ap = apply_full(lay, eq, lam, yc, yp)
        rc, rp = bc - ac, bp - ap
        dc, dp = sch.solve(rc.astype(np.float64), rp.astype(np.float64))
        yc, yp = yc + dc.astype(LD), yp + dp.astype(LD)
        size = max(np.abs(yc).max(initial=0), np.abs(yp).max(initial=0))
        if max(np.abs(dc).max(initial=0), np.abs(dp).max(initial=0)) <= 2.0 ** -62 * float(size):
            break
    return Solve(ok=True, yc=yc, yp=yp, pivot=sch.pivot, cond=sch.cond, refinements=k)


# ---------------------------------------------------------------------------------------------------------------------
# the replay
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class Step:
    """One evaluation: its cost, whether it was accepted, lambda after the control (and any re-solves), the state."""
    iteration: int
    cost: float
    accepted: bool
    lam: float
    best_cost: float
    rejected: int
    status: int | None
    reason: str | None        # ftol, floor, max_iter, cap, resolve_cap, xtol, nonfinite
    R: np.ndarray             # the accepted parameters after the control (double)
    t: np.ndarray
    X: np.ndarray
    margins: dict
    cond: float = 1.0
    resolves: int = 0         # systems found not positive definite after this evaluation
    proposal: tuple = None    # (R, t, X) of the next proposal (double)
    y: np.ndarray = None      # the scaled step solved after this evaluation (cameras then points)


@dataclasses.dataclass
class Trace:
    steps: list
    cost_start: float
    floor_sum: float          # sum(u^2 + v^2) over the list
    kappa: float              # max (|p0|_abs + |p1|_abs + |p2|_abs) / |p2| over the list at the start
    n_obs: int


def _kappa(prob, lay, R, t, X):
    P = projections(prob.K, np.asarray(R, dtype=LD), np.asarray(t, dtype=LD)).astype(np.float64)
    Pv = np.abs(P[np.asarray(prob.obs_view, dtype=np.int64)])
    Xm = np.asarray(X, dtype=np.float64)[np.asarray(prob.obs_track, dtype=np.int64)]
    Xh = np.abs(np.column_stack([Xm, np.ones(len(Xm))]))
    pa = np.einsum("mij,mj->mi", Pv, Xh).sum(axis=1)
    p = np.einsum("mij,mj->mi", P[np.asarray(prob.obs_view, dtype=np.int64)], np.column_stack([Xm, np.ones(len(Xm))]))
    with np.errstate(all="ignore"):
        k = pa / np.abs(p[:, 2])
    return float(k.max()) if len(k) else 1.0


def _apply(prob, lay, R, t, X, eq, sol):
    free = np.asarray(prob.free, dtype=np.int64)
    dc = sol.yc / eq.Dc.astype(LD)
    dp = sol.yp / eq.Dp.astype(LD)
    R2, t2, X2 = R.copy(), t.copy(), X.copy()
    if len(free):
        R2[free] = rotate(R[free], dc[:, :3])
        dt = dc[:, 3:].copy()
        if lay.anchor is not None:
            dt[lay.anchor[0], lay.anchor[1]] = 0
        t2[free] = t[free] + dt
    X2[prob.points] = X[prob.points] + dp
    return R2, t2, X2


def replay(prob, max_iter=50):
    """The bundle adjustment of ``prob`` from its start, up to ``max_iter`` evaluated proposals."""
    lay = layout(prob)
    R, t, X = (np.asarray(a, dtype=LD) for a in (prob.R, prob.t, prob.X))
    x = np.asarray(prob.obs_x, dtype=np.float64)
    try:
        floor_sum = math.fsum((x[:, 0] ** 2).tolist() + (x[:, 1] ** 2).tolist()) if len(x) else 0.0
    except OverflowError:  # the kernel's double sum is +inf too: every finite cost is at the floor
        floor_sum = math.inf
    # the kernel's floor is its double sum of fma(u, u, v v); the exactly rounded sum is within L u of it
    floor = COST_FLOOR * floor_sum
    kappa = _kappa(prob, lay, R, t, X)
    lam = LAMBDA0
    cost = math.nan
    it = rejected = evals = 0
    cur = None
    prop = (R, t, X)
    steps = []
    cost_start = math.nan
    while True:
        ev = evaluate(prob, lay, *prop)
        c = ev.cost
        margins = {}
        status = reason = None
        if evals == 0:
            cost_start = c
            if not math.isfinite(c):
                steps.append(Step(iteration=0, cost=c, accepted=False, lam=lam, best_cost=c, rejected=0,
                                  status=NONFINITE, reason="nonfinite", R=prob.R, t=prob.t, X=prob.X, margins={}))
                break
            accept = True
        else:
            it += 1
            accept = c < cost
            margins["accept"] = abs(c - cost) / cost if math.isfinite(c) and cost > 0 else math.inf
        evals += 1
        if accept:
            before = cost
            cur = (prop, equations(lay, ev))
            cost = c
            if it > 0:
                lam /= LAMBDA_FACTOR
                margins["ftol"] = abs((before - c) - FTOL * before) / before
                if before - c <= FTOL * before:
                    status, reason = CONVERGED, "ftol"
            if status is None:
                margins["floor"] = abs(c - floor) / floor if floor > 0 else math.inf
                if c <= floor:
                    status, reason = CONVERGED, "floor"
        else:
            lam *= LAMBDA_FACTOR
            rejected += 1
        if status is None and it >= max_iter:
            status, reason = MAX_ITER, "max_iter"
        if status is None and not lam <= LAMBDA_CAP:
            status, reason = STALLED, "cap"
        cond, resolves, proposal, y = 1.0, 0, None, None
        if status is None:
            eq = cur[1]
            while True:
                sol = damped_step(lay, eq, lam)
                margins["pivot"] = min(margins.get("pivot", math.inf), abs(sol.pivot))
                if sol.ok:
                    break
                resolves += 1
                lam *= LAMBDA_FACTOR
                if not (lam > 0 and lam <= LAMBDA_CAP):
                    status, reason = STALLED, "resolve_cap"
                    break
            if status is None:
                cond = sol.cond
                y = np.concatenate([sol.yc.ravel(), sol.yp.ravel()])
                ny = float(np.sqrt((y * y).sum()))
                lim = XTOL * math.sqrt(cost)
                margins["xtol"] = abs(ny - lim) / lim if lim > 0 else math.inf
                if ny <= lim:
                    status, reason = CONVERGED, "xtol"
                else:
                    prop = _apply(prob, lay, *cur[0], eq, sol)
                    proposal = tuple(a.astype(np.float64) for a in prop)
        Ra, ta, Xa = (a.astype(np.float64) for a in cur[0])
        steps.append(Step(iteration=it, cost=c, accepted=accept, lam=lam, best_cost=cost, rejected=rejected,
                          status=status, reason=reason, R=Ra, t=ta, X=Xa, margins=margins, cond=cond,
                          resolves=resolves, proposal=proposal,
                          y=None if y is None else y.astype(np.float64)))
        if status is not None:
            break
    return Trace(steps=steps, cost_start=cost_start, floor_sum=floor_sum, kappa=kappa, n_obs=len(prob.obs_track))


@dataclasses.dataclass
class Report:
    status: int
    reason: str
    iterations: int
    rejected: int
    cost_start: float
    cost_final: float
    R: np.ndarray
    t: np.ndarray
    X: np.ndarray
    min_margin: float         # the smallest decision margin up to and including the last evaluation (no pivots)
    cond: float               # the largest damped-system condition met on the way
    prior_margin: float = math.inf
    resolves: int = 0
    pivot_margin: float = math.inf  # the smallest pivot margin (eigenvalue / (1 + lambda)) of the systems solved


def report_after(trace: Trace, k: int) -> Report:
    """The report of the kernel run with max_iterations = k, from a replay run with max_iter >= k."""
    mm, pm, cond, resolves = math.inf, math.inf, 1.0, 0
    for s in trace.steps:
        prior = mm
        ms = dict(s.margins)
        if s.reason in ("ftol", "floor", "nonfinite", "max_iter"):  # made before the max_iter test
            stop, reason = s.status, s.reason
        elif s.iteration >= k:  # the capped run makes none of the later decisions
            stop, reason = MAX_ITER, "max_iter"
            for key in ("pivot", "xtol"):
                ms.pop(key, None)
        else:
            stop, reason = s.status, s.reason
            resolves += s.resolves
        pm = min(pm, ms.pop("pivot", math.inf))
        mm = min([mm] + list(ms.values()))
        if stop is None:
            cond = max(cond, s.cond)
        if stop is not None:
            return Report(status=stop, reason=reason, iterations=s.iteration, rejected=s.rejected,
                          cost_start=trace.cost_start, cost_final=s.best_cost if stop != NONFINITE else trace.cost_start,
                          R=s.R, t=s.t, X=s.X, min_margin=mm, cond=cond, prior_margin=prior, resolves=resolves,
                          pivot_margin=pm)
    raise ValueError(f"the replay stopped before iteration {k}: replay it with max_iter >= {k}")
