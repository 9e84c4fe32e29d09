"""The replay of the bundle adjustment (oracle/bundle_exact.py) against independent restatements, on the CPU: its
vectorised Jacobian blocks against oracle.bundle.jacobian, its rotation against oracle.refine.rodrigues, its first step
against the dense solve, its final cost against MINPACK, its rejected-step path, and its point steps with every view
fixed against one 3-parameter solve per point."""
import numpy as np
import pytest

from oracle import bundle as oba
from oracle import bundle_exact as bx
from oracle.refine import rodrigues
from structure_from_motion_b200.scenes import make_multi_view_scene


def _perturb(R, t, X, seed, deg, tfrac, xfrac, anchor=1):
    """Every pose but view 0 rotated by `deg` and its t moved by about `tfrac` of |t| (the anchor's largest component
    kept), every point moved by about `xfrac` of its depth."""
    rng = np.random.default_rng(seed)
    R0, t0 = R.copy(), t.copy()
    for c in range(1, len(R)):
        w = rng.normal(size=3)
        R0[c] = R[c] @ rodrigues(w / np.linalg.norm(w) * np.radians(deg))
        t0[c] = t[c] + rng.normal(size=3) * tfrac * np.linalg.norm(t[c]) / np.sqrt(3)
    if anchor is not None:
        k = int(np.argmax(np.abs(t[anchor])))
        t0[anchor, k] = t[anchor, k]
    return R0, t0, X + rng.normal(size=X.shape) * xfrac * X[:, 2:] / np.sqrt(3)


def _problem(n, V, seed, deg, frac, thr, fixed=(0,), anchor=1, K=None, pseed=4):
    K_, R, t, X, off, view, x, _ = make_multi_view_scene(n, V, seed, noise_px=0.5, outlier_frac=0.1)
    R0, t0, X0 = _perturb(R, t, X, pseed, deg, frac, frac, anchor if anchor is not None and anchor >= 0 else None)
    fmask = np.zeros(V, dtype=bool)
    fmask[list(fixed)] = True
    return oba.problem(K_ if K is None else K, np.concatenate([R0, t0[:, :, None]], 2), X0, off, view, x, thr, fmask,
                       anchor)


def _drop_anchor(prob, y):
    """The scaled step without the anchored component (oracle.bundle's parameter order)."""
    if prob.anchor is None:
        return y
    f = int(np.flatnonzero(prob.free == prob.anchor[0])[0])
    return np.delete(y, 6 * f + 3 + prob.anchor[1])


def test_rotation_is_rodrigues():
    rng = np.random.default_rng(1)
    R = rodrigues(rng.normal(size=3))
    for s in (0.0, 1e-9, 9.9e-5, 1.01e-4, 0.3, 2.0):
        w = rng.normal(size=3)
        w *= s / max(np.linalg.norm(w), 1e-300)
        assert np.abs(bx.rotate(R, w) - R @ rodrigues(w)).max() <= 4e-16


@pytest.mark.parametrize("fixed,anchor", [((0,), 1), ((2, 4), -1), ((0, 1, 2, 3, 4, 5), -1)])
def test_jacobian_blocks_equal_the_analytic_jacobian(fixed, anchor):
    prob = _problem(60, 6, 1, 2.0, 0.02, 1e4, fixed, anchor)
    Jc, Jp = bx.jacobian_blocks(prob)
    J = bx.sparse_jacobian(prob, Jc, Jp)
    J0 = oba.jacobian(prob, prob.R, prob.t, prob.X).toarray()
    assert J.shape == J0.shape and len(prob.obs_track) > 100
    assert np.abs(J - J0).max() <= 1e-14 * np.abs(J0).max()


@pytest.mark.parametrize("fixed,anchor", [((0,), 1), ((2, 5), -1), ((3,), 5)])
def test_first_step_equals_the_dense_solve(fixed, anchor):
    prob = _problem(150, 8, 2, 2.0, 0.02, 1e4, fixed, anchor)
    tr = bx.replay(prob, 1)
    R1, t1, X1, y = oba.dense_step(prob, 1e-3)
    s = tr.steps[0]
    assert s.status is None and s.proposal is not None
    assert np.abs(_drop_anchor(prob, s.y) - y).max() <= 1e-12 * np.abs(y).max()
    Rp, tp, Xp = s.proposal
    assert np.abs(Rp - R1).max() <= 1e-12
    assert np.abs(tp - t1).max() <= 1e-12 * np.abs(t1).max()
    fin = np.isfinite(X1).all(axis=1)
    assert np.abs(Xp[fin] - X1[fin]).max() <= 1e-12 * np.abs(X1[fin]).max()
    assert tr.cost_start == pytest.approx(oba.cost(prob, prob.R, prob.t, prob.X), rel=1e-14)


@pytest.mark.parametrize("n,seed", [(150, 3), (300, 4)])
def test_final_cost_equals_minpack(n, seed):
    prob = _problem(n, 8, seed, 1.0, 0.01, 16.0 * 64)
    tr = bx.replay(prob, 200)
    last = tr.steps[-1]
    assert last.status == bx.CONVERGED
    _, _, _, cm = oba.minpack_replay(prob)
    assert abs(last.best_cost - cm) <= 1e-10 * cm


def test_rejections_on_a_far_start():
    """8 degrees, 10 % of t and X, threshold 1e6 px^2: steps that put points behind views or overshoot are rejected
    and solved again from the accepted equations with lambda x 10."""
    prob = _problem(150, 6, 3, 8.0, 0.1, 1e6)
    tr = bx.replay(prob, 30)
    rej = [s for s in tr.steps if not s.accepted and s.iteration > 0]
    assert len(rej) >= 3
    # a rejected step leaves the accepted parameters and cost as they were, and lambda goes up tenfold
    for a, b in zip(tr.steps, tr.steps[1:]):
        if not b.accepted:
            assert b.best_cost == a.best_cost and np.array_equal(b.X, a.X) and b.lam == a.lam * 10
            assert b.cost > 10 * a.best_cost or not np.isfinite(b.cost) or b.cost >= a.best_cost
    # the step after a rejection is the accepted equations' step at 10 lambda
    i = next(k for k, s in enumerate(tr.steps) if not s.accepted and k > 0)
    lay = bx.layout(prob)
    acc = tr.steps[i - 1]
    eq = bx.equations(lay, bx.evaluate(prob, lay, acc.R, acc.t, acc.X))
    sol = bx.damped_step(lay, eq, tr.steps[i].lam)
    y = np.concatenate([sol.yc.ravel(), sol.yp.ravel()]).astype(np.float64)
    assert np.abs(y - tr.steps[i].y).max() <= 1e-9 * np.abs(y).max()


def test_points_only_step_is_one_solve_per_point():
    """Every view fixed (F = 0): the system is block diagonal, one 3 x 3 damped solve per point."""
    prob = _problem(120, 5, 5, 1.0, 0.02, 1e4, fixed=tuple(range(5)), anchor=-1)
    assert len(prob.free) == 0 and prob.n == 3 * len(prob.points)
    tr = bx.replay(prob, 1)
    y = tr.steps[0].y
    lay = bx.layout(prob)
    for i, p in enumerate(prob.points):
        sel = lay.pi == i
        Xp = prob.X[p]
        rows, res = [], []
        for c, uv in zip(prob.obs_view[sel], prob.obs_x[sel]):
            P = prob.K[c] @ np.column_stack([prob.R[c], prob.t[c]])
            q = P @ np.append(Xp, 1.0)
            u = q[:2] / q[2]
            rows.append((P[:2, :3] - np.outer(u, P[2, :3])) / q[2])
            res.append(u - uv)
        J, r = np.vstack(rows), np.concatenate(res)
        A = J.T @ J
        D = np.sqrt(np.diag(A))
        yi = np.linalg.solve(A / np.outer(D, D) + 1e-3 * np.eye(3), -(J.T @ r) / D)
        assert np.abs(y[3 * i:3 * i + 3] - yi).max() <= 1e-11 * max(np.abs(yi).max(), 1e-300)
