"""The bundle-adjustment oracle (oracle/bundle.py) on the CPU: the analytic Jacobian against central differences, and
the dense Levenberg-Marquardt step iterated to convergence against scipy's MINPACK from the same start."""
import numpy as np
import pytest

from oracle import bundle as oba
from oracle.refine import rodrigues
from structure_from_motion_b200.scenes import make_multi_view_scene


def _perturbed(n, V, seed, noise=0.5):
    K, R, t, X, off, view, x, _ = make_multi_view_scene(n, V, seed, noise_px=noise)
    rng = np.random.default_rng(seed + 100)
    R0, t0 = R.copy(), t.copy()
    for c in range(1, V):
        R0[c] = R[c] @ rodrigues(rng.normal(0, np.radians(0.3), 3))
        t0[c] = t[c] * (1 + rng.normal(0, 0.003, 3))
    X0 = X * (1 + rng.normal(0, 0.002, X.shape))
    Rt0 = np.concatenate([R0, t0[:, :, None]], axis=2)
    fixed = np.zeros(V, dtype=bool)
    fixed[0] = True
    return K, Rt0, X0, off, view, x, fixed


@pytest.mark.parametrize("anchor", [-1, 1])
def test_jacobian_matches_central_differences(anchor):
    K, Rt0, X0, off, view, x, fixed = _perturbed(12, 3, 5)
    prob = oba.problem(K, Rt0, X0, off, view, x, 50.0, fixed, anchor)
    assert len(prob.obs_track) > 10
    J = oba.jacobian(prob, prob.R, prob.t, prob.X).toarray()
    h = 1e-6
    Jn = np.empty_like(J)
    for k in range(prob.n):
        e = np.zeros(prob.n)
        e[k] = h
        rp = oba.residuals(prob, *oba.apply(prob, prob.R, prob.t, prob.X, e))
        rm = oba.residuals(prob, *oba.apply(prob, prob.R, prob.t, prob.X, -e))
        Jn[:, k] = (rp - rm) / (2 * h)
    assert np.abs(J - Jn).max() <= 1e-6 * max(1.0, np.abs(J).max())


def _lm(prob, max_iter=100):
    """refine_control's policy around dense_step (Ftol, cost floor, lambda cap; Xtol on the scaled step)."""
    R, t, X = prob.R, prob.t, prob.X
    c = oba.cost(prob, R, t, X)
    lam = 1e-3
    floor = 1e-24 * float(np.sum(prob.obs_x ** 2))
    for _ in range(max_iter):
        if c <= floor:
            break
        R2, t2, X2, y = oba.dense_step(prob, lam, R, t, X)
        if np.linalg.norm(y) <= 1e-9 * np.sqrt(c):
            break
        c2 = oba.cost(prob, R2, t2, X2)
        if c2 < c:
            done = c - c2 <= 1e-12 * c
            R, t, X, c, lam = R2, t2, X2, c2, lam / 10
            if done:
                break
        else:
            lam *= 10
            if lam > 1e16:
                break
    return R, t, X, c


@pytest.mark.parametrize("seed,V,n,anchor", [(1, 3, 15, 1), (2, 4, 25, -1), (3, 5, 30, 2)])
def test_dense_steps_agree_with_minpack(seed, V, n, anchor):
    K, Rt0, X0, off, view, x, fixed = _perturbed(n, V, seed)
    prob = oba.problem(K, Rt0, X0, off, view, x, 400.0, fixed, anchor)
    assert len(prob.points) > 10
    c0 = oba.cost(prob, prob.R, prob.t, prob.X)
    R, t, X, c = _lm(prob)
    Rm, tm, Xm, cm = oba.minpack_replay(prob)
    assert c < c0 and cm < c0
    assert abs(c - cm) <= 1e-9 * cm
    # the gauge: the fixed view and the anchored component do not move
    assert np.array_equal(R[0], prob.R[0]) and np.array_equal(t[0], prob.t[0])
    if anchor >= 0:
        k = oba.anchor_component(prob.t[anchor])
        assert t[anchor][k] == prob.t[anchor][k] and tm[anchor][k] == prob.t[anchor][k]


def test_list_and_parameter_points():
    K, Rt0, X0, off, view, x, fixed = _perturbed(20, 3, 9)
    X0[3] = np.nan
    inlist, param = oba.start_list(K, Rt0, X0, off, view, x, 50.0)
    assert not param[3] and not inlist[off[3]:off[4]].any()
    pt = np.repeat(np.arange(len(off) - 1), np.diff(off))
    assert np.array_equal(param, np.bincount(pt[inlist], minlength=len(off) - 1) >= 2)
