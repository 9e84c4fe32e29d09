"""CPU checks of the refinement oracle (oracle/refine.py): analytic Jacobians, stationarity of the true model on
noise-free data, and that the least-squares optimum from a minimal-sample start lowers the cost and moves toward the
truth."""
import numpy as np
import pytest

from oracle import refine as O
from structure_from_motion_b200.scenes import make_planar_scene, make_scene


def _normalised(K, x):
    return (x - K[:2, 2]) / np.diag(K)[:2]


def _e_data(seed, n=120, noise=0.5):
    K, x1, x2, R, t, out = make_scene(n, 0.0, seed, noise_px=noise)
    return _normalised(K, x1), _normalised(K, x2), R, t / np.linalg.norm(t)


def _rot_err_deg(Ra, Rb):
    return float(np.degrees(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1.0) / 2.0, -1.0, 1.0))))


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_essential_jacobian_matches_central_differences(seed):
    na, nb, R, t = _e_data(seed)
    rng = np.random.default_rng(seed)
    R0, t0 = O.retract_e(R, t, 0.05 * rng.normal(size=5))
    J = O.e_jacobian(R0, t0, na, nb)
    h = 1e-6
    for k in range(5):
        d = np.zeros(5)
        d[k] = h
        Rp, tp = O.retract_e(R0, t0, d)
        Rm, tm = O.retract_e(R0, t0, -d)
        fd = (O.e_residuals(O.skew(tp) @ Rp, na, nb) - O.e_residuals(O.skew(tm) @ Rm, na, nb)) / (2 * h)
        assert np.abs(fd - J[:, k]).max() <= 1e-6 * np.abs(J).max()


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_homography_jacobian_matches_central_differences(seed):
    K, x1, x2, H, _ = make_planar_scene(80, 0.0, seed)
    rng = np.random.default_rng(seed)
    H0 = H * (1.0 + 1e-3 * rng.normal(size=(3, 3)))
    H0 /= H0[2, 2]
    x = H0.reshape(9)[:8]
    J = O.h_jacobian(H0, x1, x2)
    for k in range(8):
        hs = 1e-6 * max(abs(x[k]), 1e-6)
        d = np.zeros(8)
        d[k] = hs
        fd = (O.h_residuals(O.h_from_params(x + d), x1, x2) - O.h_residuals(O.h_from_params(x - d), x1, x2)) / (2 * hs)
        # relative to the scale of the column: the entries span many decades (pixels vs. perspective terms)
        assert np.abs(fd - J[:, k]).max() <= 1e-5 * np.abs(J[:, k]).max()


def test_essential_residual_squares_are_the_symmetric_epipolar_distance():
    na, nb, R, t = _e_data(0)
    E = O.e_from_pose(R, t)
    a = np.column_stack([na, np.ones(len(na))])
    b = np.column_stack([nb, np.ones(len(nb))])
    la, lb = a @ E.T, b @ E
    r = np.sum(lb * a, axis=1)
    sed = r ** 2 * (1 / (la[:, 0] ** 2 + la[:, 1] ** 2) + 1 / (lb[:, 0] ** 2 + lb[:, 1] ** 2))
    np.testing.assert_allclose(O.e_residuals(E, na, nb) ** 2, sed, rtol=1e-10)
    np.testing.assert_allclose(O.e_residuals(7.0 * E, na, nb) ** 2, sed, rtol=1e-10)  # scale invariant


def test_true_models_are_stationary_with_zero_cost_on_noise_free_data():
    na, nb, R, t = _e_data(3, noise=0.0)
    r = O.e_residuals(O.e_from_pose(R, t), na, nb)
    assert O.e_cost(O.e_from_pose(R, t), na, nb) < 1e-24
    J = O.e_jacobian(R, t, na, nb)
    assert np.abs(J.T @ r).max() < 1e-12 * max(1.0, np.abs(J).max())
    K, x1, x2, H, _ = make_planar_scene(80, 0.0, 3, noise_px=0.0)
    r = O.h_residuals(H, x1, x2)
    assert O.h_cost(H, x1, x2) < 1e-16
    J = O.h_jacobian(H, x1, x2)
    assert np.all(np.abs(J.T @ r) <= 1e-8 * np.abs(J).max(axis=0) * np.sqrt(len(r)))


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_essential_optimum_from_a_minimal_sample_lowers_the_cost_and_moves_toward_the_truth(seed):
    na, nb, R, t = _e_data(seed, n=200)
    rng = np.random.default_rng(100 + seed)

    def eight_point(s):  # unnormalised DLT: enough on K-normalised data
        a = np.column_stack([na[s], np.ones(8)])
        return np.linalg.svd(np.column_stack([nb[s, 0:1] * a, nb[s, 1:2] * a, a]))[2][-1].reshape(3, 3)

    # the best of 50 minimal samples, as a RANSAC winner would be
    E8 = min((eight_point(rng.choice(len(na), 8, replace=False)) for _ in range(50)), key=lambda E: O.e_cost(E, na, nb))
    R0, t0 = O.pose_start(E8)
    E0 = O.e_from_pose(R0, t0)
    Ef, cost, (Rf, tf) = O.refine_e(R0, t0, na, nb)
    assert cost < O.e_cost(E0, na, nb)
    assert cost <= O.e_cost(O.e_from_pose(R, t), na, nb) * (1 + 1e-9)
    sv = np.linalg.svd(Ef, compute_uv=False)
    assert abs(sv[0] - sv[1]) <= 1e-12 * sv[0] and sv[2] <= 1e-12 * sv[0]
    Et = O.e_from_pose(R, t)
    assert np.linalg.norm(Ef - Et) < np.linalg.norm(E0 - Et)


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_homography_optimum_from_a_minimal_sample_lowers_the_cost_and_moves_toward_the_truth(seed):
    K, x1, x2, H, _ = make_planar_scene(200, 0.0, seed)
    rng = np.random.default_rng(200 + seed)
    s = rng.choice(len(x1), 4, replace=False)
    rows = []
    for (x, y), (u, v) in zip(x1[s], x2[s]):
        rows.append([-x, -y, -1, 0, 0, 0, u * x, u * y, u])
        rows.append([0, 0, 0, -x, -y, -1, v * x, v * y, v])
    H4 = np.linalg.svd(np.array(rows))[2][-1].reshape(3, 3)
    H4 /= H4[2, 2]
    Hf, cost = O.refine_h(H4, x1, x2)
    assert cost < O.h_cost(H4, x1, x2)
    assert cost <= O.h_cost(H, x1, x2) * (1 + 1e-9)
    # toward the truth, in the transfer of the image corners
    corners = np.array([[0.0, 0.0], [1280.0, 0.0], [0.0, 960.0], [1280.0, 960.0]])

    def warp(M):
        p = np.column_stack([corners, np.ones(4)]) @ M.T
        return p[:, :2] / p[:, 2:]

    assert np.abs(warp(Hf) - warp(H)).max() < np.abs(warp(H4) - warp(H)).max()
