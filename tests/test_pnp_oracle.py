"""CPU checks of the PnP oracle (oracle/pnp.py, oracle/reproj_exact.c): the exact P3P, the C scorer, the RANSAC loop
and the invalid-sample rules.  No GPU."""
import random

import cv2
import numpy as np
import pytest

from oracle import creproj
from oracle import pnp as op
from structure_from_motion_b200.scenes import make_pnp_scene, make_three_view_scene

pytestmark = pytest.mark.filterwarnings("ignore::RuntimeWarning")


def _rt(R, t):
    return np.column_stack([R, np.asarray(t).reshape(3)])


def _cv_candidates(X, x, K, flag):
    n, rvecs, tvecs = cv2.solveP3P(np.ascontiguousarray(X[:3]), np.ascontiguousarray(x[:3]), K, None, flags=flag)[:3]
    return [_rt(cv2.Rodrigues(r)[0], tv) for r, tv in zip(rvecs, tvecs)]


@pytest.mark.parametrize("flag", [cv2.SOLVEPNP_P3P, cv2.SOLVEPNP_AP3P])
def test_exact_p3p_matches_opencv(flag):
    """Every OpenCV P3P / AP3P candidate of a well-conditioned sample (no noise, world points spread over the scene)
    is one of the exact candidates to 1e-8 (absolute, on R and on t in scene units of ~6): OpenCV solves in float64
    with a quartic or a cubic, so its error is a few 1e-10 here; the exact candidates are good to 1e-15."""
    K, X, x, R, t, _ = make_pnp_scene(400, 0.0, seed=3, noise_px=0.0)
    rng = np.random.default_rng(0)
    checked = 0
    for _ in range(30):
        idx = rng.choice(len(X), 3, replace=False)
        if op.collinear_ratio(X[idx]) < 0.3:
            continue
        ex = [_rt(Re, te) for Re, te in op.p3p_exact(op.bearings(K, x[idx]), X[idx])]
        for c in _cv_candidates(X[idx], x[idx], K, flag):
            if np.isfinite(c).all() and (c[:, :3] @ X[idx].T + c[:, 3:])[2].min() > 0:
                assert min(np.abs(c - e).max() for e in ex) < 1e-8
                checked += 1
    assert checked >= 20


def test_exact_p3p_contains_truth_and_selection_picks_it():
    """Noise-free samples: the 4th-point rule selects the candidate that equals the truth to 1e-10 (the pixels are the
    float64 roundings of the projections; their 1e-16 relative error reaches t amplified by the sample's
    conditioning, a few 1e-12 here)."""
    K, X, x, R, t, _ = make_pnp_scene(400, 0.0, seed=5, noise_px=0.0)
    rng = np.random.default_rng(1)
    for _ in range(20):
        idx = rng.choice(len(X), 4, replace=False)
        Rt, info = op.fit_pnp_exact(K, X[idx], x[idx])
        assert Rt is not None and info["ncand"] >= 1
        assert np.abs(Rt - _rt(R, t)).max() < 1e-10


def test_c_scorer_matches_numpy_and_opencv():
    """reproj_exact.c: decisions equal the numpy restatement except within 1e-9 relative of the threshold, values
    agree to 1e-10 relative plus 1e-12 px^2 (p0 - u p2 cancels terms of ~5e3 px in 1e-16 relative steps, fused in the
    C, separate in numpy), and equal cv2.projectPoints' squared residuals to 1e-9 relative (plus
    1e-12 px^2: projectPoints divides first, then subtracts)."""
    K, X, x, R, t, _ = make_pnp_scene(5000, 0.3, seed=7)
    Rt = _rt(R, t)
    thr = 2.0
    m_c, v_c = creproj.reproj_exact_many(Rt, K, X, x, thr)
    m_n, v_n = op.reproj(Rt, K, X, x, thr)
    assert np.all(np.abs(v_c - v_n) <= 1e-10 * np.abs(v_n) + 1e-12)
    near = np.abs(v_n - thr) <= 1e-9 * thr
    assert np.array_equal(m_c[~near], m_n[~near])
    proj = cv2.projectPoints(X, cv2.Rodrigues(R)[0], t, K, None)[0].reshape(-1, 2)
    r2 = np.sum((proj - x) ** 2, axis=1)
    assert np.all(np.abs(v_c - r2) <= 1e-9 * r2 + 1e-12)


def test_c_scorer_behind_camera_and_nonfinite():
    """p2 <= 0 (on or behind the camera plane) is never an inlier, whatever F; a NaN record is never an inlier."""
    K = np.array([[800.0, 0, 640], [0, 800, 480], [0, 0, 1]])
    Rt = _rt(np.eye(3), np.zeros(3))
    X = np.array([[0, 0, 5.0], [0, 0, 0.0], [0, 0, -0.0], [0, 0, -5.0], [np.nan, 0, 5], [0, 0, np.inf]])
    x = np.array([[640, 480.0]] * 6)
    m, v = creproj.reproj_exact_many(Rt, K, X, x, 1e300)
    assert m.tolist() == [True, False, False, False, False, False]
    assert v[0] == 0.0 and v[3] == 0.0  # behind the camera: the value exists, the decision is no


@pytest.mark.parametrize("seed", [11, 12, 13])
def test_oracle_ransac_recovers_truth(seed):
    """On make_pnp_scene (300 records, 30 % outliers, 0.5 px noise), 60 iterations: R within 1e-2 (max abs entry) and
    t within 5e-2 of the truth (points at depth 4-8, the pose of a 4-point sample with 0.5 px noise)."""
    K, X, x, R, t, out = make_pnp_scene(300, 0.3, seed=seed)
    random.seed(seed)
    best = op.ransac_pnp(K, X, x, 4.0, 0, "rms", 60)
    assert np.abs(best["Rt"][:, :3] - R).max() < 1e-2
    assert np.abs(best["Rt"][:, 3] - t).max() < 5e-2
    inl = set(best["inlier_indices"].tolist())
    assert len(inl & set(out.tolist())) <= 3


def test_invalid_samples():
    """Collinear world points, three points on one camera ray (no solution with three positive depths) and a
    non-finite coordinate are invalid."""
    K, X, x, R, t, _ = make_pnp_scene(50, 0.0, seed=2, noise_px=0.0)
    Xc = X[:4].copy()
    Xc[2] = Xc[0] + 0.5 * (Xc[1] - Xc[0])  # X2 on the line X0 X1
    Rt, info = op.fit_pnp_exact(K, Xc, x[:4])
    assert Rt is None and info["collinear"] <= op.COLLINEAR
    xs = x[:4].copy()
    xs[1] = xs[2] = xs[0]  # three points on one ray: |l_i - l_j| = |X_i - X_j| has no solution for a triangle
    assert op.fit_pnp_exact(K, X[:4], xs)[0] is None
    Xn = X[:4].copy()
    Xn[1, 0] = np.nan
    assert op.fit_pnp_exact(K, Xn, x[:4])[0] is None
    xn = x[:4].copy()
    xn[3, 1] = np.inf
    assert op.fit_pnp_exact(K, X[:4], xn)[0] is None


def test_three_view_scene_consistent():
    """make_three_view_scene: the noise-free pixels of view 3 are the projections of X under (R3, t3)."""
    K, x1, x2, x3, (R2, t2), (R3, t3), X = make_three_view_scene(100, 0.0, seed=4, noise_px=0.0)
    m, v = op.reproj(_rt(R3, t3), K, X, x3, 1e-12)
    assert m.all() and v.max() < 1e-18
    m, v = op.reproj(_rt(np.eye(3), np.zeros(3)), K, X, x1, 1e-12)
    assert m.all()
