"""CPU checks of the homography oracle: the numpy 4-point fit, the C transfer-error scorer and the RANSAC loop."""
import random

import numpy as np
import pytest

from oracle import ctransfer
from oracle import homography as oh
from structure_from_motion_b200.scenes import make_planar_scene

cv2 = pytest.importorskip("cv2")


def _rel(a, b):
    return np.max(np.abs(a - b)) / np.max(np.abs(b))


def test_homography_4pt_matches_opencv():
    rng = np.random.default_rng(0)
    done = 0
    while done < 200:
        # well-conditioned quadrilaterals (corners of a unit square, jittered): OpenCV solves the 8x8 system in the
        # given coordinates, so their scale sets its condition number.  float32-representable because OpenCV takes
        # float32 points: both solvers see the same values
        sq = np.array([[0.0, 0.0], [1.0, 0.0], [1.0, 1.0], [0.0, 1.0]])
        a = (sq + rng.uniform(-0.2, 0.2, (4, 2))).astype(np.float32)
        b = (sq * rng.uniform(0.5, 1.5) + rng.uniform(-0.2, 0.2, (4, 2))).astype(np.float32)
        H, ok = oh.homography_4pt(a.astype(np.float64), b.astype(np.float64))
        if not ok:
            continue
        ref = cv2.getPerspectiveTransform(a, b)
        # OpenCV's own result carries ~1e-8 (5e-9..1e-7 from a float64 solve of the same 8x8 system)
        assert _rel(H, ref / ref[2, 2]) <= 2e-7
        A = np.zeros((8, 8))
        rhs = b.astype(np.float64).reshape(8)
        for k, ((x, y), (u, v)) in enumerate(zip(a.astype(np.float64), b.astype(np.float64))):
            A[2 * k] = [x, y, 1, 0, 0, 0, -u * x, -u * y]
            A[2 * k + 1] = [0, 0, 0, x, y, 1, -v * x, -v * y]
        assert _rel(H, np.append(np.linalg.solve(A, rhs), 1.0).reshape(3, 3)) <= 1e-9
        done += 1


def test_noise_free_planar_scene_opencv_agrees():
    _, x1, x2, H_true, out = make_planar_scene(400, 0.0, seed=2, noise_px=0.0)
    Hcv, _ = cv2.findHomography(x1, x2, method=0)
    H, ok = oh.homography_4pt(x1[[0, 50, 100, 150]], x2[[0, 50, 100, 150]])
    assert ok
    assert _rel(H, Hcv / Hcv[2, 2]) <= 1e-6
    assert _rel(H, H_true) <= 1e-9


def test_collinear_samples_are_flagged():
    a = np.array([[0.0, 0.0], [1.0, 1.0], [2.0, 2.0], [5.0, 0.0]])
    b = np.array([[3.0, 1.0], [10.0, 4.0], [1.0, 8.0], [7.0, 7.0]])
    assert not oh.homography_4pt(a, b)[1]
    assert not oh.homography_4pt(b, a)[1]  # collinear in image B
    assert not oh.homography_4pt(np.array([[0.0, 0.0], [0.0, 0.0], [1.0, 5.0], [4.0, 1.0]]), b)[1]  # coincident
    assert oh.homography_4pt(b, b)[1]


def test_c_scorer_matches_numpy_formula():
    K, x1, x2, H_true, _ = make_planar_scene(20000, 0.4, seed=3, noise_px=1.0)
    rng = np.random.default_rng(4)
    for trial in range(5):
        H = H_true + rng.normal(0, 1e-4, (3, 3)) * np.abs(H_true) if trial else H_true
        thr = [4.0, 0.5, 40.0, 1e-3, 1e4][trial]
        inl, val = ctransfer.transfer_exact_many(H, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], thr)
        ref = oh.transfer_error_vectorised(H, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1])
        # relative to the value, or to 1 px^2 where the residual itself cancels (a near-perfect inlier)
        assert np.all(np.abs(val - ref) <= 1e-12 * np.maximum(np.abs(ref), 1.0))
        clear = np.abs(ref - thr) > 1e-9 * thr
        assert np.array_equal(inl[clear], (ref <= thr)[clear])
        assert inl.sum() < len(inl) and (trial > 0 or inl.sum() > 1000)


def test_c_batch_scorer_matches_per_model_scorer():
    _, x1, x2, H_true, _ = make_planar_scene(3000, 0.3, seed=5, noise_px=1.0)
    rng = np.random.default_rng(6)
    Hs = np.stack([H_true * (1 + rng.normal(0, 1e-3, (3, 3))) for _ in range(6)])
    table = rng.integers(0, 3000, (6, 8)).astype(np.int32)
    valid = np.array([1, 1, 0, 1, 1, 1], dtype=np.uint8)
    cnt, s1, s2 = ctransfer.transfer_score_batch(Hs, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], 4.0, table, valid)
    assert cnt[2] == -1
    for h in (0, 1, 3, 4, 5):
        inl, val = ctransfer.transfer_exact_many(Hs[h], x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], 4.0)
        samp = np.zeros(3000, bool)
        samp[table[h, :4]] = True
        assert cnt[h] == int((inl & ~samp).sum())
        terms = val[inl | samp]
        assert abs(s1[h] - terms.sum()) <= 1e-12 * terms.sum()
        assert abs(s2[h] - (terms ** 2).sum()) <= 1e-12 * (terms ** 2).sum()


def test_oracle_ransac_recovers_planar_homography():
    _, x1, x2, H_true, out = make_planar_scene(600, 0.3, seed=7, noise_px=0.5)
    random.seed(5)
    # a 4-point sample is fitted exactly, so with min_extra = 0 a model through an outlier that keeps no other point
    # would win the minimum-error rule: ask for a majority of extra inliers
    res = oh.ransac_homography(x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], 16.0, 250, "rms", 100)
    assert _rel(res["H"], H_true) < 1e-2
    outliers = set(int(i) for i in out)
    inl = set(int(i) for i in res["inlier_indices"][4:])
    assert len(inl & outliers) <= 3 and len(inl) > 250
    # own sampling: the inlier list follows the permutation, and the generator advanced by 100 shuffles
    random.seed(5)
    perm = list(range(600))
    for _ in range(res["best_index"] + 1):
        random.shuffle(perm)
    assert list(res["inlier_indices"][:4]) == perm[:4]
    rest = [i for i in perm[4:] if i in inl]
    assert list(res["inlier_indices"][4:]) == rest


def test_oracle_ransac_rotation_only():
    K, x1, x2, H_true, _ = make_planar_scene(400, 0.2, seed=8, noise_px=0.0, rotation_only=True)
    R = np.linalg.inv(K) @ H_true @ K
    assert np.allclose(R @ R.T / np.cbrt(np.linalg.det(R)) ** 2, np.eye(3), atol=1e-12)
    random.seed(1)
    res = oh.ransac_homography(x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], 1.0, 200, "rms", 50)
    assert _rel(res["H"], H_true) < 1e-9
