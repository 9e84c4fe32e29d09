"""CPU checks of the homography pose oracle (oracle/homography_pose.py): the decomposition against OpenCV and the
truth, the rotation-only rule, t parallel to n, the sign fix, and the vote on a planar scene."""
import os
import re

import numpy as np
import pytest

from oracle import homography_pose as hp
from structure_from_motion_b200 import _native
from structure_from_motion_b200.scenes import euler_xyz_intrinsic, make_planar_scene

cv2 = pytest.importorskip("cv2")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
T_TRUE = np.array([-1.0, 0.05, 0.1])
N_TRUE = np.array([0.15, -0.1, 1.0]) / np.linalg.norm([0.15, -0.1, 1.0])


def _rotation(rng):
    q = rng.normal(size=4)
    w, x, y, z = q / np.linalg.norm(q)
    return np.array([[1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w)],
                     [2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w)],
                     [2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)]])


def _random_pose(rng, parallel=False):
    """(K, H, R, t, n, d) with both camera centres on the same side of the plane (1 + n^T R^T t / d > 0); H is
    scaled at random."""
    K = np.array([[rng.uniform(300, 1500), 0.0, rng.uniform(200, 800)],
                  [0.0, rng.uniform(300, 1500), rng.uniform(200, 600)], [0.0, 0.0, 1.0]])
    while True:
        R = _rotation(rng)
        n = rng.normal(size=3)
        n /= np.linalg.norm(n)
        d = rng.uniform(1.0, 10.0)
        # parallel: t along R n, the normal in camera-2 coordinates - H^T H then has the eigenvalue 1 twice, sigma_1 or
        # sigma_3 is 1 and the candidates coincide pairwise
        t = R @ n * rng.uniform(-0.8, 0.8) * d if parallel else rng.normal(size=3)
        if 1.0 + n @ R.T @ t / d > 0.05 and np.linalg.norm(t) > 1e-3:
            break
    H = K @ (R + np.outer(t, n) / d) @ np.linalg.inv(K)
    return K, H * rng.uniform(0.2, 3.0), R, t, n, d


def _set_distance(cands, R, t, n, d):
    """max over (R, t, n, d) of the distance from the truth to the nearest candidate."""
    u = t / np.linalg.norm(t)
    return min(max(np.abs(Rc - R).max(), np.abs(tc - u).max(), np.abs(nc - n).max(), abs(dc - d) / d)
               for Rc, tc, nc, dc in cands)


def test_candidates_match_opencv():
    rng = np.random.default_rng(0)
    compared = 0
    for k in range(300):
        K, H, R, t, n, d = _random_pose(rng, parallel=(k % 10 == 0))
        ours = hp.decompose_homography(H, K, rotation_tolerance=0.0)
        assert not ours["rotation_only"] and len(ours["candidates"]) == 4
        for Ro, to, no, do in ours["candidates"]:
            assert np.all(np.isfinite(Ro)) and np.all(np.isfinite(no)) and np.isfinite(do)
            assert abs(np.linalg.norm(to) - 1.0) < 1e-12
        _, Rs, Ts, Ns = cv2.decomposeHomographyMat(H, K)
        cv = [(Rs[i], Ts[i].ravel() / np.linalg.norm(Ts[i]), Ns[i].ravel()) for i in range(len(Rs))]
        # with t along R n OpenCV's unclamped square roots can give NaN; the oracle's candidates stay finite
        if all(np.all(np.isfinite(np.concatenate([Rc.ravel(), tc, nc]))) for Rc, tc, nc in cv):
            compared += 1
            for Ro, to, no, do in ours["candidates"]:
                err = min(max(np.abs(Ro - Rc).max(), np.abs(to - tc).max(), np.abs(no - nc).max()) for Rc, tc, nc in cv)
                assert err < 1e-6, (k, err)
        # one candidate is the truth, d in units of the baseline (a double eigenvalue costs digits)
        assert _set_distance(ours["candidates"], R, t, n, d / np.linalg.norm(t)) < (1e-6 if k % 10 == 0 else 1e-8), k
    assert compared >= 270


def test_noise_free_planar_scene_is_recovered():
    K, _, _, H, _ = make_planar_scene(500, 0.0, 1, noise_px=0.0)
    ours = hp.decompose_homography(H, K)
    assert not ours["rotation_only"]
    assert abs(ours["sv"][1] - 1.0) < 1e-15
    R = euler_xyz_intrinsic(2.0, -8.0, 1.0)
    assert _set_distance(ours["candidates"], R, T_TRUE, N_TRUE, 6.0 / np.linalg.norm(T_TRUE)) < 1e-8


def test_rotation_only_is_classified():
    K, _, _, H, _ = make_planar_scene(500, 0.0, 2, noise_px=0.0, rotation_only=True)
    ours = hp.decompose_homography(H, K)
    assert ours["rotation_only"] and len(ours["candidates"]) == 1
    R, t, n, d = ours["candidates"][0]
    assert np.abs(R - euler_xyz_intrinsic(2.0, -8.0, 1.0)).max() < 1e-12
    assert np.all(t == 0.0) and np.all(np.isnan(n)) and d == np.inf
    # the tolerance decides: a translating pair (sigma_1 - sigma_3 ~ 0.17) is rotation-only under a tolerance of 1
    K, _, _, H, _ = make_planar_scene(500, 0.0, 2, noise_px=0.0)
    assert not hp.decompose_homography(H, K)["rotation_only"]
    assert hp.decompose_homography(H, K, rotation_tolerance=1.0)["rotation_only"]


def test_t_parallel_to_n_stays_finite():
    rng = np.random.default_rng(5)
    for _ in range(50):
        K, H, R, t, n, d = _random_pose(rng, parallel=True)
        ours = hp.decompose_homography(H, K, rotation_tolerance=0.0)
        s = ours["sv"]
        assert min(abs(s[0] - 1.0), abs(s[2] - 1.0)) < 1e-6  # sigma_1 or sigma_3 is 1
        for Rc, tc, nc, dc in ours["candidates"]:
            assert np.all(np.isfinite(Rc)) and np.all(np.isfinite(tc)) and np.all(np.isfinite(nc)) and np.isfinite(dc)
        assert _set_distance(ours["candidates"], R, t, n, d / np.linalg.norm(t)) < 1e-6


def test_negative_determinant_is_sign_fixed():
    rng = np.random.default_rng(9)
    for _ in range(20):
        K, H, R, t, n, d = _random_pose(rng)
        a = hp.decompose_homography(H, K)
        b = hp.decompose_homography(-H, K)
        assert np.linalg.det(np.linalg.inv(K) @ -H @ K) < 0
        assert np.linalg.det(hp.normalised_homography(-H, K)) > 0
        assert np.allclose(a["sv"], b["sv"], rtol=0, atol=1e-12)
        for Rc, tc, nc, dc in b["candidates"]:
            assert abs(np.linalg.det(Rc) - 1.0) < 1e-9
            assert min(max(np.abs(Rc - Ra).max(), np.abs(tc - ta).max(), np.abs(nc - na).max(), abs(dc - da))
                       for Ra, ta, na, da in a["candidates"]) < 1e-9
        assert _set_distance(b["candidates"], R, t, n, d / np.linalg.norm(t)) < 1e-8


def test_vote_is_decisive_and_picks_the_truth():
    K, x1, x2, H, _ = make_planar_scene(300, 0.0, 3, noise_px=0.0)
    ours = hp.decompose_homography(H, K)
    bits, counts, best = hp.vote(ours["candidates"], K, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1])
    assert counts[best] == 300 and sorted(counts)[-2] < 300
    R, t, n, d = ours["candidates"][best]
    assert np.abs(R - euler_xyz_intrinsic(2.0, -8.0, 1.0)).max() < 1e-8
    assert np.abs(t - T_TRUE / np.linalg.norm(T_TRUE)).max() < 1e-8
    X = hp.triangulate(K, R, t, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], (bits >> best) & 1)
    assert np.max(np.abs(X @ n - d)) / d < 1e-8  # the points lie on the plane n^T X = d


def test_abi_declares_the_homography_pose_calls():
    header = open(os.path.join(ROOT, "include", "sfm_b200.h")).read()
    declared = set(re.findall(r"\b(sfm_[a-z0-9_]+)\s*\(", re.sub(r"/\*.*?\*/", "", header, flags=re.S)))
    new = {"sfm_decompose_homography", "sfm_homography_pose_and_triangulate", "sfm_two_view_homography"}
    assert new <= declared and new <= set(_native.EXPORTED_SYMBOLS)
