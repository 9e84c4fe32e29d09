"""GPU checks of the homography pose tail: decomposition, vote and triangulation against oracle/homography_pose.py on
the same inputs, accuracy on planar scenes, the rotation-only rule, and the RANSAC part against
ransac_homography_arrays."""
import random

import numpy as np
import pytest

from oracle import homography_pose as hp
from structure_from_motion_b200 import _native
from structure_from_motion_b200 import homography as hg
from structure_from_motion_b200.errors import EightPointCalculationError
from structure_from_motion_b200.scenes import euler_xyz_intrinsic, make_planar_scene

pytestmark = pytest.mark.gpu

THR = 16.0  # px^2 on the symmetric transfer error
# RANSAC selects the minimum aggregated error among hypotheses with enough extra inliers: without a minimum a fit that
# only explains its own 4 samples (error ~0) wins.  The scenes below have 70 % inliers.
R_TRUE = euler_xyz_intrinsic(2.0, -8.0, 1.0)
T_TRUE = np.array([-1.0, 0.05, 0.1]) / np.linalg.norm([-1.0, 0.05, 0.1])
N_TRUE = np.array([0.15, -0.1, 1.0]) / np.linalg.norm([0.15, -0.1, 1.0])
D_TRUE = 6.0 / np.linalg.norm([-1.0, 0.05, 0.1])


def _deg_r(R, Rt):
    return np.degrees(np.arccos(np.clip((np.trace(R.T @ Rt) - 1.0) / 2.0, -1.0, 1.0)))


def _deg_v(a, b):
    return np.degrees(np.arccos(np.clip(a @ b / np.linalg.norm(a) / np.linalg.norm(b), -1.0, 1.0)))


def _set_gap(gpu, ref):
    """max over the GPU's candidates of the distance to the nearest oracle candidate (d relative)."""
    return max(min(max(np.abs(Rg - Ro).max(), np.abs(tg - to).max(), np.abs(ng - no).max(), abs(dg - do) / do)
                   for Ro, to, no, do in ref) for Rg, tg, ng, dg in gpu)


def _cols(x1, x2, idx):
    return x1[idx, 0], x1[idx, 1], x2[idx, 0], x2[idx, 1]


def test_decomposition_matches_oracle(engine):
    rng = np.random.default_rng(1)
    K = np.array([[800.0, 0.0, 640.0], [0.0, 780.0, 480.0], [0.0, 0.0, 1.0]])
    done = 0
    while done < 100:
        q = rng.normal(size=3) * 0.2
        R = euler_xyz_intrinsic(*np.degrees(q))
        n = rng.normal(size=3)
        n /= np.linalg.norm(n)
        t = rng.normal(size=3)
        d = rng.uniform(2.0, 10.0)
        if not 1.0 + n @ R.T @ t / d > 0.05:
            continue
        H = K @ (R + np.outer(t, n) / d) @ np.linalg.inv(K) * rng.choice([-2.0, 0.5, 3.0])
        gpu = hg.decompose_homography_arrays(H, K, engine=engine)
        ref = hp.decompose_homography(H, K)
        assert gpu.rotation_only == ref["rotation_only"]
        assert np.abs(gpu.singular_values - ref["sv"]).max() < 1e-12
        assert _set_gap(gpu.candidates, ref["candidates"]) < 1e-9
        done += 1
    # rotation-only
    K, _, _, H, _ = make_planar_scene(100, 0.0, 1, noise_px=0.0, rotation_only=True)
    gpu = hg.decompose_homography_arrays(H, K, engine=engine)
    assert gpu.rotation_only and len(gpu.candidates) == 1
    R, t, n, d = gpu.candidates[0]
    assert np.abs(R - hp.decompose_homography(H, K)["candidates"][0][0]).max() < 1e-12
    assert np.all(t == 0.0) and np.all(np.isnan(n)) and d == np.inf


def test_decomposition_of_ransac_winners(engine):
    K, x1, x2, _, _ = make_planar_scene(2000, 0.3, 11)
    for seed in range(64):  # with and without a minimum: winners of every quality
        res = hg.ransac_homography_arrays(x1, x2, THR, 1000 * (seed % 2), max_iterations=64, sampler="device", seed=seed,
                                          engine=engine)
        gpu = hg.decompose_homography_arrays(res.H, K, engine=engine)
        ref = hp.decompose_homography(res.H, K)
        assert gpu.rotation_only == ref["rotation_only"]
        if not ref["rotation_only"]:
            assert _set_gap(gpu.candidates, ref["candidates"]) < 1e-9, seed


def test_tail_matches_mask_and_oracle(engine):
    K, x1, x2, _, _ = make_planar_scene(3000, 0.3, 4)
    res = hg.two_view_homography_arrays(K, x1, x2, THR, 1500, max_iterations=200, sampler="device", seed=3,
                                        engine=engine)
    # T1's decision and value are sfm_homography_mask's for the same winner, bit for bit
    mask, err = engine.homography_mask(res.ransac.H, THR)
    assert np.array_equal(mask, res.ransac.mask)
    assert np.array_equal(err.view(np.int64), res.ransac.err.view(np.int64))
    inl = mask.copy()
    inl[res.ransac.sample] = True
    assert np.array_equal(res.inlier_indices, np.flatnonzero(inl))
    # pass bits and counts of the oracle's vote on the GPU's candidates
    p, num, idx, ok, X = engine.homography_pose_and_triangulate(K, THR)
    assert num == len(res.inlier_indices) and np.array_equal(idx, res.inlier_indices)
    bits, counts, best = hp.vote(res.candidates, K, *_cols(x1, x2, idx))
    assert np.array_equal(ok, bits)
    assert np.array_equal(np.array(p.counts), counts) and int(p.best) == best
    assert np.array_equal(res.counts, counts) and np.array_equal(res.passing, ((bits >> best) & 1).astype(bool))
    Xo = hp.triangulate(K, res.R, res.t, *_cols(x1, x2, idx), res.passing)
    assert np.array_equal(np.isnan(Xo), np.isnan(res.points)) and res.passing.sum() > 1000
    live = res.passing
    assert np.max(np.abs(res.points[live] - Xo[live]) / np.linalg.norm(Xo[live], axis=1)[:, None]) < 1e-6


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_planar_scene_pose_and_plane(engine, seed):
    K, x1, x2, _, _ = make_planar_scene(20000, 0.3, seed)
    res = hg.two_view_homography_arrays(K, x1, x2, THR, 10000, max_iterations=500, sampler="device", seed=seed,
                                        engine=engine)
    assert not res.rotation_only
    assert _deg_r(res.R, R_TRUE) < 0.5
    assert _deg_v(res.t, T_TRUE) < 3.0 and _deg_v(res.n, N_TRUE) < 3.0
    assert abs(res.d - D_TRUE) / D_TRUE < 0.05
    X = res.points[res.passing]
    assert len(X) > 10000
    assert np.median(np.abs(X @ res.n - res.d)) / res.d < 1e-2


def test_noise_free_planar_scene_is_exact(engine):
    K, x1, x2, _, _ = make_planar_scene(20000, 0.3, 5, noise_px=0.0)
    res = hg.two_view_homography_arrays(K, x1, x2, THR, 10000, max_iterations=100, sampler="device", seed=5,
                                        engine=engine)
    assert np.abs(res.R - R_TRUE).max() < 1e-8
    assert np.abs(res.t - T_TRUE).max() < 1e-8 and np.abs(res.n - N_TRUE).max() < 1e-8
    assert abs(res.d - D_TRUE) / D_TRUE < 1e-8
    X = res.points[res.passing]
    assert np.max(np.abs(X @ res.n - res.d)) / res.d < 1e-8


def test_rotation_only(engine):
    K, x1, x2, _, _ = make_planar_scene(5000, 0.3, 6, rotation_only=True)
    res = hg.two_view_homography_arrays(K, x1, x2, THR, 2500, max_iterations=200, sampler="device", seed=6,
                                        engine=engine)
    assert res.rotation_only and _deg_r(res.R, R_TRUE) < 0.5
    assert np.all(res.t == 0.0) and np.all(np.isnan(res.n)) and res.d == np.inf
    assert len(res.inlier_indices) > 3000 and not res.passing.any() and np.all(np.isnan(res.points))
    assert np.all(res.counts == 0)
    # the threshold decides: a translating pair (s1 - s3 ~ 0.17) under a tolerance of 1
    K, x1, x2, _, _ = make_planar_scene(5000, 0.3, 6)
    res = hg.two_view_homography_arrays(K, x1, x2, THR, 2500, max_iterations=200, sampler="device", seed=6,
                                        rotation_tolerance=1.0, engine=engine)
    assert res.rotation_only and np.all(np.isnan(res.points))
    res = hg.two_view_homography_arrays(K, x1, x2, THR, 2500, max_iterations=200, sampler="reference",
                                        rotation_tolerance=1.0, engine=engine)
    assert res.rotation_only and not res.passing.any()


def test_reference_sampler_ransac_part_is_ransac_homography(engine):
    K, x1, x2, _, _ = make_planar_scene(1500, 0.3, 8)
    for sel in ["min_error", "max_inliers"]:
        random.seed(21)
        a = hg.ransac_homography_arrays(x1, x2, THR, 5, "rms", 150, selection=sel, engine=engine)
        sa = random.getstate()
        random.seed(21)
        b = hg.two_view_homography_arrays(K, x1, x2, THR, 5, "rms", 150, selection=sel, engine=engine)
        assert random.getstate() == sa
        for f in ["H", "best_index", "error", "count_extra", "inlier_indices", "mask", "err", "sample", "num_invalid",
                  "first_invalid"]:
            va, vb = getattr(a, f), getattr(b.ransac, f)
            assert np.array_equal(np.asarray(va), np.asarray(vb), equal_nan=np.asarray(va).dtype.kind == "f"), f
        assert np.array_equal(b.inlier_indices, np.sort(a.inlier_indices))


def test_fused_call_equals_ransac_then_tail(engine):
    K, x1, x2, _, _ = make_planar_scene(4000, 0.3, 9)
    for seed in [0, 1]:
        fused = hg.two_view_homography_arrays(K, x1, x2, THR, 2000, "sum", 300, 40.0, sampler="device", seed=seed,
                                              engine=engine)
        r = hg.ransac_homography_arrays(x1, x2, THR, 2000, "sum", 300, sampler="device", seed=seed, engine=engine)
        engine.set_winner(r.best_index)
        p, num, idx, ok, X = engine.homography_pose_and_triangulate(K, THR, 40.0)
        for f in ["H", "best_index", "error", "count_extra", "inlier_indices", "mask", "err", "sample"]:
            assert np.array_equal(np.asarray(getattr(r, f)), np.asarray(getattr(fused.ransac, f)), equal_nan=True), f
        b = int(p.best)
        assert b >= 0 and np.array_equal(fused.counts, np.array(p.counts))
        assert np.array_equal(fused.R, np.array(p.R).reshape(4, 3, 3)[b])
        assert np.array_equal(fused.t, np.array(p.t).reshape(4, 3)[b])
        assert np.array_equal(fused.n, np.array(p.n).reshape(4, 3)[b]) and fused.d == p.d[b]
        assert np.array_equal(fused.inlier_indices, idx)
        assert np.array_equal(fused.passing, ((ok >> b) & 1).astype(bool))
        assert np.array_equal(fused.points, X, equal_nan=True)


def test_no_passing_inlier_raises(engine):
    K, x1, x2, _, _ = make_planar_scene(2000, 0.3, 10)
    with pytest.raises(EightPointCalculationError, match="None of the transformations pass the cheirality check."):
        hg.two_view_homography_arrays(K, x1, x2, THR, 1000, max_iterations=100, distance_threshold=1e-3,
                                      sampler="device", engine=engine)
    with pytest.raises(ValueError, match="No model could be found"):
        hg.two_view_homography_arrays(K, x1, x2, THR, 5000, max_iterations=50, sampler="device", engine=engine)


def test_essential_tail_refuses_a_homography_winner(engine):
    K, x1, x2, _, _ = make_planar_scene(1000, 0.3, 12)
    hg.ransac_homography_arrays(x1, x2, THR, max_iterations=50, sampler="device", engine=engine)
    with pytest.raises(_native.NativeError, match=r"-3: .*sfm_homography_pose_and_triangulate"):
        engine.pose_and_triangulate(THR)
