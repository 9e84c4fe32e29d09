"""GPU checks of the essential-matrix / homography choice: k_score_models bit for bit against the C scorer
(oracle/select_exact.c), its refusals and degenerate inputs, the sub-result contract of two_view_select_arrays, the
choice on general, planar and rotation-only scenes, and the demo's --model auto."""
import json
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import cselect
from structure_from_motion_b200 import _native
from structure_from_motion_b200 import homography as hg
from structure_from_motion_b200 import two_view
from structure_from_motion_b200.errors import EightPointCalculationError
from structure_from_motion_b200.model_selection import model_scores_arrays, two_view_select_arrays
from structure_from_motion_b200.scenes import euler_xyz_intrinsic, make_planar_scene, make_scene

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
R_TRUE = euler_xyz_intrinsic(2.0, -8.0, 1.0)
T_TRUE = np.array([-1.0, 0.05, 0.1])
E_THR = 1e-5      # SED, K-normalised units (about 3 sigma of make_scene's 0.5 px noise at f = 800)
H_THR = 16.0      # px^2, symmetric transfer error
# of 20 000 correspondences (70 % inliers): the minimum-error winner must explain most of them, or it fits a subset
MIN_EXTRA = 10_000
# Minimal-sample winners carry the noise of their 8 (E) or 4 (H) points.  At 512 hypotheses the E winner on make_scene
# is 1.2-2.8 degrees off and planar H winners give R_H = 0.443-0.466; from 4 096 on, E is within 0.3 degrees and R_H is
# 0.461-0.470 on planar and rotation-only scenes (the true models give 0.476 at this noise).
ITERS = 4096


def _skew(t):
    return np.array([[0.0, -t[2], t[1]], [t[2], 0.0, -t[0]], [-t[1], t[0], 0.0]])


def _models(K, perturb=1e-3, seed=0):
    """E = [t]x R and the homography of the plane z = 6, slightly perturbed so that no entry is special."""
    rng = np.random.default_rng(seed)
    E = _skew(T_TRUE) @ R_TRUE * (1.0 + perturb * rng.standard_normal((3, 3)))
    H = K @ (R_TRUE + np.outer(T_TRUE, [0.0, 0.0, 1.0]) / 6.0) @ np.linalg.inv(K)
    H = H / H[2, 2] * (1.0 + perturb * rng.standard_normal((3, 3)))
    return E, H


def _deg_r(R, Rt):
    return np.degrees(np.arccos(np.clip((np.trace(R.T @ Rt) - 1.0) / 2.0, -1.0, 1.0)))


def _upload(engine, layout, x1, x2, K):
    if layout == "stride2":
        engine.upload_pairs(x1, x2, K)
    elif layout == "soa":
        engine.upload_pairs_soa(x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], K)
    else:
        import torch

        da = torch.from_numpy(np.ascontiguousarray(x1)).cuda()
        db = torch.from_numpy(np.ascontiguousarray(x2)).cuda()
        torch.cuda.synchronize()
        engine.upload_pairs_device(da.data_ptr(), da.data_ptr() + 8, db.data_ptr(), db.data_ptr() + 8, 2, len(x1), K)
        engine.synchronize()
        return da, db  # alive until the kernels that read them have run
    return None


def _assert_exact(s, pp, ref):
    np.testing.assert_array_equal(pp, ref["per_point"])  # NaN where the oracle has NaN
    assert (s.fixed_e, s.fixed_h, s.count_e, s.count_h) == (ref["fixed_e"], ref["fixed_h"], ref["count_e"],
                                                            ref["count_h"])
    assert (s.score_e, s.score_h, s.ratio_h, s.model) == (ref["score_e"], ref["score_h"], ref["ratio_h"], ref["model"])


@pytest.mark.parametrize("n", [8, 100_000])
@pytest.mark.parametrize("layout", ["stride2", "soa", "device"])
def test_bit_exact_against_c_scorer(engine, n, layout):
    K, x1, x2, *_ = make_scene(n, 0.3, seed=n % 7)
    E, H = _models(K)
    keep = _upload(engine, layout, x1, x2, K)
    for sigma, ratio in ((1.0, 0.45), (0.7, 0.3)):
        s, pp = engine.model_scores(E, H, K, sigma, ratio, per_point=True)
        _assert_exact(s, pp, cselect.score_models(K, x1, x2, E, H, sigma, ratio))
    del keep


def test_planar_scene_bit_exact(engine):
    K, x1, x2, H_true, _ = make_planar_scene(100_000, 0.3, seed=4)
    E, _ = _models(K)
    engine.upload_pairs(x1, x2, np.eye(3))  # the records' K does not matter: the scores read the pixels
    s, pp = engine.model_scores(E, H_true, K, 1.0, 0.45, per_point=True)
    ref = cselect.score_models(K, x1, x2, E, H_true)
    _assert_exact(s, pp, ref)
    assert ref["model"] == 1


def test_one_model_only(engine):
    K, x1, x2, *_ = make_scene(5000, 0.3, seed=2)
    E, H = _models(K)
    engine.upload_pairs(x1, x2, K)
    s, pp = engine.model_scores(E, None, K, 1.0, -1.0, per_point=True)  # E only: chosen although R_H = 0 > -1 fails
    _assert_exact(s, pp, cselect.score_models(K, x1, x2, E=E, ratio=-1.0))
    assert s.model == 0 and s.fixed_h == 0 and np.isnan(pp[:, 2:]).all()
    s, pp = engine.model_scores(None, H, K, 1.0, 2.0, per_point=True)  # H only: chosen although R_H <= 2
    _assert_exact(s, pp, cselect.score_models(K, x1, x2, H=H, ratio=2.0))
    assert s.model == 1 and s.fixed_e == 0 and np.isnan(pp[:, :2]).all()


def test_refusals(engine):
    K, x1, x2, *_ = make_scene(1000, 0.3, seed=3)
    E, H = _models(K)
    fresh = _native.Engine(0)
    try:
        with pytest.raises(_native.NativeError, match="-3"):
            fresh.model_scores(E, H, K)  # no correspondences
        fresh.batch_ransac(x1, x2, [0, 500, 1000], np.stack([K, K]), 64, 1, E_THR)
        with pytest.raises(_native.NativeError, match="-3"):
            fresh.model_scores(E, H, K)  # a batched context
    finally:
        fresh.close()
    engine.upload_pairs(x1, x2, K)
    bad_k = [np.zeros((3, 3)), np.diag([800.0, 0.0, 1.0]), np.where(np.eye(3) > 0, np.nan, 0.0), K * np.inf]
    bad = [dict(E=None, H=None)] + [dict(K=k) for k in bad_k]
    bad += [dict(sigma=v) for v in (0.0, -1.0, np.nan, np.inf)] + [dict(ratio=v) for v in (np.nan, np.inf, -np.inf)]
    bad += [dict(E=E * np.nan), dict(H=np.where(np.eye(3) > 0, np.inf, H))]
    for b in bad:
        args = dict(E=E, H=H, K=K, sigma=1.0, ratio=0.45)
        args.update(b)
        with pytest.raises(_native.NativeError, match="-1"):
            engine.model_scores(args["E"], args["H"], args["K"], args["sigma"], args["ratio"])


def test_degenerate_models_score_nothing_and_the_state_cleans_itself(engine):
    K, x1, x2, *_ = make_scene(3000, 0.3, seed=5)
    engine.upload_pairs(x1, x2, K)
    # E = 0: every line is 0 (0/0 = NaN); H with a zero last row maps every point of image A to infinity (F/0 = inf)
    Hz = np.array([[1.0, 0.0, 0.0], [0.0, 1.0, 0.0], [0.0, 0.0, 0.0]])
    s, pp = engine.model_scores(np.zeros((3, 3)), Hz, K, per_point=True)
    _assert_exact(s, pp, cselect.score_models(K, x1, x2, np.zeros((3, 3)), Hz))
    assert np.isnan(pp[:, :2]).all() and np.isposinf(pp[:, 3]).all()
    assert (s.fixed_e, s.count_e, s.count_h) == (0, 0, 0)
    E, H = _models(K)
    first, _ = engine.model_scores(E, H, K)
    second, _ = engine.model_scores(E, H, K)
    assert bytes(first) == bytes(second)
    ref = cselect.score_models(K, x1, x2, E, H)
    assert (second.fixed_e, second.fixed_h) == (ref["fixed_e"], ref["fixed_h"])


def test_model_scores_arrays(engine):
    K, x1, x2, H_true, _ = make_planar_scene(2000, 0.3, seed=6)
    E, _ = _models(K)
    res = model_scores_arrays(K, x1, x2, E, H_true, per_point=True, engine=engine)
    ref = cselect.score_models(K, x1, x2, E, H_true)
    assert res.model == "homography" and res.fixed_h == ref["fixed_h"] and res.fixed_e == ref["fixed_e"]
    np.testing.assert_array_equal(res.per_point, ref["per_point"])


def _eq_tree(a, b):
    """Dataclass results equal field by field, arrays bit for bit (NaN where NaN)."""
    if a is None or b is None:
        return a is b
    for k, v in vars(a).items():
        w = getattr(b, k)
        if hasattr(v, "__dataclass_fields__"):
            assert _eq_tree(v, w), k
        elif isinstance(v, np.ndarray):
            np.testing.assert_array_equal(v, w, err_msg=k)
            assert v.dtype == w.dtype, k
        elif isinstance(v, list):
            assert len(v) == len(w), k
            for x, y in zip(v, w):
                for p, q in zip(x, y):
                    np.testing.assert_array_equal(p, q, err_msg=k)
        else:
            assert v == w or (v != v and w != w), (k, v, w)
    return True


def test_sub_results_equal_standalone_calls_device(engine):
    K, x1, x2, *_ = make_planar_scene(20000, 0.3, seed=7)
    args = (K, x1, x2)
    sel = two_view_select_arrays(*args, E_THR, H_THR, MIN_EXTRA, "rms", 256, sampler="device", seed=11, engine=engine)
    e = two_view.two_view_arrays(*args, E_THR, MIN_EXTRA, "rms", 256, sampler="device", seed=11,
                                 on_degenerate="skip", engine=engine)
    h = hg.two_view_homography_arrays(*args, H_THR, MIN_EXTRA, "rms", 256, sampler="device", seed=11, engine=engine)
    assert _eq_tree(sel.essential, e) and _eq_tree(sel.homography, h)
    assert sel.model == "homography" and sel.essential_failure is None and sel.homography_failure is None


def test_sub_results_equal_standalone_calls_reference(engine):
    K, x1, x2, *_ = make_scene(600, 0.3, seed=8)
    random.seed(21)
    sel = two_view_select_arrays(K, x1, x2, E_THR, H_THR, 30, "rms", 200, engine=engine)
    after = random.getstate()
    random.seed(21)
    e = two_view.two_view_arrays(K, x1, x2, E_THR, 30, "rms", 200, on_degenerate="skip", engine=engine)
    try:
        h = hg.two_view_homography_arrays(K, x1, x2, H_THR, 30, "rms", 200, engine=engine)
    except (ValueError, EightPointCalculationError) as exc:
        h = None
        assert sel.homography_failure == str(exc)
    assert random.getstate() == after
    assert _eq_tree(sel.essential, e) and _eq_tree(sel.homography, h)
    assert sel.model == "essential"


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_general_scene_picks_essential(engine, seed):
    K, x1, x2, R, t, _ = make_scene(20000, 0.3, seed)
    sel = two_view_select_arrays(K, x1, x2, E_THR, H_THR, MIN_EXTRA, "rms", ITERS, sampler="device", seed=seed,
                                 engine=engine)
    assert sel.model == "essential", (sel.scores, sel.homography_failure)
    assert _deg_r(sel.R, R) < 0.5 and not sel.rotation_only
    assert sel.R is sel.essential.R


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_planar_scene_picks_homography(engine, seed):
    K, x1, x2, _, _ = make_planar_scene(20000, 0.3, seed)
    sel = two_view_select_arrays(K, x1, x2, E_THR, H_THR, MIN_EXTRA, "rms", ITERS, sampler="device", seed=seed,
                                 engine=engine)
    assert sel.model == "homography", (sel.scores, sel.essential_failure)
    assert _deg_r(sel.R, R_TRUE) < 0.5 and not sel.rotation_only
    assert sel.R is sel.homography.R and sel.points is sel.homography.points


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_rotation_only_picks_homography(engine, seed):
    K, x1, x2, _, _ = make_planar_scene(20000, 0.3, seed, rotation_only=True)
    sel = two_view_select_arrays(K, x1, x2, E_THR, H_THR, MIN_EXTRA, "rms", ITERS, sampler="device", seed=seed,
                                 engine=engine)
    assert sel.model == "homography", (sel.scores, sel.essential_failure)
    assert sel.rotation_only and np.all(sel.t == 0.0) and _deg_r(sel.R, R_TRUE) < 0.5


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_noise_free_planar_scene_has_no_essential_matrix(engine, seed):
    K, x1, x2, _, _ = make_planar_scene(5000, 0.0, seed, noise_px=0.0)
    sel = two_view_select_arrays(K, x1, x2, E_THR, H_THR, 500, "rms", 256, sampler="device", seed=seed, engine=engine)
    assert sel.model == "homography" and sel.essential is None and sel.essential_failure
    assert sel.scores.score_e == 0.0 and sel.scores.ratio_h == 1.0


def test_both_failing_raises(engine):
    K, x1, x2, *_ = make_scene(100, 0.0, seed=9)
    with pytest.raises(ValueError, match="essential matrix: .*homography: "):
        two_view_select_arrays(K, x1, x2, E_THR, H_THR, 10_000, "rms", 16, sampler="device", engine=engine)


def _demo(*extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "apps", "sfm.py"), "--synthetic", "0", "--seed", "1",
                          "--model", "auto", *extra], capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_demo_auto_picks_essential_on_the_layered_scene():
    res = _demo()
    assert res["model"] == "essential" and not res["rotation_only"], res
    assert res["rotation_error_deg"] < 0.5, res


def test_demo_auto_picks_homography_on_a_planar_scene():
    res = _demo("--planar")
    assert res["model"] == "homography" and res["homography_score_ratio"] > 0.45, res
    assert res["rotation_error_deg"] < 1.0, res
