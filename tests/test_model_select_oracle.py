"""CPU checks of the essential-matrix / homography choice: the C scorer (oracle/select_exact.c) against the numpy
restatement (oracle/model_select.py) and OpenCV, and the rule's choice on scenes with known models."""
import numpy as np
import pytest

from oracle import cselect
from oracle import model_select as ms
from structure_from_motion_b200.scenes import make_planar_scene, make_scene

cv2 = pytest.importorskip("cv2")


def _skew(t):
    return np.array([[0.0, -t[2], t[1]], [t[2], 0.0, -t[0]], [-t[1], t[0], 0.0]])


def _true_models(K, R, t, depth=6.0):
    """E = [t]x R and the homography of the fronto-parallel plane at ``depth`` (the middle of make_scene's depths)."""
    H = K @ (R + np.outer(t, [0.0, 0.0, 1.0]) / depth) @ np.linalg.inv(K)
    return _skew(t) @ R, H / H[2, 2]


def _scene(kind, seed, n=2000):
    if kind == "general":
        K, x1, x2, R, t, _ = make_scene(n, 0.3, seed)
        E, H = _true_models(K, R, t)
    else:
        K, x1, x2, H, _ = make_planar_scene(n, 0.3, seed, rotation_only=kind == "rotation")
        _, _, _, R, t, _ = make_scene(8, 0.0, 0)  # make_planar_scene's cameras
        E = _skew(np.zeros(3) if kind == "rotation" else t) @ R
    return K, x1, x2, E, H


def _term_scales(K, x1, x2, E):
    """Per-term size of what the errors cancel from: an inlier's residual is a small difference of large products,
    so both evaluation orders agree relative to those products, not to the residual.  Columns as per_point."""
    F = ms.fundamental(E, K)
    a = np.column_stack([x1, np.ones(len(x1))])
    b = np.column_stack([x2, np.ones(len(x2))])
    la, lb = a @ F.T, b @ F
    sb = (np.abs(la) * np.abs(b)).sum(axis=1) ** 2 / (la[:, 0] ** 2 + la[:, 1] ** 2)
    sa = (np.abs(lb) * np.abs(a)).sum(axis=1) ** 2 / (lb[:, 0] ** 2 + lb[:, 1] ** 2)
    return np.column_stack([sa, sb, np.sum(x1 ** 2, axis=1), np.sum(x2 ** 2, axis=1)])


def _rel_gap(a, b, scale):
    both = np.isfinite(a) & np.isfinite(b)
    assert np.array_equal(np.isfinite(a), np.isfinite(b))
    return np.max(np.abs(a[both] - b[both]) / (np.abs(b[both]) + scale[both])) if both.any() else 0.0


@pytest.mark.parametrize("kind", ["general", "planar"])
def test_c_scorer_matches_numpy_restatement(kind):
    K, x1, x2, E, H = _scene(kind, 3)
    c = cselect.score_models(K, x1, x2, E, H)
    o = ms.score_models(K, x1, x2, E, H)
    scale = _term_scales(K, x1, x2, E)
    for j in range(4):
        assert _rel_gap(c["per_point"][:, j], o["per_point"][:, j], scale[:, j]) <= 1e-12, j
    assert c["count_e"] == o["count_e"] and c["count_h"] == o["count_h"]
    assert abs(c["score_e"] - o["score_e"]) <= 1e-9 * o["score_e"]
    assert abs(c["score_h"] - o["score_h"]) <= 1e-9 * o["score_h"]
    assert c["model"] == o["model"]
    assert c["score_e"] == c["fixed_e"] * 2.0 ** -32 and c["score_h"] == c["fixed_h"] * 2.0 ** -32


def test_fundamental_matrix():
    K, _, _, E, _ = _scene("general", 0)
    F = cselect.fundamental(E, K)
    Ki = np.linalg.inv(K)
    assert np.max(np.abs(F - Ki.T @ E @ Ki)) <= 1e-12 * np.max(np.abs(F))


def test_epipolar_terms_match_opencv():
    K, x1, x2, E, _ = _scene("general", 1)
    F = cselect.fundamental(E, K)
    c = cselect.score_models(K, x1, x2, E=E)
    lines_b = cv2.computeCorrespondEpilines(x1.reshape(-1, 1, 2), 1, F).reshape(-1, 3)  # F a, with a^2 + b^2 = 1
    lines_a = cv2.computeCorrespondEpilines(x2.reshape(-1, 1, 2), 2, F).reshape(-1, 3)  # F^T b
    d_b = (lines_b[:, 0] * x2[:, 0] + lines_b[:, 1] * x2[:, 1] + lines_b[:, 2]) ** 2
    d_a = (lines_a[:, 0] * x1[:, 0] + lines_a[:, 1] * x1[:, 1] + lines_a[:, 2]) ** 2
    scale = _term_scales(K, x1, x2, E)
    assert np.max(np.abs(c["per_point"][:, 1] - d_b) / (d_b + scale[:, 1])) <= 1e-9
    assert np.max(np.abs(c["per_point"][:, 0] - d_a) / (d_a + scale[:, 0])) <= 1e-9
    assert np.all(np.isnan(c["per_point"][:, 2:]))


def test_transfer_terms_match_opencv():
    K, x1, x2, _, H = _scene("planar", 2)
    c = cselect.score_models(K, x1, x2, H=H)
    pb = cv2.perspectiveTransform(x1.reshape(-1, 1, 2), H).reshape(-1, 2)
    pa = cv2.perspectiveTransform(x2.reshape(-1, 1, 2), np.linalg.inv(H)).reshape(-1, 2)
    d_b = np.sum((x2 - pb) ** 2, axis=1)
    d_a = np.sum((x1 - pa) ** 2, axis=1)
    assert np.max(np.abs(c["per_point"][:, 3] - d_b) / np.maximum(d_b, 1.0)) <= 1e-9
    assert np.max(np.abs(c["per_point"][:, 2] - d_a) / np.maximum(d_a, 1.0)) <= 1e-9
    assert np.all(np.isnan(c["per_point"][:, :2]))


@pytest.mark.parametrize("seed", [0, 1, 2])
@pytest.mark.parametrize("kind, want", [("general", 0), ("planar", 1), ("rotation", 1)])
def test_true_models_are_chosen(kind, want, seed):
    K, x1, x2, E, H = _scene(kind, seed, n=5000)
    c = cselect.score_models(K, x1, x2, E, H)
    assert c["model"] == want, c["ratio_h"]
    assert ms.score_models(K, x1, x2, E, H)["model"] == want
    if kind == "rotation":  # E = 0: every epipolar error is 0/0, which scores nothing
        assert c["fixed_e"] == 0 and c["count_e"] == 0 and c["ratio_h"] == 1.0


def test_one_model_is_chosen_whatever_the_scores():
    K, x1, x2, E, H = _scene("general", 0, n=500)
    assert cselect.score_models(K, x1, x2, H=H, ratio=2.0)["model"] == 1
    assert cselect.score_models(K, x1, x2, E=E, ratio=-1.0)["model"] == 0
    assert ms.score_models(K, x1, x2, H=H, ratio=2.0)["model"] == 1
