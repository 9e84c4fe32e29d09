"""The oracle pinned: oracle/restatement.py and oracle/sed_exact.c against the golden vectors
generated from the unmodified reference (tests/golden/make_golden.py)."""
import json
import os
import random

import numpy as np
import pytest

from oracle import csed
from oracle import restatement as o
from structure_from_motion_b200.scenes import make_scene

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    with open(os.path.join(G, name)) as f:
        return json.load(f)


def test_eight_point_fixture():
    d = load("eight_point_fixture.json")
    K = np.array(d["K"])
    p1, p2 = np.array(d["cam1_points"]), np.array(d["cam2_points"])
    f = o.eight_point(p1, p2)
    assert np.array_equal(f, np.array(d["F"]))  # same numpy calls => same bits
    na = np.stack(o.k_normalise(p1[:, 0], p1[:, 1], K), 1)
    nb = np.stack(o.k_normalise(p2[:, 0], p2[:, 1], K), 1)
    e = o.eight_point(na, nb)
    assert np.array_equal(e, np.array(d["E"]))
    np.testing.assert_almost_equal(np.array(d["E_opencv"]), e, decimal=5)  # test_epipolar.py:200-203
    np.testing.assert_almost_equal(np.array(d["F_opencv"]), f, decimal=5)  # test_epipolar.py:188-191
    R1, R2, t1 = o.recover_all_r_t(e.copy())
    assert np.array_equal(R1, np.array(d["R1"])) and np.array_equal(R2, np.array(d["R2"]))
    assert np.array_equal(t1, np.array(d["t1"]))
    R, t, mask, _ = o.recover_r_t(na[:, 0], na[:, 1], nb[:, 0], nb[:, 1], e.copy())
    assert np.array_equal(R, np.array(d["R"])) and np.array_equal(t, np.array(d["t"]))
    assert mask.tolist() == d["mask"] == list(range(8))  # test_epipolar.py:240-244
    tn = t / np.linalg.norm(t)
    np.testing.assert_allclose(np.array(d["expected_t_direction"]), tn, atol=1e-5, rtol=0)  # :256-262
    np.testing.assert_allclose(np.array(d["expected_R"]), R, atol=1e-6)
    for k in range(8):  # test_epipolar.py:501-515
        s = o.sed_scalar(na[k, 0], na[k, 1], nb[k, 0], nb[k, 1], np.array(d["E_opencv"]))
        assert s == d["sed_under_E_opencv"][k] and s < 1e-20


def test_ransac_known_answer():
    d = load("ransac_known_answer.json")
    pa, pb = np.array(d["pts_a"]), np.array(d["pts_b"])
    random.seed(d["seed"])
    r = o.ransac_essential(np.array(d["K"]), pa[:, 0], pa[:, 1], pb[:, 0], pb[:, 1], d["threshold"],
                           None, d["method"], None, exact_sed=True)
    assert np.array_equal(r["E"], np.array(d["E"]))
    assert r["inlier_indices"].tolist() == d["inlier_indices"]
    assert list(random.getstate()[1]) == d["rng_state_after"]


def test_config1_known_answer():
    d = load("config1_known_answer.json")
    K, x1, x2, *_ = make_scene(**d["scene"])
    random.seed(d["seed"])
    r = o.ransac_essential(K, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], d["threshold"], d["min_extra"],
                           d["method"], d["max_iterations"])
    assert r["best_index"] == d["best_index"] == 87
    assert np.array_equal(r["E"], np.array(d["E"]))
    assert r["inlier_indices"].tolist() == d["inlier_indices"] and len(d["inlier_indices"]) == 23
    assert abs(r["error"] - d["error"]) <= 1e-12 * d["error"]


def test_sampler_known_answer():
    d = load("sampler_known_answer.json")
    random.seed(d["seed"])
    t = o.python_shuffle_table(d["n"], 3)
    assert t.tolist() == d["rows"]
    assert t[0].tolist() == [910, 516, 275, 950, 612, 970, 52, 75]  # SURVEY.md §8(c)


def test_degenerate_fixture():
    d = load("degenerate_fixture.json")
    assert d["raises"]
    with pytest.raises(o.OracleEightPointError):
        o.eight_point(np.array(d["cam1_points"]), np.array(d["cam2_points"]))


def test_triangulation_known_answer():
    d = load("triangulation_known_answer.json")
    X = o.triangulate_one(*d["feature_a"], *d["feature_b"], np.array(d["P1"]), np.array(d["P2"]))
    assert np.array_equal(X, np.array(d["reference"]))
    np.testing.assert_allclose(np.array(d["expected"]), X, atol=1e-10, rtol=0)  # test_epipolar.py:494-496


def test_sed_vectors_bit_exact():
    rows = load("sed_vectors.json")
    for r in rows:
        E = np.array(r["E"])
        assert o.sed_scalar(r["xa"], r["ya"], r["xb"], r["yb"], E) == r["sed"]
        c = csed.sed_exact_many(E, [r["xa"]], [r["ya"]], [r["xb"]], [r["yb"]])[0]
        assert c == r["sed"], (c, r["sed"])  # the C scorer reproduces numpy's evaluation order


def test_pose_known_answer():
    d = load("pose_known_answer.json")
    K, pa, pb = np.array(d["K"]), np.array(d["pts_a"]), np.array(d["pts_b"])
    R, t, mask, _ = o.recover_r_t_from_e(np.array(d["E"]), K, pa[:, 0], pa[:, 1], pb[:, 0], pb[:, 1])
    assert np.array_equal(R, np.array(d["R"])) and np.array_equal(t, np.array(d["t"]))
    assert mask.tolist() == d["mask"]
    X = o.triangulate_points(pa[:, 0], pa[:, 1], pb[:, 0], pb[:, 1], K, o.tmat(R, t))
    assert np.array_equal(X, np.array(d["X"]))


def test_c_scorer_batch_matches_restatement():
    K, x1, x2, *_ = make_scene(700, 0.4, seed=3)
    nxa, nya = o.k_normalise(x1[:, 0], x1[:, 1], K)
    nxb, nyb = o.k_normalise(x2[:, 0], x2[:, 1], K)
    rng = np.random.default_rng(0)
    table = np.stack([rng.choice(700, 8, replace=False) for _ in range(40)]).astype(np.int32)
    E = np.stack([o.eight_point(np.stack([nxa[s], nya[s]], 1), np.stack([nxb[s], nyb[s]], 1)) for s in table])
    cnt, s1, s2 = csed.score_batch(E, nxa, nya, nxb, nyb, 1.5e-6, table=table, nthreads=3)
    for h in range(40):
        sed = np.array([o.sed_scalar(nxa[i], nya[i], nxb[i], nyb[i], E[h]) for i in range(700)])
        samp = np.zeros(700, bool)
        samp[table[h]] = True
        extra = (sed <= 1.5e-6) & ~samp
        assert cnt[h] == extra.sum()
        np.testing.assert_allclose(s1[h], sed[samp | extra].sum(), rtol=1e-13)
        np.testing.assert_allclose(s2[h], (sed[samp | extra] ** 2).sum(), rtol=1e-13)


RANGE_SCALES = (1e-160, 1e-155, 1e-154, 1e-153, 1e-100, 1e-80, 1e-78, 1e-60, 1.0, 1e60, 1e77, 1e78, 1e150, 1e154,
                1e155, 1e160)


def test_c_scorer_matches_restatement_at_range_edges():
    """The C scorer, which every GPU range test compares against, must follow sed.py itself where the arithmetic leaves
    the normal range: NaN and +-inf in each coordinate, models scaled from 1e-160 to 1e160 (past the underflow knee of
    na, nb near 1e-154 and the overflow knee near 1e154), and records whose norms overflow while r^2 does not, so that
    the reference reports sed = 0."""
    K, x1, x2, R, t, _ = make_scene(48, 0.25, seed=21)
    nxa, nya = o.k_normalise(x1[:, 0], x1[:, 1], K)
    nxb, nyb = o.k_normalise(x2[:, 0], x2[:, 1], K)
    E = np.array([[0.0, -t[2], t[1]], [t[2], 0.0, -t[0]], [-t[1], t[0], 0.0]]) @ R  # the scene's own E = [t]x R
    E /= E[2, 2]
    cols = [nxa, nya, nxb, nyb]
    for c in range(4):  # one NaN, +inf and -inf record in each coordinate, and a record entirely non-finite
        for k, v in enumerate((np.nan, np.inf, -np.inf)):
            cols = [np.append(a, v if j == c else a[8 + 3 * c + k]) for j, a in enumerate(cols)]
    cols = [np.append(a, v) for a, v in zip(cols, (np.inf, np.nan, -np.inf, np.nan))]
    xa, ya, xb, yb = cols
    finite = np.isfinite(xa) & np.isfinite(ya) & np.isfinite(xb) & np.isfinite(yb)
    assert (~finite).sum() == 13
    seds = {}
    with np.errstate(all="ignore"):
        for s in RANGE_SCALES:
            Es = E * s
            c = csed.sed_exact_many(Es, xa, ya, xb, yb)
            ref = np.array([o.sed_scalar(xa[i], ya[i], xb[i], yb[i], Es) for i in range(len(xa))])
            assert np.array_equal(c, ref, equal_nan=True), s
            for thr in (0.0, 1e-12, 1.5e-6, 1e-3, 0.5, 1e100):
                assert np.array_equal(c <= thr, ref <= thr), (s, thr)
            assert not (c[~finite] <= 1e100).any(), s  # a non-finite record is never an inlier below thr = 1e100
            seds[s] = c
    # the regimes are really reached: finite inliers at unit scale, sed = 0 once na and nb overflow (while r^2 stays
    # finite), and no finite sed at all once they underflow
    assert ((seds[1.0] <= 1.5e-6) & finite).sum() >= 10
    assert ((seds[1e154] == 0.0) & finite).sum() > ((seds[1.0] <= 1.5e-6) & finite).sum()
    assert not np.isfinite(seds[1e-160][finite]).any()
    assert np.array_equal(seds[1e-100] <= 1.5e-6, seds[1.0] <= 1.5e-6)


def test_restatement_matches_live_reference():
    """The restatement against what the unmodified reference returned on the same 150 correspondences
    (tests/golden/make_golden.py): E, the inlier pairs in order and the global RNG state after the run for every
    aggregation, then the pose vote and triangulation of the last winner's inliers, all bit for bit."""
    d = load("ransac_methods_known_answer.json")
    K, x1, x2 = np.array(d["K"]), np.array(d["pts_a"]), np.array(d["pts_b"])
    for run in d["runs"]:
        random.seed(d["seed"])
        r = o.ransac_essential(K, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], d["threshold"], d["min_extra"], run["method"],
                               d["max_iterations"], exact_sed=True)
        assert list(random.getstate()[1]) == run["rng_state_after"]
        assert np.array_equal(r["E"], np.array(run["E"]))
        inl = r["inlier_indices"]
        assert np.concatenate([x1[inl], x2[inl]], 1).tolist() == run["pairs"]
    R, t, mask, _ = o.recover_r_t_from_e(r["E"].copy(), K, x1[inl, 0], x1[inl, 1], x2[inl, 0], x2[inl, 1])
    assert np.array_equal(R, np.array(d["R"])) and np.array_equal(t, np.array(d["t"]))
    assert np.array_equal(mask, np.array(d["mask"]))
    X = o.triangulate_points(x1[inl, 0], x1[inl, 1], x2[inl, 0], x2[inl, 1], K, o.tmat(R, t))
    assert np.array_equal(X, np.array(d["X"]))
