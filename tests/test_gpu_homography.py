"""GPU parity of the homography path: the CUDA fitter, scorer, K3 and mask against the oracle on the same inputs.

The scorer and the mask are bit-exact against oracle/transfer_exact.c (oracle_transfer_exact: the same pinned FMA order);
the fitter is compared with numpy's SVD route (oracle.homography.homography_4pt) under a conditioning-scaled bound.
"""
import os
import random

import numpy as np
import pytest

from oracle import ctransfer
from oracle import homography as oh
from oracle import restatement as o
from structure_from_motion_b200 import homography as hg
from structure_from_motion_b200 import _native
from structure_from_motion_b200.scenes import make_planar_scene

pytestmark = pytest.mark.gpu

THR = 16.0  # px^2 on the symmetric transfer error (noise 0.5 px per coordinate)
AGGS = ["sum", "square", "mean", "rms"]


def _rel(a, b):
    return np.max(np.abs(a - b)) / np.max(np.abs(b))


def _cols(x1, x2):
    return x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1]


def _dlt_condition(a, b):
    na, _ = o.hartley_normalise(a)
    nb, _ = o.hartley_normalise(b)
    A = []
    for (x, y), (u, v) in zip(na, nb):
        A.append([-x, -y, -1, 0, 0, 0, u * x, u * y, u])
        A.append([0, 0, 0, -x, -y, -1, v * x, v * y, v])
    s = np.linalg.svd(np.array(A), compute_uv=False)
    return s[0] / s[7]


def _scene_with_collinear(n=3000, seed=1):
    """A planar scene whose last 6 correspondences are collinear in image A (3) and in image B (3)."""
    _, x1, x2, H_true, out = make_planar_scene(n, 0.3, seed=seed)
    x1[-6:-3] = [[100.0, 100.0], [200.0, 250.0], [300.0, 400.0]]  # collinear in A
    x2[-3:] = [[50.0, 700.0], [150.0, 600.0], [250.0, 500.0]]     # collinear in B
    return x1, x2, H_true


def test_fitter_against_oracle(engine):
    x1, x2, _ = _scene_with_collinear()
    n = len(x1)
    rng = np.random.default_rng(3)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(4096)]).astype(np.int32)
    table[:8, :3] = np.arange(n - 6, n - 3)  # collinear in A
    table[8:16, 1:4] = np.arange(n - 3, n)   # collinear in B
    engine.upload_pairs(x1, x2, np.eye(3))
    engine.set_table(table)
    H, valid = engine.fit_homography()
    for i in range(len(table)):
        s = table[i, :4]
        Hr, ok = oh.homography_4pt(x1[s], x2[s])
        assert bool(valid[i]) == ok, i
        if not ok:
            assert np.all(H[i] == 0.0)
            continue
        cond = _dlt_condition(x1[s], x2[s])
        r = _rel(H[i], Hr)
        assert r <= 1e-9 * max(1.0, cond / 1e2), (i, r, cond)  # <= 1e-9 on well-conditioned samples
    assert not valid[:16].any() and valid[16:].sum() > 4000


def test_scorer_and_mask_bit_exact(engine):
    _, x1, x2, _, _ = make_planar_scene(20000, 0.4, seed=4)
    rng = np.random.default_rng(5)
    table = np.stack([rng.choice(20000, 8, replace=False) for _ in range(1024)]).astype(np.int32)
    engine.upload_pairs(x1, x2, np.eye(3))
    for agg in ("sum", "square"):
        engine.set_table(table)
        best, mask, err, cnt, err_h = engine.ransac_homography(THR, -1.0, agg, "min_error", want_arrays=True)
        Hs, valid = engine.get_models(0, 1024)
        c_cnt, s1, s2 = ctransfer.transfer_score_batch(Hs, *_cols(x1, x2), THR, table, valid.astype(np.uint8), nthreads=8)
        assert np.array_equal(cnt, c_cnt)
        ref = s1 if agg == "sum" else s2
        assert np.all(np.abs(err_h[valid] - ref[valid]) <= 1e-12 * np.abs(ref[valid]))
        assert np.all(np.isinf(err_h[~valid]))
        # the winner's mask from the one-call estimate, and the mask of a caller-supplied H
        m_ref, v_ref = ctransfer.transfer_exact_many(best.E, *_cols(x1, x2), THR)
        assert np.array_equal(mask.astype(bool), m_ref) and np.array_equal(err, v_ref)
        for t in (0, 17, 500):
            m, v = engine.homography_mask(Hs[t], THR)
            m_ref, v_ref = ctransfer.transfer_exact_many(Hs[t], *_cols(x1, x2), THR)
            assert np.array_equal(m, m_ref) and np.array_equal(v, v_ref)


@pytest.mark.parametrize("agg", AGGS)
@pytest.mark.parametrize("min_extra", [250, 300.5])
def test_reference_sampler_end_to_end(engine, agg, min_extra):
    _, x1, x2, _, _ = make_planar_scene(600, 0.3, seed=7)
    random.seed(5)
    res = hg.ransac_homography_arrays(x1, x2, THR, min_extra, agg, 100, engine=engine)
    st = random.getstate()
    random.seed(5)
    ref = oh.ransac_homography(*_cols(x1, x2), THR, min_extra, agg, 100)
    assert random.getstate() == st
    assert res.best_index == ref["best_index"]
    assert np.array_equal(res.inlier_indices, ref["inlier_indices"])
    assert abs(res.error - ref["error"]) <= 1e-12 * abs(ref["error"])
    assert _rel(res.H, ref["H"]) <= 1e-6
    assert res.count_extra == len(ref["inlier_indices"]) - 4


def test_selection_modes_against_oracle(engine):
    _, x1, x2, _, _ = make_planar_scene(600, 0.3, seed=9)
    random.seed(11)
    ref = oh.ransac_homography(*_cols(x1, x2), THR, 0, "rms", 100, return_all=True)
    random.seed(11)
    table = o.python_shuffle_table(600, 100)
    # max_inliers: most extra inliers among the valid hypotheses, earliest on ties
    res = hg.ransac_homography_arrays(x1, x2, THR, 0, "rms", sampler="table", table=table, selection="max_inliers",
                                      engine=engine)
    cnt = np.where(ref["all_valid"], ref["all_count"], -1)
    assert res.best_index == int(np.argmax(cnt)) and res.count_extra == cnt.max()
    # msac: minimum of sum_i min(value_i, thr) over all correspondences
    res = hg.ransac_homography_arrays(x1, x2, THR, 0, "rms", sampler="table", table=table, selection="msac",
                                      engine=engine)
    cost = np.full(100, np.inf)
    for t in np.nonzero(ref["all_valid"])[0]:
        _, v = ctransfer.transfer_exact_many(ref["all_H"][t], *_cols(x1, x2), THR)
        cost[t] = np.minimum(v, THR).sum()
    assert res.best_index == int(np.argmin(cost))
    assert abs(res.error - cost.min()) <= 1e-9 * cost.min()


def test_device_sampler_rows_and_split(engine):
    _, x1, x2, _, _ = make_planar_scene(5000, 0.4, seed=12)
    engine.upload_pairs(x1, x2, np.eye(3))
    engine.sample_device(77, 2048)
    rows_e = engine.get_table()
    one = hg.ransac_homography_arrays(x1, x2, THR, 1500, "rms", 2048, sampler="device", seed=77, engine=engine)
    assert np.array_equal(engine.get_table(), rows_e)  # the fit kernel drew the same rows as the E path's sampler
    parts = [hg.ransac_homography_arrays(x1, x2, THR, 1500, "rms", 1024, sampler="device", seed=77, hyp_offset=off,
                                         engine=engine) for off in (0, 1024)]
    win = min(parts, key=lambda r: (r.error, r.best_index))
    assert win.best_index == one.best_index and win.error == one.error
    assert np.array_equal(win.inlier_indices, one.inlier_indices)
    assert np.array_equal(one.sample, rows_e[one.best_index, :4])


@pytest.mark.parametrize("thr", [0.0, -1.0, np.inf, np.nan])
def test_threshold_edge_cases(engine, thr):
    _, x1, x2, _, _ = make_planar_scene(300, 0.3, seed=13)
    table = np.stack([np.random.default_rng(100 + i).choice(300, 8, replace=False) for i in range(64)]).astype(np.int32)
    res = hg.ransac_homography_arrays(x1, x2, thr, 0, "rms", sampler="table", table=table, engine=engine)
    # below 0 / NaN no extra inlier exists and the error is that of the 4 exactly fitted samples (~1e-20 px^2): its
    # winner is decided by the rounding of the fit, so the oracle selects among the GPU's models
    ref = oh.ransac_homography(*_cols(x1, x2), thr, 0, "rms", table=table, models=engine.get_models())
    assert res.best_index == ref["best_index"]
    assert np.array_equal(res.inlier_indices, ref["inlier_indices"])
    assert res.error == ref["error"] or abs(res.error - ref["error"]) <= 1e-12 * abs(ref["error"])


def test_noise_free_scene_rescore_and_near_ties(engine):
    _, x1, x2, H_true, _ = make_planar_scene(500, 0.2, seed=15, noise_px=0.0)
    random.seed(3)
    res = hg.ransac_homography_arrays(x1, x2, 4.0, 300, "rms", 200, engine=engine)
    assert engine.rescored() > 0  # sums of terms ~1e-20 px^2 against thr 4: the double-double pass
    models = engine.get_models()
    # every correct model's error is at the rounding level of its fit: the oracle selects among the GPU's models
    random.seed(3)
    ref = oh.ransac_homography(*_cols(x1, x2), 4.0, 300, "rms", 200, models=models)
    assert res.best_index == ref["best_index"]
    assert np.array_equal(res.inlier_indices, ref["inlier_indices"])
    assert _rel(res.H, H_true) <= 1e-9


def test_rotation_only_recovers_KRKinv(engine):
    K, x1, x2, H_true, _ = make_planar_scene(2000, 0.3, seed=16, noise_px=0.0, rotation_only=True)
    res = hg.ransac_homography_arrays(x1, x2, 1.0, 1000, "rms", 512, sampler="device", seed=1, engine=engine)
    assert _rel(res.H, H_true) <= 1e-6


def test_small_inputs_and_no_candidate(engine):
    _, x1, x2, H_true, _ = make_planar_scene(100, 0.0, seed=17, noise_px=0.0)
    with pytest.raises(ValueError):
        hg.ransac_homography_arrays(x1[:7], x2[:7], 4.0, engine=engine)
    with pytest.raises(ValueError, match="at least 104 inliers"):
        hg.ransac_homography_arrays(x1, x2, 4.0, 100, engine=engine)
    H = hg.fit_homography_arrays(x1[:4], x2[:4], engine=engine)
    assert _rel(H, H_true) <= 1e-9
    with pytest.raises(ValueError):
        hg.fit_homography_arrays(np.array([[0.0, 0.0], [1.0, 1.0], [2.0, 2.0], [0.0, 5.0]]), x2[:4], engine=engine)
    m, v = hg.transfer_error_arrays(H, x1, x2, 1e-6, engine=engine)
    m_ref, v_ref = ctransfer.transfer_exact_many(H, *_cols(x1, x2), 1e-6)
    assert np.array_equal(m, m_ref) and np.array_equal(v, v_ref) and m.all()


def test_full_size_parity():
    eng = _native.Engine(0)
    try:
        _, x1, x2, H_true, _ = make_planar_scene(100_000, 0.4, seed=18)
        res = hg.ransac_homography_arrays(x1, x2, 4.0, 30000, "rms", 65536, sampler="device", seed=3, engine=eng)
        eng.upload_pairs(x1, x2, np.eye(3))
        eng.sample_device(3, 65536)
        best, _, _, cnt, err_h = eng.ransac_homography(4.0, 30000, "rms", want_mask=False, want_arrays=True)
        table = eng.get_table()
        Hs, valid = eng.get_models()
        c_cnt, _, s2 = ctransfer.transfer_score_batch(Hs, *_cols(x1, x2), 4.0, table, valid.astype(np.uint8),
                                                 nthreads=os.cpu_count() or 8)
        assert np.array_equal(cnt, c_cnt)
        err = np.where(valid & (c_cnt >= 30000), np.sqrt(s2 / (4 + c_cnt)), np.inf)
        fin = np.isfinite(err)
        assert np.all(np.abs(err_h[fin] - err[fin]) <= 1e-12 * err[fin]) and np.array_equal(np.isfinite(err_h), fin)
        assert best.index == res.best_index == int(np.argmin(err))
        assert _rel(res.H, H_true) <= 1e-2
    finally:
        eng.close()
