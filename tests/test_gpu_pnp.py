"""The absolute-pose (PnP) path on the GPU against the oracles: the P3P fitter against the exact Grunert solution, the
scorer, K3 and the mask bit for bit against oracle/reproj_exact.c, the samplers end to end against the oracle's
RANSAC, a full-size run, accuracy on synthetic scenes, the composition with the two-view tail, and the refusals."""
import os
import random
import subprocess
import sys

import numpy as np
import pytest

from oracle import creproj
from oracle import pnp as op
from structure_from_motion_b200 import _native
from structure_from_motion_b200.pnp import fit_pnp_arrays, ransac_pnp_arrays, reprojection_error_arrays
from structure_from_motion_b200.scenes import make_pnp_scene, make_three_view_scene
from structure_from_motion_b200.two_view import two_view_arrays

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def eng():
    return _native.Engine(0)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def test_fitter_against_exact_p3p(eng):
    """600 samples of make_pnp_scene (1 px noise, 30 % outliers, so that some samples have several solutions near
    each other).  Outside the ambiguity band - point-3 errors of the two best solutions within 1e-6 relative, or the
    collinearity sine within 0.1 % of its tolerance - validity equals the exact oracle's and [R|t] agrees to 1e-7
    relative (Lambda Twist plus Gauss-Newton in float64 against a 50-digit solve).
    At most 2 % of the samples may fall in the band."""
    K, X, x, R, t, _ = make_pnp_scene(3000, 0.3, seed=21, noise_px=1.0)
    rng = np.random.default_rng(5)
    table = np.stack([rng.choice(len(X), 8, replace=False) for _ in range(600)]).astype(np.int32)
    eng.upload_pnp(X, x, K)
    eng.set_table(table)
    Rt, valid = eng.fit_pnp()
    band = 0
    for i, row in enumerate(table):
        ref, info = op.fit_pnp_exact(K, X[row[:4]], x[row[:4]])
        if info["gap"] < 1e-6 or abs(info["collinear"] / op.COLLINEAR - 1) < 1e-3:
            band += 1
            continue
        assert (ref is not None) == bool(valid[i]), i
        if ref is not None:
            assert np.abs(Rt[i] - ref).max() <= 1e-7 * (1 + np.abs(ref).max()), (i, np.abs(Rt[i] - ref).max())
    assert band <= 12


def test_fitter_invalid_samples(eng):
    """Collinear world points, three points on one ray and non-finite coordinates are invalid on the device too."""
    K, X, x, R, t, _ = make_pnp_scene(50, 0.0, seed=2, noise_px=0.0)
    Xc = X[:4].copy()
    Xc[2] = Xc[0] + 0.5 * (Xc[1] - Xc[0])
    xs = x[:4].copy()
    xs[1] = xs[2] = xs[0]
    Xn = X[:4].copy()
    Xn[1, 0] = np.nan
    xn = x[:4].copy()
    xn[3, 1] = np.inf
    for Xs, xs_ in ((Xc, x[:4]), (X[:4], xs), (Xn, x[:4]), (X[:4], xn)):
        with pytest.raises(ValueError):
            fit_pnp_arrays(K, Xs, xs_, engine=eng)
    R_, t_ = fit_pnp_arrays(K, X[:4], x[:4], engine=eng)
    assert np.abs(R_ - R).max() < 1e-10 and np.abs(t_ - t).max() < 1e-10


SIZES = [8, 63, 64, 65, 2047, 2048, 2049, 100_000]
THRESHOLDS = [float(np.nextafter(4.0, 0)), 4.0, float(np.nextafter(1024.0, 0)), 1024.0, 0.0, -1.0, 1.5e100]


@pytest.mark.parametrize("n", SIZES)
def test_scorer_bit_identical(eng, n):
    """Counts (K3's count_extra) and the winner's mask and values are bit-identical to reproj_exact.c; the aggregated
    errors agree to 1e-12 relative and the winner is among the oracle's best, for every aggregation, MSAC and
    max-inliers, at thresholds at and just below 2^k, 0, -1 and above 1e100, with hypothesis counts around the
    64-hypothesis group.  Records include p2 = +0, -0, < 0 and non-finite ones."""
    rng = np.random.default_rng(n)
    K, X, x, R, t, _ = make_pnp_scene(n, 0.3, seed=n, noise_px=1.0)
    if n >= 64:  # special records (never a sample: the table draws from the first n - 8)
        Rt = np.column_stack([R, t])
        c = np.linalg.solve(R, -t)  # the camera centre: X - c along the optical axis has p2 = 0
        ax = R[2]
        X[-1] = c + np.cross(ax, [1.0, 0, 0])          # p2 = +0 (or its rounding)
        X[-2] = c - np.cross(ax, [0, 1.0, 0])
        X[-3] = c - 3.0 * ax                            # behind the camera
        X[-4, 1] = np.nan
        x[-5, 0] = np.inf
        X[-6] = np.copysign(0.0, -1.0)                   # -0 coordinates
        assert np.isfinite(Rt).all()
    for h in (63, 64, 65, 129):
        m = n - 8 if n >= 64 else n
        table = np.stack([rng.choice(m, 8, replace=False) for _ in range(h)]).astype(np.int32)
        for agg, sel in (("sum", "min_error"), ("square", "min_error"), ("mean", "min_error"), ("rms", "min_error"),
                         ("rms", "max_inliers"), ("sum", "msac")):
            thr = THRESHOLDS[(h + len(agg) + len(sel)) % len(THRESHOLDS)]
            eng.upload_pnp(X, x, K)
            eng.set_table(table)
            best, Rt_w, mask, err, cnt, err_h = eng.ransac_pnp(thr, 0.0, agg, sel, want_arrays=True)
            models, valid = eng.get_pnp_models()
            exp = op.expected_selection(models, valid, K, X, x, thr, table, agg, sel)
            assert np.array_equal(cnt, np.where(valid, exp["count_extra"], -1)), (h, agg, sel, thr)
            fin = np.isfinite(exp["err"])
            assert np.array_equal(fin, np.isfinite(err_h))
            assert np.all(np.abs(err_h[fin] - exp["err"][fin]) <= 1e-12 * np.abs(exp["err"][fin]) + 1e-300)
            assert int(best.index) in exp["winners"].tolist()
            if best.index >= 0:
                assert np.array_equal(_bits(Rt_w), _bits(models[best.index]))
                m_c, v_c = creproj.reproj_exact_many(models[best.index], K, X, x, thr)
                assert np.array_equal(m_c, mask.astype(bool))
                assert np.array_equal(_bits(v_c), _bits(err))
    # the mask of a caller's pose, on every record
    m_g, v_g = reprojection_error_arrays(R, t, K, X, x, 4.0, engine=eng)
    m_c, v_c = creproj.reproj_exact_many(np.column_stack([R, t]), K, X, x, 4.0)
    assert np.array_equal(m_g, m_c) and np.array_equal(_bits(v_g), _bits(v_c))


def test_reference_sampler_end_to_end(eng):
    """The reference sampler: best_index, inlier_indices and the error equal the oracle's RANSAC run on the device's
    poses (so that the fitter's last bits do not decide), and random.getstate() afterwards equals the oracle loop's."""
    K, X, x, R, t, _ = make_pnp_scene(1500, 0.4, seed=31)
    random.seed(77)
    res = ransac_pnp_arrays(K, X, x, 4.0, 0, "rms", 200, engine=eng)
    after_gpu = random.getstate()
    models = eng.get_pnp_models()
    random.seed(77)
    ref = op.ransac_pnp(K, X, x, 4.0, 0, "rms", 200, models=models)
    assert random.getstate() == after_gpu
    assert res.best_index == ref["best_index"]
    assert np.array_equal(res.inlier_indices, ref["inlier_indices"])
    assert abs(res.error - ref["error"]) <= 1e-12 * ref["error"]
    assert np.abs(res.R - R).max() < 1e-2


def test_device_sampler_split_and_table(eng):
    """Device sampler: one run of 512 hypotheses and two runs of 256 split by hyp_offset agree (the better half holds
    the winner, with the same global index, pose and error).  Table sampler: the result equals the oracle loop on
    that table with the device's poses."""
    K, X, x, R, t, _ = make_pnp_scene(4000, 0.5, seed=41)
    full = ransac_pnp_arrays(K, X, x, 4.0, 0, "rms", 512, sampler="device", seed=9, engine=eng)
    a = ransac_pnp_arrays(K, X, x, 4.0, 0, "rms", 256, sampler="device", seed=9, hyp_offset=0, engine=eng)
    b = ransac_pnp_arrays(K, X, x, 4.0, 0, "rms", 256, sampler="device", seed=9, hyp_offset=256, engine=eng)
    win = a if (a.error, a.best_index) <= (b.error, b.best_index) else b
    assert full.best_index == win.best_index and full.error == win.error
    assert np.array_equal(full.R, win.R) and np.array_equal(full.t, win.t)
    rng = np.random.default_rng(3)
    table = np.stack([rng.choice(len(X), 4, replace=False) for _ in range(300)]).astype(np.int32)
    res = ransac_pnp_arrays(K, X, x, 4.0, 0, "mean", sampler="table", table=table, engine=eng)
    ref = op.ransac_pnp(K, X, x, 4.0, 0, "mean", 300, table=np.concatenate([table, table], 1),
                        models=eng.get_pnp_models())
    assert res.best_index == ref["best_index"]
    assert np.array_equal(res.inlier_indices, ref["inlier_indices"])


def test_full_size(eng):
    """100 000 records x 65 536 device-sampled hypotheses: every hypothesis's count equals the C scorer on the
    device's poses, and the validity of 64 of them equals the exact fitter oracle (outside its ambiguity band)."""
    K, X, x, R, t, _ = make_pnp_scene(100_000, 0.4, seed=51)
    eng.upload_pnp(X, x, K)
    eng.sample_device(123, 65_536)
    best, Rt_w, mask, err, cnt, err_h = eng.ransac_pnp(4.0, 0.0, "rms", "min_error", want_arrays=True)
    table = eng.get_table()
    models, valid = eng.get_pnp_models()
    c_cnt, _, _ = creproj.reproj_score_batch(models, K, X, x, 4.0, table, valid.astype(np.uint8),
                                             nthreads=os.cpu_count() or 8)
    assert np.array_equal(cnt, np.where(valid, c_cnt, -1))
    for i in np.random.default_rng(0).choice(65_536, 64, replace=False):
        ref, info = op.fit_pnp_exact(K, X[table[i][:4]], x[table[i][:4]])
        if info["gap"] < 1e-6 or abs(info["collinear"] / op.COLLINEAR - 1) < 1e-3:
            continue
        assert (ref is not None) == bool(valid[i])
    assert np.abs(Rt_w[:, :3] - R).max() < 5e-3


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_accuracy(eng, seed):
    """make_pnp_scene(20 000, 0.4, seed), threshold 4 px^2, 100 iterations, reference sampler seeded with ``seed``.
    The oracle's RANSAC at these seeds gave max |R - R_true| = 2.0e-3, 2.5e-3, 3.5e-3 and max |t - t_true| = 1.1e-2,
    1.4e-2, 2.1e-2; the bounds are 5e-3 and 3e-2."""
    K, X, x, R, t, _ = make_pnp_scene(20_000, 0.4, seed)
    random.seed(seed)
    res = ransac_pnp_arrays(K, X, x, 4.0, 0, "rms", 100, engine=eng)
    assert np.abs(res.R - R).max() < 5e-3
    assert np.abs(res.t - t).max() < 3e-2


def test_three_view_composition(eng):
    """two_view_arrays on views 1-2 (SED threshold 1e-5, at least 1 500 extra inliers), then ransac_pnp_arrays with its
    passing points against their view-3 pixels on the same engine, at least half of them extra inliers.  The bounds
    follow the reconstruction, not the PnP: the minimal-sample E of views 1-2 is itself 1.5e-2 (R2) and 5.8e-2 (t2) off
    the truth on this scene, and the points carry that error.  Measured on one B200: R3 within 1.3e-2 of the truth and
    t3 within 2.7e-2 of t3_true / |t12|.  The test asks for 2e-2 and 5e-2, and for R3 to be no further from the truth
    than 1.5 times R2 (the new view registered about as well as the pair was reconstructed).  A two_view_arrays call
    after the PnP call is bit-identical to the same call on a fresh engine."""
    K, x1, x2, x3, (R2, t2), (R3, t3), X = make_three_view_scene(3000, 0.2, seed=61)
    random.seed(1)
    tv = two_view_arrays(K, x1, x2, 1e-5, 1500, "rms", 200, engine=eng)
    idx = tv.inlier_indices[tv.passing]
    Xp = tv.points[tv.passing]
    random.seed(2)
    # with 0 extra inliers the smallest RMS error goes to a pose that only its own sample and a few points fit, as the
    # reference's rule allows
    res = ransac_pnp_arrays(K, Xp, x3[idx], 4.0, len(idx) // 2, "rms", 200, engine=eng)
    r3 = np.abs(res.R - R3).max()
    assert r3 < 2e-2 and r3 <= 1.5 * np.abs(tv.R - R2).max()
    assert np.abs(res.t - t3 / np.linalg.norm(t2)).max() < 5e-2
    random.seed(1)
    again = two_view_arrays(K, x1, x2, 1e-5, 1500, "rms", 200, engine=eng)
    random.seed(1)
    fresh = two_view_arrays(K, x1, x2, 1e-5, 1500, "rms", 200, engine=_native.Engine(0))
    for a, b in ((again.R, fresh.R), (again.t, fresh.t), (again.points, fresh.points), (again.ransac.E, fresh.ransac.E)):
        assert np.array_equal(_bits(a), _bits(b))
    assert np.array_equal(again.ransac.inlier_indices, fresh.ransac.inlier_indices)


def test_refusals(eng):
    K, X, x, R, t, _ = make_pnp_scene(50, 0.0, seed=1)
    with pytest.raises(ValueError):
        ransac_pnp_arrays(K, X[:7], x[:7], 4.0, engine=eng)
    with pytest.raises(ValueError):
        ransac_pnp_arrays(K, X, x[:-1], 4.0, engine=eng)
    with pytest.raises(ValueError):
        ransac_pnp_arrays(K, X[:, :2], x, 4.0, engine=eng)
    for bad in (np.diag([800.0, 800, 2]), np.array([[800.0, 0, 640], [1, 800, 480], [0, 0, 1]]), np.zeros((3, 3)),
                np.full((3, 3), np.nan), np.eye(2)):
        with pytest.raises((ValueError, RuntimeError)):
            ransac_pnp_arrays(bad, X, x, 4.0, engine=eng)
    for thr in (np.inf, np.nan):
        with pytest.raises(ValueError):
            ransac_pnp_arrays(K, X, x, thr, engine=eng)
    with pytest.raises(ValueError):
        ransac_pnp_arrays(K, X, x, 4.0, max_iterations=0, engine=eng)


def test_fuzz_cases():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_pnp.py"), "12"], capture_output=True,
                         text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0 and "mismatches: 0" in out.stdout, out.stdout[-3000:] + out.stderr[-2000:]
