"""GPU parity: the CUDA path (through the C ABI) against the oracle on the same seeded inputs.

Tolerances (BASELINE.json north_star):
  * inlier masks bit-identical except for correspondences within 1e-9 relative of the threshold
  * best E within 1e-6 (up to scale and sign)
  * triangulated points within 1e-6 relative
All fp64.  The scorer is additionally required to be *bit-exact* against oracle/sed_exact.c
(which is bit-exact against the reference's numpy evaluation, tests/test_oracle.py).
"""
import functools
import random

import numpy as np
import pytest

from oracle import csed
from oracle import restatement as o
from structure_from_motion_b200 import _native, two_view
from structure_from_motion_b200.scenes import make_scene
from test_gpu_score_range import check_against_oracle

pytestmark = pytest.mark.gpu

THR = 1.5e-6  # apps/config/config.yaml:7
BAND = 1e-9


def _norm(K, x1, x2):
    nxa, nya = o.k_normalise(x1[:, 0], x1[:, 1], K)
    nxb, nyb = o.k_normalise(x2[:, 0], x2[:, 1], K)
    return nxa, nya, nxb, nyb


def _e_close(a, b, tol=1e-6):
    a = a.reshape(-1) / np.linalg.norm(a)
    b = b.reshape(-1) / np.linalg.norm(b)
    return min(np.abs(a - b).max(), np.abs(a + b).max()) <= tol


def test_k_normalise_bit_exact(engine):
    K, x1, x2, *_ = make_scene(1000, 0.3, seed=11)
    engine.upload_pairs(x1, x2, K)
    got = engine.get_normalised()
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    assert np.array_equal(got, np.stack([nxa, nya, nxb, nyb], axis=1))


def test_sampler_table_roundtrip(engine):
    K, x1, x2, *_ = make_scene(500, 0.3, seed=0)
    engine.upload_pairs(x1, x2, K)
    engine.sample_device(seed=7, h=4096)
    t = engine.get_table()
    assert t.shape == (4096, 8) and t.min() >= 0 and t.max() < 500
    assert all(len(set(row)) == 8 for row in t.tolist())
    # same (seed, global index) => same rows, however the hypotheses are sharded
    engine.sample_device(seed=7, h=1024, hyp_offset=2048)
    assert np.array_equal(engine.get_table(), t[2048:3072])
    # roughly uniform
    counts = np.bincount(t.reshape(-1), minlength=500)
    assert counts.min() > 20 and counts.max() < 130


@pytest.mark.parametrize("variant,hpt,group", [("screen", 2, 16), ("full", 2, 16), ("screen32", 4, 8), ("screen32", 2, 16)])
def test_scorer_bit_exact_against_oracle(engine, variant, hpt, group):
    """K2+K3 with oracle-supplied E's: counts equal, sums within 1e-12 (different summation order)."""
    n, h = 3003, 700  # 3003 = 23 tiles + 59: partial last tile, partial last batch for every group size
    K, x1, x2, *_ = make_scene(n, 0.4, seed=2)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    rng = np.random.default_rng(5)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    ca, cb = np.stack([nxa, nya], 1), np.stack([nxb, nyb], 1)
    E = np.stack([o.eight_point(ca[s], cb[s]) for s in table])
    cnt_o, s1_o, s2_o = csed.score_batch(E, nxa, nya, nxb, nyb, THR, table=table, nthreads=8)

    engine.set_score_variant(variant, hpt, group)
    try:
        engine.upload_pairs(x1, x2, K)
        engine.set_table(table)
        engine.set_models(E)
        cnt, s1, s2, err = engine.score(THR, min_extra=10, aggregation="rms")
    finally:
        engine.set_score_variant("auto")
    assert np.array_equal(cnt, cnt_o)
    np.testing.assert_allclose(s1, s1_o, rtol=1e-12, atol=0)
    np.testing.assert_allclose(s2, s2_o, rtol=1e-12, atol=0)
    n_tot = 8 + cnt_o
    err_o = np.where(cnt_o >= 10, np.sqrt(s2_o / n_tot), np.inf)
    np.testing.assert_allclose(err, err_o, rtol=1e-12)
    best = engine.get_best()
    assert best.index == int(np.argmin(err_o))
    # K4: mask + SED values of the winner are bit-identical to the exact oracle scorer
    mask, sed = engine.inlier_mask(THR)
    sed_o = csed.sed_exact_many(E[best.index], nxa, nya, nxb, nyb)
    assert np.array_equal(sed, sed_o)
    assert np.array_equal(mask, sed_o <= THR)


# model scales past the underflow knee of the reference's na, nb (|E| ~ 1e-154 on unit coordinates), the knee of the
# two-sided body's degree-4 terms (~1e-77) and the overflow knee (~1e154), where the reference reports sed = 0 inliers
RANGE_SCALES = (1e-160, 1e-154, 1e-153, 1e-100, 1e-80, 1e-78, 1e-60, 1e60, 1e77, 1e78, 1e150, 1e154, 1e155, 1e160)
SCALE_CASES = ([(e, t) for e in (1.0, 1e6, 1e-7) for t in (0.0, 1e-30, 1e-18, 1e-12, 1e-9, 1.5e-6, 1e-3, 0.5, 40.0)]
               + [(e, t) for e in RANGE_SCALES for t in (0.0, 1e-12, 1.5e-6, 1e-3, 0.5)])


@functools.lru_cache(maxsize=None)
def _scale_case(escale, thr):
    n, h = 1500, 256
    K, x1, x2, *_ = make_scene(n, 0.3, seed=11)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    rng = np.random.default_rng(9)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    ca, cb = np.stack([nxa, nya], 1), np.stack([nxb, nyb], 1)
    E = np.stack([o.eight_point(ca[s], cb[s]) for s in table]) * escale
    oracle = csed.score_batch(E, nxa, nya, nxb, nyb, thr, table=table, nthreads=8)
    return K, x1, x2, (nxa, nya, nxb, nyb), table, E, oracle


@pytest.mark.parametrize("escale,thr", SCALE_CASES)
@pytest.mark.parametrize("variant", ["screen", "screen32", "full", "auto"])
def test_screen_never_drops_an_inlier(engine, thr, escale, variant):
    """Every body of the 11-slot upload is a necessary condition at EVERY threshold and model scale: counts, sums,
    K3's errors and winner and K4's mask and SED equal the exact oracle scorer's (sed.py is scale-invariant in E
    while it stays in range; the screens' guard kappa_h scales with |E_h|^2, and models outside the range guard of
    the K2 header have all their tests decided exactly).  At thr 1e-3 AUTO runs the two-sided body."""
    K, x1, x2, cols, table, E, oracle = _scale_case(escale, thr)
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    engine.set_models(E)
    engine.set_score_variant(variant)
    try:
        got = engine.score(thr, min_extra=0, aggregation="sum")
    finally:
        engine.set_score_variant("auto")
    check_against_oracle(engine, got, E, cols, thr, oracle)
    if thr == 1.5e-6 and 1e-153 <= escale <= 1e150:  # the reference's range: there are inliers to drop
        assert oracle[0].sum() > 0
    if escale == 1e154 and thr <= 1.5e-6:  # the sed = 0 regime: na, nb overflow, r^2 does not
        assert oracle[0].sum() > _scale_case(1.0, thr)[-1][0].sum()


@pytest.mark.parametrize("thr", [0.0, 1e-12, 1.5e-6, 1e-4, 1e-3, 0.03, 0.5, 40.0])
@pytest.mark.parametrize("variant,hpt,group", [("full", 2, 16), ("auto", 2, 16)])
def test_two_sided_body_at_every_inlier_rate(engine, thr, variant, hpt, group):
    """The two-sided body's survivor path (one ring entry per survivor, handed out in rounds; gathers from shared memory)
    from no survivors at all to EVERY test surviving (32 rounds per batch, ring full): counts equal and sums
    within 1e-12 of the exact oracle scorer; 1 500 correspondences = partial last tile and partial last batch."""
    n, h = 1500, 200
    K, x1, x2, *_ = make_scene(n, 0.3, seed=12)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    rng = np.random.default_rng(10)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    ca, cb = np.stack([nxa, nya], 1), np.stack([nxb, nyb], 1)
    E = np.stack([o.eight_point(ca[s], cb[s]) for s in table])
    cnt_o, s1_o, s2_o = csed.score_batch(E, nxa, nya, nxb, nyb, thr, table=table, nthreads=8)
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    engine.set_models(E)
    engine.set_score_variant(variant, hpt, group)
    try:
        cnt, s1, s2, err = engine.score(thr, min_extra=0, aggregation="sum")
    finally:
        engine.set_score_variant("auto")
    assert np.array_equal(cnt, cnt_o)
    np.testing.assert_allclose(s1, s1_o, rtol=1e-12, atol=0)
    np.testing.assert_allclose(s2, s2_o, rtol=1e-12, atol=0)
    if thr >= 40.0:
        assert cnt_o.mean() > 0.99 * (n - 8)  # (nearly) every correspondence is an inlier of every model


def test_only_shapes_with_a_kernel_are_accepted(engine):
    """K2 has kernels for fp64 2 x 16 and for the fp32 pre-filter at 4 x 8 and 2 x 16: set_score_variant refuses every
    other shape with SFM_ERR_ARG (-1), and accepts the kept shapes and 0 / 0 (the current shape, or the variant's
    default when switching to or from screen32)."""
    try:
        for variant, hpt, group in [("screen", 4, 8), ("full", 1, 32), ("auto", 4, 8), ("screen32", 8, 4)]:
            with pytest.raises(_native.NativeError, match=r"sfm_set_score_variant -> -1:"):
                engine.set_score_variant(variant, hpt, group)
        for variant, hpt, group in [("screen", 2, 16), ("full", 2, 16), ("auto", 2, 16), ("screen32", 4, 8),
                                    ("screen32", 2, 16), ("auto", 0, 0), ("screen32", 0, 0), ("full", 0, 0)]:
            engine.set_score_variant(variant, hpt, group)
    finally:
        engine.set_score_variant("auto")


@pytest.mark.parametrize("agg", ["sum", "square", "mean", "rms"])
def test_aggregation_methods(engine, agg):
    n, h = 800, 300
    K, x1, x2, *_ = make_scene(n, 0.3, seed=4)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    rng = np.random.default_rng(1)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    E, valid, _ = engine.fit()
    assert valid.all()
    cnt, s1, s2, err = engine.score(THR, min_extra=5.5, aggregation=agg)
    cnt_o, s1_o, s2_o = csed.score_batch(E, nxa, nya, nxb, nyb, THR, table=table, nthreads=4)
    assert np.array_equal(cnt, cnt_o)
    ntot = 8 + cnt_o
    exp = {"sum": s1_o, "square": s2_o, "mean": s1_o / ntot, "rms": np.sqrt(s2_o / ntot)}[agg]
    exp = np.where(cnt_o >= 5.5, exp, np.inf)  # fractional min_num_extra_inliers (test_ransac.py:109)
    np.testing.assert_allclose(err, exp, rtol=1e-12)


def test_fitter_against_oracle(engine):
    """K1 per hypothesis vs the reference's eig/svd route; tolerance scaled by conditioning (SURVEY H2)."""
    n, h = 5000, 2000
    K, x1, x2, *_ = make_scene(n, 0.4, seed=9)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    rng = np.random.default_rng(3)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    E, valid, eig = engine.fit(want_eig=True)
    assert valid.all()
    ca, cb = np.stack([nxa, nya], 1), np.stack([nxb, nyb], 1)
    rel = lambda a, b: np.linalg.norm(a - b) / np.linalg.norm(b)  # noqa: E731
    ratios = []
    for i in range(h):
        s = table[i]
        e_o = o.eight_point(ca[s], cb[s])
        w_o, sv = o.eight_point_conditioning(ca[s], cb[s])
        w = np.sort(eig[i])
        np.testing.assert_allclose(w[1:], w_o[1:], rtol=1e-9, atol=1e-13)
        d = rel(E[i], e_o)
        # How well-determined is E on this sample?  Measure it: the reference's own route (LAPACK
        # dgeev + dgesdd) against two other correct CPU solvers.  The GPU result must be as close to
        # the reference as those are (x4), with a conditioning-scaled floor (SURVEY.md H2).
        alt = max(rel(a, e_o) for a in o.eight_point_alternatives(ca[s], cb[s]))
        tol = max(4.0 * alt, 2e-14 * w_o[-1] / w_o[1] + 1e-12)
        ratios.append(d / tol)
        assert d <= tol, (i, d, tol, alt, w_o[:3], sv)
        assert d <= 1e-6  # the north_star bound, far above anything seen
        assert E[i][2, 2] == 1.0
    assert np.median(ratios) < 0.5


def test_degenerate_sample_is_flagged(engine):
    """Two coplanar rectangles (tests/golden degenerate fixture analogue): valid == 0."""
    # 8 points on a plane seen by two cameras: the 9x9 system has a 2-dimensional null space
    rng = np.random.default_rng(0)
    X = np.column_stack([rng.uniform(-1, 1, 8), rng.uniform(-1, 1, 8), np.full(8, 5.0)])
    K = np.array([[500.0, 0, 320], [0, 500.0, 240], [0, 0, 1]])
    R = np.eye(3)
    t = np.array([-0.5, 0.0, 0.0])
    x1 = (K @ X.T).T
    x1 = x1[:, :2] / x1[:, 2:]
    X2 = X @ R.T + t
    x2 = (K @ X2.T).T
    x2 = x2[:, :2] / x2[:, 2:]
    with pytest.raises(two_view.EightPointCalculationError):
        two_view.eight_point_arrays(x1, x2, K, engine=engine)


@pytest.mark.parametrize("n,h,frac,seed", [(500, 200, 0.3, 0), (2000, 500, 0.4, 1)])
def test_ransac_end_to_end_reference_sampler(engine, n, h, frac, seed):
    K, x1, x2, *_ = make_scene(n, frac, seed=seed)
    random.seed(5)
    ref = o.ransac_essential(K, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], THR, 10, "rms", h, return_all=True)
    state_after = random.getstate()
    random.seed(5)
    res = two_view.ransac_essential_arrays(K, x1, x2, THR, 10, "rms", h, engine=engine)
    assert random.getstate() == state_after  # the global RNG advanced exactly as in the reference
    assert res.best_index == ref["best_index"]
    assert _e_close(res.E, ref["E"])
    assert abs(res.error - ref["error"]) <= 1e-9 * ref["error"]
    # inlier list: same order, identical outside the guard band
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    sed_o = csed.sed_exact_many(ref["E"], nxa, nya, nxb, nyb)
    in_band = np.abs(sed_o - THR) <= BAND * THR
    a, b = list(res.inlier_indices), list(ref["inlier_indices"])
    if a != b:
        diff = set(a) ^ set(b)
        assert all(in_band[i] for i in diff), diff
    assert res.inlier_indices[:8].tolist() == ref["inlier_indices"][:8].tolist()


def test_selection_tie_and_no_candidate(engine):
    K, x1, x2, *_ = make_scene(300, 0.3, seed=5)
    random.seed(1)
    with pytest.raises(ValueError, match="No model could be found with at least 298 inliers"):
        two_view.ransac_essential_arrays(K, x1, x2, THR, 290, "rms", 20, engine=engine)
    # duplicated rows in the table: identical errors, the earliest index must win (ransac.py:83)
    rng = np.random.default_rng(2)
    row = rng.choice(300, 8, replace=False).astype(np.int32)
    table = np.stack([rng.choice(300, 8, replace=False).astype(np.int32) for _ in range(64)])
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    E, valid, _ = engine.fit()
    cnt, s1, s2, err = engine.score(THR, 0, "rms")
    w = int(np.argmin(err))
    table2 = table.copy()
    table2[w + 3 if w + 3 < 64 else w - 3] = table[w]  # a duplicate of the winner elsewhere
    dup = w + 3 if w + 3 < 64 else w - 3
    engine.set_table(table2)
    engine.fit()
    cnt2, _, _, err2 = engine.score(THR, 0, "rms")
    assert err2[dup] == err2[w]
    assert engine.get_best().index == min(w, dup)
    # max-inliers selection (non-default)
    engine.score(THR, 0, "rms", selection="max_inliers")
    b = engine.get_best()
    assert b.count_extra == cnt2.max() and b.index == int(np.argmax(cnt2))


def test_pose_and_triangulation_against_oracle(engine):
    n = 600
    K, x1, x2, R_true, t_true, out_idx = make_scene(n, 0.0, seed=8, noise_px=0.05)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    s = np.arange(8) * 50
    e = o.eight_point(np.stack([nxa[s], nya[s]], 1), np.stack([nxb[s], nyb[s]], 1))
    Rr, tr, idx_o, counts_o = o.recover_r_t(nxa, nya, nxb, nyb, e)
    res = two_view.recover_pose_arrays(e, np.stack([nxa, nya], 1), np.stack([nxb, nyb], 1), engine=engine)
    np.testing.assert_allclose(res.R, Rr, atol=1e-9)
    np.testing.assert_allclose(res.t, tr, atol=1e-9)
    assert np.array_equal(res.passing_indices, idx_o)
    assert sorted(res.counts.tolist()) == sorted(int(c) for c in counts_o)
    # the direction of t and R agree with the ground truth of the scene
    assert abs(np.dot(res.t, t_true / np.linalg.norm(t_true))) > 0.999
    np.testing.assert_allclose(res.R, R_true, atol=3e-2)
    # triangulation in pixel coordinates
    T = o.tmat(Rr, tr)
    X_o = o.triangulate_points(x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], K, T)
    P1, P2 = two_view.camera_matrices(K, T)
    X = two_view.triangulate_arrays(x1, x2, P1, P2, engine=engine)
    rel = np.linalg.norm(X - X_o, axis=1) / np.linalg.norm(X_o, axis=1)
    assert rel.max() <= 1e-6, rel.max()


def test_two_view_pipeline(engine):
    K, x1, x2, R_true, t_true, _ = make_scene(3000, 0.4, seed=12)
    res = two_view.two_view_arrays(K, x1, x2, THR, 10, "rms", 2000, sampler="device", seed=3,
                                   on_degenerate="skip", engine=engine)
    r = res.ransac
    # oracle on the same table
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    table = engine.get_table()
    ref = o.ransac_essential(K, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], THR, 10, "rms", 2000, table=table,
                             on_degenerate="skip")
    assert r.best_index == ref["best_index"]
    assert _e_close(r.E, ref["E"])
    inl = np.sort(ref["inlier_indices"])
    assert np.array_equal(res.inlier_indices, inl)
    # apps/sfm.py:118-133 hands the RANSAC inlier list (samples first, ransac.py:76) to recover_r_t_from_e, so position 0
    # of that list - the one correspondence np.count_nonzero never counts (eight_point.py:228-230) - is the winner's
    # first sample: feed the oracle in that order and require the same vote and the same passing set
    lst = ref["inlier_indices"]
    Rr, tr, idx_l, counts_o = o.recover_r_t(nxa[lst], nya[lst], nxb[lst], nyb[lst], ref["E"])
    np.testing.assert_allclose(res.R, Rr, atol=1e-6)
    np.testing.assert_allclose(res.t, tr, atol=1e-6)
    assert sorted(res.counts.tolist()) == sorted(int(c) for c in counts_o)
    assert np.array_equal(np.sort(lst[idx_l]), res.inlier_indices[res.passing])
    X_o = o.triangulate_points(x1[inl, 0], x1[inl, 1], x2[inl, 0], x2[inl, 1], K, o.tmat(Rr, tr))
    ok = res.passing
    rel = np.linalg.norm(res.points[ok] - X_o[ok], axis=1) / np.linalg.norm(X_o[ok], axis=1)
    assert rel.max() <= 1e-6
    assert np.isnan(res.points[~ok]).all()


# ---- SURVEY.md §8(f) N4: robustness extras behind non-default flags -----------------------------
@pytest.mark.parametrize("agg", ["rms", "sum"])
def test_msac_selection_against_oracle(engine, agg):
    """selection="msac": minimum of sum_i min(sed_i, thr) over ALL correspondences, candidates as in ransac.py:76."""
    n, h = 1200, 400
    K, x1, x2, *_ = make_scene(n, 0.35, seed=9)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    rng = np.random.default_rng(2)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    E, valid, _ = engine.fit()
    assert valid.all()
    cnt, _, _, err = engine.score(THR, min_extra=10, aggregation=agg, selection="msac")
    best = engine.get_best()
    cost = np.empty(h)
    for i in range(h):
        sed = csed.sed_exact_many(E[i], nxa, nya, nxb, nyb)
        cost[i] = np.minimum(sed, THR).sum()
    cnt_o, _, _ = csed.score_batch(E, nxa, nya, nxb, nyb, THR, table=table, nthreads=4)
    assert np.array_equal(cnt, cnt_o)
    want = np.where(cnt_o >= 10, cost, np.inf)
    np.testing.assert_allclose(err, want, rtol=1e-10)
    assert best.index == int(np.argmin(want)) and abs(best.err - want.min()) <= 1e-10 * want.min()
    # the default selection is untouched by the extra
    _, _, _, err_default = engine.score(THR, min_extra=10, aggregation=agg)
    assert engine.get_best().index == int(np.argmin(err_default))


def test_adaptive_early_termination(engine):
    n = 5000
    K, x1, x2, *_ = make_scene(n, 0.3, seed=12)
    res, done = two_view.ransac_essential_adaptive(K, x1, x2, THR, 10, "rms", max_iterations=65536, chunk=2048, seed=7,
                                                   engine=engine)
    assert done < 65536 and done % 2048 == 0  # 30 % outliers: a few hundred hypotheses suffice at 99 %
    w = (8 + res.count_extra) / n
    assert done >= np.log(0.01) / np.log(1 - w ** 8)
    full = two_view.ransac_essential_arrays(K, x1, x2, THR, 10, "rms", done, sampler="device", seed=7, on_degenerate="skip",
                                            selection="max_inliers", engine=engine)
    assert full.best_index == res.best_index and np.array_equal(full.E, res.E)
    assert np.array_equal(full.inlier_indices, res.inlier_indices)
    # a hopeless scene runs to the cap and reports the reference's error
    rng = np.random.default_rng(0)
    with pytest.raises(ValueError, match="No model could be found"):
        two_view.ransac_essential_adaptive(K, rng.uniform(0, 1000, (300, 2)), rng.uniform(0, 1000, (300, 2)), 1e-12, 50,
                                           "rms", max_iterations=4096, chunk=1024, engine=engine)


@pytest.mark.parametrize("min_extra", [10, 10 ** 9])
def test_fused_two_view_call_equals_the_two_step_sequence(engine, min_extra):
    """sfm_two_view (winner handed to the tail on the device) against sfm_ransac_essential + sfm_pose_and_triangulate,
    including the no-model case (min_extra that no hypothesis reaches)."""
    K, x1, x2, *_ = make_scene(3000, 0.35, seed=21)
    engine.upload_pairs(x1, x2, K)
    engine.sample_device(5, 700)
    best_a, mask_a, sed_a = engine.ransac_essential(THR, min_extra, "rms")
    engine.sample_device(5, 700)
    best_b, mask_b, sed_b, poses_b, num_b, idx_b, ok_b, X_b = engine.two_view(THR, min_extra, "rms", "min_error", 50.0)
    assert best_a.index == best_b.index and best_a.count_extra == best_b.count_extra
    assert (best_a.err == best_b.err) and list(best_a.E) == list(best_b.E)
    if min_extra > 10 ** 6:
        assert best_b.index == -1 and num_b == 0 and len(idx_b) == 0
        return
    assert np.array_equal(mask_a, mask_b) and np.array_equal(sed_a, sed_b)
    engine.sample_device(5, 700)
    engine.ransac_essential(THR, min_extra, "rms", want_mask=False, want_sed=False)
    poses_a, num_a, idx_a, ok_a, X_a = engine.pose_and_triangulate(THR, 50.0)
    assert num_a == num_b and np.array_equal(idx_a, idx_b) and np.array_equal(ok_a, ok_b)
    assert np.array_equal(X_a, X_b, equal_nan=True)
    assert poses_a.best == poses_b.best and list(poses_a.counts) == list(poses_b.counts)
    assert np.array_equal(np.array(poses_a.R), np.array(poses_b.R))


def test_two_view_stream_equals_blocking_calls(engine):
    """two_view.TwoViewStream (two contexts, un-synchronised uploads, results fetched one estimate behind) returns what
    the blocking two_view_arrays call returns, estimate by estimate."""
    K, x1, x2, *_ = make_scene(6000, 0.4, seed=14)
    want = [two_view.two_view_arrays(K, x1, x2, THR, 10, "rms", 1200, sampler="device", seed=s, on_degenerate="skip",
                                     engine=engine) for s in range(5)]
    ts = two_view.TwoViewStream(depth=2)
    try:
        got, prev = [], ts.submit(K, x1, x2, THR, 10, "rms", 1200, 50.0, seed=0)
        for s in range(1, 5):
            cur = ts.submit(K, x1, x2, THR, 10, "rms", 1200, 50.0, seed=s)
            got.append(ts.result(prev))
            prev = cur
        got.append(ts.result(prev))
    finally:
        ts.close()
    for w, g in zip(want, got):
        assert g.ransac.best_index == w.ransac.best_index and g.ransac.error == w.ransac.error
        assert np.array_equal(g.ransac.E, w.ransac.E) and g.ransac.count_extra == w.ransac.count_extra
        assert np.array_equal(g.ransac.inlier_indices, w.ransac.inlier_indices)
        assert np.array_equal(g.ransac.mask, w.ransac.mask) and np.array_equal(g.ransac.sed, w.ransac.sed)
        assert np.array_equal(g.R, w.R) and np.array_equal(g.t, w.t) and np.array_equal(g.counts, w.counts)
        assert np.array_equal(g.inlier_indices, w.inlier_indices) and np.array_equal(g.passing, w.passing)
        assert np.array_equal(g.points, w.points, equal_nan=True)


@pytest.mark.parametrize("thr", [1.5e-6, 1.5e-4, 1.5e-2])
def test_auto_variant_matches_explicit_screens(engine, thr):
    """variant "auto" (the default): a pilot on the device measures the survivor rate of the one-sided screen and one of
    the two fp64 scoring kernels runs.  Whichever it picks, counts, sums, errors and the winner are bit-identical to
    both explicit variants (every decision and every summed value comes from the exact scorer)."""
    K, x1, x2, *_ = make_scene(20_000, 0.4, seed=27)
    engine.upload_pairs(x1, x2, K)
    engine.sample_device(seed=2, h=2048)
    engine.fit(want_E=False)
    got = {}
    try:
        for variant in ("auto", "screen", "full"):
            engine.set_score_variant(variant, 2, 16)
            got[variant] = engine.score(thr, min_extra=10, aggregation="rms") + (engine.get_best().index,)
    finally:
        engine.set_score_variant("auto")
    for variant in ("screen", "full"):
        for a, b in zip(got["auto"][:4], got[variant][:4]):
            assert np.array_equal(a, b, equal_nan=True), (variant, thr)
        assert got["auto"][4] == got[variant][4]
    assert got["auto"][0].max() > 10


def test_tail_state_survives_changing_shapes(engine):
    """The tail's look-back words, tickets and counters clean up behind themselves, whatever the sequence of problem
    shapes (regression: a flag left behind by a one-block launch once sat where a two-block launch keeps its ticket)."""
    for n in (700, 1025, 3000, 500, 2049, 64, 5000):
        K, x1, x2, *_ = make_scene(n, 0.3, seed=n)
        engine.upload_pairs(x1, x2, K)
        engine.sample_device(seed=1, h=300)
        best, mask, sed, poses, num, idx, ok, X = engine.two_view(THR, 5, "rms", "min_error", 50.0)
        if best.index < 0:
            assert num == 0
            continue
        want = mask.astype(bool)
        want[np.array(best.sample)] = True
        assert num == int(want.sum()) and np.array_equal(idx, np.nonzero(want)[0])
        assert X.shape == (num, 3) and np.isfinite(X[((ok >> poses.best) & 1).astype(bool)]).all()
