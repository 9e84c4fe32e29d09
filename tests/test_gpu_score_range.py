"""K2's screening bodies where the arithmetic leaves the normal range: records with NaN or infinite coordinates, in
single pairs of both upload kinds (below 65 536 records the 11-slot screen, above it the 9-slot screen over K2's
Morton-sorted copy) and in batches.  Every body is only a screen: counts must equal the exact C scorer's, sums agree to
1e-12, and K3's errors and winner and K4's mask and SED follow.  The model-scale sweep lives in
test_gpu_parity.py::test_screen_never_drops_an_inlier and test_gpu_tile_screen.py::test_tile_screen_never_drops_an_inlier,
which use check_against_oracle below."""
import functools

import numpy as np
import pytest

from oracle import csed
from oracle import restatement as o
from structure_from_motion_b200.scenes import make_scene

pytestmark = pytest.mark.gpu
SORT_MIN = 65_536  # kK2SortMin in csrc/sfm_ransac.cu: single pairs from here on get the 9-slot screen
SIZES = {"11-slot": 3_003, "9-slot": SORT_MIN + 7_000}
VARIANTS = ("screen", "full", "screen32", "auto")
THRS = (0.0, 1.5e-6, 1e-3, 0.5)  # at 1e-3 AUTO picks the two-sided body
H = 200


def expected_winner(s1_o):
    """K3 with sum aggregation and min_extra 0: a hypothesis is a candidate iff its error (S1) is not NaN; the smallest
    error wins, the lowest index on ties.  Returns (candidate mask, winner or -1, indices the winner may be when the
    runner-up is within the 1e-12 the sums are compared to)."""
    cand = ~np.isnan(s1_o)
    if not cand.any():
        return cand, -1, [-1]
    key = np.where(cand, s1_o, np.inf)
    m = key.min()
    near = np.flatnonzero(cand & (key <= m + 2e-12 * abs(m)))
    exact = np.flatnonzero(cand & (key == m))
    return cand, int(exact[0]), [int(i) for i in near]


def check_against_oracle(engine, got, E, cols, thr, oracle):
    """got = engine.score(thr, min_extra=0, aggregation="sum"); oracle = csed.score_batch on the same models."""
    cnt, s1, s2, err = got
    cnt_o, s1_o, s2_o = oracle
    assert np.array_equal(cnt, cnt_o)
    np.testing.assert_allclose(s1, s1_o, rtol=1e-12, atol=0)
    np.testing.assert_allclose(s2, s2_o, rtol=1e-12, atol=0)
    cand, win, near = expected_winner(s1_o)
    np.testing.assert_allclose(err, np.where(cand, s1_o, np.inf), rtol=1e-12, atol=0)
    best = engine.get_best()
    assert best.index == win or (len(near) > 1 and best.index in near), (best.index, win, near)
    if best.index >= 0:
        mask, sed = engine.inlier_mask(thr)
        sed_o = csed.sed_exact_many(E[best.index], *cols)
        assert np.array_equal(sed, sed_o, equal_nan=True)
        assert np.array_equal(mask, sed_o <= thr)


def score(engine, x1, x2, K, table, E, thr, variant, hpt=0, group=0):
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    engine.set_models(E)
    engine.set_score_variant(variant, hpt, group)
    try:
        return engine.score(thr, min_extra=0, aggregation="sum")
    finally:
        engine.set_score_variant("auto")


def fit_models(cols, rows, seed, h=H):
    """h eight-point models, each from 8 records drawn from `rows` (finite ones), and the sample table."""
    rng = np.random.default_rng(seed)
    table = np.stack([rng.choice(rows, 8, replace=False) for _ in range(h)]).astype(np.int32)
    ca, cb = np.stack(cols[:2], 1), np.stack(cols[2:], 1)
    return table, np.stack([o.eight_point(ca[s], cb[s]) for s in table])


def morton_order(xb, yb):
    """K2's sorted copy in numpy (k2_order_bbox, k2_quantise, k2_order_keys and the stable radix sort): the box is over
    the non-NaN values, and an infinite coordinate collapses its axis of the key to 0."""
    def quant(x):
        f = x[~np.isnan(x)]
        lo, hi = f.min(), f.max()
        with np.errstate(all="ignore"):
            sc = 65535.0 / (hi - lo)
            q = (x - lo) * sc if 0.0 < sc < 1e308 else np.zeros_like(x)
        q = np.where(np.isnan(q), 0.0, q)
        return np.clip(q, 0.0, 65535.0).astype(np.uint64)

    def spread(v):
        v = (v | (v << 8)) & 0x00FF00FF
        v = (v | (v << 4)) & 0x0F0F0F0F
        v = (v | (v << 2)) & 0x33333333
        return (v | (v << 1)) & 0x55555555

    key = (spread(quant(yb)) << 1) | spread(quant(xb))
    return np.argsort(key, kind="stable")


@functools.lru_cache(maxsize=None)
def _scene(kind):
    K, x1, x2, *_ = make_scene(SIZES[kind], 0.3, seed=61)
    cols = (*o.k_normalise(x1[:, 0], x1[:, 1], K), *o.k_normalise(x2[:, 0], x2[:, 1], K))
    return K, x1, x2, cols


def _corrupt(kind, how):
    """Pixel arrays with non-finite records, their K-normalised columns and the rows left finite."""
    K, x1, x2, _ = _scene(kind)
    x1, x2 = x1.copy(), x2.copy()
    n = len(x1)
    bad = np.zeros(n, bool)
    if how == "nan_runs":  # a warp-aligned run of 32 NaN records in xa, another in yb: each poisons a warp's bound
        x1[64:96, 0] = np.nan
        x2[1024:1056, 1] = np.nan
        bad[64:96] = bad[1024:1056] = True
    elif how == "scattered":  # single NaN, +inf and -inf records in each coordinate
        idx = np.random.default_rng(5).choice(n, 12, replace=False)
        for k, i in enumerate(idx):
            arr, c = (x1, x2)[k // 6], (k // 3) % 2
            arr[i, c] = (np.nan, np.inf, -np.inf)[k % 3]
        bad[idx] = True
    cols = (*o.k_normalise(x1[:, 0], x1[:, 1], K), *o.k_normalise(x2[:, 0], x2[:, 1], K))
    return K, x1, x2, cols, np.flatnonzero(~bad)


@functools.lru_cache(maxsize=None)
def _case(kind, how):
    K, x1, x2, cols, rows = _corrupt(kind, how)
    table, E = fit_models(cols, rows, seed=7)
    oracle = {thr: csed.score_batch(E, *cols, thr, table=table, nthreads=8) for thr in THRS}
    return K, x1, x2, cols, table, E, oracle


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("how", ["nan_runs", "scattered"])
@pytest.mark.parametrize("kind", list(SIZES))
def test_non_finite_records_match_exact_scorer(engine, kind, how, variant):
    """A record with a NaN or infinite coordinate is never an inlier (its sed is NaN or inf), and it must not take the
    finite records' inliers with it: the coordinate bounds behind kappa are taken over finite records only."""
    K, x1, x2, cols, table, E, oracle = _case(kind, how)
    for thr in THRS:
        got = score(engine, x1, x2, K, table, E, thr, variant)
        check_against_oracle(engine, got, E, cols, thr, oracle[thr])
    assert (oracle[1.5e-6][0] > 0).sum() > H // 4  # the finite records do have inliers


@functools.lru_cache(maxsize=None)
def _nan_tile_case():
    """9-slot upload whose first sorted tile holds 64 records with both B coordinates NaN (its box is the non-finite
    default: centre 0, half-widths DBL_MAX)."""
    K, x1, x2, _ = _scene("9-slot")
    x2 = x2.copy()
    x2[:64] = np.nan
    cols = (*o.k_normalise(x1[:, 0], x1[:, 1], K), *o.k_normalise(x2[:, 0], x2[:, 1], K))
    order = morton_order(cols[2], cols[3])
    assert np.array_equal(np.sort(order[:64]), np.arange(64))  # they share key 0 and come first in input order
    table, E = fit_models(cols, np.arange(64, len(x1)), seed=8)
    return K, x1, x2, cols, table, E


@functools.lru_cache(maxsize=None)
def _inf_tile_case():
    """9-slot upload (K = I) with one sorted tile of 40 records at a = b = (0, 0) and 24 with an infinite B
    coordinate, and models with e_8 = 0: r = 0 and sed = 0 exactly at (0, 0), inliers even at thr = 0, in a tile whose
    box is the non-finite default."""
    K, x1, x2, _ = _scene("9-slot")
    cols = [np.array(c) for c in (*o.k_normalise(x1[:, 0], x1[:, 1], K), *o.k_normalise(x2[:, 0], x2[:, 1], K))]
    cols[3] = cols[3] - cols[3].min() + 0.25  # every other B point above y = 0: the special tile has key 0
    for c in cols:
        c[:64] = 0.0
    cols[2][40:52] = np.inf
    cols[2][52:64] = -np.inf
    order = morton_order(cols[2], cols[3])
    assert np.array_equal(np.sort(order[:64]), np.arange(64))
    table, E = fit_models(cols, np.arange(64, len(cols[0])), seed=9)
    E[:, 2, 2] = 0.0
    x1 = np.stack(cols[:2], 1)
    x2 = np.stack(cols[2:], 1)
    return np.eye(3), x1, x2, tuple(cols), table, E


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("case", ["nan_tile", "inf_tile"])
def test_non_finite_tiles_of_the_sorted_copy(engine, case, variant):
    K, x1, x2, cols, table, E = (_nan_tile_case if case == "nan_tile" else _inf_tile_case)()
    for thr in THRS:
        oracle = csed.score_batch(E, *cols, thr, table=table, nthreads=8)
        got = score(engine, x1, x2, K, table, E, thr, variant)
        check_against_oracle(engine, got, E, cols, thr, oracle)
        if case == "inf_tile":
            assert (oracle[0] >= 40).all()  # every model has the 40 exact inliers of the special tile


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("kind", list(SIZES))
def test_sample_row_with_a_nan_record_never_wins(engine, kind, variant):
    """A hypothesis whose minimal sample holds a NaN record has a NaN error (its samples always enter the error): it is
    no candidate, however many inliers it has."""
    K, x1, x2, cols, table, E, _ = _case(kind, "nan_runs")
    table = table.copy()
    cnt0 = csed.score_batch(E, *cols, 1.5e-6, table=table, nthreads=8)[0]
    top = int(np.argmax(cnt0))  # the model with the most inliers gets the poisoned row
    table[top, 3] = 70
    for thr in (1.5e-6, 1e-3):
        oracle = csed.score_batch(E, *cols, thr, table=table, nthreads=8)
        assert np.isnan(oracle[1][top])
        got = score(engine, x1, x2, K, table, E, thr, variant)
        check_against_oracle(engine, got, E, cols, thr, oracle)
        assert got[3][top] == np.inf and engine.get_best().index != top


@pytest.mark.parametrize("variant", VARIANTS)
def test_batch_pair_with_nan_records_leaves_the_others_alone(engine, variant):
    """In a batch, one pair's coordinate bounds are everyone's: a warp-aligned NaN run in one pair must leave every
    other pair's estimate bit for bit as it is with that pair finite."""
    sizes = [1500, 2100, 900, 1700, 1200]
    scenes = [make_scene(s, 0.3, seed=400 + p) for p, s in enumerate(sizes)]
    xa = np.concatenate([sc[1] for sc in scenes])
    xb = np.concatenate([sc[2] for sc in scenes])
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    Ks = np.stack([sc[0] for sc in scenes])
    bad = 2
    xa_nan = xa.copy()
    xa_nan[off[bad] + 32:off[bad] + 64, 0] = np.nan  # records 32..63 of pair 2: one warp of k_normalise
    engine.set_score_variant(variant)
    try:
        clean = engine.batch_ransac(xa, xb, off, Ks, 400, 5, 1.5e-6, 0, "rms")
        dirty = engine.batch_ransac(xa_nan, xb, off, Ks, 400, 5, 1.5e-6, 0, "rms")
    finally:
        engine.set_score_variant("auto")
    others = [p for p in range(len(sizes)) if p != bad]
    for k in ("E", "best_index", "best_err", "count_extra"):
        assert np.array_equal(np.asarray(clean[k])[others], np.asarray(dirty[k])[others], equal_nan=True), k
    assert (np.asarray(clean["count_extra"])[others] > 0).any()
