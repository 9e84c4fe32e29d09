"""The one-sided bodies' survivor drain: every drain takes up to 32 ring records, one per lane, and evaluates each
record's lowest set bit; records with bits left go back to the ring behind its tail.  These cases make that
write-back the common case rather than the rare one: records with most of their 32 bits set, a ring that stays
nearly full and wraps on every drain, items that end with 1, 31 or 32 records pending, models outside the range
guard (every test survives) and partial last batches.  Each runs the 11-slot body (< 65 536 correspondences), the
9-slot body (>= 65 536, sorted copy) and the fp32 pre-filter, with the variant set explicitly so that `auto` does not
hand the survivor-rich cases to the two-sided body.  Counts and sums are checked against the exact C scorer, and
counts, sums and errors bit for bit against the two-sided body, whose drain is a different one."""
import functools

import numpy as np
import pytest

from oracle import csed
from oracle import restatement as o
from structure_from_motion_b200.scenes import euler_xyz_intrinsic, make_scene

pytestmark = pytest.mark.gpu
SORT_MIN = 65_536  # kK2SortMin in csrc/sfm_ransac.cu: from here a single pair runs the 9-slot body
IDENT = np.eye(3)
VARIANTS = [("screen", 2, 16), ("screen32", 4, 8), ("screen32", 2, 16)]  # the kept one-sided shapes


def _skew(t):
    return np.array([[0.0, -t[2], t[1]], [t[2], 0.0, -t[0]], [-t[1], t[0], 0.0]])


@functools.lru_cache(maxsize=None)
def _exact_geometry(n):
    """Noise-free correspondences in normalised coordinates (K = I), the model they satisfy and one they do not."""
    K, x1, x2, R, t, _ = make_scene(n, 0.0, seed=5, noise_px=0.0)
    nxa, nya = o.k_normalise(x1[:, 0], x1[:, 1], K)
    nxb, nyb = o.k_normalise(x2[:, 0], x2[:, 1], K)
    good = _skew(t) @ R
    bad = _skew(np.array([0.2, 1.0, -0.3])) @ euler_xyz_intrinsic(-6.0, 3.0, 9.0)
    return (nxa, nya, nxb, nyb), (good / np.linalg.norm(good)).ravel(), (bad / np.linalg.norm(bad)).ravel()


def _run(engine, cols, table, E, thr, variant):
    x1, x2 = np.stack(cols[:2], 1), np.stack(cols[2:], 1)
    engine.upload_pairs(x1, x2, IDENT)
    engine.set_table(table)
    engine.set_models(E)
    engine.set_score_variant(*variant)
    try:
        return engine.score(thr, min_extra=0, aggregation="sum")
    finally:
        engine.set_score_variant("auto")


def _check(engine, cols, table, E, thr, variant):
    """K2 through `variant` against the exact scorer, and bit for bit against the two-sided body."""
    got = _run(engine, cols, table, E, thr, variant)
    cnt_o, s1_o, s2_o = csed.score_batch(E, *cols, thr, table=table, nthreads=8)
    assert np.array_equal(got[0], cnt_o)
    np.testing.assert_allclose(got[1], s1_o, rtol=1e-12, atol=0)
    np.testing.assert_allclose(got[2], s2_o, rtol=1e-12, atol=0)
    ref = _run(engine, cols, table, E, thr, ("full", 2, 16))
    for a, b in zip(got, ref):
        assert np.array_equal(a, b, equal_nan=True)
    return cnt_o


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("n", [16, 1_000 + 5, SORT_MIN + 16, SORT_MIN + 37])
@pytest.mark.parametrize("lanes", [1, 31, 32])
def test_full_records_from_some_lanes(engine, lanes, n, variant):
    """64 hypotheses, one warp's item group: the first `lanes` lanes hold the model every correspondence satisfies
    (both slots of the even ones, slot 0 of the odd ones), the rest one that none comes near.  Every batch then
    pushes exactly `lanes` records with 16 or 32 bits set.  n = 16 is a single batch in a single item, so the item
    ends with 1, 31 or 32 records pending (32: the push drains, the write-backs remain); longer pairs end every
    item with a few records and keep the ring at 62-63 records while 31 or 32 lanes push full records."""
    cols, good, bad = _exact_geometry(n)
    sed_good = csed.sed_exact_many(good, *cols)
    sed_bad = csed.sed_exact_many(bad, *cols)
    thr = float(np.sqrt(sed_good.max() * sed_bad.min())) if sed_good.max() > 0 else sed_bad.min() * 1e-6
    assert sed_good.max() < thr * 1e-3 and sed_bad.min() > thr * 1e3
    E = np.stack([bad] * 64)
    for lane in range(lanes):
        E[lane] = good
        if lane % 2 == 0:
            E[32 + lane] = good
    table = np.tile(np.arange(8, dtype=np.int32), (64, 1))
    cnt = _check(engine, cols, table, E, thr, variant)
    assert np.array_equal(cnt, np.where((E == good).all(1), n - 8, 0))


@functools.lru_cache(maxsize=None)
def _noisy_scene(n, h, seed):
    K, x1, x2, *_ = make_scene(n, 0.3, seed=seed)
    nxa, nya = o.k_normalise(x1[:, 0], x1[:, 1], K)
    nxb, nyb = o.k_normalise(x2[:, 0], x2[:, 1], K)
    rng = np.random.default_rng(seed)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    ca, cb = np.stack([nxa, nya], 1), np.stack([nxb, nyb], 1)
    return (nxa, nya, nxb, nyb), table, np.stack([o.eight_point(ca[s], cb[s]) for s in table])


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("n", [4_000 + 9, SORT_MIN + 37])
@pytest.mark.parametrize("thr", [1e-3, 0.5, 40.0])
def test_survivor_rich_thresholds(engine, n, thr, variant):
    """Eight-point models of a noisy scene at thresholds where a large share (1e-3) up to nearly all (40) of the tests
    survive: records carry most of their 32 bits and nearly every drain writes 32 records back.  200 hypotheses (a
    partly filled last warp) and a partial last batch."""
    cols, table, E = _noisy_scene(n, 200, seed=n % 97)
    cnt = _check(engine, cols, table, E, thr, variant)
    if thr >= 0.5:
        assert np.median(cnt) > 0.6 * n


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("n", [2_000 + 3, SORT_MIN + 37])
@pytest.mark.parametrize("scale", [1e-160, 1e160])
def test_models_outside_the_range_guard(engine, n, scale, variant):
    """Every third model scaled out of the range guard, so all of its tests survive the screen and the exact scorer
    decides each: full records from some lanes next to sparse ones from the others, at the reference's threshold."""
    cols, table, E = _noisy_scene(n, 200, seed=n % 89)
    E = E.copy()
    E[::3] *= scale
    _check(engine, cols, table, E, 1.5e-6, variant)
