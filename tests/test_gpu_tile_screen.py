"""K2's one-sided screen in 9 FP64 slots: a single pair of >= 65 536 correspondences is sorted by the Morton code of its
image-B positions at upload, and every test is made against one bound on the line norm per (hypothesis, tile).  The
bound must never drop an inlier of the exact scorer, the sort must change no output, and padding must never survive.
Shorter pairs and batches keep the 11-slot screen on the scaled copy (tests/test_gpu_parity.py covers it at 1 500)."""
import functools

import numpy as np
import pytest

from oracle import csed
from oracle import restatement as o
from structure_from_motion_b200.scenes import make_scene
from test_gpu_parity import SCALE_CASES
from test_gpu_score_range import check_against_oracle

pytestmark = pytest.mark.gpu
THR = 1.5e-6
IDENT = np.eye(3)
SORT_MIN = 65_536  # kK2SortMin in csrc/sfm_ransac.cu


def _norm(K, x1, x2):
    nxa, nya = o.k_normalise(x1[:, 0], x1[:, 1], K)
    nxb, nyb = o.k_normalise(x2[:, 0], x2[:, 1], K)
    return nxa, nya, nxb, nyb


def _models(nxa, nya, nxb, nyb, h, seed):
    rng = np.random.default_rng(seed)
    n = len(nxa)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    ca, cb = np.stack([nxa, nya], 1), np.stack([nxb, nyb], 1)
    return table, np.stack([o.eight_point(ca[s], cb[s]) for s in table])


def _score(engine, x1, x2, K, table, E, thr, variant="screen", aggregation="rms", min_extra=10):
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    engine.set_models(E)
    engine.set_score_variant(variant, 2, 16)
    try:
        return engine.score(thr, min_extra=min_extra, aggregation=aggregation)
    finally:
        engine.set_score_variant("auto")


def test_shuffled_input_gives_identical_results(engine):
    """The sort key ties keep input order, so a shuffled upload sorts differently inside ties; counts and sums are
    integers and must not move, nor the winner, its inlier list or its SED values (read in input order)."""
    n, h = 40_000, 1024
    K, x1, x2, *_ = make_scene(n, 0.4, seed=31)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    table, E = _models(nxa, nya, nxb, nyb, h, seed=4)
    base = _score(engine, x1, x2, K, table, E, THR)
    best = engine.get_best()
    mask, sed = engine.inlier_mask(THR)
    cnt_o, s1_o, s2_o = csed.score_batch(E, nxa, nya, nxb, nyb, THR, table=table, nthreads=8)
    assert np.array_equal(base[0], cnt_o)
    np.testing.assert_allclose(base[2], s2_o, rtol=1e-12, atol=0)

    perm = np.random.default_rng(8).permutation(n)
    inv = np.empty(n, dtype=np.int64)
    inv[perm] = np.arange(n)
    got = _score(engine, x1[perm], x2[perm], K, inv[table].astype(np.int32), E, THR)
    for a, b in zip(base, got):
        assert np.array_equal(a, b, equal_nan=True)
    best2 = engine.get_best()
    assert best2.index == best.index and best2.err == best.err
    mask2, sed2 = engine.inlier_mask(THR)
    assert np.array_equal(mask2, mask[perm]) and np.array_equal(sed2, sed[perm])
    assert np.array_equal(np.sort(perm[np.flatnonzero(mask2)]), np.flatnonzero(mask))


@pytest.mark.parametrize("n", [8, 63, SORT_MIN - 1, SORT_MIN, SORT_MIN + 1, SORT_MIN + 63, SORT_MIN + 64, SORT_MIN + 65])
def test_pair_lengths_match_exact_scorer(engine, n):
    """Both sides of the sort threshold and partial last tiles of the 9-slot body, whose box covers only its own
    records; counts equal and sums within 1e-12 of the exact oracle at several thresholds."""
    K, x1, x2, *_ = make_scene(max(n, 8), 0.3, seed=50 + n)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    table, E = _models(nxa, nya, nxb, nyb, 150, seed=n)
    for thr in (0.0, 1e-9, THR, 1e-3, 40.0):
        cnt, s1, s2, _ = _score(engine, x1, x2, K, table, E, thr, aggregation="sum", min_extra=0)
        cnt_o, s1_o, s2_o = csed.score_batch(E, nxa, nya, nxb, nyb, thr, table=table, nthreads=8)
        assert np.array_equal(cnt, cnt_o), thr
        np.testing.assert_allclose(s1, s1_o, rtol=1e-12, atol=0)
        np.testing.assert_allclose(s2, s2_o, rtol=1e-12, atol=0)


def test_batched_ragged_pairs_match_full_body(engine):
    """Batches keep the 11-slot screen (no sorted copy, whatever the pair lengths); explicitly selected, it must pick the
    same winners with the same errors and counts as the two-sided body, pair by pair, for pairs of 8 to 63 records and
    lengths that are not multiples of the tile."""
    sizes = [8, 63, 9, 64, 65, 40, 1025, 17, 700, 130, 2000, 31]
    scenes = [make_scene(s, 0.3, seed=300 + p) for p, s in enumerate(sizes)]
    xa = np.concatenate([sc[1] for sc in scenes])
    xb = np.concatenate([sc[2] for sc in scenes])
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    Ks = np.stack([sc[0] for sc in scenes])
    out = {}
    try:
        for variant in ("screen", "full"):
            engine.set_score_variant(variant, 2, 16)
            out[variant] = engine.batch_ransac(xa, xb, off, Ks, 500, 5, THR, 0, "rms")
    finally:
        engine.set_score_variant("auto")
    for k in ("E", "best_index", "best_err", "count_extra", "num_invalid"):
        assert np.array_equal(out["screen"][k], out["full"][k], equal_nan=True), k
    assert out["screen"]["count_extra"].sum() > 100


def _adversarial_scene(kind, rng):
    """Correspondences in normalised coordinates (K = I) that stress the box bound, and models to score them with."""
    K, x1, x2, *_ = make_scene(SORT_MIN + 7_000, 0.3, seed=77)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    table, E = _models(nxa, nya, nxb, nyb, 200, seed=3)
    if kind == "corners":  # B points on a coarse lattice: many records sit exactly on their tile's box corners
        nxb = np.round(nxb * 8) / 8
        nyb = np.round(nyb * 8) / 8
    elif kind == "epipole":  # B points at and around the epipole of model 0, where lb0^2 + lb1^2 -> 0
        u, _, _ = np.linalg.svd(E[0])
        ep = u[:, 2] / u[2, 2]  # E^T ep = 0
        m = 1500
        r = 10.0 ** rng.uniform(-12, -2, m) * rng.choice([-1, 1], m)
        ang = rng.uniform(0, 2 * np.pi, m)
        nxb[:m] = ep[0] + r * np.cos(ang)
        nyb[:m] = ep[1] + r * np.sin(ang)
        nxb[0], nyb[0] = ep[0], ep[1]
        nxa[:m] = rng.uniform(-1, 1, m)
        nya[:m] = rng.uniform(-1, 1, m)
    elif kind == "wide":  # a few far outliers in image B widen every box they fall into
        idx = rng.choice(len(nxb), 60, replace=False)
        nxb[idx] = rng.uniform(-1e4, 1e4, 60)
        nyb[idx] = rng.uniform(-1e4, 1e4, 60)
    return nxa, nya, nxb, nyb, table, E


@pytest.mark.parametrize("kind", ["corners", "epipole", "wide"])
@pytest.mark.parametrize("thr", [0.0, 1e-12, THR, 1e-3, 0.5])
def test_adversarial_tiles_match_exact_scorer(engine, kind, thr):
    rng = np.random.default_rng({"corners": 1, "epipole": 2, "wide": 3}[kind])
    nxa, nya, nxb, nyb, table, E = _adversarial_scene(kind, rng)
    x1 = np.stack([nxa, nya], 1)
    x2 = np.stack([nxb, nyb], 1)
    cnt, s1, s2, _ = _score(engine, x1, x2, IDENT, table, E, thr, aggregation="sum", min_extra=0)
    cnt_o, s1_o, s2_o = csed.score_batch(E, nxa, nya, nxb, nyb, thr, table=table, nthreads=8)
    assert np.array_equal(cnt, cnt_o)
    np.testing.assert_allclose(s1, s1_o, rtol=1e-12, atol=0)
    np.testing.assert_allclose(s2, s2_o, rtol=1e-12, atol=0)


@functools.lru_cache(maxsize=1)
def _sweep_scene():
    n, h = SORT_MIN + 7_000, 256
    K, x1, x2, *_ = make_scene(n, 0.3, seed=11)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    table, E = _models(nxa, nya, nxb, nyb, h, seed=9)
    return K, x1, x2, (nxa, nya, nxb, nyb), table, E


@functools.lru_cache(maxsize=None)
def _sweep_oracle(escale, thr):
    K, x1, x2, cols, table, E = _sweep_scene()
    return csed.score_batch(E * escale, *cols, thr, table=table, nthreads=8)


@pytest.mark.parametrize("escale,thr", SCALE_CASES)
def test_tile_screen_never_drops_an_inlier(engine, thr, escale):
    """Every body of the 9-slot upload is a necessary condition at every threshold and model scale (the grid of
    test_gpu_parity.py::test_screen_never_drops_an_inlier, whose 1 500 correspondences run the 11-slot screen): T's
    kappa scales with |E_h|^2 and its thr' with the threshold; outside the range guard every test is decided exactly.
    Counts, sums, K3's errors and winner and K4's mask and SED against the exact oracle, for every variant."""
    K, x1, x2, cols, table, E = _sweep_scene()
    E = E * escale
    oracle = _sweep_oracle(escale, thr)
    for variant in ("screen", "full", "screen32", "auto"):
        engine.upload_pairs(x1, x2, K)
        engine.set_table(table)
        engine.set_models(E)
        engine.set_score_variant(variant)
        try:
            got = engine.score(thr, min_extra=0, aggregation="sum")
        finally:
            engine.set_score_variant("auto")
        check_against_oracle(engine, got, E, cols, thr, oracle)
    if thr == 1.5e-6 and 1e-153 <= escale <= 1e150:
        assert oracle[0].sum() > 0
    if escale == 1e154 and thr <= 1.5e-6:
        assert oracle[0].sum() > _sweep_oracle(1.0, thr)[0].sum()


@pytest.mark.parametrize("variant,hpt,group,thr", [("screen", 2, 16, THR), ("screen", 2, 16, 1e-3),
                                                   ("auto", 2, 16, THR), ("auto", 2, 16, 1e-3)])
def test_every_tiled_shape_matches_exact_scorer(engine, variant, hpt, group, thr):
    """The 9-slot body (ScoreWarpSmemBox<HPT>: boxes and per-lane kappa in shared memory), and AUTO on
    either side of its pilot's decision (1.5e-6: the 9-slot body; 1e-3: the two-sided one), against the exact oracle:
    72 573 records (a partial last tile) and 300 hypotheses (not a multiple of 32 HPT), with K3 and the K4 mask."""
    n, h = SORT_MIN + 7_037, 300
    K, x1, x2, *_ = make_scene(n, 0.3, seed=13)
    cols = _norm(K, x1, x2)
    table, E = _models(*cols, h, seed=14)
    oracle = csed.score_batch(E, *cols, thr, table=table, nthreads=8)
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    engine.set_models(E)
    engine.set_score_variant(variant, hpt, group)
    try:
        got = engine.score(thr, min_extra=0, aggregation="sum")
    finally:
        engine.set_score_variant("auto")
    check_against_oracle(engine, got, E, cols, thr, oracle)
