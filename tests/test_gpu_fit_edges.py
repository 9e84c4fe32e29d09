"""K1's production fitter — k_fit_qr (Householder QR of Y^T in registers) and the k_fit fallback it hands the samples
its validity test cannot call — against the exact fit of oracle/fit_exact.py, through ``fit()`` without eigenvalues
(the path every estimate takes), on samples fed in by ``set_table`` and on the same samples fitted inside a batch.

Bounds (u = 2^-53, E compared as a direction: Frobenius-normalised, sign-aligned):
- the direction of E is within C_DIR u kappa(Y) rho(F*) amp of E*, with C_DIR = 16: a backward-stable null vector
  errs by O(u kappa(Y)) — linear in kappa, where the reference's route through Y^T Y errs by O(u kappa^2) — the
  rank-2 projection multiplies that by rho = sigma_1(F) / (sigma_2(F) - sigma_3(F)), the denormalisation
  E = T2^T F' T1 by amp = |T1| |T2| |F'| / |E*| (fit_exact.ExactFit);
- validity: k_fit_qr decides from 1 / |R^-1|_F^2 <= sigma_8^2 <= min r_ii^2 against 1e-10 with a 0.1 % margin and
  flags the rest ambiguous; k_fit then redoes them in the reference's arithmetic (Y^T Y, eigenvalues), whose lambda_2
  errs by about u lambda_max.  So ``valid`` must equal the exact decision (sigma_8^2 > 1e-10) outside the 0.1 % band
  (plus QR rounding, ~1e-10 relative here; 1e-6 is allowed) unless the sample may have gone to k_fit and lies within
  4 u lambda_max of the threshold; it must equal the reference's decision wherever the reference's lambda_2 is further
  than 4 u lambda_max from 1e-10; and a sample the exact bounds prove ambiguous must come back bit-identical to a
  ``want_eig=True`` fit (k_fit for every hypothesis), which shows the fallback ran and rewrote E and the status byte.
  Scoring after the fast fit must equal scoring ``set_models`` with the returned E bit for bit (K2's screen evaluates
  its survivors from K1's padded rows, which must hold that E)."""
import json
import os
import random

import numpy as np
import pytest

from oracle import fit_exact as fx
from oracle import restatement as o
from structure_from_motion_b200 import _native, two_view
from structure_from_motion_b200.scenes import make_scene

pytestmark = pytest.mark.gpu
U = fx.U
C_DIR = 16
THR = 1e100  # scoring threshold: every record with a finite SED is an inlier, so stale rows change the counts
SLACK = 1e-6
I3 = np.eye(3)
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.uint64)


def same(a, b):
    return np.array_equal(bits(a), bits(b))


def normalised_scene(n, outliers, seed):
    K, x1, x2, *_ = make_scene(n, outliers, seed=seed)
    return K, x1, x2, np.stack(o.k_normalise(x1[:, 0], x1[:, 1], K), 1), np.stack(o.k_normalise(x2[:, 0], x2[:, 1], K), 1)


def fit_rows(engine, ca, cb, table, want_eig=False):
    """K-normalised records (uploaded with an identity camera: x / 1 = x) and a table -> (E [h,3,3], valid [h])."""
    engine.upload_pairs(ca, cb, I3)
    engine.set_table(table)
    E, valid, _ = engine.fit(want_eig=want_eig)
    return E, valid


def batch_rows(engine, pairs, h, seed=7):
    """Fit h device-drawn hypotheses for every pair of K-normalised records in one batch; per pair (table, E, valid)."""
    P = len(pairs)
    offsets = np.concatenate([[0], np.cumsum([len(a) for a, _ in pairs])]).astype(np.int64)
    pa = np.vstack([a for a, _ in pairs])
    pb = np.vstack([b for _, b in pairs])
    engine.batch_ransac(pa, pb, offsets, np.tile(I3.reshape(1, 9), (P, 1)), h, seed, 1e-3)
    E, valid = engine.get_models(0, P * h)
    table = engine.get_table(P * h, 0)
    return [(table[p * h:(p + 1) * h], E[p * h:(p + 1) * h], valid[p * h:(p + 1) * h]) for p in range(P)]


def check_direction(E, valid, fits, worst):
    """Every row valid, E[2,2] == 1 and the direction within C_DIR u kappa rho amp of E*; worst[0] keeps the largest
    error / bound."""
    for i, f in enumerate(fits):
        assert valid[i] and f.valid, i
        d = fx.direction_error(E[i], f)
        bound = C_DIR * U * f.kappa * f.rho * f.amp
        worst[0] = max(worst[0], d / bound)
        assert d <= bound, (i, d, bound, f.kappa, f.rho, f.amp)
        assert E[i][2, 2] == 1.0


# ---------------------------------------------------------------------------------------------------------------------
# generic samples
# ---------------------------------------------------------------------------------------------------------------------
def test_generic_samples_within_a_bound_linear_in_kappa(engine):
    n, h = 4000, 1500
    K, x1, x2, ca, cb = normalised_scene(n, 0.5, seed=21)
    rng = np.random.default_rng(4)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    engine.upload_pairs(x1, x2, K)  # the camera applied on the device: bit-identical to o.k_normalise
    engine.set_table(table)
    E, valid, _ = engine.fit()
    fits = [fx.fit_exact(ca[s], cb[s]) for s in table]
    worst = [0.0]
    check_direction(E, valid, fits, worst)
    # DESIGN's claim: error O(u kappa) against the reference's O(u kappa^2) — on the best-conditioned fifth of the
    # samples the two are both at rounding level; on the worst-conditioned fifth the GPU must be the closer one
    kap = np.array([f.kappa for f in fits])
    hi = np.flatnonzero(kap >= np.quantile(kap, 0.8))
    d_gpu = np.array([fx.direction_error(E[i], fits[i]) for i in hi])
    d_ref = np.array([fx.direction_error(o.eight_point(ca[table[i]], cb[table[i]]), fits[i]) for i in hi])
    ratio = np.median(d_gpu / np.maximum(d_ref, 1e-300))
    assert ratio < 1.0, ratio
    # the same kind of samples fitted inside a batch, next to a pair too short to sample from
    got = batch_rows(engine, [(ca[:1000], cb[:1000]), (ca[:5], cb[:5])], 300)
    (tb, Eb, vb), (ts, Es, vs) = got
    check_direction(Eb, vb, [fx.fit_exact(ca[s], cb[s]) for s in tb], worst)
    assert not vs.any() and not Es.any() and not ts.any()
    print(f"generic: largest error / (u kappa rho amp) = {worst[0] * C_DIR:.3g} (bound {C_DIR}); "
          f"kappa {kap.min():.3g}..{kap.max():.3g}; high-kappa median d_gpu / d_ref = {ratio:.3g}")


# ---------------------------------------------------------------------------------------------------------------------
# the validity ladder
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def ladder():
    return [(geo, seed, delta, ca, cb, fx.fit_exact(ca, cb)) for geo, seed, delta, ca, cb in fx.ladder(seeds=(0, 1, 2))]


def ladder_expectations(f):
    """(rows must equal the exact decision, rows must equal the reference's decision, rows must be bit-identical to
    the Jacobi fit) for a sample of exact fit f."""
    sure_valid = f.qr_lo > 1.001 * fx.VERY_SMALL * (1 + SLACK)
    sure_invalid = f.qr_hi < 0.999 * fx.VERY_SMALL * (1 - SLACK)
    sure_ambiguous = f.qr_lo < 1.001 * fx.VERY_SMALL * (1 - SLACK) and f.qr_hi > 0.999 * fx.VERY_SMALL * (1 + SLACK)
    jacobi_band = abs(f.s8sq - fx.VERY_SMALL) <= 4 * U * f.lam_max_ref
    outside_qr_band = abs(f.s8sq / fx.VERY_SMALL - 1.0) > 1e-3 + SLACK
    exact = outside_qr_band and (sure_valid or sure_invalid or not jacobi_band)
    ref = abs(f.lam2_ref - fx.VERY_SMALL) > 4 * U * f.lam_max_ref
    return exact, ref, sure_ambiguous


def check_ladder_rows(f, E, valid, E_eig=None, valid_eig=None):
    exact, ref, ambiguous = ladder_expectations(f)
    if exact:
        assert (valid == f.valid).all()
    if ref:
        assert (valid == f.ref_valid).all()
    if ambiguous and E_eig is not None:
        assert same(E, E_eig) and np.array_equal(valid, valid_eig)
    zero = ~E.reshape(len(E), 9).any(axis=1)
    assert not (valid & zero).any()  # no "valid" all-zero model (an unresolved status byte 2)
    assert zero[~valid].all()
    return exact, ref, ambiguous


def test_validity_ladder(engine, ladder):
    """sigma_8(Y)^2 = 1e-10 (1 + delta), delta in +-{0.5, 0.05, 5e-3, 1.5e-3, 1e-3, 5e-4, 1e-4}, clustered and with one
    far point, three seeds; each sample as 8 rows (its own order and 7 permutations) over its 8 records followed by
    300 scene records to score."""
    _, _, _, sa, sb = normalised_scene(300, 0.3, seed=5)
    rng = np.random.default_rng(8)
    table = np.stack([np.arange(8)] + [rng.permutation(8) for _ in range(7)]).astype(np.int32)
    n_exact = n_ref = n_amb = 0
    for geo, seed, delta, ca, cb, f in ladder:
        ra, rb = np.vstack([ca, sa]), np.vstack([cb, sb])
        E_eig, valid_eig = fit_rows(engine, ra, rb, table, want_eig=True)
        # the one-sided screen evaluates its survivors (here: every record) from K1's padded rows
        for variant in ("screen", "auto"):
            engine.set_score_variant(variant)
            try:
                E, valid = fit_rows(engine, ra, rb, table)
                got = engine.score(THR, aggregation="sum")
                best = engine.get_best().index
                engine.set_models(E.reshape(-1, 9), valid.astype(np.uint8))
                again = engine.score(THR, aggregation="sum")
            finally:
                engine.set_score_variant("auto")
            for a, b in zip(got, again):
                assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8)), (geo, seed, delta)
            assert engine.get_best().index == best
            assert (got[0][valid] > 0).all(), (geo, seed, delta, variant)
        exact, ref, amb = check_ladder_rows(f, E, valid, E_eig, valid_eig)
        n_exact += exact
        n_ref += ref
        n_amb += amb
    assert n_amb >= len(ladder) // 3  # the fallback did run on a good share of the ladder
    print(f"ladder: {len(ladder)} samples; exact decision asserted on {n_exact}, the reference's on {n_ref} "
          f"(skipped {len(ladder) - n_ref} inside 4 u lambda_max of 1e-10); {n_amb} bit-identical to the Jacobi fit")


def test_validity_ladder_in_a_batch(engine, ladder):
    """Every ladder sample as its own pair of 8 records (so each device-drawn row is a permutation of the sample),
    with a pair too short to sample from in the middle: the rows equal single-pair fits of the same rows bit for bit
    and satisfy the same decisions."""
    pairs = [(ca, cb) for *_, ca, cb, _ in ladder]
    pairs.insert(len(pairs) // 2, (pairs[0][0][:6], pairs[0][1][:6]))
    got = batch_rows(engine, pairs, 16)
    short = got.pop(len(ladder) // 2)
    assert not short[2].any() and not short[1].any()
    for (geo, seed, delta, ca, cb, f), (tb, Eb, vb) in zip(ladder, got):
        assert (np.sort(tb, axis=1) == np.arange(8)).all()
        E, valid = fit_rows(engine, ca, cb, tb)
        assert same(E, Eb) and np.array_equal(valid, vb), (geo, seed, delta)
        check_ladder_rows(f, Eb, vb)


# ---------------------------------------------------------------------------------------------------------------------
# exactly degenerate samples
# ---------------------------------------------------------------------------------------------------------------------
def coplanar_pair():
    rng = np.random.default_rng(0)
    X = np.column_stack([rng.uniform(-1, 1, 8), rng.uniform(-1, 1, 8), np.full(8, 5.0)])
    X2 = X + np.array([-0.5, 0.0, 0.0])
    return X[:, :2] / X[:, 2:], X2[:, :2] / X2[:, 2:]


def test_exactly_degenerate_samples_are_invalid(engine):
    """A repeated index in a row (rank 7) and eight coplanar points (rank 6) are invalid with E = 0, in single pairs
    and in a batch; so are eight exactly coincident points in one image and a NaN record (non-finite normalised
    coordinates), whose exceptions test_nonfinite_samples_raise_what_the_reference_raises pins."""
    _, _, _, ca, cb = normalised_scene(100, 0.0, seed=3)
    rep = np.array([[0, 1, 2, 3, 4, 5, 6, 0], [9, 9, 1, 2, 3, 4, 5, 6], [7, 6, 5, 4, 3, 2, 1, 1]], dtype=np.int32)
    E, valid = fit_rows(engine, ca, cb, rep)
    assert not valid.any() and not E.any()
    pa, pb = coplanar_pair()
    coinc = np.repeat([[0.5, -0.25]], 8, axis=0)
    nan_a = ca[:8].copy()
    nan_a[5, 0] = np.nan
    cases = [(pa, pb), (coinc, cb[:8]), (ca[:8], coinc), (nan_a, cb[:8])]
    for a, b in cases:
        E, valid = fit_rows(engine, a, b, np.arange(8, dtype=np.int32).reshape(1, 8))
        assert not valid.any() and not E.any()
    for tb, Eb, vb in batch_rows(engine, cases + [(ca, cb)], 32)[:-1]:
        assert not vb.any() and not Eb.any()


def test_nonfinite_samples_raise_what_the_reference_raises(engine):
    """tests/golden/nonfinite_sample_fixture.json, from the unmodified reference: numpy's LinAlgError where the
    normalised coordinates are not finite, EightPointCalculationError where they are; RANSAC (reference sampler)
    stops with the global random state where the reference leaves it."""
    with open(os.path.join(GOLDEN, "nonfinite_sample_fixture.json")) as fh:
        d = json.load(fh)
    K = np.array(d["K"])
    kinds = {"numpy.linalg.LinAlgError": np.linalg.LinAlgError,
             "lib.epipolar.eight_point.EightPointCalculationError": two_view.EightPointCalculationError}
    for case in d["eight_point"]:
        with pytest.raises(kinds[case["raises"]]) as info:
            two_view.eight_point_arrays(np.array(case["pts_a"]), np.array(case["pts_b"]), K, engine=engine)
        assert type(info.value) is kinds[case["raises"]] and str(info.value) == case["message"], case["name"]
    for case in d["ransac"]:
        random.seed(case["seed"])
        with pytest.raises(kinds[case["raises"]]) as info:
            two_view.ransac_essential_arrays(K, np.array(case["pts_a"]), np.array(case["pts_b"]), case["threshold"],
                                             None, "rms", case["max_iterations"], engine=engine)
        assert type(info.value) is kinds[case["raises"]] and str(info.value) == case["message"], case["name"]
        assert list(random.getstate()[1]) == case["state_after"], case["name"]


# ---------------------------------------------------------------------------------------------------------------------
# extreme inputs
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("spread", [1e-3, 1e-1, 1e2, 1e4, 1e6])
def test_pixel_spread_extremes(engine, spread):
    """The scene's samples squeezed or stretched about their centroid to a pixel spread of 1e-3 .. 1e6 (Hartley
    normalisation undoes the scale): E's direction within the same bound of the exact fit of those coordinates."""
    K, x1, x2, *_ = make_scene(400, 0.3, seed=13)
    rng = np.random.default_rng(2)
    rows = [rng.choice(400, 8, replace=False) for _ in range(40)]
    pa, pb = [], []
    for s in rows:
        for src, dst in ((x1, pa), (x2, pb)):
            c = src[s].mean(axis=0)
            dst.append(c + (src[s] - c) * (spread / np.ptp(src[s], axis=0).max()))
    pa, pb = np.vstack(pa), np.vstack(pb)
    table = np.arange(8 * len(rows), dtype=np.int32).reshape(-1, 8)
    engine.upload_pairs(pa, pb, K)
    engine.set_table(table)
    E, valid, _ = engine.fit()
    ca = np.stack(o.k_normalise(pa[:, 0], pa[:, 1], K), 1)
    cb = np.stack(o.k_normalise(pb[:, 0], pb[:, 1], K), 1)
    fits = [fx.fit_exact(ca[s], cb[s]) for s in table]
    worst = [0.0]
    check_direction(E, valid, fits, worst)
    (tb, Eb, vb), = batch_rows(engine, [(ca[:8], cb[:8])], 8)
    check_direction(Eb, vb, [fx.fit_exact(ca[s], cb[s]) for s in tb], worst)
    print(f"spread {spread:g} px: largest error / (u kappa rho amp) = {worst[0] * C_DIR:.3g}")


def test_pure_horizontal_translation(engine):
    """Noise-free, R = I, t along x (rectified stereo): E* = [t]x has E*[2,2] = 0, so K1's E / E[2,2] divides by
    rounding noise or by 0.  Finite rows keep E*'s direction; a valid row with a non-finite E scores no inlier and
    never wins, as in the reference (its SED is NaN, its error NaN, and NaN < best is false)."""
    rng = np.random.default_rng(6)
    n = 400
    X = np.column_stack([rng.uniform(-2, 2, n), rng.uniform(-1.5, 1.5, n), rng.uniform(4, 8, n)])
    K = np.array([[800.0, 0, 640], [0, 800.0, 480], [0, 0, 1]])
    x1 = (K @ X.T).T
    x2 = (K @ (X + np.array([-1.0, 0.0, 0.0])).T).T
    x1, x2 = x1[:, :2] / x1[:, 2:], x2[:, :2] / x2[:, 2:]
    ca = np.stack(o.k_normalise(x1[:, 0], x1[:, 1], K), 1)
    cb = np.stack(o.k_normalise(x2[:, 0], x2[:, 1], K), 1)
    table = np.stack([rng.choice(n, 8, replace=False) for _ in range(200)]).astype(np.int32)
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    E, valid, _ = engine.fit()
    cnt, s1, _, err = engine.score(1.5e-6, aggregation="rms")
    best = engine.get_best().index
    finite = np.isfinite(E.reshape(-1, 9)).all(axis=1)
    worst = [0.0]
    for i in np.flatnonzero(valid & finite):
        f = fx.fit_exact(ca[table[i]], cb[table[i]])
        d = fx.direction_error(E[i], f)
        bound = C_DIR * U * f.kappa * f.rho * f.amp
        worst[0] = max(worst[0], d / bound)
        assert d <= bound, (i, d, bound)
    bad = np.flatnonzero(valid & ~finite)
    assert (cnt[bad] == 0).all() and np.isinf(err[bad]).all()
    assert best not in set(bad.tolist())
    print(f"pure translation: {valid.sum()} valid rows, {len(bad)} with a non-finite E; "
          f"largest error / (u kappa rho amp) of the finite ones = {worst[0] * C_DIR:.3g}")


# ---------------------------------------------------------------------------------------------------------------------
# draws and call sequences
# ---------------------------------------------------------------------------------------------------------------------
def test_rows_drawn_inside_the_fit_equal_k_sample(engine):
    """sample_device is lazy: the fit kernel draws the rows itself.  The rows (hyp_offset included) and the fit equal
    those of k_sample, which runs when the table is read before the fit."""
    K, x1, x2, *_ = make_scene(3000, 0.3, seed=17)
    for off in (0, 12_345):
        engine.upload_pairs(x1, x2, K)
        engine.sample_device(3, 700, hyp_offset=off)
        E1, v1, _ = engine.fit()
        t1 = engine.get_table(700)
        engine.upload_pairs(x1, x2, K)
        engine.sample_device(3, 700, hyp_offset=off)
        t2 = engine.get_table(700)
        E2, v2, _ = engine.fit()
        assert np.array_equal(t1, t2) and same(E1, E2) and np.array_equal(v1, v2)


def test_call_sequences_equal_fresh_contexts(engine, ladder):
    """With rows the fast path flags ambiguous in the table: fit -> fit (no score between, so K3 never reset the
    ambiguous counter), fit -> score -> fit, and a batch followed by a single pair all give what a fresh context
    gives: E and validity bit for bit, and the scores after them."""
    amb = [(ca, cb) for _, _, delta, ca, cb, f in ladder if ladder_expectations(f)[2]]
    ca, cb = amb[0]
    _, _, _, sa, sb = normalised_scene(300, 0.3, seed=5)
    ra, rb = np.vstack([ca, sa]), np.vstack([cb, sb])
    rng = np.random.default_rng(1)
    table = np.vstack([np.stack([rng.permutation(8) for _ in range(12)]),
                       np.stack([8 + rng.choice(300, 8, replace=False) for _ in range(20)])]).astype(np.int32)

    def run(eng):
        E, valid = fit_rows(eng, ra, rb, table)
        return E, valid

    fresh = _native.Engine(0)
    try:
        E0, v0 = run(fresh)
        s0 = fresh.score(THR, aggregation="sum")
    finally:
        fresh.close()

    def agree(E, v, s=None):
        assert same(E, E0) and np.array_equal(v, v0)
        if s is not None:
            for a, b in zip(s, s0):
                assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))

    agree(*run(engine))
    E, v, _ = engine.fit()  # fit -> fit
    agree(E, v, engine.score(THR, aggregation="sum"))
    E, v, _ = engine.fit()  # fit -> score -> fit
    agree(E, v, engine.score(THR, aggregation="sum"))
    batch_rows(engine, [(ca, cb), (sa, sb), (ca[:3], cb[:3])], 64)  # batched -> single
    E, v = run(engine)
    agree(E, v, engine.score(THR, aggregation="sum"))
