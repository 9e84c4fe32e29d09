"""GPU parity at the BASELINE.json configuration sizes.

config 2 (10k correspondences x 16k hypotheses): full-size comparison with the oracle on the
  reference-RNG sample table.
config 3 (100k x 64k): size-independent properties — run-to-run determinism, invariance under
  hypothesis sharding and under the scoring variant, K2's count of the winner against K4's mask.
config 4 (batch of image pairs): the batched call against per-pair calls, ragged and empty pairs.
"""
import random

import numpy as np
import pytest

from oracle import csed
from oracle import restatement as o
from structure_from_motion_b200 import _native, two_view
from structure_from_motion_b200.scenes import make_scene

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


def test_config2_full_size_against_oracle(engine):
    """10 000 correspondences x 16 384 hypotheses, 40 % outliers, sample table drawn by the
    CPython-exact sampler from random.seed(5) (what ransac.py:62 would draw)."""
    n, h = 10_000, 16_384
    K, x1, x2, *_ = make_scene(n, 0.4, seed=0)
    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    random.seed(5)
    state = random.getstate()
    st = np.array(state[1], dtype=np.uint32)
    table, _ = _native.mt_shuffle_table(st, n, h)
    # spot-check the table against CPython itself on a prefix
    random.setstate(state)
    perm = list(range(n))
    for it in range(3):
        random.shuffle(perm)
        assert perm[:8] == table[it].tolist()

    # (1) the scorer alone, with the oracle's models: counts bit-exact, sums to 1e-12
    ca, cb = np.stack([nxa, nya], 1), np.stack([nxb, nyb], 1)
    E_o = np.stack([o.eight_point(ca[s], cb[s]) for s in table])
    cnt_o, s1_o, s2_o = csed.score_batch(E_o, nxa, nya, nxb, nyb, THR, table=table, nthreads=16)
    engine.upload_pairs(x1, x2, K)
    engine.set_table(table)
    engine.set_models(E_o)
    cnt, s1, s2, err = engine.score(THR, min_extra=10, aggregation="rms")
    assert np.array_equal(cnt, cnt_o)
    np.testing.assert_allclose(s1, s1_o, rtol=1e-12, atol=0)
    np.testing.assert_allclose(s2, s2_o, rtol=1e-12, atol=0)
    err_o = np.where(cnt_o >= 10, np.sqrt(s2_o / (8 + cnt_o)), np.inf)
    win_o = int(np.argmin(err_o))
    assert engine.get_best().index == win_o

    # (2) the whole GPU pipeline (own fitter) from the same global RNG state
    random.setstate(state)
    res = two_view.ransac_essential_arrays(K, x1, x2, THR, 10, "rms", h, engine=engine)
    assert res.best_index == win_o
    assert _e_close(res.E, E_o[win_o])
    assert abs(res.error - err_o[win_o]) <= 1e-9 * err_o[win_o]
    sed_o = csed.sed_exact_many(E_o[win_o], nxa, nya, nxb, nyb)
    in_band = np.abs(sed_o - THR) <= BAND * THR
    mask_o = sed_o <= THR
    mask_o[table[win_o]] = True  # samples are always part of the model's inliers (ransac.py:76)
    got = np.zeros(n, dtype=bool)
    got[res.inlier_indices] = True
    assert not ((got != mask_o) & ~in_band).any()
    assert res.inlier_indices[:8].tolist() == table[win_o].tolist()
    # per-hypothesis fitted models against the oracle's, on a subsample (conditioning-scaled)
    engine.set_table(table)
    E_g, valid, _ = engine.fit()
    assert valid.all()
    worst = 0.0
    for i in range(0, h, 37):
        d = np.linalg.norm(E_g[i] / np.linalg.norm(E_g[i]) - E_o[i] / np.linalg.norm(E_o[i]))
        worst = max(worst, d)
    assert worst <= 1e-6, worst


@pytest.fixture(scope="module")
def config3(engine):
    n, h = 100_000, 65_536
    K, x1, x2, *_ = make_scene(n, 0.4, seed=0)
    engine.upload_pairs(x1, x2, K)
    engine.sample_device(seed=3, h=h)
    engine.fit(want_E=False)
    cnt, s1, s2, err = engine.score(THR, min_extra=10, aggregation="rms")
    best = engine.get_best()
    return dict(n=n, h=h, K=K, x1=x1, x2=x2, cnt=cnt, s1=s1, s2=s2, err=err, best=best)


def test_config3_deterministic_and_variant_invariant(engine, config3):
    c = config3
    for variant, hpt, group in [("screen", 2, 16), ("full", 2, 16), ("screen32", 4, 8)]:
        engine.set_score_variant(variant, hpt, group)
        try:
            cnt, s1, s2, err = engine.score(THR, min_extra=10, aggregation="rms")
        finally:
            engine.set_score_variant("auto")
        assert np.array_equal(cnt, c["cnt"]), variant
        # integer accumulation: the sums are bit-identical whatever the schedule or the variant
        assert np.array_equal(s1, c["s1"]) and np.array_equal(s2, c["s2"]), variant
        assert np.array_equal(err, c["err"]), variant
        assert engine.get_best().index == c["best"].index


def test_config3_hypothesis_sharding_invariant(engine, config3):
    """Scoring the hypothesis range in four shards (what bench.py --gpus 4 does per rank) gives
    the same per-hypothesis results and, merged by the reference's rule, the same winner."""
    c = config3
    h, parts = c["h"], 4
    rows = []
    for r in range(parts):
        lo = r * h // parts
        engine.sample_device(seed=3, h=h // parts, hyp_offset=lo)
        engine.fit(want_E=False)
        cnt, s1, s2, err = engine.score(THR, min_extra=10, aggregation="rms", idx_offset=lo)
        assert np.array_equal(cnt, c["cnt"][lo:lo + h // parts])
        assert np.array_equal(err, c["err"][lo:lo + h // parts])
        b = engine.get_best()
        rows.append((b.err, b.index))
    # strict <, earliest index on ties (ransac.py:83)
    win = min(rows, key=lambda t: (t[0], t[1]))
    assert win[1] == c["best"].index
    engine.sample_device(seed=3, h=h)
    engine.fit(want_E=False)
    engine.score(THR, min_extra=10, aggregation="rms", want_arrays=False)


def test_config3_winner_count_equals_mask(engine, config3):
    c = config3
    best = engine.get_best()
    assert best.index == c["best"].index
    mask, sed = engine.inlier_mask(THR)
    table = engine.get_table()
    samples = table[best.index]
    assert np.array_equal(mask, sed <= THR)
    # ransac.py:63-64,70-76: samples are not thresholded but always part of the model's inliers
    n_extra = int(mask.sum()) - int(mask[samples].sum())
    assert n_extra == best.count_extra == c["cnt"][best.index]
    s2 = float(np.sum(sed[mask] ** 2) + np.sum(sed[samples][~mask[samples]] ** 2))
    assert abs(np.sqrt(s2 / (8 + n_extra)) - best.err) <= 1e-12 * best.err
    # and the exact C scorer agrees bit for bit with K4 on every correspondence
    nxa, nya, nxb, nyb = _norm(c["K"], c["x1"], c["x2"])
    E = np.array(best.E, dtype=np.float64).reshape(3, 3)
    assert np.array_equal(sed, csed.sed_exact_many(E, nxa, nya, nxb, nyb))


def test_config3_full_size_inlier_rich_against_oracle(engine, config3):
    """The same at a threshold where 7 % of the correspondences are inliers of a typical model: the AUTO pilot picks
    the two-sided body (survivor gathers from shared memory, one ring entry per survivor).  All 65 536 models x 100 000
    correspondences against the exact C scorer: counts bit-exact, sums to 1e-12, same winner; and bit-identical to the
    one-sided body's results."""
    import os

    c = config3
    thr = 1.5e-4
    E, valid = engine.get_models()
    table = engine.get_table()
    nxa, nya, nxb, nyb = _norm(c["K"], c["x1"], c["x2"])
    cnt_o, s1_o, s2_o = csed.score_batch(E.reshape(-1, 9), nxa, nya, nxb, nyb, thr, table=table,
                                         nthreads=os.cpu_count() or 8)
    assert cnt_o.mean() > 0.05 * c["n"]
    got = {}
    try:
        for variant in ("auto", "screen"):
            engine.set_score_variant(variant, 2, 16)
            got[variant] = engine.score(thr, min_extra=10, aggregation="rms") + (engine.get_best().index,)
    finally:
        engine.set_score_variant("auto")
    cnt, s1, s2, err, win = got["auto"]
    assert np.array_equal(cnt, cnt_o)
    np.testing.assert_allclose(s2, s2_o, rtol=1e-12, atol=0)
    err_o = np.where(cnt_o >= 10, np.sqrt(s2_o / (8 + cnt_o)), np.inf)
    assert win == int(np.argmin(err_o))
    for a, b in zip(got["auto"][:4], got["screen"][:4]):
        assert np.array_equal(a, b, equal_nan=True)
    assert got["screen"][4] == win
    engine.score(THR, min_extra=10, aggregation="rms", want_arrays=False)  # leave the engine as the fixture left it


def test_config3_full_size_counts_against_oracle(engine, config3):
    """BASELINE.json configs[2] at full size against the oracle, not against itself: ALL 65 536 models the GPU fitted
    are scored by the exact C scorer over all 100 000 correspondences (6.5e9 evaluations, threaded): extra-inlier
    counts bit-exact, sum of squares to 1e-12, the same winner as the oracle's arg-min, and the triangulated points of
    the winner's inliers within 1e-6 relative of the oracle's DLT (lib/epipolar/triangulation.py:9-62)."""
    import os

    c = config3
    n, h = c["n"], c["h"]
    engine.upload_pairs(c["x1"], c["x2"], c["K"])
    engine.sample_device(seed=3, h=h)
    best, _, _, poses, num, idx, ok, X = engine.two_view(THR, 10, "rms", "min_error", 50.0)
    E, valid = engine.get_models()
    table = engine.get_table()
    assert valid.all()
    nxa, nya, nxb, nyb = _norm(c["K"], c["x1"], c["x2"])
    cnt_o, s1_o, s2_o = csed.score_batch(E.reshape(-1, 9), nxa, nya, nxb, nyb, THR, table=table,
                                         nthreads=os.cpu_count() or 8)
    assert np.array_equal(c["cnt"], cnt_o)
    np.testing.assert_allclose(c["s2"], s2_o, rtol=1e-12, atol=0)
    err_o = np.where(cnt_o >= 10, np.sqrt(s2_o / (8 + cnt_o)), np.inf)
    win = int(np.argmin(err_o))
    assert best.index == win == c["best"].index
    assert abs(best.err - err_o[win]) <= 1e-12 * err_o[win]
    # the winner's inliers (samples included, ransac.py:76), ascending
    sed_o = csed.sed_exact_many(E[win], nxa, nya, nxb, nyb)
    m = sed_o <= THR
    m[table[win]] = True
    assert num == int(m.sum()) and np.array_equal(idx, np.nonzero(m)[0])
    # pose: the oracle's candidates from the same E; ours is one of them, the vote picked the one most points pass
    R1, R2, t1 = o.recover_all_r_t(E[win])
    b = int(poses.best)
    Rg = np.array(poses.R, dtype=np.float64).reshape(4, 3, 3)[b]
    tg = np.array(poses.t, dtype=np.float64).reshape(4, 3)[b]
    assert min(np.abs(Rg - R).max() for R in (R1, R2)) <= 1e-9
    assert min(np.abs(tg - t).max() for t in (t1, -t1)) <= 1e-9
    sub = idx[:: max(1, len(idx) // 400)]  # the oracle's per-point python check on a sample of the inliers
    passing_sub = ((ok >> b) & 1).astype(bool)[:: max(1, len(idx) // 400)]
    want = [o.cheirality_check(nxa[i], nya[i], nxb[i], nyb[i], Rg, tg, 50.0) for i in sub]
    assert passing_sub.tolist() == [bool(w) for w in want]
    # triangulation of every passing inlier against the oracle's DLT
    passing = ((ok >> b) & 1).astype(bool)
    pi = idx[passing]
    X_o = o.triangulate_points(c["x1"][pi, 0], c["x1"][pi, 1], c["x2"][pi, 0], c["x2"][pi, 1], c["K"], o.tmat(Rg, tg))
    rel = np.linalg.norm(X[passing] - X_o, axis=1) / np.linalg.norm(X_o, axis=1)
    assert rel.max() <= 1e-6, rel.max()
    assert np.isnan(X[~passing]).all()
    # leave the engine as the fixture left it
    engine.sample_device(seed=3, h=h)
    engine.fit(want_E=False)
    engine.score(THR, min_extra=10, aggregation="rms", want_arrays=False)


def test_config4_batch_matches_single_pairs(engine):
    """Ragged batch (a pair with too few correspondences and an empty pair included): every pair's
    winner equals the single-pair pipeline on the same (seed, pair id) sample table."""
    sizes = [2000, 1500, 5, 0, 2000, 700, 8, 33]
    h, seed, pair0 = 2000, 9, 40
    scenes = [make_scene(max(s, 8), 0.4, seed=100 + p) for p, s in enumerate(sizes)]
    K = scenes[0][0]
    xa = np.concatenate([sc[1][:s] for sc, s in zip(scenes, sizes)])
    xb = np.concatenate([sc[2][:s] for sc, s in zip(scenes, sizes)])
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    Ks = np.stack([K] * len(sizes))
    out = engine.batch_ransac(xa, xb, offsets, Ks, h, seed, THR, 10, "rms", pair_id0=pair0)
    for p, s in enumerate(sizes):
        if s < 8 + 10:  # cannot have 10 extra inliers
            assert out["best_index"][p] == -1, (p, s)
            continue
        a, b = xa[offsets[p]:offsets[p + 1]], xb[offsets[p]:offsets[p + 1]]
        engine.upload_pairs(a, b, K)
        engine.sample_device(seed=seed, h=h, stream=pair0 + p)
        best, _, _ = engine.ransac_essential(THR, 10, "rms", want_mask=False, want_sed=False)
        assert best.index == out["best_index"][p], p
        if best.index < 0:  # no model with enough inliers (ransac.py:88-91)
            assert np.isinf(out["best_err"][p])
            continue
        assert best.count_extra == out["count_extra"][p]
        assert best.err == out["best_err"][p]
        assert np.array_equal(np.array(best.E).reshape(3, 3), out["E"][p])
        # and against the oracle on that table
        table = engine.get_table()
        try:
            ref = o.ransac_essential(K, a[:, 0], a[:, 1], b[:, 0], b[:, 1], THR, 10, "rms", h, table=table,
                                     on_degenerate="skip")
        except ValueError:  # ransac.py:88-91: no model with enough inliers
            assert best.index == -1
            continue
        assert ref["best_index"] == best.index
        assert _e_close(out["E"][p], ref["E"])


def test_pair_pipeline_equals_single_call(engine):
    """distributed.PairPipeline (two contexts, chunks of pairs, H2D overlapped with compute) returns exactly what one
    batch_ransac call over all pairs returns, for ragged pairs and any chunking."""
    from structure_from_motion_b200.distributed import PairPipeline

    sizes = [700, 64, 333, 9, 1200, 500, 8, 410, 77]
    scenes = [make_scene(max(s, 8), 0.35, seed=40 + p) for p, s in enumerate(sizes)]
    xa = np.concatenate([sc[1][:s] for sc, s in zip(scenes, sizes)])
    xb = np.concatenate([sc[2][:s] for sc, s in zip(scenes, sizes)])
    off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    Ks = np.stack([sc[0] for sc in scenes])
    want = engine.batch_ransac(xa, xb, off, Ks, 300, 11, 1.5e-6, 5, "rms", pair_id0=1000)
    pipe = PairPipeline(depth=2)
    try:
        for chunk in (None, 1, 4, 100):
            got = pipe.batch_ransac(xa, xb, off, Ks, 300, 11, 1.5e-6, 5, "rms", pair_id0=1000, chunk_pairs=chunk)
            for k in want:
                assert np.array_equal(got[k], want[k], equal_nan=True) if got[k].dtype.kind == "f" else np.array_equal(got[k], want[k]), (chunk, k)
    finally:
        pipe.close()


def test_config5_scale_invariants(engine):
    """BASELINE.json configs[4] sizes on one GPU: 1 048 576 correspondences and one rank's share (1/64 here) of the
    1 048 576 hypotheses.  Size-independent properties: shard invariance, count == mask, the error from the mask, the
    exact C scorer on a sample of hypotheses, and the whole tail (pose vote + triangulation of ~400k inliers)."""
    n, h_total, shard = 1_048_576, 1_048_576, 16_384
    K, x1, x2, R_true, t_true, _ = make_scene(n, 0.4, seed=5)
    engine.upload_pairs(x1, x2, K)
    lo = 37 * shard  # rank 37 of 64
    engine.sample_device(seed=9, h=shard, hyp_offset=lo)
    E, valid, _ = engine.fit()
    cnt, s1, s2, err = engine.score(THR, min_extra=10, aggregation="rms", idx_offset=lo)
    best = engine.get_best()
    assert lo <= best.index < lo + shard and best.index - lo == int(np.argmin(err))
    # the same hypotheses scored as two half shards
    for part in range(2):
        plo = lo + part * shard // 2
        engine.sample_device(seed=9, h=shard // 2, hyp_offset=plo)
        engine.fit(want_E=False)
        c2, _, _, e2 = engine.score(THR, min_extra=10, aggregation="rms", idx_offset=plo)
        sl = slice(part * shard // 2, (part + 1) * shard // 2)
        assert np.array_equal(c2, cnt[sl]) and np.array_equal(e2, err[sl])
    engine.sample_device(seed=9, h=shard, hyp_offset=lo)
    engine.fit(want_E=False)
    engine.score(THR, min_extra=10, aggregation="rms", idx_offset=lo, want_arrays=False)
    best = engine.get_best()
    mask, sed = engine.inlier_mask(THR)
    samples = engine.get_table()[best.index - lo]
    n_extra = int(mask.sum()) - int(mask[samples].sum())
    assert n_extra == best.count_extra == cnt[best.index - lo]
    ssum = float(np.sum(sed[mask] ** 2) + np.sum(sed[samples][~mask[samples]] ** 2))
    assert abs(np.sqrt(ssum / (8 + n_extra)) - best.err) <= 1e-11 * best.err
    # exact C scorer on EVERY hypothesis of this rank's shard, all 1M correspondences (1.7e10 evaluations, threaded)
    import os

    nxa, nya, nxb, nyb = _norm(K, x1, x2)
    table = engine.get_table()
    cnt_o, s1_o, s2_o = csed.score_batch(E.reshape(-1, 9), nxa, nya, nxb, nyb, THR, table=table,
                                         nthreads=os.cpu_count() or 8)
    assert np.array_equal(cnt, cnt_o)
    np.testing.assert_allclose(s2, s2_o, rtol=1e-12, atol=0)
    err_o = np.where(cnt_o >= 10, np.sqrt(s2_o / (8 + cnt_o)), np.inf)
    assert best.index - lo == int(np.argmin(err_o))
    # tail: cheirality vote + triangulation of the winner's inliers; the pose is the scene's (to the accuracy of an
    # eight-point fit on one minimal sample selected by min-RMS, which is what the reference computes)
    poses, num, idx, ok, X = engine.pose_and_triangulate(THR, 50.0)
    assert num == int(mask.sum() + (~mask[samples]).sum()) and num > 300_000
    b = poses.best
    Rg = np.array(poses.R, dtype=np.float64).reshape(4, 3, 3)[b]
    tg = np.array(poses.t, dtype=np.float64).reshape(4, 3)[b]
    assert np.degrees(np.arccos(np.clip((np.trace(Rg.T @ R_true) - 1) / 2, -1, 1))) < 2.5
    assert np.degrees(np.arccos(np.clip(tg @ t_true / np.linalg.norm(t_true), -1, 1))) < 10.0
    passing = ((ok >> b) & 1).astype(bool)
    assert passing.mean() > 0.95 and np.isfinite(X[passing]).all() and (X[passing][:, 2] > 0).all()


def test_device_side_merge_of_sharded_records(engine):
    """sfm_sharded_tail's merge kernel against distributed.merge_best (the host rule the gloo tests pin) on crafted
    records, and the fused sharded path with world = 1 against the plain fused call."""
    import torch

    from structure_from_motion_b200 import distributed

    K, x1, x2, *_ = make_scene(4000, 0.35, seed=31)
    engine.set_stream(torch.cuda.current_stream().cuda_stream)
    try:
        engine.upload_pairs(x1, x2, K)
        r = distributed.two_view_sharded(THR, 10, "rms", 600, 4, engine=engine, rank=0, world=1)
        engine.sample_device(4, 600)
        best, _, _, poses, num, idx, ok, X = engine.two_view(THR, 10, "rms", "min_error", 50.0)
        assert r["index"] == best.index and r["owner"] == 0 and r["err"] == best.err
        assert r["num_inliers"] == num and np.array_equal(r["inlier_idx"], idx) and np.array_equal(r["pass_bits"], ok)
        assert np.array_equal(r["points"], X, equal_nan=True)
        # crafted gather: rank 2 of 4 holds the winner (a tie on the error with rank 3: the earlier global index wins),
        # rank 0 has no candidate
        H = 600
        engine.sample_device(4, H, hyp_offset=1 * H)
        ptr = engine.score_async(THR, 10, "rms")
        mine = torch.as_tensor(distributed._DeviceBuffer(ptr, engine.RECORD_BYTES // 8), device="cuda").clone()
        torch.cuda.synchronize()
        rec = mine.cpu().numpy().copy()  # [err, idx(bits), count|pad(bits), ninv, first, E[9], sample int32[8]]
        as_i64 = rec.view(np.int64)
        rows = []
        for rank_r, (err_scale, idx_local) in enumerate([(None, -1), (1.0, int(as_i64[1])), (0.5, 7), (0.5, 3)]):
            row = rec.copy()
            ri = row.view(np.int64)
            if err_scale is None:
                ri[1] = -1
            else:
                row[0] = rec[0] * err_scale
                ri[1] = idx_local
                row[5:14] = rec[5:14] * (1.0 + rank_r)  # a recognisable E per rank
                row[14:].view(np.int32)[:] = np.arange(8) + 10 * rank_r  # and a recognisable sample row
            rows.append(row)
        gathered = torch.from_numpy(np.concatenate(rows)).cuda()
        engine.sharded_tail(gathered.data_ptr(), 4, 1, H, THR, 50.0)
        b, owner, poses, num, idx, ok, X = engine.sharded_fetch()
        want = distributed.merge_best(np.array([distributed.pack_local_best(
            rows[k][0], (k * H + int(rows[k].view(np.int64)[1])) if rows[k].view(np.int64)[1] >= 0 else -1,
            int(rows[k].view(np.int32)[4]), rows[k][5:14]) for k in range(4)]))
        assert owner == want[0] == 2 and b.index == want[2] == 2 * H + 7 and b.err == want[1]
        assert np.array_equal(np.array(b.E), rows[2][5:14])
        # the winner's sample row (rank 2's: 20..27) was forced into the inlier set on this non-owner rank (ransac.py:76)
        assert set(range(20, 28)) <= set(idx.tolist())
        # all ranks empty
        for row in rows:
            row.view(np.int64)[1] = -1
        gathered = torch.from_numpy(np.concatenate(rows)).cuda()
        engine.sharded_tail(gathered.data_ptr(), 4, 1, H, THR, 50.0)
        b, owner, poses, num, idx, ok, X = engine.sharded_fetch()
        assert owner == -1 and b.index == -1 and num == 0 and np.isinf(b.err)
    finally:
        engine.set_stream(None)
