"""GPU checks of the batched homography path and the batched choice between the essential matrix and a homography:
every pair of sfm_batch_two_view_homography and sfm_batch_score_models is bit for bit what the single-pair calls return
on that pair alone (ragged sizes around the 64-record tile and the 2 048-record item, short and empty pairs, every
aggregation and selection mode, thresholds outside the fixed-point range), the scores also against oracle/cselect, the
per-pair rule of batch_two_view_select_arrays, its classification of general, planar and rotation-only pairs, the
refusals, PairPipeline's chunking and the randomised sweep of tools/fuzz_batch_homography.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import cselect
from structure_from_motion_b200 import _native, batch_two_view_select_arrays
from structure_from_motion_b200.distributed import PairPipeline
from structure_from_motion_b200.model_selection import two_view_select_arrays
from structure_from_motion_b200.scenes import make_planar_scene, make_scene

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import fuzz_batch_homography as fz  # noqa: E402

pytestmark = pytest.mark.gpu

SIZES = [0, 5, 7, 8, 33, 63, 64, 65, 1024, 1025, 2047, 2048, 2049]
KINDS = "epreprepreper"
H_THR = 4.0   # px^2
E_THR = 1e-5  # SED, K-normalised


def _mixed(seed=7, skew=False, sizes=SIZES, kinds=KINDS):
    return fz.batch(sizes, kinds, seed, skew=skew)


@pytest.mark.parametrize("skew", [False, True])
def test_equal_to_single_pair_calls(engine, skew):
    xa, xb, offsets, Ks = _mixed(skew=skew)
    bad, r = fz.compare_homography(engine, xa, xb, offsets, Ks, 300, 11, 17, H_THR)
    assert not bad, bad[:10]
    assert (r["best_index"][np.diff(offsets) >= 33] >= 0).all()


@pytest.mark.parametrize("thr", [H_THR, 0.0, -1.0, 1e101])
def test_every_aggregation_and_selection(engine, thr):
    xa, xb, offsets, Ks = _mixed(seed=9, sizes=[0, 7, 40, 300, 2049], kinds="eprpe")
    modes = [(a, "min_error") for a in fz.AGGS] + [("sum", "max_inliers"), ("rms", "msac")]
    for agg, sel in modes:
        min_extra = 3.0 if sel == "max_inliers" else 0.0
        bad, _ = fz.compare_homography(engine, xa, xb, offsets, Ks, 130, 5, 3, thr, min_extra, agg, sel)
        assert not bad, bad[:10]


def test_scores_equal_single_pair_and_oracle(engine):
    # a skewed K: the E path's camera Kd (no skew) differs from K
    xa, xb, offsets, Ks = _mixed(seed=13, skew=True, sizes=[40, 300, 7, 2049, 65, 500],
                                 kinds="eprepe")
    r = engine.batch_two_view_homography(xa, xb, offsets, Ks, 200, 3, H_THR)
    P = len(offsets) - 1
    rng = np.random.default_rng(1)
    E = rng.normal(size=(P, 3, 3))
    H = np.where(r["best_index"][:, None, None] >= 0, r["H"], np.eye(3))
    cases = [(np.ones(P, bool), np.ones(P, bool)), (np.ones(P, bool), np.zeros(P, bool)),
             (np.zeros(P, bool), np.ones(P, bool)), (np.array([1, 0, 0, 1, 0, 1], bool), np.array([0, 1, 0, 1, 0, 0], bool))]
    for he, hh in cases:
        bad = fz.compare_scores(engine, xa, xb, offsets, Ks, E, H, he, hh)
        assert not bad, bad[:10]
        engine.batch_two_view_homography(xa, xb, offsets, Ks, 1, 3, H_THR)  # back to the batched upload
        s, pp = engine.batch_score_models(E, H, he, hh, 1.0, 0.45, per_point=True)
        for p in range(P):
            lo, hi = offsets[p], offsets[p + 1]
            if not (he[p] or hh[p]):
                assert s[p].model == -1
                continue
            ref = cselect.score_models(Ks[p], xa[lo:hi], xb[lo:hi], E=E[p] if he[p] else None,
                                       H=H[p] if hh[p] else None)
            np.testing.assert_array_equal(pp[lo:hi], ref["per_point"])
            assert (s[p].fixed_e, s[p].fixed_h, s[p].count_e, s[p].count_h, s[p].model) == (
                ref["fixed_e"], ref["fixed_h"], ref["count_e"], ref["count_h"], ref["model"])
    # NULL flag arrays: every model given
    s_all, _ = engine.batch_score_models(E, H)
    s_one, _ = engine.batch_score_models(E, H, np.ones(P, bool), np.ones(P, bool))
    assert bytes(s_all) == bytes(s_one)


def test_selection_sides_and_rule(engine):
    xa, xb, offsets, Ks = _mixed(seed=21, sizes=[0, 7, 300, 600, 1025, 400, 64], kinds="epepere")
    h, seed, pid0 = 256, 4, 9
    sel = batch_two_view_select_arrays(xa, xb, offsets, Ks, E_THR, H_THR, h, seed, pair_id0=pid0, engine=engine)
    ess = engine.batch_two_view(xa, xb, offsets, Ks, h, seed, E_THR, pair_id0=pid0)
    hom = engine.batch_two_view_homography(xa, xb, offsets, Ks, h, seed, H_THR, pair_id0=pid0)
    for side, ref in (("essential", ess), ("homography", hom)):
        for k, v in ref.items():
            np.testing.assert_array_equal(sel[side][k], v, err_msg=f"{side}.{k}")
    for p in range(len(offsets) - 1):
        lo, hi = offsets[p], offsets[p + 1]
        if hi - lo < 8:
            assert sel["model"][p] is None and sel["essential_status"][p] and sel["homography_status"][p]
            continue
        # the single-pair call with the device sampler draws stream 0: run it on a batch of one pair with that id
        one = batch_two_view_select_arrays(xa[lo:hi], xb[lo:hi], [0, hi - lo], Ks[p:p + 1], E_THR, H_THR, h, seed,
                                           pair_id0=pid0 + p, engine=engine)
        assert one["model"][0] == sel["model"][p]
        for k in ("fixed_e", "fixed_h", "count_e", "count_h", "essential_status", "homography_status"):
            assert one[k][0] == sel[k][p]


def test_selection_matches_single_pair_rule(engine):
    # pair_id0 = 0 and one pair: the batch draws stream 0, as two_view_select_arrays(sampler="device") does
    for kind, seed in [("e", 1), ("p", 2), ("r", 3), ("p", 4)]:
        xa, xb, offsets, Ks = fz.batch([700], kind, seed)
        sel = batch_two_view_select_arrays(xa, xb, offsets, Ks, E_THR, H_THR, 512, seed, engine=engine)
        one = two_view_select_arrays(Ks[0], xa, xb, E_THR, H_THR, None, "rms", 512, None, sampler="device", seed=seed,
                                     engine=engine)
        assert sel["model"][0] == one.model
        assert (sel["essential_status"][0] is None) == (one.essential is not None)
        assert (sel["homography_status"][0] is None) == (one.homography is not None)
        assert (sel["fixed_e"][0], sel["fixed_h"][0]) == (one.scores.fixed_e, one.scores.fixed_h)
        np.testing.assert_array_equal(sel["R"][0], one.R)
        np.testing.assert_array_equal(sel["inlier_idx"], one.inlier_indices)
        np.testing.assert_array_equal(sel["passing"], one.passing)
        np.testing.assert_array_equal(sel["points"], one.points)
        assert bool(sel["rotation_only"][0]) == one.rotation_only


def test_classification(engine):
    # the scenes, thresholds and 4 096 hypotheses of the single-pair classification tests (test_gpu_model_select.py)
    kinds = "eeeppprrr"
    scenes = [make_scene(20000, 0.3, s)[:3] for s in range(3)] + [make_planar_scene(20000, 0.3, s)[:3] for s in range(3)]
    scenes += [make_planar_scene(20000, 0.3, s, rotation_only=True)[:3] for s in range(3)]
    xa, xb = np.concatenate([x1 for _, x1, _ in scenes]), np.concatenate([x2 for _, _, x2 in scenes])
    offsets, Ks = np.arange(10) * 20000, np.stack([K for K, _, _ in scenes])
    sel = batch_two_view_select_arrays(xa, xb, offsets, Ks, 1e-5, 16.0, 4096, 7, min_extra=10_000, engine=engine)
    want = {"e": "essential", "p": "homography", "r": "homography"}
    assert list(sel["model"]) == [want[k] for k in kinds], (list(sel["model"]), sel["ratio_h"])
    assert list(sel["rotation_only"]) == [k == "r" for k in kinds]


def test_refusals(engine):
    xa, xb, offsets, Ks = _mixed(seed=3, sizes=[100, 200, 300], kinds="epr")

    def call(**kw):
        args = dict(pts_a=xa, pts_b=xb, offsets=offsets, Ks=Ks, h=64, seed=1, threshold=H_THR)
        args.update(kw)
        return engine.batch_two_view_homography(**args)

    for bad_k in (np.array([[800, 0, 640], [1e-3, 800, 480], [0, 0, 1.0]]), 2 * Ks[1], Ks[1] * np.nan):
        Kb = Ks.copy()
        Kb[1] = bad_k
        with pytest.raises(_native.NativeError, match=r"-1: pair 1"):
            call(Ks=Kb)
    for off in ([1, 100, 300, 600], [0, 200, 100, 600], [0, 100, 300, 0]):
        with pytest.raises(_native.NativeError, match="-1"):
            call(offsets=np.array(off))
    with pytest.raises(_native.NativeError, match="-1"):
        call(rotation_tolerance=np.nan)
    big = np.zeros(65537, dtype=np.int64)
    big[-1] = 600
    with pytest.raises(_native.NativeError, match="-1"):
        call(offsets=big, Ks=np.tile(Ks[:1], (65536, 1, 1)))
    r = call()
    P = 3
    E, H = np.tile(np.eye(3), (P, 1, 1)), r["H"]
    for kw in (dict(E=E * np.nan), dict(H=np.where(np.eye(3) > 0, np.inf, H)), dict(E=None, H=None),
               dict(sigma=0.0), dict(sigma=np.inf), dict(homography_ratio=np.nan)):
        args = dict(E=E, H=H, sigma=1.0, homography_ratio=0.45)
        args.update(kw)
        with pytest.raises(_native.NativeError, match="-1"):
            engine.batch_score_models(**args)
    # a non-finite model that is not given is not read
    s, _ = engine.batch_score_models(E * np.nan, H, np.zeros(P, bool), None)
    assert [x.model for x in s[:P]] == [1, 1, 1]
    engine.upload_pairs(xa[:100], xb[:100], np.eye(3))
    out = (_native.ModelScores * P)()
    rc = engine.lib.sfm_batch_score_models(engine.h, E.ctypes.data, None, np.ascontiguousarray(H).ctypes.data, None,
                                           1.0, 0.45, _native.C.cast(out, _native.C.c_void_p), None)
    assert rc == -3  # not a batched upload


@pytest.mark.parametrize("chunk", [None, 1, 4, 100])
def test_pipeline_chunks_equal_one_call(engine, chunk):
    # no empty pair: a chunk of empty pairs alone has no correspondences to upload
    xa, xb, offsets, Ks = _mixed(seed=41, sizes=[5, 300, 7, 900, 65, 2049, 8, 400, 33, 1500], kinds="eprepreper")
    pipe = PairPipeline(depth=2)
    try:
        got = pipe.batch_two_view_homography(xa, xb, offsets, Ks, 200, 8, H_THR, pair_id0=5, chunk_pairs=chunk)
        want = engine.batch_two_view_homography(xa, xb, offsets, Ks, 200, 8, H_THR, pair_id0=5)
        assert got.keys() == want.keys()
        for k in want:
            np.testing.assert_array_equal(got[k], want[k], err_msg=k)
        got = pipe.batch_two_view_select(xa, xb, offsets, Ks, E_THR, H_THR, 200, 8, pair_id0=5, chunk_pairs=chunk)
        want = batch_two_view_select_arrays(xa, xb, offsets, Ks, E_THR, H_THR, 200, 8, pair_id0=5, engine=engine)
        for k in want:
            if isinstance(want[k], dict):
                for kk in want[k]:
                    np.testing.assert_array_equal(got[k][kk], want[k][kk], err_msg=f"{k}.{kk}")
            else:
                np.testing.assert_array_equal(got[k], want[k], err_msg=k)
        got = pipe.batch_two_view(xa, xb, offsets, Ks, 200, 8, E_THR, pair_id0=5, chunk_pairs=chunk)
        want = engine.batch_two_view(xa, xb, offsets, Ks, 200, 8, E_THR, pair_id0=5)
        for k in want:
            np.testing.assert_array_equal(got[k], want[k], err_msg=k)
    finally:
        pipe.close()


def test_fuzz_batch_homography():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_batch_homography.py"), "30"],
                         capture_output=True, text=True, timeout=1200, cwd=ROOT)
    assert out.returncode == 0 and "mismatches: 0" in out.stdout, out.stdout[-3000:] + out.stderr[-2000:]
