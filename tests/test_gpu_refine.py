"""GPU checks of the least-squares refinement of essential-matrix and homography winners (sfm_set_refinement,
csrc/sfm_refine.cuh): refinement off changes nothing and leaves the RANSAC side untouched, the optimum against scipy's
Levenberg-Marquardt (oracle/refine.py) from the same start, the invariants and statuses, the tail on the refined model
against the existing calls for a caller-supplied model, determinism across runs, batches and PairPipeline chunks,
accuracy against the truth, the refusals, and a reduced sweep of tools/fuzz_refine.py."""
import os
import random
import sys

import numpy as np
import pytest

from oracle import refine as O
from oracle.restatement import triangulate_one
from structure_from_motion_b200 import _native
from structure_from_motion_b200.distributed import PairPipeline
from structure_from_motion_b200.homography import two_view_homography_arrays
from structure_from_motion_b200.scenes import make_planar_scene, make_scene
from structure_from_motion_b200.two_view import two_view_arrays

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import fuzz_refine as fz  # noqa: E402

pytestmark = pytest.mark.gpu

E_THR = 1e-5   # SED, K-normalised
H_THR = 4.0    # px^2
RAGGED = [0, 5, 8, 63, 64, 65, 1024, 1025, 2047, 2048, 2049]


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _rot_deg(Ra, Rb):
    return float(np.degrees(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1.0) / 2.0, -1.0, 1.0))))


def _dir_deg(a, b):
    a, b = a / np.linalg.norm(a), b / np.linalg.norm(b)
    return float(np.degrees(np.arccos(np.clip(abs(a @ b), 0.0, 1.0))))


# ---- off means off --------------------------------------------------------------------------------
@pytest.mark.parametrize("sampler", ["reference", "device"])
def test_refinement_leaves_the_ransac_result_untouched(engine, sampler):
    K, x1, x2, _, _, _ = make_scene(600, 0.4, 3)
    kw = dict(sampler=sampler, seed=5, engine=engine, on_degenerate="skip")
    random.seed(11)
    a = two_view_arrays(K, x1, x2, E_THR, 0, "rms", 300, **kw)
    st_a = random.getstate()
    random.seed(11)
    b = two_view_arrays(K, x1, x2, E_THR, 0, "rms", 300, refine_iterations=0, **kw)
    random.seed(11)
    c = two_view_arrays(K, x1, x2, E_THR, 0, "rms", 300, refine_iterations=20, **kw)
    assert random.getstate() == st_a
    assert b.refinement is None and c.refinement is not None
    for r in (b, c):
        assert np.array_equal(_bits(r.ransac.E), _bits(a.ransac.E))
        assert r.ransac.best_index == a.ransac.best_index and _bits(r.ransac.error) == _bits(a.ransac.error)
        assert np.array_equal(r.ransac.mask, a.ransac.mask) and np.array_equal(_bits(r.ransac.sed), _bits(a.ransac.sed))
        assert np.array_equal(r.ransac.inlier_indices, a.ransac.inlier_indices)
    assert np.array_equal(_bits(b.R), _bits(a.R)) and np.array_equal(_bits(b.points), _bits(a.points))


def test_homography_refinement_leaves_the_ransac_result_untouched(engine):
    K, x1, x2, _, _ = make_planar_scene(500, 0.3, 4)
    a = two_view_homography_arrays(K, x1, x2, H_THR, sampler="device", seed=2, engine=engine)
    c = two_view_homography_arrays(K, x1, x2, H_THR, sampler="device", seed=2, engine=engine, refine_iterations=20)
    assert np.array_equal(_bits(c.ransac.H), _bits(a.ransac.H))
    assert np.array_equal(c.ransac.mask, a.ransac.mask) and np.array_equal(_bits(c.ransac.err), _bits(a.ransac.err))
    assert c.refinement.cost_final <= c.refinement.cost_start


@pytest.mark.parametrize("kind", ["E", "H"])
def test_batch_without_refinement_is_unchanged_and_the_ransac_keys_stay(engine, kind):
    xa, xb, offsets, Ks = fz.batch([300, 65, 7, 1025], "epep", 5)
    call = engine.batch_two_view if kind == "E" else engine.batch_two_view_homography
    thr = E_THR if kind == "E" else H_THR
    a = call(xa, xb, offsets, Ks, 200, 3, thr)
    b = call(xa, xb, offsets, Ks, 200, 3, thr, refine_iterations=0)
    c = call(xa, xb, offsets, Ks, 200, 3, thr, refine_iterations=10)
    assert set(a) == set(b) and not any(k.startswith("refine") for k in a)
    for k in a:
        va, vb = np.asarray(a[k]), np.asarray(b[k])
        assert np.array_equal(_bits(va) if va.dtype == np.float64 else va, _bits(vb) if vb.dtype == np.float64 else vb), k
    key = "E" if kind == "E" else "H"
    for k in (key, "best_index", "best_err", "count_extra", "num_invalid"):
        va, vc = np.asarray(a[k]), np.asarray(c[k])
        assert np.array_equal(_bits(va) if va.dtype == np.float64 else va, _bits(vc) if vc.dtype == np.float64 else vc), k
    assert {"refined_" + key, "refine_cost_ransac", "refine_cost_start", "refine_cost_final", "refine_num",
            "refine_iterations", "refine_status", "refine_rejected"} <= set(c)


# ---- optimum against the oracle ---------------------------------------------------------------
@pytest.mark.parametrize("seed", [0, 1, 2])
def test_essential_optimum_matches_the_oracle(engine, seed):
    K, x1, x2, _, _, _ = make_scene(800, 0.3, seed)
    bad, rep, o = fz.oracle_check(engine, "E", x1, x2, K, 300, seed, E_THR, iters=100)
    assert not bad, bad
    assert _native.REFINE_STATUS[rep.status] == "converged"
    assert o["dmodel"] < 1e-5


@pytest.mark.parametrize("seed,rot", [(0, False), (1, False), (2, False), (3, True), (4, True)])
def test_homography_optimum_matches_the_oracle(engine, seed, rot):
    K, x1, x2, _, _ = make_planar_scene(800, 0.3, seed, rotation_only=rot)
    # a floor of extra inliers: the bare minimum-error winner is an exact fit through its own 4 samples
    bad, rep, o = fz.oracle_check(engine, "H", x1, x2, K, 300, seed, H_THR, iters=100, min_extra=200)
    assert not bad, bad
    assert _native.REFINE_STATUS[rep.status] == "converged"
    assert o["dmodel"] < 1e-5


# ---- statuses -----------------------------------------------------------------------------------
def test_statuses_at_the_edges(engine):
    K, x1, x2, _, _, _ = make_scene(300, 0.3, 1)
    engine.upload_pairs(x1, x2, K)
    for thr in (-1.0, float("nan"), 0.0, float("inf")):
        engine.sample_device(1, 200)
        best, *_ = engine.two_view(thr, refine_iterations=10)
        rep = engine.get_refinement(1)[0]
        st = _native.REFINE_STATUS[rep.status]
        assert not fz.invariants(rep, "E")
        if best.index < 0:
            assert st == "no_model"
        else:
            assert st in ("converged", "max_iterations", "stalled", "nonfinite")
            if thr < 0 or thr != thr:
                assert rep.num == 8  # only the sample
    # no model: min_extra beyond the data
    engine.sample_device(1, 50)
    best, *_ = engine.two_view(E_THR, 1e9, refine_iterations=5)
    assert best.index < 0 and _native.REFINE_STATUS[engine.get_refinement(1)[0].status] == "no_model"
    # H at threshold 0: the 4 exactly fitted samples
    K, x1, x2, _, _ = make_planar_scene(300, 0.0, 2)
    engine.upload_pairs(x1, x2, np.eye(3))
    engine.sample_device(2, 100)
    engine.two_view_homography(K, 0.0, refine_iterations=10)
    rep = engine.get_refinement(1)[0]
    assert rep.num == 4 and _native.REFINE_STATUS[rep.status] == "converged" and rep.iterations == 0
    assert rep.cost_final <= rep.cost_start


def test_refusals(engine):
    K, x1, x2, _, _, _ = make_scene(200, 0.2, 0)
    engine.upload_pairs(x1, x2, K)
    engine.sample_device(0, 64)
    engine.set_refinement(5)
    rec = engine.score_async(E_THR)
    with pytest.raises(_native.NativeError):
        engine.sharded_tail(rec, 1, 0, 64, E_THR)
    engine.set_refinement(0)
    with pytest.raises(ValueError):
        two_view_arrays(K, x1, x2, E_THR, refine_iterations=-1, engine=engine)
    with pytest.raises(ValueError):
        engine.batch_two_view(x1, x2, [0, 200], K[None], 64, 0, E_THR, refine_iterations=-2)


# ---- the tail on the refined model ---------------------------------------------------------------
def test_essential_tail_equals_a_caller_supplied_model(engine):
    K, x1, x2, R, t, _ = make_scene(700, 0.3, 6)
    engine.upload_pairs(x1, x2, K)
    engine.sample_device(6, 300)
    _, _, _, p, num, idx, ok, X = engine.two_view(E_THR, refine_iterations=30)
    rep = engine.get_refinement(1)[0]
    engine.set_winner(-1, np.array(rep.model))
    p2, num2, idx2, ok2, X2 = engine.pose_and_triangulate(E_THR)
    assert num == num2 and np.array_equal(idx, idx2) and np.array_equal(ok, ok2)
    assert np.array_equal(_bits(X), _bits(X2)) and int(p.best) == int(p2.best)
    assert np.array_equal(_bits(np.array(p.R)), _bits(np.array(p2.R)))
    # points against the oracle's DLT under the refined pose
    b = int(p.best)
    P1 = np.hstack([K, np.zeros((3, 1))])
    P2 = K @ np.hstack([np.array(p.R[b]).reshape(3, 3), np.array(p.t[b]).reshape(3, 1)])
    m = ((ok >> b) & 1).astype(bool)
    for k in np.flatnonzero(m)[:50]:
        (xa, ya), (xb, yb) = x1[idx[k]], x2[idx[k]]
        Xo = np.asarray(triangulate_one(xa, ya, xb, yb, P1, P2), dtype=np.float64).reshape(-1)[:3]
        assert np.allclose(X[k], Xo, rtol=1e-6, atol=1e-9 * np.abs(Xo).max())


def test_homography_tail_on_the_refined_model(engine):
    K, x1, x2, _, _ = make_planar_scene(700, 0.3, 7)
    engine.upload_pairs(x1, x2, np.eye(3))
    engine.sample_device(7, 300)
    _, _, _, p, num, idx, ok, X = engine.two_view_homography(K, H_THR, refine_iterations=30)
    Hr = np.array(engine.get_refinement(1)[0].model).reshape(3, 3)
    dec, _ = engine.homography_mask(Hr, H_THR)
    assert np.array_equal(idx, np.flatnonzero(dec))
    d = engine.decompose_homography(Hr, K)
    for f in ("R", "t", "n", "d", "sv"):
        assert np.array_equal(_bits(np.array(getattr(p, f))), _bits(np.array(getattr(d, f)))), f
    # points against the oracle's DLT under the voted candidate of the refined H (P1 = K[I|0], P2 = K[R|t], pixels)
    b = int(p.best)
    assert b >= 0 and not p.rotation_only
    P1 = np.hstack([K, np.zeros((3, 1))])
    P2 = K @ np.hstack([np.array(p.R[b]).reshape(3, 3), np.array(p.t[b]).reshape(3, 1)])
    m = ((ok >> b) & 1).astype(bool)
    assert m.sum() > 0 and np.isnan(X[~m]).all()
    for k in np.flatnonzero(m)[:50]:
        (xa, ya), (xb, yb) = x1[idx[k]], x2[idx[k]]
        Xo = np.asarray(triangulate_one(xa, ya, xb, yb, P1, P2), dtype=np.float64).reshape(-1)[:3]
        assert np.allclose(X[k], Xo, rtol=1e-6, atol=1e-9 * np.abs(Xo).max())


# ---- determinism -----------------------------------------------------------------------------------
def test_two_runs_are_bit_identical(engine):
    K, x1, x2, _, _, _ = make_scene(3000, 0.4, 8)
    out = []
    for _ in range(2):
        engine.upload_pairs(x1, x2, K)
        engine.sample_device(8, 500)
        engine.two_view(E_THR, refine_iterations=15)
        rep = engine.get_refinement(1)[0]
        out.append(np.frombuffer(bytes(rep), dtype=np.uint8).copy())
    assert np.array_equal(out[0], out[1])


@pytest.mark.parametrize("kind", ["E", "H"])
def test_batch_pairs_equal_single_pair_calls(engine, kind):
    xa, xb, offsets, Ks = fz.batch(RAGGED, "epeperepepe", 9, skew=True)
    bad, r = fz.compare_batch(engine, kind, xa, xb, offsets, Ks, 300, 21, 5, E_THR if kind == "E" else H_THR, 12)
    assert not bad, bad[:10]
    assert (r["refine_status"][np.diff(offsets) >= 63] != 3).all()


@pytest.mark.parametrize("kind", ["E", "H"])
def test_pair_pipeline_chunks_equal_one_call(engine, kind):
    xa, xb, offsets, Ks = fz.batch([300, 65, 2049, 5, 1024, 500, 80, 257], "epeprepe", 10)
    thr = E_THR if kind == "E" else H_THR
    call = engine.batch_two_view if kind == "E" else engine.batch_two_view_homography
    one = call(xa, xb, offsets, Ks, 200, 4, thr, refine_iterations=10)
    pipe = PairPipeline(device=0)
    try:
        for cp in (1, 4, 100):
            f = pipe.batch_two_view if kind == "E" else pipe.batch_two_view_homography
            r = f(xa, xb, offsets, Ks, 200, 4, thr, chunk_pairs=cp, refine_iterations=10)
            for k in one:
                va, vb = np.asarray(one[k]), np.asarray(r[k])
                assert np.array_equal(_bits(va) if va.dtype == np.float64 else va,
                                      _bits(vb) if vb.dtype == np.float64 else vb), (cp, k)
    finally:
        pipe.close()


def test_fuzz_sweep(engine):
    rng = np.random.default_rng(7)
    bad = []
    for case in range(6):
        bad += fz.one_case(engine, rng, case)
    assert not bad, bad[:10]


# ---- accuracy (direction only; the numbers are in DESIGN.md) ----------------------------------------
@pytest.mark.parametrize("selection", ["min_error", "max_inliers"])
def test_refinement_improves_the_essential_pose(engine, selection):
    er0, er1, et0, et1 = [], [], [], []
    for seed in range(8):
        K, x1, x2, R, t, _ = make_scene(1000, 0.4, 100 + seed, noise_px=0.5)
        kw = dict(sampler="device", seed=seed, engine=engine, on_degenerate="skip", selection=selection)
        # a floor of extra inliers, as in the config-4 timing shape: the bare minimum-error winner explains ~10 points
        a = two_view_arrays(K, x1, x2, E_THR, 300, "rms", 500, **kw)
        b = two_view_arrays(K, x1, x2, E_THR, 300, "rms", 500, refine_iterations=30, **kw)
        er0.append(_rot_deg(a.R, R)), er1.append(_rot_deg(b.R, R))
        et0.append(_dir_deg(a.t, t)), et1.append(_dir_deg(b.t, t))
    assert np.median(er1) < np.median(er0)
    assert np.median(et1) < np.median(et0)


def test_refinement_improves_the_homography_pose(engine):
    er0, er1, en0, en1 = [], [], [], []
    for seed in range(8):
        K, x1, x2, H, _ = make_planar_scene(1000, 0.4, 200 + seed, noise_px=0.5)
        a = two_view_homography_arrays(K, x1, x2, H_THR, 300, sampler="device", seed=seed, engine=engine,
                                       max_iterations=500)
        b = two_view_homography_arrays(K, x1, x2, H_THR, 300, sampler="device", seed=seed, engine=engine,
                                       max_iterations=500, refine_iterations=30)
        # the truth's pose and normal from the exact homography's own decomposition
        d = engine.decompose_homography(H, K)
        c = int(np.argmin([_rot_deg(np.array(d.R[k]).reshape(3, 3), a.R) for k in range(4)]))
        Rt, nt = np.array(d.R[c]).reshape(3, 3), np.array(d.n[c])
        er0.append(_rot_deg(a.R, Rt)), er1.append(_rot_deg(b.R, Rt))
        en0.append(_dir_deg(a.n, nt)), en1.append(_dir_deg(b.n, nt))
    assert np.median(er1) < np.median(er0)
    assert np.median(en1) < np.median(en0)


# ---- the demo ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("model", ["essential", "auto"])
def test_demo_refines_before_the_pose(capsys, model):
    import json

    from apps import sfm as app

    res = app.main(["--synthetic", "0", "--seed", "1", "--refine", "20", "--model", model])
    out = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    rep = out["refinement"]
    assert rep["status"] in ("converged", "max_iterations", "stalled") and rep["num"] >= 8
    assert rep["cost_final"] <= rep["cost_start"]
    assert "rotation_error_deg" in out and np.isfinite(out["rotation_error_deg"])
    assert res.refinement == rep
