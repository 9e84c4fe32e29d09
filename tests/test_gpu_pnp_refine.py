"""The PnP pose refinement (sfm_refine_pnp, csrc/sfm_refine.cuh MODEL_P) on the GPU: off means off, the RANSAC state
is untouched, agreement with scipy's LM from the same start on the same list, the statuses, determinism, exact
rescaling, accuracy, and the refusals."""
import random

import numpy as np
import pytest

from oracle import pnp as opnp
from oracle import pnp_refine as opr
from oracle.refine import rodrigues
from structure_from_motion_b200 import _native
from structure_from_motion_b200.pnp import ransac_pnp_arrays, refine_pnp_arrays
from structure_from_motion_b200.scenes import make_pnp_scene, make_scene, make_three_view_scene
from structure_from_motion_b200.two_view import two_view_arrays

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]


@pytest.fixture(scope="module")
def eng():
    return _native.Engine(0)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _report_tuple(r):
    return (_bits(r.R).tobytes(), _bits(r.t).tobytes(), _bits([r.cost_ransac, r.cost_start, r.cost_final]).tobytes(),
            r.num, r.iterations, r.status, r.rejected)


def _rot_err(Ra, Rb):
    c = (np.trace(Ra @ Rb.T) - 1) / 2
    return float(np.degrees(np.arccos(np.clip(c, -1, 1))))


def _ransac_fields(res):
    return (res.R, res.t, res.best_index, res.error, res.count_extra, res.inlier_indices, res.mask, res.err, res.sample,
            res.num_invalid, res.first_invalid)


def _assert_same_ransac(a, b):
    for u, v in zip(_ransac_fields(a), _ransac_fields(b)):
        u, v = np.asarray(u), np.asarray(v)
        if u.dtype.kind == "f":
            assert _same(u, v)
        else:
            assert np.array_equal(u, v)


# ---- off means off; the RANSAC result and state are untouched -------------------------------------------------------
@pytest.mark.parametrize("sampler", ["reference", "device"])
def test_off_means_off(eng, sampler):
    K, X, x, _, _, _ = make_pnp_scene(800, 0.3, seed=11)
    random.seed(4)
    a = ransac_pnp_arrays(K, X, x, 4.0, 100, "rms", 300, sampler=sampler, seed=3, engine=eng)
    sa = random.getstate()
    random.seed(4)
    b = ransac_pnp_arrays(K, X, x, 4.0, 100, "rms", 300, sampler=sampler, seed=3, engine=eng, refine_iterations=0)
    assert random.getstate() == sa
    _assert_same_ransac(a, b)
    assert a.refinement is None and b.refinement is None
    random.seed(4)
    c = ransac_pnp_arrays(K, X, x, 4.0, 100, "rms", 300, sampler=sampler, seed=3, engine=eng, refine_iterations=20)
    assert random.getstate() == sa
    _assert_same_ransac(a, c)
    assert c.refinement is not None and c.refinement.status in ("converged", "max_iterations")
    assert c.refinement.cost_final <= c.refinement.cost_start


def test_ransac_state_untouched(eng):
    K, x1, x2, _, _, _ = make_scene(600, 0.3, seed=3)
    e2 = _native.Engine(0)
    random.seed(5)
    two_view_arrays(K, x1, x2, 1.5e-6, 10, "rms", 64, engine=e2, refine_iterations=10)
    before_ref = bytes(e2.get_refinement(1))
    Kp, X, x, _, _, _ = make_pnp_scene(700, 0.3, seed=12)
    e2.upload_pnp(X, x, Kp)
    e2.sample_device(7, 256)
    best, Rt, mask, err, cnt, errh = e2.ransac_pnp(4.0, 50.0, "rms", "min_error", want_arrays=True)
    ties0 = e2.near_ties(1e-3, 64)
    m0, v0 = e2.pnp_mask(None, 4.0)
    models0, valid0 = e2.get_pnp_models(0, 256)
    rep, rmask, rerr = e2.refine_pnp(4.0, 20)
    assert rep.status in (0, 1)
    ties1 = e2.near_ties(1e-3, 64)
    m1, v1 = e2.pnp_mask(None, 4.0)
    models1, valid1 = e2.get_pnp_models(0, 256)
    assert np.array_equal(np.asarray(ties0[0]), np.asarray(ties1[0])) and ties0[1] == ties1[1]
    assert np.array_equal(m0, m1) and _same(v0, v1)
    assert _same(models0, models1) and np.array_equal(valid0, valid1)
    assert bytes(e2.get_refinement(1)) == before_ref
    # a later two-view call equals one on a fresh engine
    random.seed(6)
    again = two_view_arrays(K, x1, x2, 1.5e-6, 10, "rms", 64, engine=e2)
    random.seed(6)
    fresh = two_view_arrays(K, x1, x2, 1.5e-6, 10, "rms", 64, engine=_native.Engine(0))
    for a, b in ((again.R, fresh.R), (again.t, fresh.t), (again.points, fresh.points), (again.ransac.E, fresh.ransac.E)):
        assert _same(a, b)


# ---- agreement with scipy's LM from the same start on the same list -------------------------------------------------
def _list_scene(m, n_out, seed):
    """m records with 0.5 px noise about the true pose, then n_out records 300 px off: at threshold 100 px^2 the list
    of a pose near the truth is exactly the first m."""
    K, X, x, R, t, _ = make_pnp_scene(m + n_out, 0.0, seed=seed, noise_px=0.5)
    rng = np.random.default_rng(seed)
    x = x.copy()
    if n_out:
        ang = rng.uniform(0, 2 * np.pi, n_out)
        x[m:] += 300.0 * np.column_stack([np.cos(ang), np.sin(ang)])
    return K, X, x, R, t


@pytest.mark.parametrize("m", [4, 5, 63, 255, 256, 257, 2049, 60000])
def test_matches_scipy_on_the_same_list(eng, m):
    K, X, x, R, t = _list_scene(m, 37, seed=100 + m)
    rng = np.random.default_rng(m)
    R0 = R @ rodrigues(rng.normal(0, 5e-4, 3))
    t0 = t + rng.normal(0, 5e-4, 3)
    lst = opr.inlier_list(np.column_stack([R0, t0]), K, X, x, 100.0)
    assert np.array_equal(lst, np.arange(m))
    rep = refine_pnp_arrays(R0, t0, K, X, x, 100.0, max_iterations=50, engine=eng)
    assert rep.num == m and rep.status == "converged", rep
    Rs, ts, cs = opr.refine(opr.nearest_rotation(R0), t0, K, X[lst], x[lst])
    assert abs(rep.cost_final - cs) <= 1e-9 * cs + 1e-20, (rep.cost_final, cs)
    assert rep.cost_final <= rep.cost_start
    assert abs(rep.cost_start - opr.cost(opr.nearest_rotation(R0), t0, K, X[lst], x[lst])) <= 1e-9 * rep.cost_start
    _, v = opnp.reproj(np.column_stack([R0, t0]), K, X[lst], x[lst], 100.0)
    assert abs(rep.cost_ransac - v.sum()) <= 1e-9 * v.sum()


# ---- statuses -------------------------------------------------------------------------------------------------------
def test_empty_list_is_converged_at_the_projected_start(eng):
    K, X, x, R, t = _list_scene(50, 0, seed=1)
    Rn = R + 1e-4 * np.arange(9).reshape(3, 3)
    rep = refine_pnp_arrays(Rn, t, K, X, x, -1.0, max_iterations=5, engine=eng)
    assert rep.status == "converged" and rep.iterations == 0 and rep.num == 0 and rep.cost_final == 0.0
    assert np.allclose(rep.R, opr.nearest_rotation(Rn), atol=1e-14) and _same(rep.t, t)
    assert not rep.mask.any()


def test_nonfinite_pose_keeps_the_pose(eng):
    K, X, x, R, t = _list_scene(50, 0, seed=2)
    Rb = R.copy()
    Rb[1, 2] = np.nan
    rep = refine_pnp_arrays(Rb, t, K, X, x, 25.0, sample=[0, 1, 2, 3], max_iterations=5, engine=eng)
    assert rep.status == "nonfinite"
    assert _same(rep.R, Rb) and _same(rep.t, t)


def test_reflection_is_projected_onto_a_rotation(eng):
    K, X, x, R, t = _list_scene(300, 0, seed=3)
    U, _, Vt = np.linalg.svd(R)
    M = U @ np.diag([1.0, 1.0, -0.02]) @ Vt  # det < 0; its nearest rotation is R
    rep = refine_pnp_arrays(M, t, K, X, x, 1e9, sample=[0, 1, 2, 3], max_iterations=30, engine=eng)
    assert rep.status in ("converged", "max_iterations")
    assert abs(np.linalg.det(rep.R) - 1) < 1e-12 and np.allclose(rep.R @ rep.R.T, np.eye(3), atol=1e-12)
    assert _rot_err(rep.R, R) < 0.1


def test_noise_free_list_converges_at_the_floor(eng):
    K, X, x, R, t, _ = make_pnp_scene(500, 0.0, seed=4, noise_px=0.0)
    R0 = R @ rodrigues([1e-3, -2e-3, 1e-3])
    rep = refine_pnp_arrays(R0, t + 1e-3, K, X, x, 100.0, max_iterations=50, engine=eng)
    assert rep.status == "converged" and rep.num == 500
    assert rep.cost_final <= 1e-20 * np.sum(x * x)
    assert np.abs(rep.R - R).max() < 1e-9 and np.abs(rep.t - t).max() < 1e-9


def test_proposal_behind_the_camera_is_rejected(eng):
    """A forced record just in front of the camera plane (p2 ~ 1e-9) whose pixel disagrees with its projection: a
    step that would cross the plane costs +inf and is rejected; the reported pose keeps the record in front."""
    K, X, x, R, t = _list_scene(200, 0, seed=5)
    X = X.copy()
    x = x.copy()
    c = -R.T @ t  # camera centre; a point 1e-9 in front of it along the optical axis, 0.5 to the side
    X[7] = c + R.T @ np.array([0.5, 0.0, 1e-9])
    x[7] = [700.0, 500.0]
    R0 = R @ rodrigues([2e-3, 1e-3, -1e-3])
    rep = refine_pnp_arrays(R0, t, K, X, x, 25.0, sample=[7, 8, 9, 10], max_iterations=30, engine=eng)
    assert rep.rejected >= 1 and np.isfinite(rep.cost_final)
    assert (rep.R @ X[7] + rep.t)[2] > 0


# ---- determinism ----------------------------------------------------------------------------------------------------
def test_determinism(eng):
    K, X, x, _, _, _ = make_pnp_scene(5000, 0.4, seed=21)
    random.seed(3)
    a = ransac_pnp_arrays(K, X, x, 4.0, 300, "rms", 500, sampler="device", seed=9, engine=eng, refine_iterations=20)
    random.seed(3)
    b = ransac_pnp_arrays(K, X, x, 4.0, 300, "rms", 500, sampler="device", seed=9, engine=_native.Engine(0),
                          refine_iterations=20)
    assert _report_tuple(a.refinement) == _report_tuple(b.refinement)
    assert np.array_equal(a.refinement.mask, b.refinement.mask) and _same(a.refinement.err, b.refinement.err)
    # Rt = NULL equals the explicit winner with its sample
    eng.upload_pnp(X, x, K)
    eng.sample_device(9, 500)
    best, Rt, _, _, _, _ = eng.ransac_pnp(4.0, 300.0, "rms", "min_error")
    r_null = eng.refine_pnp(4.0, 20)[0]
    r_expl = eng.refine_pnp(4.0, 20, Rt=Rt, sample=np.array(best.sample[:4]))[0]
    assert bytes(r_null) == bytes(r_expl)
    assert bytes(r_null)[:96] == bytes(_bits(np.concatenate([a.refinement.R, a.refinement.t[:, None]], 1)))
    # appended outliers outside the list leave the report bit-identical
    rng = np.random.default_rng(1)
    Xo = np.concatenate([X, rng.uniform(-2, 2, (3000, 3)) + [0, 0, 6]])
    xo = np.concatenate([x, rng.uniform(0, 1280, (3000, 2)) + 5000])
    R0 = a.R
    ra = refine_pnp_arrays(R0, a.t, K, X, x, 4.0, sample=a.sample, engine=eng)
    rb = refine_pnp_arrays(R0, a.t, K, Xo, xo, 4.0, sample=a.sample, engine=eng)
    assert _report_tuple(ra) == _report_tuple(rb)


# ---- exact rescaling -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [-300, -100, -30, -1, 1, 30, 100, 300])
def test_world_scale_is_exact(eng, k):
    K, X, x, R, t = _list_scene(400, 20, seed=31)
    R0 = R @ rodrigues([2e-3, -1e-3, 1e-3])
    base = refine_pnp_arrays(R0, t, K, X, x, 25.0, engine=eng)
    sc = refine_pnp_arrays(R0, np.ldexp(t, k), K, np.ldexp(X, k), x, 25.0, engine=eng)
    assert _same(sc.R, base.R) and _same(sc.t, np.ldexp(base.t, k))
    assert (sc.cost_final, sc.num, sc.iterations, sc.status) == (base.cost_final, base.num, base.iterations, base.status)


@pytest.mark.parametrize("k", [-200, -60, -10, 10, 60, 200])
def test_pixel_scale_is_exact(eng, k):
    K, X, x, R, t = _list_scene(400, 20, seed=32)
    R0 = R @ rodrigues([2e-3, -1e-3, 1e-3])
    base = refine_pnp_arrays(R0, t, K, X, x, 25.0, engine=eng)
    Ks = K.copy()
    Ks[:2] = np.ldexp(Ks[:2], k)
    sc = refine_pnp_arrays(R0, t, Ks, X, np.ldexp(x, k), np.ldexp(25.0, 2 * k), engine=eng)
    assert _same(sc.R, base.R) and _same(sc.t, base.t)
    assert sc.cost_final == np.ldexp(base.cost_final, 2 * k) and sc.num == base.num and sc.iterations == base.iterations


# ---- accuracy -------------------------------------------------------------------------------------------------------
def test_accuracy_halves_the_median_errors(eng):
    off_r, off_t, on_r, on_t = [], [], [], []
    for s in range(8):
        K, X, x, R, t, _ = make_pnp_scene(1000, 0.4, s, noise_px=0.5)
        random.seed(s)
        res = ransac_pnp_arrays(K, X, x, 4.0, 300, "rms", 500, engine=eng, refine_iterations=20)
        off_r.append(_rot_err(res.R, R))
        off_t.append(np.linalg.norm(res.t - t))
        on_r.append(_rot_err(res.refinement.R, R))
        on_t.append(np.linalg.norm(res.refinement.t - t))
    print("median rotation error off / on (deg):", np.median(off_r), np.median(on_r))
    print("median translation error off / on:", np.median(off_t), np.median(on_t))
    assert np.median(on_r) <= 0.5 * np.median(off_r)
    assert np.median(on_t) <= 0.5 * np.median(off_t)


def test_three_view_composition_refined(eng):
    K, x1, x2, x3, (R2, t2), (R3, t3), X = make_three_view_scene(3000, 0.2, seed=61)
    out = {}
    for n_it in (0, 20):
        random.seed(1)
        tv = two_view_arrays(K, x1, x2, 1e-5, 1500, "rms", 200, engine=eng, refine_iterations=n_it)
        idx = tv.inlier_indices[tv.passing]
        random.seed(2)
        res = ransac_pnp_arrays(K, tv.points[tv.passing], x3[idx], 4.0, len(idx) // 2, "rms", 200, engine=eng,
                                refine_iterations=n_it)
        R = res.refinement.R if n_it else res.R
        out[n_it] = np.abs(R - R3).max()
    print("three-view R3 error, refinement off / on:", out[0], out[20])
    assert out[20] <= out[0]


# ---- refusals -------------------------------------------------------------------------------------------------------
def test_refusals(eng):
    K, X, x, R, t, _ = make_pnp_scene(50, 0.0, seed=1)
    Rt = np.column_stack([R, t])
    fresh = _native.Engine(0)
    with pytest.raises(_native.NativeError):
        fresh.refine_pnp(4.0, 5, Rt=Rt)  # no PnP records
    fresh.upload_pnp(X, x, K)
    with pytest.raises(_native.NativeError):
        fresh.refine_pnp(4.0, 5)  # no winner
    with pytest.raises(_native.NativeError):
        fresh.refine_pnp(4.0, 0, Rt=Rt)
    with pytest.raises(_native.NativeError):
        fresh.refine_pnp(np.nan, 5, Rt=Rt)
    with pytest.raises(_native.NativeError):
        fresh.refine_pnp(4.0, 5, Rt=Rt, sample=[0, 1, 2, 50])
    with pytest.raises(_native.NativeError):
        fresh.refine_pnp(4.0, 5, Rt=Rt, sample=[-1, 1, 2, 3])
    with pytest.raises(ValueError):
        ransac_pnp_arrays(K, X, x, 4.0, engine=eng, refine_iterations=-1)
    with pytest.raises(ValueError):
        refine_pnp_arrays(R, t, K, X, x, 4.0, max_iterations=0, engine=eng)
