"""The PnP path at its edges on the GPU: random poses and cameras against the exact P3P, bit-exact equivariance under
power-of-two world and pixel scales, world and pixel scales beyond the float64 range of the plain formulas, skewed
anisotropic cameras, near-degenerate samples, and records whose reprojection terms overflow."""
import random

import numpy as np
import pytest

from oracle import creproj
from oracle import pnp as op
from structure_from_motion_b200 import _native
from structure_from_motion_b200.pnp import ransac_pnp_arrays, reprojection_error_arrays
from structure_from_motion_b200.scenes import make_pnp_samples, make_pnp_scene

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]

PAIRS = (("sum", "min_error"), ("square", "min_error"), ("mean", "min_error"), ("rms", "min_error"),
         ("rms", "max_inliers"), ("sum", "msac"))
# a skewed, anisotropic camera with an off-centre principal point
K_SKEW = np.array([[912.5, 3.75, 598.25], [0.0, 871.0, 517.5], [0.0, 0.0, 1.0]])


@pytest.fixture(scope="module")
def eng():
    return _native.Engine(0)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _fit_batch(eng, K, Xs, xs):
    """Device fits of samples (Xs [m,4,3], xs [m,4,2]) under one K: records 4 i .. 4 i + 3 are sample i."""
    m = len(Xs)
    eng.upload_pnp(np.concatenate(Xs).reshape(-1, 3), np.concatenate(xs).reshape(-1, 2), K)
    base = 4 * np.arange(m, dtype=np.int32)[:, None] + np.arange(4, dtype=np.int32)
    eng.set_table(np.concatenate([base, base], axis=1))
    Rt, valid = eng.fit_pnp()
    return Rt, valid.astype(bool)


def _in_band(info):
    return info["gap"] < 1e-6 or abs(info["collinear"] / op.COLLINEAR - 1) < 1e-3


def _tol(ref, y):
    """The fitter's tolerance against the 50-digit solve: 1e-7 (1 + max |ref|), times 1e-2 / theta for a sample whose
    smallest bearing angle theta is below 1e-2 rad.  Why: the bearings enter the distance equations only through
    their cosines; a rounding of ~1e-16 in a cosine moves the angle between two bearings by ~1e-16 / sin(theta), and
    the depths - hence R and t - move in proportion to that relative change of theta.  Lambda Twist's cubic, eigen
    step and Gauss-Newton polish then keep the float64 solve within ~1e-9 relative of the exact one at theta ~ 1
    (the existing 1e-7 bound on make_pnp_scene leaves that margin), so 1e-7 / theta keeps a factor of ~100 above the
    rounding for narrow cameras (f = 20 000) and tight spreads (1e-3 of the depth)."""
    return 1e-7 * (1.0 + np.abs(ref).max()) * max(1.0, 1e-2 / max(op.bearing_angles(y), 1e-300))


def _compare_fits(Rt, valid, samples, truth_noise_free):
    """(band, branches, worst): compares every device fit with fit_pnp_exact; failures are collected, not raised."""
    band, branches, fails, worst = 0, {0: 0, 1: 0, 3: 0}, [], 0.0
    for i, (K, X, x, R, t) in enumerate(samples):
        ref, info = op.fit_pnp_exact(K, X, x)
        y = op.bearings(K, x[:3])
        branches[op.cubic_branch(y, X[:3])] += 1
        if _in_band(info):
            band += 1
            continue
        if (ref is not None) != bool(valid[i]):
            fails.append((i, "validity", ref is not None, info))
            continue
        if ref is None:
            continue
        tol = _tol(ref, y)
        err = np.abs(Rt[i] - ref).max()
        worst = max(worst, err / tol)
        if err > tol:
            fails.append((i, "pose", err, tol, info))
        if truth_noise_free:
            e_true = np.abs(ref - np.column_stack([R, t])).max()
            if e_true > tol:
                fails.append((i, "truth", e_true, tol, info))
    return band, branches, fails, worst


@pytest.mark.parametrize("noise", [0.0, 1.0])
def test_random_geometry_against_exact(eng, noise):
    """1 000 random samples per noise level (make_pnp_samples: uniform rotations including cameras along every world
    axis and near-180-degree rotations, depths 0.5-100, spreads 1e-3 to 10 times the depth, f from 150 to 20 000).
    Outside the ambiguity band of test_fitter_against_exact_p3p, validity equals fit_pnp_exact's and [R|t] agrees to
    _tol; noise-free samples also agree with the true pose to _tol.  At most 2 % fall in the band, and both the one-
    and the three-root branch of the cubic (oracle.pnp.cubic_branch) are reached."""
    samples = make_pnp_samples(1000, seed=100 + int(noise), noise_px=noise)
    by_k = {}
    for i, s in enumerate(samples):
        by_k.setdefault(s[0].tobytes(), []).append(i)
    Rt = np.zeros((len(samples), 3, 4))
    valid = np.zeros(len(samples), dtype=bool)
    for idx in by_k.values():  # one upload per camera
        K = samples[idx[0]][0]
        r, v = _fit_batch(eng, K, [samples[i][1] for i in idx], [samples[i][2] for i in idx])
        Rt[idx], valid[idx] = r, v
    band, branches, fails, worst = _compare_fits(Rt, valid, samples, noise == 0.0)
    print(f"noise {noise}: band {band}, cubic branches {branches}, worst error / tolerance {worst:.3g}")
    assert not fails, fails[:10]
    assert band <= 20
    assert branches[1] > 0 and branches[3] > 0


def _scene_table(n, h, seed, K=None):
    K_, X, x, R, t, _ = make_pnp_scene(n, 0.3, seed=seed, noise_px=1.0, K=K)
    rng = np.random.default_rng(seed)
    table = np.stack([rng.choice(n - 8 if n >= 64 else n, 8, replace=False) for _ in range(h)]).astype(np.int32)
    return K_, X, x, R, t, table


def _run(eng, K, X, x, table, thr, agg, sel):
    eng.upload_pnp(X, x, K)
    eng.set_table(table)
    best, Rt_w, mask, err, cnt, err_h = eng.ransac_pnp(thr, 0.0, agg, sel, want_arrays=True)
    models, valid = eng.get_pnp_models()
    return dict(best=int(best.index), mask=np.asarray(mask).astype(bool), err=np.asarray(err), cnt=np.asarray(cnt),
                err_h=np.asarray(err_h), models=models, valid=np.asarray(valid).astype(bool))


@pytest.mark.parametrize("k", [-100, -40, -7, 0, 9, 40, 100])
def test_world_scale_bit_exact(eng, k):
    """World x 2^k, table, K and pixels unchanged: every step of the fitter is homogeneous in the world scale and
    every rounding commutes with a power of two, so R is bit-identical and t is bit-identical to 2^k t; the scorer's
    F and W scale by 4^k together, so best index, counts, mask, values and err_h are bit-identical for every
    aggregation and selection."""
    K, X, x, R, t, table = _scene_table(2049, 129, seed=3)
    s = 2.0 ** k
    for agg, sel in PAIRS:
        a = _run(eng, K, X, x, table, 4.0, agg, sel)
        b = _run(eng, K, X * s, x, table, 4.0, agg, sel)
        assert np.array_equal(a["valid"], b["valid"])
        assert np.array_equal(_bits(a["models"][:, :, :3]), _bits(b["models"][:, :, :3]))
        assert np.array_equal(_bits(a["models"][:, :, 3] * s), _bits(b["models"][:, :, 3]))
        assert a["best"] == b["best"] and a["best"] >= 0
        assert np.array_equal(a["cnt"], b["cnt"]) and np.array_equal(a["mask"], b["mask"])
        assert np.array_equal(_bits(a["err"]), _bits(b["err"])) and np.array_equal(_bits(a["err_h"]), _bits(b["err_h"]))


@pytest.mark.parametrize("k", [-20, -3, 5, 20])
def test_pixel_scale_bit_exact(eng, k):
    """Pixels and the first two rows of K x 2^k, thr x 4^k: the bearings are bit-identical (so are the fits), p0 and
    p1 scale by 2^k, F by 4^k and W not at all, so decisions are identical and values exactly x 4^k; the fixed-point
    exponent moves by 2k, so the chunks are identical and err_h is exactly x 4^k (sum, mean, rms) or x 16^k
    (square)."""
    K, X, x, R, t, table = _scene_table(2049, 129, seed=4)
    s = 2.0 ** k
    Ks = K.copy()
    Ks[:2] *= s
    err_scale = {"sum": 4.0 ** k, "mean": 4.0 ** k, "rms": 4.0 ** k, "square": 16.0 ** k}
    for agg, sel in PAIRS:
        a = _run(eng, K, X, x, table, 4.0, agg, sel)
        b = _run(eng, Ks, X, x * s, table, 4.0 * 4.0 ** k, agg, sel)
        assert np.array_equal(a["valid"], b["valid"])
        assert np.array_equal(_bits(a["models"]), _bits(b["models"]))
        assert a["best"] == b["best"] and a["best"] >= 0
        assert np.array_equal(a["cnt"], b["cnt"]) and np.array_equal(a["mask"], b["mask"])
        assert np.array_equal(_bits(a["err"] * 4.0 ** k), _bits(b["err"]))
        if sel == "min_error":
            assert np.array_equal(_bits(a["err_h"] * err_scale[agg]), _bits(b["err_h"]))


def _reprojects(Rt, K, X, x):
    """The angle between R X_i + t and the exact bearing of x_i, for the three sample points (radians, inf for a point
    not in front of the camera)."""
    y = op.bearings(K, x[:3])
    c = X[:3] @ Rt[:, :3].T + Rt[:, 3]
    # a point within ~1e-6 rad of the camera plane: the pose's rounding decides the sign of its depth, not the solve
    edge = y[:, 2] < 1e-6
    # scale each camera point by a power of two first: at world scales near the float64 limits |c|^2 overflows
    c = c / np.exp2(np.floor(np.log2(np.abs(c).max(axis=1, keepdims=True))))
    cn = c / np.linalg.norm(c, axis=1, keepdims=True)
    ang = np.arctan2(np.linalg.norm(np.cross(cn, y), axis=1), np.sum(cn * y, axis=1))
    return np.where((c[:, 2] > 0) | edge, ang, np.inf)


@pytest.mark.parametrize("k", [-300, -160, -130, 130, 160, 300])
def test_world_scale_beyond_range(eng, k):
    """World x 2^k beyond the range of the unscaled formulas (eigvec3's degree-8 norm overflows near 2^+-128, the
    cubic's degree-6 coefficients near 2^+-170).  48 noise-free samples of make_pnp_scene: validity equals
    fit_pnp_exact's; a valid pose is finite, puts the three sample points within 1e-9 rad of their exact bearings,
    and - the fitter being equivariant - has R bit-identical to the unscaled fit's and t = 2^k times its t."""
    K, X, x, R, t, _ = make_pnp_scene(400, 0.0, seed=9, noise_px=0.0)
    rng = np.random.default_rng(9)
    rows = [rng.choice(len(X), 4, replace=False) for _ in range(48)]
    s = 2.0 ** k
    Rt0, v0 = _fit_batch(eng, K, [X[r] for r in rows], [x[r] for r in rows])
    Rt1, v1 = _fit_batch(eng, K, [X[r] * s for r in rows], [x[r] for r in rows])
    for i, r in enumerate(rows):
        ref, info = op.fit_pnp_exact(K, X[r] * s, x[r])
        if _in_band(info):
            continue
        assert bool(v1[i]) == (ref is not None), (i, info)
        if v1[i]:
            assert np.isfinite(Rt1[i]).all()
            assert _reprojects(Rt1[i], K, X[r] * s, x[r]).max() <= 1e-9, i
            assert np.array_equal(_bits(Rt1[i][:, :3]), _bits(Rt0[i][:, :3]))
            assert np.array_equal(_bits(Rt1[i][:, 3]), _bits(Rt0[i][:, 3] * s))
    assert v1.sum() >= 40


def test_pixels_beyond_range(eng):
    """One sample column with a pixel near 1e160 (a world point 1e-157 of a unit in front of the camera plane):
    xn^2 overflows, and the bearing must still be the unit vector the oracle computes.  Validity equals
    fit_pnp_exact's in every column, a valid pose is finite and puts the three sample points within 1e-9 rad of
    their exact bearings."""
    K, X, _, _, _, _ = make_pnp_scene(50, 0.0, seed=12, noise_px=0.0)
    x = (X[:, :2] / X[:, 2:]) @ K[:2, :2].T + K[:2, 2]  # the world frame is the camera's: x_cam = X exactly
    Xs, xs = [], []
    for col in range(4):
        for j in range(6):
            rows = np.arange(4 * j, 4 * j + 4)
            Xj, xj = X[rows].copy(), x[rows].copy()
            Xj[col] = [1.0 + 0.1 * j, 0.5 - 0.2 * j, 1e-157]
            xj[col] = K[:2, :2] @ (Xj[col, :2] / Xj[col, 2]) + K[:2, 2]
            assert np.abs(xj[col]).max() > 1e159
            Xs.append(Xj)
            xs.append(xj)
    Rt, valid = _fit_batch(eng, K, Xs, xs)
    nvalid = 0
    for i, (Xj, xj) in enumerate(zip(Xs, xs)):
        ref, info = op.fit_pnp_exact(K, Xj, xj)
        if _in_band(info):
            continue
        assert bool(valid[i]) == (ref is not None), (i, info)
        if valid[i]:
            nvalid += 1
            assert np.isfinite(Rt[i]).all()
            assert _reprojects(Rt[i], K, Xj, xj).max() <= 1e-9, i
    assert nvalid >= 6


def test_skewed_camera_fitter(eng):
    """The comparison of test_random_geometry_against_exact (300 samples, 1 px noise and none) under K_SKEW: the
    bearings subtract the skew's share of y before dividing by fx."""
    for noise in (0.0, 1.0):
        samples = make_pnp_samples(150, seed=200 + int(noise), noise_px=noise, K=K_SKEW)
        Rt, valid = _fit_batch(eng, K_SKEW, [s[1] for s in samples], [s[2] for s in samples])
        band, branches, fails, worst = _compare_fits(Rt, valid, samples, noise == 0.0)
        print(f"skewed K, noise {noise}: band {band}, branches {branches}, worst error / tolerance {worst:.3g}")
        assert not fails, fails[:10]
        assert band <= 6


@pytest.mark.parametrize("n", [63, 64, 65, 2049])
def test_skewed_camera_scorer_bit_identical(eng, n):
    """Under K_SKEW (pnp_projection pins K[r][1] into its FMA chain), for hypothesis counts 63, 64, 65 and every
    aggregation / selection pair: counts, the winner's mask and values bit-identical to reproj_exact.c, err_h to
    1e-12 relative, the winner among the oracle's best; and reprojection_error_arrays bit for bit."""
    K, X, x, R, t, _ = make_pnp_scene(n, 0.3, seed=n + 7, noise_px=1.0, K=K_SKEW)
    rng = np.random.default_rng(n)
    for h in (63, 64, 65):
        table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
        for agg, sel in PAIRS:
            r = _run(eng, K, X, x, table, 4.0, agg, sel)
            exp = op.expected_selection(r["models"], r["valid"], K, X, x, 4.0, table, agg, sel)
            assert np.array_equal(r["cnt"], np.where(r["valid"], exp["count_extra"], -1)), (h, agg, sel)
            fin = np.isfinite(exp["err"])
            assert np.array_equal(fin, np.isfinite(r["err_h"]))
            assert np.all(np.abs(r["err_h"][fin] - exp["err"][fin]) <= 1e-12 * np.abs(exp["err"][fin]) + 1e-300)
            assert r["best"] in exp["winners"].tolist()
            if r["best"] >= 0:
                m_c, v_c = creproj.reproj_exact_many(r["models"][r["best"]], K, X, x, 4.0)
                assert np.array_equal(m_c, r["mask"]) and np.array_equal(_bits(v_c), _bits(r["err"]))
    m_g, v_g = reprojection_error_arrays(R, t, K, X, x, 4.0, engine=eng)
    m_c, v_c = creproj.reproj_exact_many(np.column_stack([R, t]), K, X, x, 4.0)
    assert np.array_equal(m_g, m_c) and np.array_equal(_bits(v_g), _bits(v_c))


def _collinear_sample(rng, sine, K, R, t):
    """Four noise-free records whose first three world points have the collinearity sine ``sine`` at X0 (to ~1e-10
    relative), in front of the camera (R, t)."""
    X0 = R.T @ (np.array([rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(5, 7)]) - t)
    d = rng.normal(size=3)
    d /= np.linalg.norm(d)
    nrm = np.cross(d, rng.normal(size=3))
    nrm /= np.linalg.norm(nrm)
    X1 = X0 - rng.uniform(0.5, 1.5) * d
    X2 = X0 - rng.uniform(0.5, 1.5) * (np.sqrt(1 - sine * sine) * d + sine * nrm)
    X3 = R.T @ (np.array([rng.uniform(-1, 1), rng.uniform(-1, 1), rng.uniform(4, 8)]) - t)
    Xs = np.stack([X0, X1, X2, X3])
    p = (K @ (Xs @ R.T + t).T).T
    return Xs, p[:, :2] / p[:, 2:]


def _collinear_tol(ref, y, sine):
    """_tol times (1e-2 / sine)^2 below sine 1e-2.  A near-collinear world triple is
    conditioned twice by its sine: the three distance equations become dependent (their Jacobian in the depths is
    singular for collinear points), so the depths are good to ~1 / sine of their rounding, and R = [d1 d2 d1 x d2]
    [w1 w2 w1 x w2]^-1 divides by the small cross products once more."""
    return _tol(ref, y) * max(1.0, 1e-2 / sine) ** 2


@pytest.mark.parametrize("side", ["below", "above"])
def test_collinearity_boundary(eng, side):
    """Triples at collinearity sine 1e-6 (1 +- 1e-6).  The band is narrowed from the 0.1 % of the other fitter tests
    to 1e-6 relative: the test compares |w1 x w2|^2 with 1e-12 |w1|^2 |w2|^2, and the cross product cancels terms of
    size |w1| |w2| to leave |w1| |w2| sin, so its rounding is ~1e-16 / 1e-6 = 1e-10 relative to the sine -
    FMA-contracted or not (the device's dot3 and cross3 may be), which is why the exact boundary is not pinned.  1e-6
    leaves a factor of 1e4 over that.  Below: invalid on the device and in the oracle.  Above: the device either
    reports the sample invalid (at this sine its R is not orthonormal to 1e-6) or returns the oracle's pose to
    _collinear_tol.  The oracle itself may find no pose here: its two roots nearly coincide, and it drops roots whose
    imaginary part it cannot resolve."""
    K, _, _, R, t, _ = make_pnp_scene(10, 0.0, seed=1, noise_px=0.0)
    rng = np.random.default_rng(13)
    Xs, xs = [], []
    for j in range(16):
        sine = op.COLLINEAR * (1 + (1e-6 if side == "above" else -1e-6))
        Xj, xj = _collinear_sample(rng, sine, K, R, t)
        Xs.append(Xj)
        xs.append(xj)
        assert (op.collinear_ratio(Xj[:3]) > op.COLLINEAR) == (side == "above")
    Rt, valid = _fit_batch(eng, K, Xs, xs)
    for i in range(len(Xs)):
        ref, _ = op.fit_pnp_exact(K, Xs[i], xs[i])
        if side == "below":
            assert ref is None and not valid[i], i
        elif valid[i]:
            assert ref is not None, i
            tol = _collinear_tol(ref, op.bearings(K, xs[i][:3]), op.COLLINEAR)
            assert np.abs(Rt[i] - ref).max() <= tol, (i, np.abs(Rt[i] - ref).max(), tol)


# the fewest valid fits per decade of sine, of 48 samples (measured on one B200: 2, 40 and 47)
NEAR_COLLINEAR_MIN_VALID = {-5: 1, -4: 33, -3: 45}


@pytest.mark.parametrize("decade", [-5, -4, -3])
def test_near_collinear_valid(eng, decade):
    """Near-collinear triples (48 per decade of sine from 1e-5 to 1e-2, noise-free).  Every fit the device reports
    valid agrees with fit_pnp_exact to _collinear_tol: a wrong pose returned as valid fails.  A sample the oracle
    solves may be invalid on the device only by its orthonormality rule, which drops the samples float64 cannot
    solve; at least NEAR_COLLINEAR_MIN_VALID[decade] stay valid, and invalid samples are never reported valid."""
    K, _, _, R, t, _ = make_pnp_scene(10, 0.0, seed=2, noise_px=0.0)
    rng = np.random.default_rng(14 + decade)
    Xs, xs, sines = [], [], []
    for j in range(48):
        sine = 10.0 ** rng.uniform(decade, decade + 1)
        Xj, xj = _collinear_sample(rng, sine, K, R, t)
        Xs.append(Xj)
        xs.append(xj)
        sines.append(sine)
    Rt, valid = _fit_batch(eng, K, Xs, xs)
    checked = 0
    for i in range(len(Xs)):
        ref, info = op.fit_pnp_exact(K, Xs[i], xs[i])
        if info["gap"] < 1e-6 or not valid[i]:
            continue
        assert ref is not None, (i, info)
        tol = _collinear_tol(ref, op.bearings(K, xs[i][:3]), sines[i])
        assert np.abs(Rt[i] - ref).max() <= tol, (i, sines[i], np.abs(Rt[i] - ref).max(), tol)
        R_ = Rt[i][:, :3]
        assert np.abs(R_ @ R_.T - np.eye(3)).max() <= 1e-6
        checked += 1
    print(f"sine 1e{decade}: {checked} valid of 48")
    assert checked >= NEAR_COLLINEAR_MIN_VALID[decade]


def test_repeated_and_coincident_points(eng):
    """A table row repeating an index among columns 0-2 is invalid (two coincident world points); a fourth column
    equal to one of the first three gives a valid fit (which solution is chosen is not checked)."""
    K, X, x, R, t, _ = make_pnp_scene(64, 0.0, seed=5, noise_px=0.5)
    rows = []
    for a, b, c in ((0, 0, 1), (2, 3, 2), (4, 5, 5), (6, 6, 6)):
        rows.append([a, b, c, 7])
    valid_rows = [[8, 9, 10, 8], [11, 12, 13, 12], [14, 15, 16, 16]]
    table = np.array(rows + valid_rows, dtype=np.int32)
    eng.upload_pnp(X, x, K)
    eng.set_table(np.concatenate([table, table], axis=1))
    _, valid = eng.fit_pnp()
    assert valid.astype(bool).tolist() == [False] * 4 + [True] * 3
    for row in valid_rows:
        assert op.fit_pnp_exact(K, X[row], x[row])[0] is not None


def test_four_candidates(eng):
    """Samples with four positive-depth solutions (rejection-sampled from make_pnp_samples until the oracle reports
    ncand == 4 with a point-3 gap >= 1e-3, 1 px noise) match the oracle's pick to _tol."""
    found = []
    for seed in range(300, 340):
        for s in make_pnp_samples(40, seed=seed, noise_px=1.0):
            ref, info = op.fit_pnp_exact(s[0], s[1], s[2])
            if ref is not None and info["ncand"] == 4 and info["gap"] >= 1e-3:
                found.append((s, ref))
        if len(found) >= 24:
            break
    assert len(found) >= 3
    for s, ref in found:
        Rt, valid = _fit_batch(eng, s[0], [s[1]], [s[2]])
        assert valid[0]
        assert np.abs(Rt[0] - ref).max() <= _tol(ref, op.bearings(s[0], s[2][:3]))


def _overflow_scene(seed):
    """make_pnp_scene(2049) with its last 8 records (never a sample) replaced by finite records at |X| = 1e150, 1e152,
    1e160 and 1e300: four on the true ray of a scene pixel (F finite or inf, W finite or inf) and four off every ray
    in front of the camera (F and W inf from 1e160 on)."""
    K, X, x, R, t, out = make_pnp_scene(2049, 0.3, seed=seed)
    C = -R.T @ t
    for j, s in enumerate((1e150, 1e152, 1e160, 1e300)):
        d = R.T @ np.linalg.solve(K, np.array([x[j, 0], x[j, 1], 1.0]))
        X[-1 - j] = C + s * d / np.linalg.norm(d)  # on the ray of x[-1 - j] (the pixel set below)
        x[-1 - j] = x[j]
        X[-5 - j] = C + s * (R.T @ np.array([0.3, -0.2, 1.0]))  # pixel of a different ray
        x[-5 - j] = x[j]
    return K, X, x, R, t


def test_overflowing_records_bit_identical(eng):
    """The overflow scene, 129 hypotheses of a table over the first 2 041 records, every aggregation / selection pair
    at thr 4 and 1e100: counts, mask, values and err_h as reproj_exact.c computes them, and no inlier - of any
    hypothesis's mask, or of the winner's - carries a non-finite value."""
    K, X, x, R, t = _overflow_scene(17)
    rng = np.random.default_rng(17)
    table = np.stack([rng.choice(2041, 8, replace=False) for _ in range(129)]).astype(np.int32)
    for thr in (4.0, 1e100):
        for agg, sel in PAIRS:
            r = _run(eng, K, X, x, table, thr, agg, sel)
            exp = op.expected_selection(r["models"], r["valid"], K, X, x, thr, table, agg, sel)
            assert np.array_equal(r["cnt"], np.where(r["valid"], exp["count_extra"], -1)), (agg, sel, thr)
            fin = np.isfinite(exp["err"])
            assert np.array_equal(fin, np.isfinite(r["err_h"])), (agg, sel, thr)
            assert np.all(np.abs(r["err_h"][fin] - exp["err"][fin]) <= 1e-12 * np.abs(exp["err"][fin]) + 1e-300)
            assert r["best"] in exp["winners"].tolist() and r["best"] >= 0
            m_c, v_c = creproj.reproj_exact_many(r["models"][r["best"]], K, X, x, thr)
            assert np.array_equal(m_c, r["mask"]) and np.array_equal(_bits(v_c), _bits(r["err"]))
            assert np.isfinite(r["err"][r["mask"]]).all()
    for i in np.flatnonzero(r["valid"]):
        m, v = creproj.reproj_exact_many(r["models"][i], K, X, x, 1e100)
        assert np.isfinite(v[m]).all(), i


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_overflowing_records_accuracy(eng, seed):
    """RANSAC on the overflow scene (reference sampler seeded with ``seed``, 200 iterations, thr 4 px^2, RMS) finds
    the true pose within test_accuracy's bounds (5e-3 on R, 3e-2 on t) and no inlier carries a non-finite error."""
    K, X, x, R, t = _overflow_scene(seed)
    random.seed(seed)
    res = ransac_pnp_arrays(K, X, x, 4.0, 0, "rms", 200, engine=eng)
    assert np.abs(res.R - R).max() < 5e-3
    assert np.abs(res.t - t).max() < 3e-2
    assert np.isfinite(res.err[res.mask]).all()
