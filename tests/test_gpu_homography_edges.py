"""GPU checks of the homography paths at their edges: the fixed-point range of k_score_homography (thresholds at and
just below powers of two, the exponent clamp, the range where K2 is skipped), correspondences whose transfer error is
the threshold to within a few ulps, the decomposition at repeated singular values, close planes, extreme scales of H
and the rotation-tolerance boundary, one camera K^-1 for the decomposition, the vote and the triangulation (skewed K;
non-upper-triangular or scaled K refused), F built from the E path's camera in k_score_models, the three upload
layouts of the one-call two-view homography, and the randomised sweep of tools/fuzz_homography.py."""
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import cselect, ctransfer
from oracle import homography as oh
from oracle import homography_pose as hp
from oracle import model_select as ms
from structure_from_motion_b200 import _native
from structure_from_motion_b200 import homography as hg
from structure_from_motion_b200.scenes import euler_xyz_intrinsic, make_planar_scene, make_scene

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

AGGS = ["sum", "square", "mean", "rms"]
R_TRUE = euler_xyz_intrinsic(2.0, -8.0, 1.0)
T_TRUE = np.array([-1.0, 0.05, 0.1]) / np.linalg.norm([-1.0, 0.05, 0.1])
N_TRUE = np.array([0.15, -0.1, 1.0]) / np.linalg.norm([0.15, -0.1, 1.0])


def _cols(x1, x2, idx=slice(None)):
    return x1[idx, 0], x1[idx, 1], x2[idx, 0], x2[idx, 1]


def _table(n, h, seed):
    rng = np.random.default_rng(seed)
    return np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)


def _check_estimate(engine, x1, x2, table, thr, agg, sel, min_extra=0.0):
    """One ransac_homography call against oracle.homography.expected_selection on the GPU's own models: counts bit
    for bit, the error of every hypothesis within 1e-12 (finite exactly where the oracle's is), the winner among the
    oracle's best, and the winner's mask and errors bit for bit."""
    engine.set_table(table)
    best, mask, err, cnt, err_h = engine.ransac_homography(thr, min_extra, agg, sel, want_arrays=True)
    Hs, valid = engine.get_models()
    ref = oh.expected_selection(Hs, valid, *_cols(x1, x2), thr, table, agg, sel, min_extra)
    assert np.array_equal(np.where(valid, cnt, -1), np.where(valid, ref["count_extra"], -1)), (thr, agg, sel)
    fin = np.isfinite(ref["err"])
    assert np.array_equal(np.isfinite(err_h), fin), (thr, agg, sel)
    assert np.all(np.abs(err_h[fin] - ref["err"][fin]) <= 1e-12 * np.abs(ref["err"][fin])), (thr, agg, sel)
    assert int(best.index) in ref["winners"], (thr, agg, sel, best.index, ref["winners"][:4])
    if best.index >= 0:
        m_ref, v_ref = ctransfer.transfer_exact_many(Hs[best.index], *_cols(x1, x2), thr)
        assert np.array_equal(mask.astype(bool), m_ref) and np.array_equal(err.view(np.int64), v_ref.view(np.int64))
    return Hs, valid


# ---- fixed-point range of k_score_homography -------------------------------------------------------------------
FIXED_POINT_THRESHOLDS = [v for k in (-3, 2, 4, 10) for v in (float(np.nextafter(2.0 ** k, 0.0)), 2.0 ** k)]
FIXED_POINT_THRESHOLDS += [1e-130, 1e100, float(np.nextafter(1e100, np.inf))]


@pytest.mark.parametrize("thr", FIXED_POINT_THRESHOLDS)
def test_fixed_point_range(engine, thr):
    # 2 600 correspondences: items of 2 048 records and a partial one; 200 hypotheses: a padded last group
    _, x1, x2, _, _ = make_planar_scene(2600, 0.3, seed=21)
    table = _table(len(x1), 200, 22)
    engine.upload_pairs(x1, x2, np.eye(3))
    for agg in AGGS:
        _check_estimate(engine, x1, x2, table, thr, agg, "min_error")
    _check_estimate(engine, x1, x2, table, thr, "rms", "msac")
    _check_estimate(engine, x1, x2, table, thr, "sum", "max_inliers", min_extra=3.0)


# ---- correspondences on the threshold --------------------------------------------------------------------------
def _on_threshold(H, x1, x2, thr, rows):
    """Image-B points of ``rows`` moved along a fixed direction away from pi(H a) until their transfer error under H
    (the C oracle's value) is as close to thr as the pixel grid allows: bisection on the displacement down to adjacent
    doubles."""
    x2 = x2.copy()
    a = np.column_stack([x1[rows], np.ones(len(rows))]) @ H.T
    base = a[:, :2] / a[:, 2:]
    ang = np.linspace(0.0, 2.0 * np.pi, len(rows), endpoint=False)
    u = np.column_stack([np.cos(ang), np.sin(ang)])

    def value(s):
        p = base + s[:, None] * u
        return ctransfer.transfer_exact_many(H, x1[rows, 0], x1[rows, 1], p[:, 0], p[:, 1], thr)[1]

    lo, hi = np.zeros(len(rows)), np.full(len(rows), 2.0 * np.sqrt(thr))
    assert np.all(value(hi) > thr)
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        live = (mid > lo) & (mid < hi)
        if not live.any():
            break
        above = value(mid) > thr
        hi = np.where(live & above, mid, hi)
        lo = np.where(live & ~above, mid, lo)
    vlo, vhi = value(lo), value(hi)
    s = np.where(np.abs(vlo - thr) <= np.abs(vhi - thr), lo, hi)
    x2[rows] = base + s[:, None] * u
    return x2


@pytest.mark.parametrize("thr", [float(np.nextafter(16.0, 0.0)), 16.0])
def test_correspondences_on_the_threshold(engine, thr):
    _, x1, x2, _, _ = make_planar_scene(6000, 0.0, seed=23, noise_px=0.0)
    table = _table(len(x1), 64, 24)
    engine.upload_pairs(x1, x2, np.eye(3))
    engine.set_table(table)
    engine.ransac_homography(thr, 0.0, "rms", "min_error")
    H_fit = engine.get_models(0, 1)[0][0].copy()
    rows = np.setdiff1d(np.arange(len(x1)), table[0, :4])
    x2t = _on_threshold(H_fit, x1, x2, thr, rows)
    m, v = ctransfer.transfer_exact_many(H_fit, *_cols(x1, x2t, rows), thr)
    # a pixel coordinate near 1 000 moves in steps of 1e-13 px, which moves the error by ~1e-12 px^2: a few hundred
    # ulps of 16 is as close as a displaced point can get
    assert np.max(np.abs(v - thr)) <= 2048 * np.spacing(thr) and len(rows) >= 4096
    assert (v > thr).any() and (v <= thr).any()
    assert (m & (v > thr)).any() or (~m & (v <= thr)).any()  # where the division-free decision and the value disagree
    engine.upload_pairs(x1, x2t, np.eye(3))
    for agg in AGGS:
        Hs, _ = _check_estimate(engine, x1, x2t, table, thr, agg, "min_error")
        assert np.array_equal(Hs[0].view(np.int64), H_fit.view(np.int64))  # the samples did not move: the same fit
    _check_estimate(engine, x1, x2t, table, thr, "rms", "msac")
    m, v = engine.homography_mask(H_fit, thr)
    m_ref, v_ref = ctransfer.transfer_exact_many(H_fit, *_cols(x1, x2t), thr)
    assert np.array_equal(m, m_ref) and np.array_equal(v.view(np.int64), v_ref.view(np.int64))


# ---- decomposition geometry ------------------------------------------------------------------------------------
K_DEC = np.array([[800.0, 0.0, 640.0], [0.0, 780.0, 480.0], [0.0, 0.0, 1.0]])
R_DEC = euler_xyz_intrinsic(3.0, -5.0, 2.0)
N_DEC = np.array([0.1, -0.2, 1.0]) / np.linalg.norm([0.1, -0.2, 1.0])
_RN = R_DEC @ N_DEC
# (t, d, H scale, repeated singular value)
GEOMETRY = {
    "forward": (-_RN * 0.5, 4.0, 1.0, True),
    "backward": (_RN * 0.5, 4.0, 1.0, True),
    "near_forward_1e-7": (-_RN * 0.5 + 1e-7 * np.cross(_RN, [0.0, 1.0, 0.0]), 4.0, 1.0, True),
    "near_forward_1e-4": (-_RN * 0.5 + 1e-4 * np.cross(_RN, [0.0, 1.0, 0.0]), 4.0, 1.0, False),
    "in_plane": (np.cross(_RN, [0.0, 1.0, 0.0]), 4.0, 1.0, False),
    "close_plane": (np.array([0.3, 0.1, 0.2]), 0.05, 1.0, False),
    "negative_scale": (np.array([0.4, -0.2, 0.3]), 3.0, -1.0, False),
    "tiny_scale": (np.array([0.4, -0.2, 0.3]), 3.0, 1e-6, False),
    "huge_scale": (np.array([0.4, -0.2, 0.3]), 3.0, 1e6, False),
}


def _set_gap(a, b):
    return max(min(max(np.abs(Ra - Rb).max(), np.abs(ta - tb).max(), np.abs(na - nb).max(), abs(da - db) / db)
                   for Rb, tb, nb, db in b) for Ra, ta, na, da in a)


@pytest.mark.parametrize("case", list(GEOMETRY))
def test_decomposition_geometry(engine, case):
    t, d, scale, repeated = GEOMETRY[case]
    assert 1.0 + N_DEC @ R_DEC.T @ t / d > 0.0  # both cameras on the same side of the plane
    H = K_DEC @ (R_DEC + np.outer(t, N_DEC) / d) @ np.linalg.inv(K_DEC) * scale
    gpu = hg.decompose_homography_arrays(H, K_DEC, rotation_tolerance=0.0, engine=engine)
    ref = hp.decompose_homography(H, K_DEC, rotation_tolerance=0.0)
    tol = 1e-6 if repeated else 1e-9  # sqrt(eps) where two singular values coincide
    assert not gpu.rotation_only and len(gpu.candidates) == 4
    assert np.abs(gpu.singular_values - ref["sv"]).max() < 1e-12
    Hn = hp.normalised_homography(H, K_DEC)
    for R, tc, n, dc in gpu.candidates:
        assert np.abs(Hn - (R + np.outer(tc, n) / dc)).max() <= 1e-12 * max(1.0, np.abs(Hn).max())
        assert np.abs(R @ R.T - np.eye(3)).max() < 1e-12 and abs(np.linalg.det(R) - 1.0) < 1e-12
        assert abs(np.linalg.norm(tc) - 1.0) < 1e-12 and abs(np.linalg.norm(n) - 1.0) < 1e-12
    truth = [(R_DEC, t / np.linalg.norm(t), N_DEC, d / np.linalg.norm(t))]
    assert _set_gap(truth, gpu.candidates) < tol
    assert _set_gap(gpu.candidates, ref["candidates"]) < tol and _set_gap(ref["candidates"], gpu.candidates) < tol


def test_rotation_tolerance_boundary(engine):
    t, d, _, _ = GEOMETRY["in_plane"]
    for scale in (1.0, -1.0):
        H = K_DEC @ (R_DEC + np.outer(0.05 * t, N_DEC) / d) @ np.linalg.inv(K_DEC) * scale
        sv = hp.decompose_homography(H, K_DEC)["sv"]
        for f, rot in ((1.0 - 1e-9, False), (1.0 + 1e-9, True)):
            tol = (sv[0] - sv[2]) * f
            gpu = hg.decompose_homography_arrays(H, K_DEC, rotation_tolerance=tol, engine=engine)
            ref = hp.decompose_homography(H, K_DEC, rotation_tolerance=tol)
            assert gpu.rotation_only == ref["rotation_only"] == rot, (scale, f)
            if rot:
                assert np.abs(gpu.candidates[0][0] - ref["candidates"][0][0]).max() < 1e-12


# ---- one camera for the homography pose; the E path's camera for model selection -------------------------------
K_BASE = np.array([[800.0, 0.0, 610.0], [0.0, 790.0, 500.0], [0.0, 0.0, 1.0]])


def _skewed(s):
    K = K_BASE.copy()
    K[0, 1] = s
    return K


def _bad_cameras():
    k10 = K_BASE.copy()
    k10[1, 0] = 2.0
    k20 = K_BASE.copy()
    k20[2, 0] = 1e-4
    k21 = K_BASE.copy()
    k21[2, 1] = -1e-4
    return {"2K": 2.0 * K_BASE, "K/2": 0.5 * K_BASE, "K[1,0]": k10, "K[2,0]": k20, "K[2,1]": k21}


def test_hpose_refuses_a_camera_it_cannot_read_consistently(engine):
    K, x1, x2, H, _ = make_planar_scene(2000, 0.3, seed=31)
    for name, Kb in _bad_cameras().items():
        with pytest.raises(_native.NativeError, match=r"-1: .*upper triangular"):
            engine.decompose_homography(H, Kb)
        engine.upload_pairs(x1, x2, np.eye(3))
        engine.sample_device(1, 256)
        with pytest.raises(_native.NativeError, match=r"-1: .*upper triangular"):
            engine.two_view_homography(Kb, 16.0, 500.0)
        hg.ransac_homography_arrays(x1, x2, 16.0, 500, max_iterations=256, sampler="device", engine=engine)
        with pytest.raises(_native.NativeError, match=r"-1: .*upper triangular"):
            engine.homography_pose_and_triangulate(Kb, 16.0)
        with pytest.raises(_native.NativeError, match=r"-1: .*upper triangular"):
            hg.two_view_homography_arrays(Kb, x1, x2, 16.0, 500, max_iterations=256, sampler="device", engine=engine)
    # the same K, well formed, is accepted on every path
    hg.two_view_homography_arrays(K, x1, x2, 16.0, 500, max_iterations=256, sampler="device", engine=engine)


def _deg_r(R, Rt):
    return np.degrees(np.arccos(np.clip((np.trace(R.T @ Rt) - 1.0) / 2.0, -1.0, 1.0)))


def _deg_v(a, b):
    return np.degrees(np.arccos(np.clip(a @ b / np.linalg.norm(a) / np.linalg.norm(b), -1.0, 1.0)))


@pytest.mark.parametrize("skew", [5.0, 40.0])
def test_skewed_camera_pose_and_vote(engine, skew):
    K = _skewed(skew)
    _, x1, x2, _, _ = make_planar_scene(6000, 0.3, seed=32, K=K)
    res = hg.two_view_homography_arrays(K, x1, x2, 16.0, 3000, max_iterations=500, sampler="device", seed=4,
                                        engine=engine)
    assert not res.rotation_only
    assert _deg_r(res.R, R_TRUE) < 0.5 and _deg_v(res.t, T_TRUE) < 3.0 and _deg_v(res.n, N_TRUE) < 3.0
    bits, counts, best = hp.vote(res.candidates, K, *_cols(x1, x2, res.inlier_indices))
    p, _, idx, ok, _ = engine.homography_pose_and_triangulate(K, 16.0)
    assert np.array_equal(idx, res.inlier_indices) and np.array_equal(ok, bits)
    assert np.array_equal(res.counts, counts) and int(p.best) == best
    assert res.passing.sum() >= 0.9 * len(res.inlier_indices)


@pytest.mark.parametrize("skew", [5.0, 40.0])
def test_skewed_camera_model_scores(engine, skew):
    K = _skewed(skew)
    K, x1, x2, R, t, out = make_scene(20000, 0.3, seed=33, K=K)
    Kd, Ki = ms.essential_camera(K), np.linalg.inv(K)
    E = Kd.T @ Ki.T @ np.array([[0.0, -t[2], t[1]], [t[2], 0.0, -t[0]], [-t[1], t[0], 0.0]]) @ R @ Ki @ Kd
    H = K @ (R + np.outer(t, [0.0, 0.0, 1.0]) / 6.0) @ Ki
    engine.upload_pairs(x1, x2, K)
    s, pp = engine.model_scores(E, H / H[2, 2], K, per_point=True)
    ref = cselect.score_models(K, x1, x2, E, H / H[2, 2])
    np.testing.assert_array_equal(pp, ref["per_point"])
    assert (s.fixed_e, s.fixed_h, s.count_e, s.count_h) == (ref["fixed_e"], ref["fixed_h"], ref["count_e"],
                                                            ref["count_h"])
    assert (s.score_e, s.score_h, s.ratio_h, s.model) == (ref["score_e"], ref["score_h"], ref["ratio_h"], ref["model"])
    assert s.count_e >= 0.95 * (len(x1) - len(out)) and s.model == 0


# ---- upload layouts --------------------------------------------------------------------------------------------
def _fields(st):
    """The bytes of every field of a ctypes result except the reserved ones, as one array."""
    raw = bytes(st)
    parts = [raw[getattr(type(st), f).offset:][:getattr(type(st), f).size] for f, _ in st._fields_ if f != "reserved"]
    return np.frombuffer(b"".join(parts), dtype=np.uint8)


def test_two_view_homography_is_the_same_for_every_upload_layout(engine):
    import torch

    K, x1, x2, _, _ = make_planar_scene(5000, 0.3, seed=34)
    da = torch.from_numpy(np.ascontiguousarray(x1)).cuda()
    db = torch.from_numpy(np.ascontiguousarray(x2)).cuda()
    torch.cuda.synchronize()
    uploads = {
        "stride2": lambda: engine.upload_pairs(x1, x2, np.eye(3)),
        "soa": lambda: engine.upload_pairs_soa(x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], np.eye(3)),
        "device": lambda: engine.upload_pairs_device(da.data_ptr(), da.data_ptr() + 8, db.data_ptr(),
                                                     db.data_ptr() + 8, 2, len(x1), np.eye(3)),
    }
    out = {}
    for name, up in uploads.items():
        up()
        engine.sample_device(5, 512)
        b, mask, err, p, num, idx, ok, X = engine.two_view_homography(K, 16.0, 2000.0)
        engine.synchronize()
        assert b.index >= 0 and num > 2000 and p.best >= 0
        out[name] = [_fields(b), mask, err.view(np.int64), _fields(p), idx, ok, X.view(np.int64)]
    del da, db
    for name in ("soa", "device"):
        for a, b in zip(out["stride2"], out[name]):
            assert np.array_equal(a, b), name


# ---- randomised sweep ------------------------------------------------------------------------------------------
def test_fuzz_homography():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_homography.py"), "25"], capture_output=True,
                         text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0 and "mismatches: 0" in out.stdout, out.stdout[-3000:] + out.stderr[-2000:]
