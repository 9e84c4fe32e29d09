"""Generate tests/golden/*.json from the UNMODIFIED reference (build container only).

Run:  python tests/golden/make_golden.py
Needs /root/reference (through oracle/reference_shims.py) and OpenCV (only to build the
reference's own test fixtures exactly as lib/epipolar/tests/test_epipolar.py does).
The JSON files are committed; nothing at test time reads /root/reference.
json stores floats with repr(), which round-trips IEEE doubles exactly.
"""
import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from oracle import reference_shims  # noqa: E402
from oracle import restatement as o  # noqa: E402
from structure_from_motion_b200.scenes import make_scene  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
ref = reference_shims.load()
F, M = ref.feature.Feature, ref.matching.Match


def dump(name, obj):
    def conv(x):
        if isinstance(x, np.ndarray):
            return x.tolist()
        if isinstance(x, (np.floating,)):
            return float(x)
        if isinstance(x, (np.integer,)):
            return int(x)
        if isinstance(x, dict):
            return {k: conv(v) for k, v in x.items()}
        if isinstance(x, (list, tuple)):
            return [conv(v) for v in x]
        return x

    with open(os.path.join(OUT, name), "w") as f:
        json.dump(conv(obj), f, indent=1)
    print("wrote", name)


def camera_matrix(f, w, h):
    return np.array([[f, 0.0, w / 2.0], [0.0, f, h / 2.0], [0.0, 0.0, 1.0]])


def eight_point_fixture():
    """lib/epipolar/tests/test_epipolar.py:109-143."""
    import cv2 as cv
    from scipy.spatial.transform import Rotation

    K = camera_matrix(50.0, 512, 256)
    rng = np.random.default_rng(seed=6)
    pts = rng.random((8, 3), dtype=np.float64) + np.array([1.0, 0.0, 0.0])
    c1 = np.array([1.5, 0.25, -1.0])
    R1 = np.eye(3)
    c2 = np.array([2.5, 0.1, -1.5])
    R2 = Rotation.from_euler("XY", [-20.0, -50.0], degrees=True).as_matrix()
    p1, _ = cv.projectPoints(pts, cv.Rodrigues(R1)[0], R1 @ -c1, K, None)
    p2, _ = cv.projectPoints(pts, cv.Rodrigues(R2)[0], R2 @ -c2, K, None)
    return K, pts, p1.squeeze(), p2.squeeze(), rng, (c1, R1, c2, R2)


def main():
    import cv2 as cv

    # ---------------- eight-point fixture: F, E, decomposition, pose (test_epipolar.py:151-269)
    K, world, p1, p2, rng, (c1, R1w, c2, R2w) = eight_point_fixture()
    fa = [F(x=p[0], y=p[1]) for p in p1]
    fb = [F(x=p[0], y=p[1]) for p in p2]
    ms = ref.eight_point.create_trivial_matches(8)
    f_ref = ref.eight_point.estimate_fundamental_mat(fa, fb, ms)
    e_ref = ref.eight_point.estimate_essential_mat(camera_matrix=K, features_a=fa, features_b=fb, matches=ms)
    e_cv, _ = cv.findEssentialMat(p1, p2, K)
    e_cv /= e_cv[2][2]
    f_cv, _ = cv.findFundamentalMat(p1, p2, method=cv.FM_8POINT)
    R1d, R2d, t1d = ref.eight_point._recover_all_r_t(e_ref.copy())
    na = [ref.eight_point.to_normalized_image_coords(f, K) for f in fa]
    nb = [ref.eight_point.to_normalized_image_coords(f, K) for f in fb]
    Rr, tr, mask = ref.eight_point._recover_r_t(na, nb, e_ref.copy())
    sed_cv = [ref.sed.calculate_symmetric_epipolar_distance(a, b, e_cv) for a, b in zip(na, nb)]
    world_t = c1 - c2
    exp_t = R2w @ world_t
    exp_t /= np.linalg.norm(exp_t)
    dump("eight_point_fixture.json", dict(
        K=K, cam1_points=p1, cam2_points=p2, F=f_ref, E=e_ref, E_opencv=e_cv, F_opencv=f_cv,
        R1=R1d, R2=R2d, t1=t1d, R=Rr, t=tr, mask=mask, sed_under_E_opencv=sed_cv,
        expected_t_direction=exp_t, expected_R=R2w @ R1w.T))

    # ---------------- RANSAC known answer (test_epipolar.py:367-415)
    xs, ys = [f.x for f in fa], [f.y for f in fa]
    nx = rng.random(4) * (max(xs) - min(xs)) + min(xs)
    ny = rng.random(4) * (max(ys) - min(ys)) + min(ys)
    fa10 = fa + [F(x=x, y=y) for x, y in zip(nx[:2], ny[:2])]
    fb10 = fb + [F(x=x, y=y) for x, y in zip(nx[2:], ny[2:])]
    ms10 = ref.eight_point.create_trivial_matches(10)
    random.seed(5)
    e10, pairs10 = ref.epipolar_ransac.estimate_essential_mat_with_ransac(
        camera_matrix=K, features_a=fa10, features_b=fb10, matches=ms10, sed_inlier_threshold=0.01,
        error_aggregation_method=ref.ransac.ErrorAggregationMethod.SUM)
    state_words = list(random.getstate()[1])
    coords = {(f.x, f.y): i for i, f in enumerate(fa10)}
    dump("ransac_known_answer.json", dict(
        K=K, pts_a=[[f.x, f.y] for f in fa10], pts_b=[[f.x, f.y] for f in fb10], threshold=0.01,
        method="sum", seed=5, E=e10, inlier_indices=[coords[(p[0].x, p[0].y)] for p in pairs10],
        rng_state_after=state_words))

    # ---------------- config 1 (BASELINE.json configs[0]): N=500, 30 % outliers, H=1000
    Kc, x1, x2, _, _, _ = make_scene(500, 0.3, seed=0)
    fa1 = [F(x=float(p[0]), y=float(p[1])) for p in x1]
    fb1 = [F(x=float(p[0]), y=float(p[1])) for p in x2]
    ms1 = [M(a_index=i, b_index=i) for i in range(500)]
    random.seed(5)
    e1, pairs1 = ref.epipolar_ransac.estimate_essential_mat_with_ransac(
        Kc, fa1, fb1, ms1, 1.5e-6, min_num_extra_inliers=10,
        error_aggregation_method=ref.ransac.ErrorAggregationMethod.RMS, max_iterations=1000)
    coords = {(f.x, f.y): i for i, f in enumerate(fa1)}
    inl1 = [coords[(p[0].x, p[0].y)] for p in pairs1]
    random.seed(5)
    rest = o.ransac_essential(Kc, x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1], 1.5e-6, 10, "rms", 1000, exact_sed=True)
    assert np.array_equal(rest["E"], e1) and list(rest["inlier_indices"]) == inl1
    dump("config1_known_answer.json", dict(
        scene=dict(n=500, outlier_frac=0.3, seed=0), threshold=1.5e-6, min_extra=10, method="rms",
        max_iterations=1000, seed=5, E=e1, inlier_indices=inl1, best_index=rest["best_index"],
        error=rest["error"]))

    # ---------------- sampler known answer (SURVEY.md §8(c))
    random.seed(5)
    perm = list(range(1000))
    rows = []
    for _ in range(3):
        random.shuffle(perm)
        rows.append(perm[:8])
    dump("sampler_known_answer.json", dict(seed=5, n=1000, rows=rows, state_after=list(random.getstate()[1])))

    # ---------------- degenerate fixture (test_epipolar.py:272-364)
    from scipy.spatial.transform import Rotation

    w_, h_ = np.array([1.0, 0.0, 0.0]), np.array([0.0, 0.5, 0.0])
    ra = np.array([np.zeros(3), w_, w_ + h_, h_])
    rb = ra + np.array([2.0, 0.0, 0.0])

    def rot(rect, r):
        c = rect.mean(axis=0)
        return r.apply(rect - c) + c

    ra = rot(ra, Rotation.from_euler("y", -40.0, degrees=True))
    rb = rot(rb, Rotation.from_euler("y", 40.0, degrees=True))
    base = np.radians((180 - 100) / 2.0)
    fdeg = min(np.tan(base) * 512 / 2, np.tan(base) * 256 / 2)
    Kd = camera_matrix(fdeg, 512, 256)
    allp = np.vstack([ra, rb])
    d1, _ = cv.projectPoints(allp, cv.Rodrigues(np.eye(3))[0], -c1, Kd, None)
    d2, _ = cv.projectPoints(allp, cv.Rodrigues(R2w)[0], -c2, Kd, None)
    d1, d2 = d1.squeeze(), d2.squeeze()
    try:
        ref.eight_point.estimate_fundamental_mat([F(x=p[0], y=p[1]) for p in d1], [F(x=p[0], y=p[1]) for p in d2], ms)
        raised = False
    except ref.eight_point.EightPointCalculationError:
        raised = True
    dump("degenerate_fixture.json", dict(K=Kd, cam1_points=d1, cam2_points=d2, raises=raised))

    # ---------------- triangulation known answer (test_epipolar.py:418-496)
    Kt = camera_matrix(50.0, 512, 256)
    P = np.array([0.0, 0.0, 10.0])
    cw1 = np.array([0.0, 0.0, 5.0])
    cw2 = np.array([3.0, 0.0, 5.0])
    Rw2 = Rotation.from_euler("XYZ", [0.0, 30.0, 0.0], degrees=True).as_matrix()
    T1 = ref.transforms.Transform3D.from_rmat_t(np.eye(3), -cw1).Tmat
    T2 = ref.transforms.Transform3D.from_rmat_t(Rw2.T, -cw2).Tmat
    q1, _ = cv.projectPoints(P.reshape(1, 3), cv.Rodrigues(np.eye(3))[0], -cw1, Kt, distCoeffs=None)
    q2, _ = cv.projectPoints(P.reshape(1, 3), cv.Rodrigues(Rw2.T)[0], -cw2, Kt, distCoeffs=None)
    q1, q2 = q1.reshape(2), q2.reshape(2)
    Kext = np.hstack((Kt, np.zeros((3, 1))))
    P1, P2 = Kext @ T1, Kext @ T2
    Xr = ref.triangulation.triangulate_point_correspondence(F(x=q1[0], y=q1[1]), F(x=q2[0], y=q2[1]), P1, P2)
    dump("triangulation_known_answer.json", dict(feature_a=q1, feature_b=q2, P1=P1, P2=P2, expected=P, reference=Xr))

    # ---------------- SED bit vectors: sed.py on random and near-inlier inputs
    r = np.random.default_rng(7)
    rows = []
    for k in range(300):
        if k % 2 == 0:
            E = r.normal(size=(3, 3))
            E /= E[2, 2]
            xa, ya, xb, yb = (r.normal(size=4) * 0.5).tolist()
        else:
            t = r.normal(size=3)
            E = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
            if abs(E[2, 2]) > 1e-3:
                E = E / E[2, 2]
            X = r.normal(size=3) + np.array([0, 0, 5.0])
            a = X / X[2]
            X2 = X + t
            b = X2 / X2[2]
            b[:2] += r.normal(size=2) * 1e-3
            xa, ya, xb, yb = float(a[0]), float(a[1]), float(b[0]), float(b[1])
        s = ref.sed.calculate_symmetric_epipolar_distance(F(xa, ya), F(xb, yb), E)
        rows.append(dict(E=E, xa=xa, ya=ya, xb=xb, yb=yb, sed=s))
    dump("sed_vectors.json", rows)

    # ---------------- pose + triangulation on a noisy scene (recover_r_t_from_e, triangulate_points)
    Kp, y1, y2, Rt, tt, _ = make_scene(60, 0.0, seed=21, noise_px=0.1)
    fa2 = [F(x=float(p[0]), y=float(p[1])) for p in y1]
    fb2 = [F(x=float(p[0]), y=float(p[1])) for p in y2]
    ep = ref.eight_point.estimate_essential_mat(camera_matrix=Kp, features_a=fa2, features_b=fb2,
                                                matches=[M(a_index=i * 7, b_index=i * 7) for i in range(8)])
    Rp, tp, maskp = ref.eight_point.recover_r_t_from_e(ep.copy(), Kp, fa2, fb2)
    Tp = ref.transforms.Transform3D.from_rmat_t(Rp, tp)
    Xp = ref.triangulation.triangulate_points(fa2, fb2, Kp, Tp)
    dump("pose_known_answer.json", dict(K=Kp, pts_a=y1, pts_b=y2, E=ep, R=Rp, t=tp, mask=maskp, X=Xp))

    # ---------------- generic fit_with_ransac with a Python line model (test_ransac.py:70-123)
    line_start, slope, npts, dx = np.array([4, 5]), 0.6, 50, 0.3
    line_points = np.array([line_start + np.array([i * dx, i * slope * dx]) for i in range(npts)]).reshape((-1, 2))
    rng2 = np.random.default_rng(seed=6)
    noise = rng2.random(size=(25, 2))
    noise[:, 0] = noise[:, 0] * (line_points[:, 0].max() - line_points[:, 0].min()) + line_points[:, 0].min()
    noise[:, 1] = noise[:, 1] * (line_points[:, 1].max() - line_points[:, 1].min()) + line_points[:, 1].min()
    allp = np.vstack([line_points, noise])

    def fitter(pts):
        dxx = pts[1][0] - pts[0][0]
        if abs(dxx) <= 1e-6:
            return (1.0, 0.0, -pts[0][0])
        s = (pts[1][1] - pts[0][1]) / dxx
        return (s, -1.0, pts[0][1] - s * pts[0][0])

    def scorer(m, p):
        return abs(m[0] * p[0] + m[1] * p[1] + m[2]) / (m[0] ** 2 + m[1] ** 2) ** 0.5

    random.seed(5)
    model, inl = ref.ransac.fit_with_ransac(list(allp), 2, fitter, scorer, 0.2, len(allp) / 2,
                                            ref.ransac.ErrorAggregationMethod.RMS)
    dump("line_ransac_known_answer.json", dict(points=allp, model=list(model), inliers=np.array(inl),
                                               state_after=list(random.getstate()[1])))
    front_end_golden()
    reference_outputs_golden()
    nonfinite_golden()


def synthetic_image_pair(seed, h=72, w=96):
    """A textured uint8 image and a shifted, noisy second view of it (what cv.cvtColor would hand over)."""
    rng = np.random.default_rng(seed)
    base = rng.random((h + 16, w + 16))
    # smooth a little so that windows carry structure, keep it integer-valued like a camera image
    k = np.ones((3, 3)) / 9.0
    sm = sum(base[i:i + h + 14, j:j + w + 14] * k[i, j] for i in range(3) for j in range(3))
    img = np.clip(np.round(255 * (sm - sm.min()) / (sm.max() - sm.min())), 0, 255)
    a = img[4:4 + h, 4:4 + w]
    b = np.clip(img[6:6 + h, 7:7 + w] + np.round(rng.normal(0, 2.0, (h, w))), 0, 255)
    return a.astype(np.uint8), b.astype(np.uint8)


def front_end_golden():
    """SURVEY.md §8(f) N1: brute-force matcher + NCC / SSD on the unmodified reference."""
    import functools

    img_a, img_b = synthetic_image_pair(3)
    rng = np.random.default_rng(11)
    h, w = img_a.shape
    na, nb = 40, 37
    # Harris returns integer-valued float coordinates (+ block_size/2); include border cases and x.5 positions
    fa = np.stack([rng.integers(0, w, na), rng.integers(0, h, na)], 1).astype(np.float64)
    fb = np.stack([np.clip(fa[:nb, 0] - 3 + rng.integers(-1, 2, nb), 0, w - 1),
                   np.clip(fa[:nb, 1] - 2 + rng.integers(-1, 2, nb), 0, h - 1)], 1).astype(np.float64)
    fb = fb[rng.permutation(nb)]
    fa[5] += 0.5
    fb[7] += 0.5
    fa[0] = [0.0, 0.0]
    fb[1] = [w - 1.0, h - 1.0]
    feats_a = [F(x=float(x), y=float(y)) for x, y in fa]
    feats_b = [F(x=float(x), y=float(y)) for x, y in fb]
    out = dict(image_a=img_a.astype(int), image_b=img_b.astype(int), feats_a=fa, feats_b=fb, cases=[])
    VS = ref.matching.ValidationStrategy
    for kind, window in [("ncc", 9), ("ncc", 3), ("ssd", 5)]:
        base_fn = ref.ncc.calculate_ncc if kind == "ncc" else ref.ssd.calculate_ssd
        score = functools.partial(base_fn, img_a, img_b, window_size=window)
        S = np.array([[score(a, b) for b in feats_b] for a in feats_a])
        for strategies, thr in [(None, 0.5), (VS.RATIO_TEST, 0.7), (VS.CROSSCHECK, 0.5),
                                ({VS.RATIO_TEST, VS.CROSSCHECK}, 0.7), ({VS.RATIO_TEST, VS.CROSSCHECK}, 0.95)]:
            m = ref.matching.match_brute_force(feats_a, feats_b, score, validation_strategies=strategies,
                                               ratio_test_threshold=thr)
            names = [] if strategies is None else sorted(x.name for x in (strategies if isinstance(strategies, set) else {strategies}))
            out["cases"].append(dict(kind=kind, window=window, strategies=names, ratio=thr,
                                     matches=[[x.a_index, x.b_index, x.match_score] for x in m],
                                     scores=S if not names else None))
    dump("matching_known_answer.json", out)
    harris_golden()


def harris_golden():
    """SURVEY.md §8(f) N2: Harris detector + cross-correlation + Gaussian kernel on the unmodified reference."""
    img_a, _ = synthetic_image_pair(3)
    img = img_a[:48, :64]
    # a few bright rectangles so that there are real corners (and flat areas with zero cornerness)
    img = img.copy()
    img[10:22, 12:30] = 230
    img[28:40, 36:58] = 20
    out = dict(image=img.astype(int), cases=[])
    for num, bs, k in [(50, 2, 0.04), (20, 3, 0.06), (100000, 2, 0.04)]:
        cim = ref.harris._calculate_cornerness_image(img, bs, k)
        raw = cim.copy()
        cim[cim < 0] = 0.0
        ref.harris._non_max_suppress(cim)
        corners = ref.harris.detect_harris_corners(img, num_corners=num, block_size=bs, k=k)
        out["cases"].append(dict(num_corners=num, block_size=bs, k=k, cornerness_raw=raw, cornerness=cim,
                                 corners=[[float(c.x), float(c.y)] for c in corners]))
    # the reference's own fixture (test_harris_detector.py:14-32): a white square on black
    sq = np.zeros((20, 20), dtype=np.uint8)
    sq[5:15, 5:15] = 255
    corners = ref.harris.detect_harris_corners(sq, num_corners=4)
    out["square"] = dict(image=sq.astype(int), corners=[[float(c.x), float(c.y)] for c in corners])
    # test_harris_detector.py:14-32: cv.rectangle(zeros((100, 200)), (50, 25), (150, 75), 255, -1) fills both corners inclusively
    rect = np.zeros((100, 200), dtype=float)
    rect[25:76, 50:151] = 255.0
    corners = ref.harris.detect_harris_corners(rect)
    out["rectangle"] = dict(fill=[25, 76, 50, 151], shape=[100, 200],
                            corners=[[float(c.x), float(c.y)] for c in corners],
                            expected_yx=[[75, 50], [75, 150], [25, 50], [25, 150]])
    fimg = img.astype(np.float64) / 255.0
    kern = ref.gaussian.create_gaussian_kernel(5, 1.2)
    out["correlate"] = dict(kernel=kern, result=ref.correlate.cross_correlate(fimg[:20, :24], kern),
                            sobel_u8=ref.correlate.cross_correlate(img[:20, :24], ref.harris._sobel_x_kernel))
    dump("harris_known_answer.json", out)


def reference_outputs_golden():
    """What tests/test_oracle.py::test_restatement_matches_live_reference and
    tests/test_front_end_oracle.py::test_front_end_matches_live_reference compare against: the reference's
    estimate_essential_mat_with_ransac for every aggregation, its pose and triangulation of the winner's inliers, and
    its matcher and Harris detector on small crops of the front-end fixtures."""
    import functools

    K, x1, x2, *_ = make_scene(150, 0.3, seed=2)
    fa = [F(x=float(p[0]), y=float(p[1])) for p in x1]
    fb = [F(x=float(p[0]), y=float(p[1])) for p in x2]
    ms = [M(a_index=i, b_index=i) for i in range(150)]
    runs = []
    for method in ("sum", "square", "mean", "rms"):
        random.seed(9)
        e, pairs = ref.epipolar_ransac.estimate_essential_mat_with_ransac(
            K, fa, fb, ms, 1.5e-6, min_num_extra_inliers=4,
            error_aggregation_method=ref.ransac.ErrorAggregationMethod(method), max_iterations=40)
        runs.append(dict(method=method, E=e, pairs=[[a.x, a.y, b.x, b.y] for a, b in pairs],
                         rng_state_after=list(random.getstate()[1])))
    ia, ib = [a for a, _ in pairs], [b for _, b in pairs]
    R, t, mask = ref.eight_point.recover_r_t_from_e(e.copy(), K, ia, ib)
    X = ref.triangulation.triangulate_points(ia, ib, K, ref.transforms.Transform3D.from_rmat_t(R, t))
    dump("ransac_methods_known_answer.json", dict(
        K=K, pts_a=x1, pts_b=x2, seed=9, threshold=1.5e-6, min_extra=4, max_iterations=40, runs=runs,
        R=R, t=t, mask=np.asarray(mask), X=X))

    with open(os.path.join(OUT, "matching_known_answer.json")) as f:
        m = json.load(f)
    img_a, img_b = np.array(m["image_a"], dtype=np.uint8), np.array(m["image_b"], dtype=np.uint8)
    feats_a, feats_b = np.array(m["feats_a"])[:12], np.array(m["feats_b"])[:11]
    fa = [F(x=float(x), y=float(y)) for x, y in feats_a]
    fb = [F(x=float(x), y=float(y)) for x, y in feats_b]
    VS = ref.matching.ValidationStrategy
    cases = []
    for kind, fn, w in [("ncc", ref.ncc.calculate_ncc, 5), ("ssd", ref.ssd.calculate_ssd, 3)]:
        score = functools.partial(fn, img_a, img_b, window_size=w)
        matches = []
        for strategies in [None, VS.RATIO_TEST, {VS.RATIO_TEST, VS.CROSSCHECK}]:
            got = ref.matching.match_brute_force(fa, fb, score, validation_strategies=strategies, ratio_test_threshold=0.8)
            names = [] if strategies is None else sorted(x.name for x in (strategies if isinstance(strategies, set) else {strategies}))
            matches.append(dict(strategies=names, matches=[[x.a_index, x.b_index, x.match_score] for x in got]))
        cases.append(dict(kind=kind, window=w, scores=[[score(a, b) for b in fb] for a in fa], matching=matches))
    with open(os.path.join(OUT, "harris_known_answer.json")) as f:
        img = np.array(json.load(f)["image"], dtype=np.uint8)[:24, :30]
    corners = ref.harris.detect_harris_corners(img, num_corners=15)
    dump("front_end_known_answer.json", dict(
        num_features=[12, 11], ratio=0.8, cases=cases, harris=dict(rows=24, cols=30, num_corners=15,
                                                                    corners=[[float(c.x), float(c.y)] for c in corners])))


def nonfinite_golden():
    """What the reference raises when a sample's Hartley-normalised coordinates are not finite (a coordinate is NaN,
    or all eight points of one image coincide and their mean rounds back to the point: scale sqrt(2)/0):
    np.linalg.eig refuses Y^T Y (eight_point.py:410) with numpy's LinAlgError, which nothing in ransac.py catches.
    Coincident points whose mean does not round back to the point leave tiny finite offsets, a finite scale and a
    rank-deficient Y: EightPointCalculationError.  For the RANSAC cases the global random state after the exception
    is recorded too: the loop stops inside the iteration of the first such sample."""
    K = camera_matrix(800.0, 1280, 960)
    _, x1, x2, _, _, _ = make_scene(30, 0.0, seed=4)

    def outcome(call):
        try:
            call()
        except Exception as exc:  # the exception's type and message are the fixture
            return dict(raises=type(exc).__module__ + "." + type(exc).__qualname__, message=str(exc))
        return dict(raises=None, message=None)

    def feats(pts):
        return [F(x=float(p[0]), y=float(p[1])) for p in pts]

    eight = []
    coincident = np.repeat(x1[:1], 8, axis=0)
    exact = np.repeat([[K[0, 2] + 0.5 * K[0, 0], K[1, 2] - 0.25 * K[1, 1]]], 8, axis=0)  # K-normalised (0.5, -0.25)
    nan_rec = x1[:8].copy()
    nan_rec[3, 1] = np.nan
    for name, pa, pb in (("coincident_a", coincident, x2[:8]), ("coincident_b", x1[:8], coincident[:, ::-1]),
                         ("exact_coincident_a", exact, x2[:8]), ("exact_coincident_b", x1[:8], exact),
                         ("nan", nan_rec, x2[:8])):
        res = outcome(lambda: ref.eight_point.estimate_essential_mat(
            camera_matrix=K, features_a=feats(pa), features_b=feats(pb), matches=ref.eight_point.create_trivial_matches(8)))
        eight.append(dict(name=name, pts_a=pa, pts_b=pb, **res))

    ransac = []
    nan_scene = x1.copy()
    nan_scene[17, 0] = np.nan
    all_same = np.repeat(x1[:1], len(x1), axis=0)
    all_exact = np.repeat(exact[:1], len(x1), axis=0)
    for name, pa, pb in (("nan_record", nan_scene, x2), ("coincident_a", all_same, x2),
                         ("exact_coincident_b", x1, all_exact)):
        random.seed(5)
        res = outcome(lambda: ref.epipolar_ransac.estimate_essential_mat_with_ransac(
            K, feats(pa), feats(pb), [M(a_index=i, b_index=i) for i in range(len(pa))], 1.5e-6,
            error_aggregation_method=ref.ransac.ErrorAggregationMethod.RMS, max_iterations=50))
        ransac.append(dict(name=name, pts_a=pa, pts_b=pb, seed=5, max_iterations=50, threshold=1.5e-6,
                           state_after=list(random.getstate()[1]), **res))
    dump("nonfinite_sample_fixture.json", dict(K=K, eight_point=eight, ransac=ransac))


def pose_nonfinite_golden():
    """What the reference's pose functions do with a NaN or an infinity in E, in one correspondence, or in P1 / P2:
    _recover_all_r_t (eight_point.py:245-280), _recover_r_t (:181-242, normalised coordinates) and
    triangulate_point_correspondence (triangulation.py:9-39) applied to every correspondence.  Recorded: the
    exception's type and message, or the result (R, t and passing indices; the points)."""
    rng = np.random.default_rng(11)
    R = np.array([[0.9950041652780258, -0.09983341664682815, 0.0], [0.09983341664682815, 0.9950041652780258, 0.0],
                  [0.0, 0.0, 1.0]])
    t = np.array([1.0, 0.2, 0.1])
    X = np.stack([rng.uniform(-1, 1, 6), rng.uniform(-1, 1, 6), rng.uniform(2, 8, 6)], 1)
    na = X[:, :2] / X[:, 2:3]
    Xb = X @ R.T + t
    nb = Xb[:, :2] / Xb[:, 2:3]
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    E = tx @ R
    P1 = np.eye(4)[:3]
    P2 = np.hstack([R, t[:, None]])

    def outcome(call):
        try:
            out = call()
        except Exception as exc:
            return dict(raises=type(exc).__module__ + "." + type(exc).__qualname__, message=str(exc), result=None)
        return dict(raises=None, message=None, result=out)

    def feats(a):
        return [F(x=float(p[0]), y=float(p[1])) for p in a]

    def recover_all(e):
        R1, R2, t1 = ref.eight_point._recover_all_r_t(e.copy())
        return dict(R1=R1, R2=R2, t1=t1)

    def recover(e, a, b):
        Rr, tr, idx = ref.eight_point._recover_r_t(feats(a), feats(b), e.copy())
        return dict(R=Rr, t=tr, passing=[int(i) for i in idx])

    def triangulate(a, b, p1, p2):
        return [ref.triangulation.triangulate_point_correspondence(fa, fb, p1, p2)
                for fa, fb in zip(feats(a), feats(b))]

    cases = []
    for val, vname in ((np.nan, "nan"), (np.inf, "inf"), (-np.inf, "-inf")):
        e = E.copy()
        e[1, 2] = val
        cases.append(dict(name=f"E_{vname}", call="recover_all_r_t", E=e, **outcome(lambda: recover_all(e))))
        cases.append(dict(name=f"E_{vname}", call="recover_r_t", E=e, pts_a=na, pts_b=nb,
                          **outcome(lambda: recover(e, na, nb))))
        for side, col in (("a", 0), ("b", 1)):
            a, b = na.copy(), nb.copy()
            (a if side == "a" else b)[2, col] = val
            cases.append(dict(name=f"pts_{side}_{vname}", call="recover_r_t", E=E, pts_a=a, pts_b=b,
                              **outcome(lambda: recover(E, a, b))))
            cases.append(dict(name=f"pts_{side}_{vname}", call="triangulate", P1=P1, P2=P2, pts_a=a, pts_b=b,
                              **outcome(lambda: triangulate(a, b, P1, P2))))
        for which in ("P1", "P2"):
            p1, p2 = P1.copy(), P2.copy()
            (p1 if which == "P1" else p2)[1, 3] = val
            cases.append(dict(name=f"{which}_{vname}", call="triangulate", P1=p1, P2=p2, pts_a=na, pts_b=nb,
                              **outcome(lambda: triangulate(na, nb, p1, p2))))
    # an infinite coordinate against a camera whose third row has no zero: the DLT row is infinite, NaN-free
    Rg = np.array([[0.936, -0.28, 0.2136], [0.3104, 0.9464, -0.0896], [-0.1770, 0.1608, 0.9710]])
    Pg = np.hstack([Rg, np.array([[1.0], [0.2], [0.1]])])
    a, b = na.copy(), nb.copy()
    b[2, 1] = np.inf
    cases.append(dict(name="pts_b_inf_generic_camera", call="triangulate", P1=P1, P2=Pg, pts_a=a, pts_b=b,
                      **outcome(lambda: triangulate(a, b, P1, Pg))))
    # E of rank 3 with a NaN coordinate: the decomposition's error comes before any point is triangulated
    e3 = E.copy()
    e3[2, 2] += 0.5
    a = na.copy()
    a[1, 0] = np.nan
    cases.append(dict(name="E_rank3_pts_a_nan", call="recover_r_t", E=e3, pts_a=a, pts_b=nb,
                      **outcome(lambda: recover(e3, a, nb))))
    dump("pose_nonfinite_fixture.json", dict(cases=cases))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "nonfinite":
        nonfinite_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "pose_nonfinite":
        pose_nonfinite_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "front_end":
        front_end_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "harris":
        harris_golden()
    elif len(sys.argv) > 1 and sys.argv[1] == "reference_outputs":
        reference_outputs_golden()
    else:
        main()
