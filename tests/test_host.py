"""Host-side logic that needs no GPU: the C-ABI library loads and exports every declared
symbol, the CPython-exact sampler, the generic RANSAC driver, value types, import paths."""
import ctypes
import functools
import json
import os
import random
import re

import numpy as np
import pytest

from structure_from_motion_b200 import _native
from structure_from_motion_b200.ransac import ransac

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = os.path.join(ROOT, "tests", "golden")


def load(name):
    with open(os.path.join(G, name)) as f:
        return json.load(f)


def test_abi_exports_every_declared_symbol():
    header = open(os.path.join(ROOT, "include", "sfm_b200.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(sfm_[a-z0-9_]+)\s*\(", header))
    assert len(declared) >= 30
    lib = ctypes.CDLL(_native.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/sfm_b200.h but not exported"
    assert declared == set(_native.EXPORTED_SYMBOLS), declared ^ set(_native.EXPORTED_SYMBOLS)
    assert _native.load_library().sfm_version() >= 100


def test_struct_layouts_match_header():
    assert ctypes.sizeof(_native.Best) == 8 + 8 + 4 + 4 + 8 + 8 + 72 + 32
    assert ctypes.sizeof(_native.Poses) == 4 * 72 + 4 * 24 + 24 + 32 + 8


def test_no_gpu_fails_loudly():
    lib = _native.load_library()
    if lib.sfm_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(_native.NativeUnavailableError, match="no CPU fallback"):
        _native.Engine(0)
    from lib.epipolar.sed import calculate_symmetric_epipolar_distance
    from lib.common.feature import Feature

    with pytest.raises(_native.NativeUnavailableError):
        calculate_symmetric_epipolar_distance(Feature(0.1, 0.2), Feature(0.3, 0.1), np.eye(3))


@pytest.mark.parametrize("seed,n,h", [(5, 1000, 3), (0, 8, 5), (123, 9, 40), (7, 4097, 6), (11, 65536, 2)])
def test_mt_sampler_matches_cpython(seed, n, h):
    random.seed(seed)
    perm = list(range(n))
    rows = []
    for _ in range(h):
        random.shuffle(perm)
        rows.append(perm[:8])
    expected_state = random.getstate()
    random.seed(seed)
    version, words, gauss = random.getstate()
    st = np.array(words, dtype=np.uint32)
    table, p = _native.mt_shuffle_table(st, n, h, perm_at=h - 1)
    assert table.tolist() == rows
    assert p.tolist() == perm
    assert (version, tuple(int(w) for w in st), gauss) == expected_state


def test_mt_sampler_golden_and_midstream_state():
    d = load("sampler_known_answer.json")
    random.seed(d["seed"])
    random.random()  # advance: position inside the 624-word block must be honoured
    random.getrandbits(17)
    v, words, g = random.getstate()
    st = np.array(words, dtype=np.uint32)
    table, _ = _native.mt_shuffle_table(st, 50, 30)
    perm = list(range(50))
    for i in range(30):
        random.shuffle(perm)
        assert table[i].tolist() == perm[:8]
    assert tuple(int(w) for w in st) == random.getstate()[1]
    random.seed(d["seed"])
    st = np.array(random.getstate()[1], dtype=np.uint32)
    table, _ = _native.mt_shuffle_table(st, d["n"], 3)
    assert table.tolist() == d["rows"] and st.tolist() == d["state_after"]


def test_mt_sampler_argument_errors():
    st = np.zeros(625, dtype=np.uint32)
    with pytest.raises(_native.NativeError):
        _native.mt_shuffle_table(st, 7, 1)  # fewer than 8 correspondences
    st[624] = 700
    with pytest.raises(_native.NativeError):
        _native.mt_shuffle_table(st, 100, 1)


def _line_fitter(pts):
    dx = pts[1][0] - pts[0][0]
    if abs(dx) <= 1e-6:
        return (1.0, 0.0, -pts[0][0])
    s = (pts[1][1] - pts[0][1]) / dx
    return (s, -1.0, pts[0][1] - s * pts[0][0])


def _line_scorer(m, p):
    return abs(m[0] * p[0] + m[1] * p[1] + m[2]) / (m[0] ** 2 + m[1] ** 2) ** 0.5


def test_generic_ransac_line_model_matches_reference():
    """lib/ransac/tests/test_ransac.py:70-123 — golden produced by the reference's fit_with_ransac."""
    d = load("line_ransac_known_answer.json")
    pts = np.array(d["points"])
    data = list(pts)
    random.seed(5)
    model, inliers = ransac.fit_with_ransac(
        data=data, model_fit_data_count=2, model_fitter=_line_fitter, inlier_scorer=_line_scorer,
        inlier_threshold=0.2, min_num_extra_inliers=len(data) / 2,
        error_aggregation_method=ransac.ErrorAggregationMethod.RMS)
    assert list(model) == d["model"]
    assert np.array_equal(np.array(inliers), np.array(d["inliers"]))
    assert list(random.getstate()[1]) == d["state_after"]
    assert all(a is not b for a in inliers for b in data)  # copies, as ransac.py:59
    assert abs(-model[0] / model[1] - 0.6) <= 1e-7  # test_ransac.py:119-120
    assert 0 <= len(inliers) - 50 <= 3


def test_generic_ransac_defaults_and_failure():
    random.seed(0)
    pts = [np.array([float(i), 2.0 * i + 1.0]) for i in range(20)]
    model, inl = ransac.fit_with_ransac(pts, 2, _line_fitter, _line_scorer, 1e-9)
    assert abs(model[0] - 2.0) < 1e-12 and len(inl) == 20
    with pytest.raises(ValueError, match="No model could be found with at least 32 inliers"):
        ransac.fit_with_ransac(pts, 2, _line_fitter, _line_scorer, 1e-9, min_num_extra_inliers=30)
    for m, exp in [(ransac.ErrorAggregationMethod.SUM, 6.0), (ransac.ErrorAggregationMethod.SQUARE, 14.0),
                   (ransac.ErrorAggregationMethod.MEAN, 2.0), (ransac.ErrorAggregationMethod.RMS, (14 / 3) ** 0.5)]:
        assert ransac._aggregate_error([1.0, 2.0, 3.0], m) == pytest.approx(exp, rel=1e-15)


def test_epipolar_partials_are_recognised():
    from lib.epipolar import epipolar_ransac as er

    K = np.eye(3)
    f = functools.partial(er.eight_point_model_fitter, camera_matrix=K)
    s = functools.partial(er.calculate_sed_inlier_score, camera_matrix=K)
    assert ransac._epipolar_camera_matrix(8, f, s) is not None
    assert ransac._epipolar_camera_matrix(7, f, s) is None
    assert ransac._epipolar_camera_matrix(8, f, _line_scorer) is None
    s2 = functools.partial(er.calculate_sed_inlier_score, camera_matrix=2 * K)
    assert ransac._epipolar_camera_matrix(8, f, s2) is None


def test_reference_import_paths_and_value_types():
    from lib.common.feature import Feature
    from lib.epipolar.eight_point import (EightPointCalculationError, _get_matching_coordinates, _get_y_col,
                                          _normalize_coords, create_trivial_matches, to_normalized_image_coords)
    from lib.epipolar.epipolar_ransac import estimate_essential_mat_with_ransac  # noqa: F401
    from lib.epipolar.triangulation import triangulate_points  # noqa: F401
    from lib.feature_matching.matching import Match
    from lib.ransac.ransac import ErrorAggregationMethod
    from lib.transforms.transforms import Transform3D
    import structure_from_motion_b200.epipolar.eight_point as impl
    import lib.epipolar.eight_point as alias

    assert alias is impl
    assert issubclass(EightPointCalculationError, Exception)
    assert [m.value for m in ErrorAggregationMethod] == ["sum", "square", "mean", "rms"]
    assert Match().a_index == -1 and Match().match_score == float("inf") and Match(0, 1, 0.1) < Match(0, 1, 0.2)
    ms = create_trivial_matches(3)
    assert [(m.a_index, m.b_index, m.match_score) for m in ms] == [(0, 0, 0.0), (1, 1, 0.0), (2, 2, 0.0)]
    # test_epipolar.py:30-46
    fa, fb = [Feature(256, 128), Feature(128, 64)], [Feature(32, 64), Feature(16, 8)]
    ca, cb = _get_matching_coordinates(fa, fb, [Match(0, 1), Match(1, 0)])
    assert ca.tolist() == [[256, 128], [128, 64]] and cb.tolist() == [[16, 8], [32, 64]]
    # test_epipolar.py:49-61
    nc, t = _normalize_coords(np.array([[10, 10], [15, 10], [5, 10]]))
    d = np.sqrt(2.0) * 3.0 / 2.0
    np.testing.assert_allclose(nc, [[0, 0], [d, 0], [-d, 0]], atol=1e-15)
    back = (np.hstack([nc, np.ones((3, 1))]) @ np.linalg.inv(t).T)[:, :2]
    np.testing.assert_allclose(back, [[10, 10], [15, 10], [5, 10]])
    # test_epipolar.py:64-85
    assert _get_y_col(np.array([2.0, 3.0]), np.array([7.0, 6.0])).tolist() == [14, 21, 7, 12, 18, 6, 2, 3, 1]
    # test_epipolar.py:95-106
    K = np.array([[50.0, 0, 256], [0, 50.0, 128], [0, 0, 1]])
    nf = to_normalized_image_coords(Feature(x=50, y=60), K)
    exp = np.linalg.inv(K) @ np.array([50, 60, 1.0])
    np.testing.assert_allclose([nf.x, nf.y], exp[:2] / exp[2])
    # Transform3D (transforms.py:10-66)
    T = Transform3D.from_rmat_t(np.eye(3), np.array([1.0, 2.0, 3.0]))
    assert T.t.tolist() == [1, 2, 3] and np.array_equal(T.Rmat, np.eye(3))
    assert np.allclose((T @ T.inv()).Tmat, np.eye(4)) and np.array_equal(Transform3D.identity().Tmat, np.eye(4))
    with pytest.raises(ValueError):
        Transform3D(np.eye(3))
    with pytest.raises(ValueError):
        Transform3D.from_rmat_t(np.eye(2))
    with pytest.raises(TypeError):
        T * 3


def test_argument_errors_before_any_gpu_work():
    from lib.common.feature import Feature
    from lib.epipolar import eight_point, epipolar_ransac, triangulation
    from lib.transforms.transforms import Transform3D

    f = [Feature(1.0, 2.0)] * 3
    with pytest.raises(ValueError, match="Exactly eight matches are needed"):
        eight_point.estimate_fundamental_mat(f, f, eight_point.create_trivial_matches(3))
    with pytest.raises(ValueError, match="Exactly eight matches are needed"):
        eight_point.estimate_essential_mat(camera_matrix=np.eye(3), features_a=f, features_b=f,
                                           matches=eight_point.create_trivial_matches(3))
    with pytest.raises(ValueError, match="Need some matching features"):
        eight_point.estimate_r_t(np.eye(3), [], [], [])
    with pytest.raises(ValueError, match="Eight feature pairs are expected"):
        epipolar_ransac.eight_point_model_fitter([(f[0], f[0])] * 3, np.eye(3))
    with pytest.raises(ValueError, match="not 3x3"):
        triangulation.triangulate_points(f, f, np.eye(4), Transform3D.identity())
    random.seed(3)
    with pytest.raises(ValueError, match="Eight feature pairs are expected"):
        epipolar_ransac.estimate_essential_mat_with_ransac(np.eye(3), f, f, eight_point.create_trivial_matches(3), 0.01)
    st = random.getstate()
    random.seed(3)
    random.shuffle(list(range(3)))
    assert random.getstate() == st  # one shuffle happened, as in the reference, before the fitter raised


def test_scene_generator_is_deterministic():
    from structure_from_motion_b200.scenes import euler_xyz_intrinsic, make_scene

    a, b = make_scene(100, 0.4, 3), make_scene(100, 0.4, 3)
    assert all(np.array_equal(u, v) for u, v in zip(a, b))
    K, x1, x2, R, t, idx = a
    assert len(idx) == 40 and np.allclose(R @ R.T, np.eye(3)) and abs(np.linalg.det(R) - 1) < 1e-12
    assert x1.shape == (100, 2) and np.isfinite(x2).all()
    assert np.allclose(euler_xyz_intrinsic(0, 0, 90), [[0, -1, 0], [1, 0, 0], [0, 0, 1]])


def test_middlebury_parameter_file(tmp_path):
    """lib/data_utils/tests/test_middlebury_utils.py with the same two-entry file."""
    from lib.data_utils.middlebury_utils import load_camera_k_r_t
    from lib.transforms.transforms import Transform3D

    par = tmp_path / "test_par.txt"
    par.write_text("2\nfile01.png 1 2 3 4 5 6 7 8 9 1 2 3 4 5 6 7 8 9 1 2 3\n"
                   "file02.png 9 8 7 6 5 4 3 2 1 9 8 7 6 5 4 3 2 1 3 2 1\n")
    k, transform = load_camera_k_r_t(par, 1)
    np.testing.assert_almost_equal(np.arange(1, 10).reshape(3, 3), k)
    expected = Transform3D.from_rmat_t(np.arange(1.0, 10.0).reshape(3, 3), np.arange(1.0, 4.0).reshape(3, 1))
    np.testing.assert_almost_equal(expected.Tmat, transform.Tmat)
    k2, t2 = load_camera_k_r_t(par, 2)
    assert k2[0, 0] == 9 and t2.t.tolist() == [3, 2, 1]
    with pytest.raises(ValueError, match="There are 2 entries"):
        load_camera_k_r_t(par, 3)
    par.write_text("5\nfile01.png 1 2 3 4 5 6 7 8 9 1 2 3 4 5 6 7 8 9 1 2 3\n")
    with pytest.raises(ValueError, match="Could not find"):
        load_camera_k_r_t(par, 4)
    par.write_text("1\nnonsense 1 2 3\n")
    with pytest.raises(RuntimeError, match="Could not decode"):
        load_camera_k_r_t(par, 1)


def test_front_end_host_logic():
    """What the front-end mirrors decide on the host: window bookkeeping, the Gaussian table, which score functions
    the GPU may evaluate itself, validation-strategy normalisation, errors raised before any GPU work."""
    from lib.blur import gaussian
    from lib.common.feature import Feature
    from lib.feature_matching import matching, ncc, ssd, util
    from lib.harris import harris_detector as harris

    # util.py:8-27 (test_util.py): float comparison for the bounds, int() for the slice
    assert util.is_within_bounds(Feature(1, 1), (3, 3), 3) and not util.is_within_bounds(Feature(0, 1), (3, 3), 3)
    assert not util.is_within_bounds(Feature(1, 2), (3, 3), 3) and util.is_within_bounds(Feature(1.9, 1.0), (3, 3), 3)
    img = np.arange(25).reshape(5, 5)
    assert util.select_window(img, Feature(2.7, 1.2), 3).tolist() == [[1, 2, 3], [6, 7, 8], [11, 12, 13]]
    # gaussian.py:4-26 (test_gaussian.py)
    g = gaussian.create_gaussian_kernel(3, 1.0)
    assert g.shape == (3, 3) and abs(g.sum() - 1.0) < 1e-15 and g[1, 1] == g.max() and np.allclose(g, g.T)
    for bad in (2, 4, 1):
        with pytest.raises(ValueError):
            gaussian.create_gaussian_kernel(bad, 1.0)
    # score-function recognition
    a, b = np.zeros((8, 8), dtype=np.uint8), np.ones((8, 8), dtype=np.uint8)
    p = matching._recognise(functools.partial(ncc.calculate_ncc, a, b, window_size=5))
    assert p is not None and (p.kind, p.window_size) == ("ncc", 5) and p.image_a is a and p.image_b is b
    p = matching._recognise(functools.partial(ssd.calculate_ssd, image_a=a, image_b=b))
    assert p is not None and (p.kind, p.window_size) == ("ssd", 5)

    def create(image_a, image_b, full):  # apps/sfm.py:266-277
        def score(fa, fb):
            return full(image_a, image_b, fa, fb)
        return score

    p = matching._recognise(create(a, b, functools.partial(ncc.calculate_ncc, window_size=9)))
    assert p is not None and (p.kind, p.window_size) == ("ncc", 9) and p.image_a is a
    assert matching._recognise(create(a, b, ncc.calculate_ncc)).window_size == 3
    assert matching._recognise(lambda fa, fb: 0.0) is None
    assert matching._recognise(functools.partial(ncc.calculate_ncc, a)) is None            # one image only
    assert matching._recognise(functools.partial(ncc.calculate_ncc, a, b[:4])) is None     # shapes differ: the call raises later
    assert matching._recognise(create(a, b, lambda *x: 0.0)) is None
    # enum values and the trivial outcomes that need no GPU
    assert matching.ValidationStrategy.CROSSCHECK.value == 1 and matching.ValidationStrategy.RATIO_TEST.value == 2
    assert matching.match_brute_force([], [Feature(1, 1)], lambda fa, fb: 0.0) == []
    with pytest.raises(IndexError):
        matching.match_brute_force([Feature(1, 1)], [], lambda fa, fb: 0.0)
    assert matching.match_brute_force([Feature(1, 1)], [], lambda fa, fb: 0.0,
                                      validation_strategies=matching.ValidationStrategy.RATIO_TEST) == []
    with pytest.raises(ValueError, match="at least 1"):
        harris.detect_harris_corners(np.zeros((8, 8)), num_corners=0)


@pytest.mark.parametrize("n,h,budget", [(500, 300, 64 << 20), (40, 1000, 4096), (1000, 77, 100_000)])
def test_reference_sampler_snapshots(n, h, budget, monkeypatch):
    """_native.ReferenceSampler (chunked, snapshot + short replay) against the one-shot sampler and CPython itself."""
    monkeypatch.setattr(_native.ReferenceSampler, "SNAPSHOT_BYTES", budget)
    random.seed(17)
    st0 = np.array(random.getstate()[1], dtype=np.uint32)
    rs = _native.ReferenceSampler(st0, n, h)
    assert rs.stride == max(1, -(-h // 64), -(-(h * n * 4) // budget)) and len(rs._states) <= 64
    w = st0.copy()
    table, _ = _native.mt_shuffle_table(w, n, h)
    assert np.array_equal(rs.table, table) and np.array_equal(rs.final_state, w)
    assert np.array_equal(st0, np.array(random.getstate()[1], dtype=np.uint32))  # the caller's state is not touched
    data = list(range(n))
    for it in range(h):
        random.shuffle(data)
        if it in (0, 1, h // 3, h - 2, h - 1):
            st, perm = rs.after(it)
            assert perm.tolist() == data and st.tolist() == list(random.getstate()[1])


def test_reference_error_matches_the_reference_aggregation():
    """two_view._reference_error is what settles near-ties (SURVEY H1): the same floating-point value as
    _aggregate_error (lib/ransac/ransac.py:96-108) on the same list, for every aggregation."""
    from oracle import restatement as o
    from structure_from_motion_b200 import two_view

    rng = np.random.default_rng(3)
    for n in (1, 8, 9, 130, 4097):
        errs = [float(v) for v in rng.uniform(0, 1e-6, n) ** 2]
        for agg in ("sum", "square", "mean", "rms"):
            assert two_view._reference_error(errs, agg) == o.aggregate_error(errs, agg)


def test_aggregation_name_accepts_any_enum_with_the_reference_values():
    """ransac.py:99-105 compares ``.value``: an Enum of another module with the same values must work (ADVICE r1)."""
    import enum

    from structure_from_motion_b200 import two_view
    from structure_from_motion_b200.ransac.ransac import ErrorAggregationMethod

    class Foreign(enum.Enum):
        SUM = "sum"
        RMS = "rms"

    assert two_view._agg_name(Foreign.SUM) == "sum" and two_view._agg_name(Foreign.RMS) == "rms"
    assert two_view._agg_name(ErrorAggregationMethod.MEAN) == "mean" and two_view._agg_name(None) == "rms"
    assert two_view._agg_name("square") == "square"


def test_near_tie_replay_with_a_scripted_engine():
    """_resolve_near_ties: strict < in iteration order on list-order sums (ransac.py:83), from per-hypothesis scores."""
    from structure_from_motion_b200 import two_view

    class Fake:
        def __init__(self, seds):
            self.seds, self.cur = seds, None

        def set_winner(self, t):
            self.cur = t

        def inlier_mask(self, thr):
            s = self.seds[self.cur]
            return s <= thr, s

    thr = 1.0
    base = np.array([0.25, 0.5, 0.125, 2.0, 0.0625, 0.5, 0.25, 0.125, 0.5, 0.75])
    seds = {3: base, 7: base.copy(), 9: base * (1 - 2 ** -40)}
    rows = lambda t: np.arange(8)  # noqa: E731
    after = lambda t: np.array([8, 9])  # noqa: E731
    t, e = two_view._resolve_near_ties(Fake(seds), [3, 7, 9], thr, "sum", rows, after)
    assert t == 9 and e == sum(float(v) for v in seds[9][[0, 1, 2, 3, 4, 5, 6, 7, 8, 9]] if True)
    seds[9] = base.copy()
    t, e = two_view._resolve_near_ties(Fake(seds), [3, 7, 9], thr, "rms", rows, after)
    assert t == 3  # exact ties keep the earliest iteration


def test_near_tie_replay_and_inlier_order_for_4_point_samples():
    """The shared replay and inlier-order helpers at the homography path's sample size: the list order is the first
    four table columns, then the rest (columns 4-7 are not part of the sample); the replay runs only for 2..64 near-ties
    of min_error on a host-side sampler."""
    import types

    from structure_from_motion_b200 import two_view

    class Fake:
        def __init__(self, ties, total):
            self.ties, self.total = ties, total

        def near_ties(self, rel_tol, cap):
            return np.array(self.ties), self.total

    class Ref:  # ReferenceSampler.after(t) -> (state, permutation of iteration t); it starts with table[t][:4]
        def after(self, t):
            return None, np.array({1: [1, 2, 3, 4, 9, 8, 7, 6, 5, 0], 2: [2, 3, 4, 5, 9, 0, 7, 1, 6, 8]}[t])

    n, thr = 10, 1.0
    table = np.array([[t, t + 1, t + 2, t + 3, 9, 9, 9, 9] for t in range(4)], dtype=np.int32)
    errs = {1: np.full(n, 0.5), 2: np.array([0.5, 2.0, 0.25, 0.5, 0.5, 0.5, 0.125, 0.5, 3.0, 0.0625])}
    errs[1][9] = 0.0625 * (1 + 2 ** -45)
    score = lambda t: (errs[t] <= thr, errs[t])  # noqa: E731

    def list_order_error(t, rest):
        e, inl = errs[t], errs[t] <= thr
        return sum([float(v) for v in e[table[t][:4]]] + [float(v) for v in e[rest][inl[rest]]])

    eng = Fake([1, 2], 2)
    for ref, sampler in ((None, "table"), ((Ref(), 3, None), "reference")):
        t, e = two_view._replay_near_ties(eng, sampler, "min_error", table, ref, n, 4, thr, "sum", score)
        rest = {1: np.array([0, 5, 6, 7, 8, 9]), 2: np.array([0, 1, 6, 7, 8, 9])}
        if ref is not None:
            rest = {1: np.array([9, 8, 7, 6, 5, 0]), 2: np.array([9, 0, 7, 1, 6, 8])}
        want = min((1, 2), key=lambda u: (list_order_error(u, rest[u]), u))
        assert t == want and e == list_order_error(want, rest[want])
    assert two_view._replay_near_ties(eng, "device", "min_error", table, None, n, 4, thr, "sum", score) is None
    assert two_view._replay_near_ties(eng, "table", "max_inliers", table, None, n, 4, thr, "sum", score) is None
    for total in (1, 65):
        assert two_view._replay_near_ties(Fake([1], total), "table", "min_error", table, None, n, 4, thr, "sum",
                                          score) is None

    mask = errs[2] <= thr
    best = types.SimpleNamespace(index=2, sample=[7, 0, 3, 5, 1, 2, 4, 6])
    sample, inl = two_view._inlier_order(best, "table", table, None, mask, 4)
    assert sample.dtype == np.int32 and sample.tolist() == [2, 3, 4, 5] and inl.tolist() == [2, 3, 4, 5, 0, 6, 7, 9]
    sample, inl = two_view._inlier_order(best, "reference", table, (Ref(), 3, None), mask, 4)
    assert sample.tolist() == [2, 3, 4, 5] and inl.tolist() == [2, 3, 4, 5, 9, 0, 7, 6]
    sample, inl = two_view._inlier_order(best, "device", table, None, mask, 4)
    assert sample.tolist() == [7, 0, 3, 5] and inl.tolist() == [7, 0, 3, 5, 2, 4, 6, 9]
    sample, inl = two_view._tail_inliers(best, np.array([0, 2, 3, 5, 7, 9], dtype=np.int64), 4)
    assert sample.tolist() == [7, 0, 3, 5] and inl.dtype == np.int64 and inl.tolist() == [7, 0, 3, 5, 2, 9]
