"""The front-end oracle (oracle/front_end.py: brute-force matcher, NCC/SSD, Harris, cross-correlation) pinned
against golden vectors generated from the unmodified reference (tests/golden/make_golden.py).  No GPU needed."""
import json
import os

import numpy as np
import pytest

from oracle import front_end as fe

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def load(name):
    with open(os.path.join(G, name)) as f:
        return json.load(f)


@pytest.fixture(scope="module")
def matching_golden():
    d = load("matching_known_answer.json")
    d["image_a"] = np.array(d["image_a"], dtype=np.uint8)
    d["image_b"] = np.array(d["image_b"], dtype=np.uint8)
    d["feats_a"], d["feats_b"] = np.array(d["feats_a"]), np.array(d["feats_b"])
    return d


def test_patch_scores_match_reference(matching_golden):
    d = matching_golden
    for case in d["cases"]:
        if case["scores"] is None:
            continue
        S = fe.score_matrix(d["image_a"], d["image_b"], d["feats_a"], d["feats_b"], case["kind"], case["window"])
        assert np.array_equal(S, np.array(case["scores"]))  # the same numpy calls => the same bits
    # both kinds of "outside" are present in the fixture
    S = fe.score_matrix(d["image_a"], d["image_b"], d["feats_a"], d["feats_b"], "ssd", 5)
    assert np.isinf(S[0]).all() and np.isfinite(S).any()


def test_matcher_matches_reference(matching_golden):
    d = matching_golden
    scores = {}
    for case in d["cases"]:
        key = (case["kind"], case["window"])
        if case["scores"] is not None:
            scores[key] = np.array(case["scores"])
        got = fe.match_from_scores(scores[key], "RATIO_TEST" in case["strategies"], "CROSSCHECK" in case["strategies"],
                                   case["ratio"])
        assert [[a, b, s] for a, b, s in got] == case["matches"], (case["kind"], case["strategies"])


def test_heap_closed_form_equals_heapq():
    rng = np.random.default_rng(0)
    for trial in range(300):
        n = int(rng.integers(1, 70))
        if trial % 3 == 0:
            s = rng.integers(0, 4, n).astype(float)  # many ties
        elif trial % 3 == 1:
            s = rng.random(n)
            s[rng.random(n) < 0.2] = np.inf
        else:
            s = np.sort(rng.random(n))[::(-1 if trial % 2 else 1)]
        assert fe.heap_top2(s) == fe.heap_top2_closed_form(s), s


@pytest.fixture(scope="module")
def harris_golden():
    d = load("harris_known_answer.json")
    d["image"] = np.array(d["image"], dtype=np.uint8)
    return d


def test_harris_matches_reference(harris_golden):
    d = harris_golden
    for case in d["cases"]:
        raw = fe.cornerness_image(d["image"], case["block_size"], case["k"])
        assert np.array_equal(raw, np.array(case["cornerness_raw"]))
        xy, score, cim = fe.harris_corners(d["image"], case["num_corners"], case["block_size"], case["k"])
        assert np.array_equal(cim, np.array(case["cornerness"]))
        ref = np.array(case["corners"]).reshape(-1, 2)
        assert len(xy) == len(ref)
        _assert_same_corners(xy, score, ref, cim, case["block_size"])


def _assert_same_corners(xy, score, ref_xy, cim, block_size):
    """Same sequence wherever the cornerness values are distinct; the same set inside a group of exact ties."""
    off = block_size / 2.0
    ref_score = np.array([cim[int(y - off), int(x - off)] for x, y in ref_xy])
    assert np.array_equal(ref_score, score)  # descending values agree position by position
    for v in np.unique(score):
        g = score == v
        assert sorted(map(tuple, xy[g])) == sorted(map(tuple, ref_xy[g]))


def test_harris_reference_fixtures(harris_golden):
    d = harris_golden
    sq = np.array(d["square"]["image"], dtype=np.uint8)
    xy, _, _ = fe.harris_corners(sq, 4)
    assert sorted(map(tuple, xy)) == sorted(map(tuple, d["square"]["corners"]))
    r = d["rectangle"]
    img = np.zeros(r["shape"])
    img[r["fill"][0]:r["fill"][1], r["fill"][2]:r["fill"][3]] = 255.0
    xy, _, _ = fe.harris_corners(img)
    assert sorted(map(tuple, xy)) == sorted(map(tuple, r["corners"]))
    # test_harris_detector.py:27-31: each expected corner within one pixel of a detected one
    for ey, ex in r["expected_yx"]:
        assert min(max(abs(x - ex), abs(y - ey)) for x, y in xy) <= 1.0


def test_nms_fixed_point_equals_sequential_scan():
    rng = np.random.default_rng(1)
    for trial in range(40):
        shape = (int(rng.integers(1, 24)), int(rng.integers(1, 24)))
        v = rng.integers(0, 5, shape).astype(float) if trial % 2 else rng.random(shape)
        if trial % 5 == 0:
            v = np.sort(v.ravel())[::-1].reshape(shape)  # long dependency chains
        seq = v.copy()
        fe.non_max_suppress(seq)
        fp, sweeps = fe.non_max_suppress_fixed_point(v)
        assert np.array_equal(seq, fp), (trial, sweeps)


def test_cross_correlate_matches_reference(harris_golden):
    d = harris_golden["correlate"]
    img = harris_golden["image"]
    kern = np.array(d["kernel"])
    assert np.array_equal(fe.cross_correlate(img[:20, :24].astype(np.float64) / 255.0, kern), np.array(d["result"]))
    assert np.array_equal(fe.cross_correlate(img[:20, :24], fe.SOBEL_X), np.array(d["sobel_u8"]))
    with pytest.raises(ValueError):
        fe.cross_correlate(img, np.ones((2, 2)))
    with pytest.raises(ValueError):
        fe.cross_correlate(img[:2, :2], np.ones((3, 3)))


def test_front_end_matches_live_reference(matching_golden, harris_golden):
    """Score matrices, matches and Harris corners on crops of the fixtures against what the unmodified reference
    returned for them (front_end_known_answer.json, tests/golden/make_golden.py)."""
    d = matching_golden
    g = load("front_end_known_answer.json")
    na, nb = g["num_features"]
    for case in g["cases"]:
        S = fe.score_matrix(d["image_a"], d["image_b"], d["feats_a"][:na], d["feats_b"][:nb], case["kind"], case["window"])
        assert np.array_equal(S, np.array(case["scores"]))
        for m in case["matching"]:
            got = fe.match_from_scores(S, "RATIO_TEST" in m["strategies"], "CROSSCHECK" in m["strategies"], g["ratio"])
            assert [[a, b, s] for a, b, s in got] == m["matches"], (case["kind"], m["strategies"])
    h = g["harris"]
    xy, _, _ = fe.harris_corners(harris_golden["image"][:h["rows"], :h["cols"]], h["num_corners"])
    assert sorted(map(tuple, h["corners"])) == sorted(map(tuple, xy))


# ---- property-based checks (the reference's own suite uses hypothesis for its geometry tests) ----
from hypothesis import given, settings  # noqa: E402
from hypothesis import strategies as st  # noqa: E402

_scores = st.lists(st.one_of(st.integers(0, 6).map(float), st.floats(0, 2, allow_nan=False), st.just(float("inf"))),
                   min_size=1, max_size=80)


@settings(max_examples=150, deadline=None)
@given(_scores)
def test_heap_closed_form_property(scores):
    """heap[0] / heap[1] of the reference's per-feature heapq, without the heap: any length, ties, infinities."""
    assert fe.heap_top2(scores) == fe.heap_top2_closed_form(scores)


@settings(max_examples=60, deadline=None)
@given(st.integers(1, 14), st.integers(1, 14), st.integers(0, 2 ** 32 - 1), st.booleans())
def test_nms_fixed_point_property(rows, cols, seed, ties):
    """The parallel fixed point equals the reference's in-place row-major scan on arbitrary non-negative images."""
    rng = np.random.default_rng(seed)
    v = rng.integers(0, 4, (rows, cols)).astype(float) if ties else rng.random((rows, cols))
    seq = v.copy()
    fe.non_max_suppress(seq)
    fp, sweeps = fe.non_max_suppress_fixed_point(v)
    assert np.array_equal(seq, fp) and sweeps <= rows * cols + 1


@settings(max_examples=40, deadline=None)
@given(st.integers(2, 12), st.integers(1, 12), st.integers(0, 2 ** 32 - 1), st.booleans(), st.booleans(),
       st.floats(0.05, 1.5))
def test_matcher_cross_check_is_an_injection(na, nb, seed, ratio, many_ties, thr):
    """With CROSSCHECK every feature of B is used at most once and each kept match is the lowest-scored (earliest on
    ties) surviving match of its B feature (matching.py:100-118)."""
    rng = np.random.default_rng(seed)
    S = rng.integers(0, 3, (na, nb)).astype(float) if many_ties else rng.random((na, nb))
    kept = fe.match_from_scores(S, ratio, True, thr)
    bs = [b for _, b, _ in kept]
    assert len(set(bs)) == len(bs)
    survivors = fe.match_from_scores(S, ratio, False, thr)
    for a, b, s in kept:
        rivals = [(s2, a2) for a2, b2, s2 in survivors if b2 == b]
        assert (s, a) == min(rivals)
