"""oracle/fit_exact.py, the exact eight-point fit K1 is tested against, checked against the reference's own route and
itself; and the reference's exception for samples whose normalised coordinates are not finite, pinned by
tests/golden/nonfinite_sample_fixture.json (generated from the unmodified reference by make_golden.py)."""
import json
import os
import random

import numpy as np
import pytest

from oracle import fit_exact as fx
from oracle import restatement as o
from structure_from_motion_b200 import two_view
from structure_from_motion_b200.scenes import make_scene

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def generic_samples(count, seed=11, n=400):
    K, x1, x2, *_ = make_scene(n, 0.5, seed=seed)
    ca = np.stack(o.k_normalise(x1[:, 0], x1[:, 1], K), 1)
    cb = np.stack(o.k_normalise(x2[:, 0], x2[:, 1], K), 1)
    rng = np.random.default_rng(seed)
    return [(ca[s], cb[s]) for s in (rng.choice(n, 8, replace=False) for _ in range(count))]


def test_exact_fit_agrees_with_the_reference_route():
    """restatement.eight_point (np.linalg.eig of Y^T Y, then svd) lands within its own conditioning of E*: its
    null vector errs by O(u kappa(Y)^2), the rank-2 projection multiplies that by rho(F), the denormalisation by amp.
    And E* is what it claims: rank 2, with Y's null vector behind it (sigma_8 > 0 here, E* from the exact null space)."""
    worst = 0.0
    for ca, cb in generic_samples(60):
        f = fx.fit_exact(ca, cb)
        assert f.valid and f.ref_valid and np.isfinite(f.kappa)
        assert f.sv[0] >= f.sv[-1] > 0 and f.kappa == pytest.approx(f.sv[0] / f.sv[-1], rel=1e-12)
        assert f.s8sq == pytest.approx(f.sv[-1] ** 2, rel=1e-12)
        assert f.qr_lo <= f.s8sq * (1 + 1e-12) and f.s8sq <= f.qr_hi * (1 + 1e-12)
        assert abs(f.lam2_ref - f.s8sq) <= 4 * fx.U * f.lam_max_ref  # the reference's lambda_2 near the exact one
        s = np.linalg.svd(f.E_dir, compute_uv=False)
        assert s[2] <= 1e-15 * s[0] and np.linalg.norm(f.E_dir) == pytest.approx(1.0, rel=1e-14)
        d = fx.direction_error(o.eight_point(ca, cb), f)
        bound = 64 * fx.U * f.kappa ** 2 * f.rho * f.amp
        worst = max(worst, d / bound)
        assert d <= bound, (d, bound, f.kappa, f.rho, f.amp)
    print(f"largest reference-route error / (64 u kappa^2 rho amp): {worst:.3g}")


def test_exact_fit_of_an_exactly_degenerate_sample():
    """A repeated correspondence: Y has rank 7, sigma_8 = 0 (to the working precision) and the sample is invalid."""
    ca, cb = generic_samples(1)[0]
    ca[7], cb[7] = ca[2], cb[2]
    f = fx.fit_exact(ca, cb)
    assert not f.valid and not f.ref_valid
    assert f.s8sq <= 1e-60 and f.qr_lo <= 1e-60


def test_design_matrix_is_the_reference_one():
    ca, cb = generic_samples(1)[0]
    Y, _, _ = fx.design(ca, cb)
    na, _ = o.hartley_normalise(ca)
    nb, _ = o.hartley_normalise(cb)
    for i in range(8):
        assert np.array_equal(Y[i], o.y_col(na[i], nb[i]))


def test_ladder_lands_where_it_says():
    """Every ladder sample has sigma_8(Y)^2 = 1e-10 (1 + delta) in exact arithmetic to 1e-6 relative, far inside the
    smallest step (1e-4); the clustered geometry keeps lambda_max(Y^T Y) below 180, the far-point one above it and
    near 1e3; and both geometries are the duplicated-and-nudged kind: sigma_7 stays far above sigma_8."""
    lam = {"clustered": [], "far": []}
    for geo, seed, delta, ca, cb in fx.ladder(seeds=(0, 1)):
        f = fx.fit_exact(ca, cb)
        assert f.s8sq / fx.VERY_SMALL - 1.0 == pytest.approx(delta, abs=1e-6), (geo, seed, delta)
        assert f.valid == (delta > 0)
        assert f.sv[-2] > 1e3 * f.sv[-1]
        lam[geo].append(f.lam_max_ref)
    assert max(lam["clustered"]) <= 180.0
    assert 180.0 < min(lam["far"]) and max(lam["far"]) <= 2e3


def _fixture():
    with open(os.path.join(GOLDEN, "nonfinite_sample_fixture.json")) as f:
        return json.load(f)


def test_degenerate_sample_error_matches_the_reference():
    """The host decision between numpy's LinAlgError and EightPointCalculationError for one degenerate sample
    gives the reference's exception type and message on every eight-point case of the fixture."""
    d = _fixture()
    K = np.array(d["K"])
    for case in d["eight_point"]:
        exc = two_view._degenerate_sample_error(np.array(case["pts_a"]), np.array(case["pts_b"]), K)
        assert case["raises"].split(".")[-1] == type(exc).__name__, case["name"]
        if isinstance(exc, np.linalg.LinAlgError):
            assert case["raises"] == "numpy.linalg.LinAlgError"
        assert str(exc) == case["message"], case["name"]


def test_restatement_reproduces_the_nonfinite_fixture():
    """The numpy restatement raises what the reference raised, and leaves the global random state where it did."""
    d = _fixture()
    K = np.array(d["K"])
    for case in d["eight_point"]:
        ca = np.stack(o.k_normalise(*np.array(case["pts_a"]).T, K), 1)
        cb = np.stack(o.k_normalise(*np.array(case["pts_b"]).T, K), 1)
        with np.errstate(all="ignore"), pytest.raises((np.linalg.LinAlgError, o.OracleEightPointError)) as info:
            o.eight_point(ca, cb)
        want = np.linalg.LinAlgError if case["raises"] == "numpy.linalg.LinAlgError" else o.OracleEightPointError
        assert isinstance(info.value, want) and str(info.value) == case["message"], case["name"]
    for case in d["ransac"]:
        pa, pb = np.array(case["pts_a"]), np.array(case["pts_b"])
        random.seed(case["seed"])
        with np.errstate(all="ignore"), pytest.raises((np.linalg.LinAlgError, o.OracleEightPointError)) as info:
            o.ransac_essential(K, pa[:, 0], pa[:, 1], pb[:, 0], pb[:, 1], case["threshold"], None, "rms",
                               case["max_iterations"])
        assert str(info.value) == case["message"], case["name"]
        assert list(random.getstate()[1]) == case["state_after"], case["name"]
