"""CPU checks of the helpers behind tests/test_gpu_pnp_edges.py: make_pnp_samples, the overflow-safe bearings, the
cubic-branch restatement and the inlier rule's range terms in reproj_exact.c and its numpy restatement.  No GPU."""
import numpy as np
import pytest

from oracle import creproj
from oracle import pnp as op
from structure_from_motion_b200.scenes import make_pnp_samples, random_rotation

pytestmark = pytest.mark.filterwarnings("ignore::RuntimeWarning")


def test_samples_are_consistent():
    """make_pnp_samples: R is a rotation, every point is in front of the camera and projects to its pixel, the first
    six samples look along +-x, +-y, +-z, and the exact fit of a noise-free sample is the true pose to 1e-6."""
    samples = make_pnp_samples(60, seed=1)
    axes = [s[3][2] for s in samples[:6]]
    assert np.allclose(np.abs(np.array(axes)).sum(axis=0), 2.0)
    for K, X, x, R, t in samples:
        assert abs(np.linalg.det(R) - 1) < 1e-12 and np.abs(R @ R.T - np.eye(3)).max() < 1e-12
        cam = X @ R.T + t
        assert (cam[:, 2] > 0).all()
        p = cam @ K.T
        assert np.allclose(p[:, :2] / p[:, 2:], x, rtol=0, atol=1e-6)
        Rt, info = op.fit_pnp_exact(K, X, x)
        assert Rt is not None
        assert np.abs(Rt - np.column_stack([R, t])).max() <= 1e-6 * (1 + np.abs(t).max())


def test_random_rotation_is_uniform():
    """The trace of a uniform rotation has mean 0 (E[1 + 2 cos angle] over the Haar measure)."""
    rng = np.random.default_rng(0)
    tr = [np.trace(random_rotation(rng)) for _ in range(4000)]
    assert abs(np.mean(tr)) < 0.05


def test_bearings_beyond_overflow():
    """A pixel 1e160 off axis: the plain norm overflows, the bearing is still the unit vector (exact to 1 ulp)."""
    K = np.array([[800.0, 0, 640], [0, 800, 480], [0, 0, 1]])
    b = op.bearings(K, np.array([[8e159 + 640, 4e159 + 480], [700.0, 500.0]]))
    assert np.allclose(np.linalg.norm(b, axis=1), 1.0, rtol=0, atol=2e-16)
    assert np.allclose(b[0], np.array([2, 1, 2e-157]) / np.sqrt(5), rtol=1e-15, atol=0)
    assert op.bearings(K, np.array([[np.inf, 0.0]]))[0][0] != op.bearings(K, np.array([[np.inf, 0.0]]))[0][0]


def test_cubic_branch_reaches_both():
    """Both branches of cubic_roots occur among 400 random samples, and a sample's branch does not depend on its
    world scale (the cubic's coefficients all scale by the same power)."""
    seen = set()
    for K, X, x, R, t in make_pnp_samples(400, seed=3):
        y = op.bearings(K, x[:3])
        b = op.cubic_branch(y, X[:3])
        assert b == op.cubic_branch(y, X[:3] * 2.0 ** 40)
        seen.add(b)
    assert seen == {1, 3}


def test_inlier_rule_range_terms():
    """The decision's range terms, in the C scorer and its numpy restatement alike: a finite record with F = W = inf
    (far off the ray), one with F finite and W inf (on the ray, value 0), and p2 below 2^-537 (W = 0)."""
    K = np.array([[800.0, 0, 640], [0, 800, 480], [0, 0, 1]])
    Rt = np.column_stack([np.eye(3), np.zeros(3)])
    X = np.array([[0.0, 0.0, 5.0], [3e159, 0.0, 1e160], [0.0, 0.0, 1e160], [0.0, 0.0, 2.0 ** -538],
                  [0.0, 0.0, 2.0 ** -537], [1e300, 1e300, 1e300]])
    x = np.array([[640.0, 480.0]] * 6)
    for thr in (4.0, 1e100):
        m_c, v_c = creproj.reproj_exact_many(Rt, K, X, x, thr)
        m_n, v_n = op.reproj(Rt, K, X, x, thr)
        assert m_c.tolist() == m_n.tolist() == [True, False, True, False, True, False]
        assert np.isfinite(v_c[m_c]).all()
        assert np.isnan(v_c[1]) and v_c[2] == 0.0
