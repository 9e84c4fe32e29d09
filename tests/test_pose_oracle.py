"""CPU checks of oracle/pose_exact.py — the exact decomposition, null vector and cheirality quantities the pose-tail
edge tests measure the GPU against — against numpy's SVD route (oracle/restatement.py) on well-conditioned inputs, and
the host build of csrc/sfm_fastsvd.cuh on the sweeps those tests run, to confirm by construction that both routes of
svd3_rank2_frames and of null_vector4_fast are taken (the device uses rsqrt where the host uses 1 / sqrt, so the host
build only says which route a case takes well away from the switch)."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import pose_exact as px
from oracle import restatement as o

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
U = px.U


def test_decomposition_matches_numpy_on_well_conditioned_e():
    rng = np.random.default_rng(1)
    for E in [px.true_essential(rng) for _ in range(6)] + [px.rank2(r, rng) for r in (1.0, 0.5, 0.1) for _ in range(4)]:
        ex = px.decompose_exact(E)
        R1, R2, t = o.recover_all_r_t(E)
        er, et = px.candidate_error(R1, R2, t, ex)
        assert er <= 64 * U * ex.cond and et <= 64 * U * ex.cond, (er, et, ex.cond)
        assert ex.accepted and abs(ex.s[2]) < 1e-15
        for R in (ex.R1, ex.R2):
            assert np.abs(R.T @ R - np.eye(3)).max() < 4 * U and abs(np.linalg.det(R) - 1) < 8 * U
        assert abs(np.linalg.norm(ex.t) - 1) < 4 * U
        assert np.allclose(ex.s, np.linalg.svd(E, compute_uv=False), rtol=0, atol=8 * U * ex.s[0])


def test_decision_follows_isclose():
    rng = np.random.default_rng(2)
    for f in (0.5, 0.99, 1.01, 2.0):
        E = px.with_singular_values([1.0, 0.6, f * px.SV_LIMIT], rng)
        ex = px.decompose_exact(E)
        assert ex.accepted == (f < 1), (f, ex.s)
        assert ex.accepted == bool(np.isclose(0.0, np.linalg.svd(E, compute_uv=False)[-1]))


def test_null_vector_matches_numpy_on_well_conditioned_systems():
    rng = np.random.default_rng(3)
    for s in ([1.0, 0.3, 1e-2, 5e-3], [1.0, 0.9, 0.8, 0.4], [2.0, 1.0, 0.5, 0.0]):
        for _ in range(4):
            A = px.with_singular_values(s, rng)
            ex = px.null_exact(A)
            assert np.allclose(ex.s, np.linalg.svd(A, compute_uv=False), rtol=0, atol=8 * U * ex.s[0])
            vh = np.linalg.svd(A)[2][-1]
            X = vh[:3] / vh[3]
            assert px.direction_error(X, ex) <= 64 * U / ex.gap
            assert abs(px.residual_excess(A, X)) <= 16 * U * ex.s[0]
            assert abs(np.linalg.norm(ex.x) - 1) < 4 * U and ex.x[3] >= 0
            P1, P2 = px.cameras_for(A)
            assert np.array_equal(px.dlt_system(0.0, 0.0, 0.0, 0.0, P1, P2), A)
            assert np.array_equal(px.dlt_system(0.3, -0.2, 0.1, 0.7, np.eye(4)[:3], P2[:3]),
                                  np.array([-0.2 * np.eye(4)[2] - np.eye(4)[1], np.eye(4)[0] - 0.3 * np.eye(4)[2],
                                            0.7 * P2[2] - P2[1], P2[0] - 0.1 * P2[2]]))


def test_cheirality_quantities_follow_the_reference():
    rng = np.random.default_rng(4)
    R, t, na, nb = px.scene(40, rng, parallax=0.05, noise=1e-4)
    E = px.essential_of(R, t)
    R1, R2, t1 = o.recover_all_r_t(E)
    clear = 0
    for Rc, tc in ((R1, t1), (R1, -t1), (R2, t1), (R2, -t1)):
        for i in range(len(na)):
            c = px.cheirality_exact(na[i, 0], na[i, 1], nb[i, 0], nb[i, 1], Rc, tc, lambda ex: 1e-9)
            if c.clear(50.0):
                clear += 1
                assert c.passes(50.0) == o.cheirality_check(na[i, 0], na[i, 1], nb[i, 0], nb[i, 1], Rc, tc)
    assert clear >= 150


def test_sweeps_are_reproducible():
    a = px.null_sweep()
    b = px.null_sweep()
    assert all(np.array_equal(x[2], y[2]) for x, y in zip(a, b))
    assert len(px.decomposition_sweep()) == len(px.decomposition_sweep())


def _host_build(tmp_path_factory):
    from structure_from_motion_b200 import build as b

    try:
        nvcc = b._nvcc()
    except RuntimeError:
        pytest.skip("no nvcc: the host build of sfm_fastsvd.cuh cannot be made")
    out = str(tmp_path_factory.mktemp("fastsvd") / "libfastsvd.so")
    subprocess.check_call([nvcc, "-O2", "-shared", "-Xcompiler", "-fPIC", "-Wno-deprecated-gpu-targets", "-o", out,
                           os.path.join(ROOT, "tools", "fastsvd_check.cu")])
    return ctypes.CDLL(out)


def test_sweeps_take_both_routes_on_the_host_build(tmp_path_factory):
    lib = _host_build(tmp_path_factory)
    P = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    fast = fallback = 0
    for fam, r, A in px.null_sweep():
        A = np.ascontiguousarray(A)
        x = np.empty(4)
        ok = bool(lib.null4(P(A), P(x)))
        if r <= px.NULL_FAST_MAX:
            assert ok, (fam, r)
            fast += 1
        elif r >= px.NULL_FALLBACK_MIN:
            assert not ok, (fam, r)
            fallback += 1
    assert fast and fallback
    closed = jac = 0
    for name, E in px.decomposition_sweep():
        E = np.ascontiguousarray(E)
        Uf, Vf, s = np.empty(9), np.empty(9), np.empty(3)
        ok = bool(lib.frames3(P(E), P(Uf), P(Vf), P(s)))
        if name == "fallback":
            assert not ok
            jac += 1
        elif name.startswith("essential_") or (name.startswith("rank2_") and float(name[6:]) >= 1e-6):
            assert ok, name
            closed += 1
    assert closed and jac
