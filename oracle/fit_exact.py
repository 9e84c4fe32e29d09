"""TEST INFRASTRUCTURE ONLY — the eight-point fit of one sample in exact arithmetic, and samples placed where K1's
validity test is hard to call.

The design matrix Y (8x9) is built in double exactly as the reference builds it (restatement.hartley_normalise and
y_col, eight_point.py:308-393; K1 and numpy produce the same rounded Y) and is then taken as exact.  Everything after
it is computed in mpmath at ``DPS`` digits: the singular values of Y, its null vector, the rank-2 projection
(eight_point.py:430-446) and E* = T2^T F' T1 (:163).  What that gives a test:

- ``E_dir``: E* / |E*|_F, sign fixed so that its largest entry is positive — the direction any fitter should find
  (E[2,2] can be 0 or rounding noise, so directions are compared, not E / E[2,2]);
- ``sv``: sigma_1..sigma_8(Y) and ``kappa`` = sigma_1 / sigma_8: a backward-stable null-vector solver (Householder QR
  of Y^T, K1's k_fit_qr) errs by O(u kappa), the reference's route through Y^T Y by O(u kappa^2);
- ``rho`` = sigma_1(F) / (sigma_2(F) - sigma_3(F)) of the rank-3 estimate F: how much the rank-2 projection amplifies
  an error in F;
- ``valid``: sigma_8^2 > 1e-10, the reference's test (eight_point.py:414-421) in exact arithmetic
  (lambda_2(Y^T Y) = sigma_8(Y)^2);
- ``qr_lo``, ``qr_hi``: 1 / |R^-1|_F^2 <= sigma_8^2 <= min r_ii^2 for R of Y^T = QR, the two bounds k_fit_qr decides
  validity from;
- ``lam2_ref``, ``lam_max_ref``, ``ref_valid``: what the reference itself computes (np.linalg.eig of Y^T Y, :410) —
  its lambda_2 errs by about u * lambda_max, so near 1e-10 its decision is decided by rounding.

Never imported by the product path.
"""
from __future__ import annotations

import dataclasses

import mpmath as mp
import numpy as np

from . import restatement as o

DPS = 50
U = 2.0 ** -53  # unit roundoff of binary64
VERY_SMALL = o.VERY_SMALL


def design(ca, cb):
    """(Y [8,9], T1, T2) of K-normalised coordinates ca, cb [8,2], in the reference's double arithmetic."""
    na, T1 = o.hartley_normalise(np.asarray(ca, dtype=np.float64))
    nb, T2 = o.hartley_normalise(np.asarray(cb, dtype=np.float64))
    return np.stack([o.y_col(na[i], nb[i]) for i in range(8)]), T1, T2


def _mp(a):
    return mp.matrix(np.asarray(a, dtype=np.float64).tolist())


def _np(m):
    return np.array([[float(m[i, j]) for j in range(m.cols)] for i in range(m.rows)])


@dataclasses.dataclass
class ExactFit:
    Y: np.ndarray
    T1: np.ndarray
    T2: np.ndarray
    sv: np.ndarray          # sigma_1..sigma_8(Y), descending (rounded from DPS digits)
    s8sq: float             # sigma_8(Y)^2
    kappa: float            # sigma_1 / sigma_8 (inf for an exactly rank-deficient Y)
    rho: float              # sigma_1(F) / (sigma_2(F) - sigma_3(F))
    E_dir: np.ndarray       # E* / |E*|_F, largest entry positive
    valid: bool             # sigma_8^2 > 1e-10
    qr_lo: float            # 1 / |R^-1|_F^2
    qr_hi: float            # min r_ii^2
    amp: float              # |T1|_2 |T2|_2 |F'|_F / |E*|_F: how much the denormalisation E = T2^T F' T1 can amplify a
                            # relative error in F' (1 <= amp <= cond(T1) cond(T2))
    lam2_ref: float         # the reference's sorted eigenvalues of Y^T Y: [1] and [-1]
    lam_max_ref: float
    ref_valid: bool         # compute_f_est does not raise


def fit_exact(ca, cb, dps=DPS) -> ExactFit:
    """The exact fit of one sample of K-normalised coordinates ca, cb [8,2]; the sample must be finite."""
    Y, T1, T2 = design(ca, cb)
    if not np.isfinite(Y).all():
        raise ValueError("the design matrix is not finite")
    with mp.workdps(dps):
        Q, R = mp.qr(_mp(Y).T)  # Y^T = Q R, Q 9x9: its last column spans Y's null space
        R8 = R[0:8, 0:8]
        z = Q[0:9, 8]
        rdiag2 = [R8[i, i] ** 2 for i in range(8)]
        qr_hi = min(rdiag2)
        try:
            Ri = mp.inverse(R8)
            qr_lo = 1 / sum(Ri[i, j] ** 2 for i in range(8) for j in range(8))
        except ZeroDivisionError:  # R singular to the working precision: sigma_8 = 0
            qr_lo = mp.mpf(0)
        sv = mp.svd_r(R8, compute_uv=False)
        sv = sorted([abs(s) for s in sv], reverse=True)
        F = mp.matrix(3, 3)
        for i in range(9):
            F[i // 3, i % 3] = z[i]
        Uf, Sf, Vf = mp.svd_r(F)
        Sf = [Sf[i] for i in range(3)]
        D = mp.diag([Sf[0], Sf[1], 0])
        Fp = Uf * D * Vf
        E = _mp(T2).T * Fp * _mp(T1)
        nrm = mp.sqrt(sum(E[i, j] ** 2 for i in range(3) for j in range(3)))
        amp = np.linalg.norm(T1, 2) * np.linalg.norm(T2, 2) * float(mp.sqrt(Sf[0] ** 2 + Sf[1] ** 2) / nrm)
        E_dir = _np(E / nrm)
        s8sq = sv[7] ** 2
        rho = Sf[0] / (Sf[1] - Sf[2]) if Sf[1] > Sf[2] else mp.inf
        kappa = sv[0] / sv[7] if sv[7] > 0 else mp.inf
        valid = bool(s8sq > VERY_SMALL)
        out = dict(sv=np.array([float(s) for s in sv]), s8sq=float(s8sq), kappa=float(kappa), rho=float(rho),
                   valid=valid, qr_lo=float(qr_lo), qr_hi=float(qr_hi), amp=float(amp))
    k = np.argmax(np.abs(E_dir))
    E_dir *= np.sign(E_dir.flat[k])
    w = np.sort(np.linalg.eig(o.yT_y(*_normalised(ca, cb)))[0])
    try:
        o.compute_f_est(o.yT_y(*_normalised(ca, cb)))
        ref_valid = True
    except o.OracleEightPointError:
        ref_valid = False
    return ExactFit(Y=Y, T1=T1, T2=T2, E_dir=E_dir, lam2_ref=float(np.real(w[1])),
                    lam_max_ref=float(np.real(w[-1])), ref_valid=ref_valid, **out)


def _normalised(ca, cb):
    return (o.hartley_normalise(np.asarray(ca, dtype=np.float64))[0],
            o.hartley_normalise(np.asarray(cb, dtype=np.float64))[0])


def direction(E):
    """E / |E|_F with its largest entry positive (the convention of ExactFit.E_dir)."""
    E = np.asarray(E, dtype=np.float64).reshape(3, 3)
    d = E / np.linalg.norm(E)
    return d * np.sign(d.flat[np.argmax(np.abs(d))])


def direction_error(E, fit: ExactFit) -> float:
    """|dir(E) - E*_dir|_F, with the sign of E chosen to match (the two can differ in sign only by convention when
    the largest entries are near-equal in magnitude)."""
    d = direction(E)
    return float(min(np.linalg.norm(d - fit.E_dir), np.linalg.norm(d + fit.E_dir)))


# ---------------------------------------------------------------------------------------------------------------------
# Samples at the validity boundary
# ---------------------------------------------------------------------------------------------------------------------
def s8sq_double(ca, cb) -> float:
    """sigma_8(Y)^2 from np.linalg.svd: accurate to about u * sigma_1 absolute, i.e. to ~1e-11 relative at sigma_8
    ~ 1e-5 — fine for placing a sample, which fit_exact then measures exactly."""
    return float(np.linalg.svd(design(ca, cb)[0], compute_uv=False)[-1] ** 2)


def ladder_sample(base_a, base_b, target, seed, dup=0):
    """8 K-normalised correspondences (ca, cb [8,2]) whose design matrix has sigma_8(Y)^2 = target (to ~1e-9
    relative): the 7 distinct correspondences of base_a, base_b [7,2] and a copy of correspondence ``dup`` nudged by
    t d, with d a random unit direction in (xa, ya, xb, yb) and t found by bisection (sigma_8 grows from 0 at t = 0).
    The nudged copy is the last correspondence."""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=4)
    d /= np.linalg.norm(d)
    base_a = np.asarray(base_a, dtype=np.float64)
    base_b = np.asarray(base_b, dtype=np.float64)

    def sample(t):
        ca = np.vstack([base_a, base_a[dup] + t * d[:2]])
        cb = np.vstack([base_b, base_b[dup] + t * d[2:]])
        return ca, cb

    lo, hi = 0.0, 1e-7
    while s8sq_double(*sample(hi)) < target:
        lo, hi = hi, 2.0 * hi
    for _ in range(200):
        mid = 0.5 * (lo + hi)
        if mid in (lo, hi):
            break
        if s8sq_double(*sample(mid)) < target:
            lo = mid
        else:
            hi = mid
    return sample(hi)


LADDER_DELTAS = (0.5, 0.05, 5e-3, 1.5e-3, 1e-3, 5e-4, 1e-4)


def ladder_bases(seed):
    """Two geometries of 7 distinct K-normalised correspondences from a make_scene scene: ``clustered`` (the scene's
    own spread, lambda_max(Y^T Y) in the low hundreds) and ``far`` (one of the seven moved 4x further from the others'
    centroid in both images, lambda_max ~ 1e3)."""
    from structure_from_motion_b200.scenes import make_scene

    K, x1, x2, *_ = make_scene(40, 0.0, seed=seed)
    ca = np.stack(o.k_normalise(x1[:, 0], x1[:, 1], K), 1)[:7]
    cb = np.stack(o.k_normalise(x2[:, 0], x2[:, 1], K), 1)[:7]
    fa, fb = ca.copy(), cb.copy()
    for c in (fa, fb):
        m = c[:6].mean(axis=0)
        c[6] = m + 4.0 * (c[6] - m) / np.linalg.norm(c[6] - m) * np.abs(c[:6] - m).max()
    return {"clustered": (ca, cb), "far": (fa, fb)}


def ladder(seeds=(0, 1, 2)):
    """[(geometry, seed, delta, ca, cb)] with sigma_8^2 = 1e-10 (1 + delta) for every delta in +-LADDER_DELTAS."""
    out = []
    for seed in seeds:
        for geo, (ba, bb) in ladder_bases(seed).items():
            for k, mag in enumerate(LADDER_DELTAS):
                for sgn in (1.0, -1.0):
                    delta = sgn * mag
                    ca, cb = ladder_sample(ba, bb, VERY_SMALL * (1.0 + delta), seed=1000 * seed + 10 * k + (sgn > 0))
                    out.append((geo, seed, delta, ca, cb))
    return out
