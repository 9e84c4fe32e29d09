"""TEST INFRASTRUCTURE ONLY — the essential-matrix pose tail in exact arithmetic, and inputs placed at its edges.

The inputs (E, the 4x4 DLT system, the correspondences) are doubles and are taken as exact; everything after them is
computed in mpmath at ``DPS`` digits.  What that gives a test:

- ``decompose_exact(E)``: the singular values of E, and the four pose candidates of _recover_all_r_t
  (eight_point.py:245-280) from a proper exact SVD (third columns of U and V = cross products of the first two, which is
  what the reference's sign fixes achieve).  The candidate SET is unique: another proper SVD swaps R1 and R2 and/or
  negates t (the reference's own test accepts exactly that).  ``cond`` = s0 / (s1 - s2) bounds how far a backward-stable
  SVD can move the frames, in units of u;
- ``null_exact(A)``: the four singular values of a 4x4 system, its smallest right singular vector x (sign: x[3] >= 0)
  and the dehomogenised X = x[:3] / x[3] (triangulation.py:34-39);
- ``cheirality_exact``: the depth of the exact X in both cameras and |X| (eight_point.py:473-487), each with the margin
  by which an X within a given distance of the exact one can move it: a decision is "clear" when the quantity lies
  further than its margin from -1e-8 (depths) or from the distance threshold (|X|);
- constructors: matrices with prescribed singular values through random orthogonal factors, rank-2 and true essential
  matrices, DLT systems that ``triangulate_arrays`` turns into any 4x4 matrix (with xa = ya = xb = yb = 0 and
  P1[2] = P2[2] = 0 the rows are -P1[1], P1[0], -P2[1], P2[0]), and scenes with a prescribed parallax.

Never imported by the product path.
"""
from __future__ import annotations

import dataclasses

import mpmath as mp
import numpy as np

from . import restatement as o

DPS = 50
U = 2.0 ** -53  # unit roundoff of binary64
CHEIRALITY_TOLERANCE = o.CHEIRALITY_TOLERANCE
# np.isclose(0.0, s, rtol=1e-5, atol=1e-8) (eight_point.py:268) holds exactly when s <= 1e-8 / (1 - 1e-5)
SV_LIMIT = 1e-8 / (1.0 - 1e-5)
W = np.array([[0, -1, 0], [1, 0, 0], [0, 0, 1]], dtype=float)   # eight_point.py:273
Z = np.array([[0, 1, 0], [-1, 0, 0], [0, 0, 0]], dtype=float)   # :274


def _mp(a):
    return mp.matrix(np.asarray(a, dtype=np.float64).tolist())


def _np(m):
    return np.array([[float(m[i, j]) for j in range(m.cols)] for i in range(m.rows)])


def _svd_sorted(A):
    """(U, s, V) of an mp matrix with s descending (A = U diag(s) V^T)."""
    Um, S, Vt = mp.svd_r(A)
    n = A.cols
    order = sorted(range(n), key=lambda i: -S[i])
    Uo = mp.matrix(A.rows, n)
    Vo = mp.matrix(n, n)
    for k, i in enumerate(order):
        for r in range(A.rows):
            Uo[r, k] = Um[r, i]
        for r in range(n):
            Vo[r, k] = Vt[i, r]
    return Uo, [S[i] for i in order], Vo


def _cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


# ---------------------------------------------------------------------------------------------------------------------
# the decomposition of E
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class ExactDecomposition:
    s: np.ndarray        # s0 >= s1 >= s2 (rounded from DPS digits)
    R1: np.ndarray       # U W^T V^T
    R2: np.ndarray       # U W V^T
    t: np.ndarray        # t_1 of eight_point.py:275-276 (unit)
    cond: float          # s0 / (s1 - s2): inf when s1 == s2
    accepted: bool       # the exact s2 passes np.isclose(0, s2)


def decompose_exact(E, dps=DPS) -> ExactDecomposition:
    """The exact candidates of a finite 3x3 E (any scale: mpmath has no exponent range to leave)."""
    E = np.asarray(E, dtype=np.float64).reshape(3, 3)
    if not np.isfinite(E).all():
        raise ValueError("E is not finite")
    with mp.workdps(dps):
        Um, S, Vm = _svd_sorted(_mp(E))
        u = [[Um[r, c] for r in range(3)] for c in range(3)]
        v = [[Vm[r, c] for r in range(3)] for c in range(3)]
        u[2] = _cross(u[0], u[1])
        v[2] = _cross(v[0], v[1])
        Up = mp.matrix([[u[c][r] for c in range(3)] for r in range(3)])
        Vp = mp.matrix([[v[c][r] for c in range(3)] for r in range(3)])
        R1 = Up * _mp(W).T * Vp.T
        R2 = Up * _mp(W) * Vp.T
        tx = Up * _mp(Z) * Up.T
        t = [-tx[1, 2], tx[0, 2], -tx[0, 1]]
        cond = S[0] / (S[1] - S[2]) if S[1] > S[2] else mp.inf
        return ExactDecomposition(s=np.array([float(x) for x in S]), R1=_np(R1), R2=_np(R2),
                                  t=np.array([float(x) for x in t]), cond=float(cond),
                                  accepted=bool(S[2] <= mp.mpf(1e-8) / (1 - mp.mpf(1e-5))))


def candidate_error(R1, R2, t, ex: ExactDecomposition):
    """(rotation error, translation error) in max-abs entries between the candidate set (R1, R2, +-t) and the exact
    one, under the (R1, R2) swap and the t sign that fit best."""
    R1, R2, t = (np.asarray(a, dtype=np.float64) for a in (R1, R2, t))
    er = min(max(np.abs(R1 - ex.R1).max(), np.abs(R2 - ex.R2).max()),
             max(np.abs(R1 - ex.R2).max(), np.abs(R2 - ex.R1).max()))
    et = min(np.abs(t - ex.t).max(), np.abs(t + ex.t).max())
    return float(er), float(et)


# ---------------------------------------------------------------------------------------------------------------------
# the DLT null vector
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class ExactNull:
    A: np.ndarray
    s: np.ndarray        # sigma_1..sigma_4, descending
    x: np.ndarray        # unit right singular vector of sigma_4, x[3] >= 0
    X: np.ndarray        # x[:3] / x[3] (inf / nan when x[3] == 0)
    x_mp: list           # x at DPS digits

    @property
    def gap(self) -> float:
        """(sigma_3 - sigma_4) / sigma_1: a backward-stable null vector errs by O(u / gap)."""
        return float((self.s[2] - self.s[3]) / self.s[0]) if self.s[0] > 0 else 0.0


def null_exact(A, dps=DPS) -> ExactNull:
    A = np.asarray(A, dtype=np.float64).reshape(4, 4)
    with mp.workdps(dps):
        _, S, Vm = _svd_sorted(_mp(A))
        x = [Vm[r, 3] for r in range(4)]
        if x[3] < 0:
            x = [-c for c in x]
        with np.errstate(divide="ignore", invalid="ignore"):
            X = np.array([float(x[i] / x[3]) if x[3] != 0 else np.sign(float(x[i])) * np.inf for i in range(3)])
        return ExactNull(A=A, s=np.array([float(c) for c in S]), x=np.array([float(c) for c in x]), X=X, x_mp=x)


def residual_excess(A, X, dps=DPS) -> float:
    """|A xh| - sigma_4 for xh = [X, 1] / |[X, 1]| (the device returns X only), in exact arithmetic."""
    with mp.workdps(dps):
        xh = [mp.mpf(float(c)) for c in X] + [mp.mpf(1)]
        n = mp.sqrt(sum(c * c for c in xh))
        Am = _mp(A)
        r = mp.sqrt(sum(sum(Am[i, j] * xh[j] for j in range(4)) ** 2 for i in range(4))) / n
        _, S, _ = _svd_sorted(Am)
        return float(r - S[3])


def direction_error(X, ex: ExactNull, dps=DPS) -> float:
    """|xh - x| for xh = [X, 1] / |[X, 1]|, sign-aligned, in exact arithmetic."""
    with mp.workdps(dps):
        xh = [mp.mpf(float(c)) for c in X] + [mp.mpf(1)]
        n = mp.sqrt(sum(c * c for c in xh))
        d1 = mp.sqrt(sum((xh[i] / n - ex.x_mp[i]) ** 2 for i in range(4)))
        d2 = mp.sqrt(sum((xh[i] / n + ex.x_mp[i]) ** 2 for i in range(4)))
        return float(min(d1, d2))


def dlt_system(xa, ya, xb, yb, P1, P2):
    """triangulation.py:24-31 in double, the rows as the reference (and dlt_triangulate) round them."""
    P1 = np.asarray(P1, dtype=np.float64)
    P2 = np.asarray(P2, dtype=np.float64)
    return np.array([ya * P1[2] - P1[1], P1[0] - xa * P1[2], yb * P2[2] - P2[1], P2[0] - xb * P2[2]])


def cameras_for(A):
    """(P1, P2) 3x4 with P1[2] = P2[2] = 0 whose DLT system at xa = ya = xb = yb = 0 is exactly A."""
    A = np.asarray(A, dtype=np.float64).reshape(4, 4)
    P1 = np.zeros((3, 4))
    P2 = np.zeros((3, 4))
    P1[1], P1[0] = -A[0], A[1]
    P2[1], P2[0] = -A[2], A[3]
    return P1, P2


# ---------------------------------------------------------------------------------------------------------------------
# cheirality
# ---------------------------------------------------------------------------------------------------------------------
@dataclasses.dataclass
class ExactCheirality:
    z1: float            # depth in camera 1 (X[2])
    z2: float            # depth in camera 2 ((R X + t)[2])
    norm: float          # |X|
    m1: float            # margins: how far each quantity can move when X moves by dX
    m2: float
    mn: float
    finite: bool         # the exact x[3] != 0

    def clear(self, dist_thr) -> bool:
        """Every one of the three comparisons of eight_point.py:478-487 decided with room to spare."""
        return (self.finite and abs(self.z1 + CHEIRALITY_TOLERANCE) > self.m1
                and abs(self.z2 + CHEIRALITY_TOLERANCE) > self.m2 and abs(self.norm - dist_thr) > self.mn)

    def passes(self, dist_thr) -> bool:
        return (self.finite and self.z1 >= -CHEIRALITY_TOLERANCE and self.z2 >= -CHEIRALITY_TOLERANCE
                and self.norm <= dist_thr)


def cheirality_exact(xa, ya, xb, yb, R, t, dX_of=None) -> ExactCheirality:
    """The quantities _cheirality_check compares (normalised coordinates, P1 = [I|0], P2 = [R|t]) at the exact X.
    ``dX_of(ex)`` -> how far the computed X may lie from the exact one (default: the null-vector bound of the tests);
    the margins are that distance times the Lipschitz constants (1 for z1 and |X|, |R[2]| = 1 for z2) plus the
    rounding of the comparison's own arithmetic."""
    R = np.asarray(R, dtype=np.float64)
    t = np.asarray(t, dtype=np.float64).reshape(3)
    P2 = np.hstack([R, t[:, None]])
    ex = null_exact(dlt_system(xa, ya, xb, yb, np.eye(4)[:3], P2))
    if not np.isfinite(ex.X).all():
        return ExactCheirality(np.nan, np.nan, np.inf, np.inf, np.inf, np.inf, False)
    with mp.workdps(DPS):
        Xm = [ex.x_mp[i] / ex.x_mp[3] for i in range(3)]
        z2 = sum(_mp(R)[2, j] * Xm[j] for j in range(3)) + mp.mpf(float(t[2]))
        nrm = mp.sqrt(sum(c * c for c in Xm))
    d = float(dX_of(ex)) if dX_of is not None else 0.0
    rnd = 8 * U * (float(nrm) + abs(float(t[2])))
    return ExactCheirality(z1=float(Xm[2]), z2=float(z2), norm=float(nrm), m1=d + rnd,
                           m2=d * float(np.linalg.norm(R[2])) + rnd, mn=d + rnd, finite=True)


# ---------------------------------------------------------------------------------------------------------------------
# constructors
# ---------------------------------------------------------------------------------------------------------------------
def orthogonal(n, rng, proper=True):
    q, r = np.linalg.qr(rng.normal(size=(n, n)))
    q = q * np.sign(np.diag(r))
    if proper and np.linalg.det(q) < 0:
        q[:, -1] *= -1
    return q


def with_singular_values(s, rng):
    """Q1 diag(s) Q2^T in double with random proper orthogonal Q1, Q2 (the rounded product's exact singular values
    differ from s by about u |s|; the tests measure the matrix they pass, not s)."""
    s = np.asarray(s, dtype=np.float64)
    n = len(s)
    return orthogonal(n, rng) @ np.diag(s) @ orthogonal(n, rng).T


def rank2(ratio, rng):
    """E = U diag(1, ratio, 0) V^T: ratio = 1 is a true essential matrix, a small ratio one close to rank 1."""
    return with_singular_values([1.0, ratio, 0.0], rng)


def true_essential(rng, scale=1.0):
    """[t]_x R of a random pose: s0 = s1 = |t|."""
    R = orthogonal(3, rng)
    t = rng.normal(size=3)
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    return scale * tx @ R


def rotation(axis, angle):
    axis = np.asarray(axis, dtype=np.float64)
    axis = axis / np.linalg.norm(axis)
    K = np.array([[0, -axis[2], axis[1]], [axis[2], 0, -axis[0]], [-axis[1], axis[0], 0]])
    return np.eye(3) + np.sin(angle) * K + (1 - np.cos(angle)) * K @ K


def scene(n, rng, parallax=0.1, depth=(2.0, 8.0), noise=0.0, baseline=None):
    """(R, t, na, nb) K-normalised correspondences of n points seen from camera 1 = [I|0] and camera 2 = [R|t], with
    the baseline |t| chosen so that the typical angle between the rays is ``parallax`` rad; ``noise`` is added to the
    normalised coordinates of image B."""
    R = rotation(rng.normal(size=3), 0.1)
    zmid = float(np.mean(depth))
    tdir = np.array([1.0, 0.2, 0.1]) if baseline is None else np.asarray(baseline, dtype=np.float64)
    t = tdir / np.linalg.norm(tdir) * parallax * zmid
    X = np.stack([rng.uniform(-1, 1, n), rng.uniform(-1, 1, n), rng.uniform(*depth, n)], 1)
    X[:, :2] *= X[:, 2:3] * 0.5
    Xb = X @ R.T + t
    na = X[:, :2] / X[:, 2:3]
    nb = Xb[:, :2] / Xb[:, 2:3] + noise * rng.normal(size=(n, 2))
    return R, t, na, nb


def essential_of(R, t):
    t = np.asarray(t, dtype=np.float64)
    tx = np.array([[0, -t[2], t[1]], [t[2], 0, -t[0]], [-t[1], t[0], 0]])
    return tx @ np.asarray(R, dtype=np.float64)


# ---------------------------------------------------------------------------------------------------------------------
# the sweeps the GPU tests run (one definition, so that the host build can confirm which route each case takes)
# ---------------------------------------------------------------------------------------------------------------------
# sigma_4 / sigma_3 across null_vector4_fast's fallback switch (~0.7): at most 0.6 the inverse iteration converges
# within its 40 steps, from 0.8 on the Jacobi SVD takes over
NULL_RATIOS = (0.0, 1e-3, 0.1, 0.3, 0.5, 0.6, 0.8, 0.9, 0.99, 1.0 - 1e-6)
NULL_FAST_MAX, NULL_FALLBACK_MIN = 0.6, 0.8
NULL_SPECTRA = {"normalised": (1.0, 0.9, 0.8), "pixel": (1.0, 0.3, 1e-2)}  # sigma_1..3; sigma_4 = ratio * sigma_3


def null_sweep(trials=6, seed=3):
    """[(family, ratio, A)]: 4x4 systems with prescribed singular values."""
    rng = np.random.default_rng(seed)
    out = []
    for fam, (s1, s2, s3) in NULL_SPECTRA.items():
        for r in NULL_RATIOS:
            for _ in range(trials):
                out.append((fam, r, with_singular_values([s1, s2, s3, s3 * r], rng)))
    return out


# s1 / s0 of rank-2 E (1 = a true essential matrix) down to nearly rank 1
RANK2_RATIOS = (1.0, 0.5, 1e-2, 1e-4, 1e-6, 1e-9, 1e-12)


def decomposition_sweep(trials=5, seed=5):
    """[(name, E)]: rank-2 E over RANK2_RATIOS, true essentials at several scales, and E whose exact s2 lies around
    np.isclose's limit (with s0 = 1, and with s0 = 4 where the closed form takes them), and the Jacobi-fallback case: s2 above 1e-8 s0 (svd3_rank2_frames refuses it) but below 1e-8
    (the reference accepts it)."""
    rng = np.random.default_rng(seed)
    out = []
    for r in RANK2_RATIOS:
        out += [(f"rank2_{r:g}", rank2(r, rng)) for _ in range(trials)]
    for sc in (1e-3, 1.0, 1e3):
        out += [(f"essential_{sc:g}", true_essential(rng, sc)) for _ in range(trials)]
    for f in (0.5, 0.9, 0.99, 1.01, 1.1, 2.0):
        out += [(f"s2_limit_{f:g}", with_singular_values([1.0, 0.6, f * SV_LIMIT], rng)) for _ in range(trials)]
    # s0 > 1: the closed form's route test (s2 <= 1e-8 s0) admits s2 around the absolute limit, where a residual
    # |E v3| of up to sqrt(3) s2 would decide the reference's test differently
    for f in (0.6, 0.7, 0.8, 0.9, 0.95, 0.99):
        out += [(f"s2_band_{f:g}", with_singular_values([4.0, 2.4, f * SV_LIMIT], rng)) for _ in range(2 * trials)]
    out += [("fallback", fallback_case(rng)) for _ in range(trials)]
    return out


def fallback_case(rng):
    """s0 = 0.5, s2 = 0.6e-8: s2 > 1e-8 s0, s2 < 1e-8."""
    return with_singular_values([0.5, 0.3, 0.6e-8], rng)
