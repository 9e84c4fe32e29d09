"""Bundle adjustment (csrc/sfm_bundle.cuh) against a replay of its own iteration (oracle/bundle_exact.py): trajectories
with rejected steps, per-view cameras and every gauge, the first step at every Cholesky panel count up to 255 free
views, the structure edges of the reduced system and its sums, and world and pixel scales out to where the normal
equations leave the double range.  The worst observed ratio of every bounded check is printed (run with -s) and kept
in profiles/bundle_edges_pytest_gpu_1xB200.log.

Notation: u = 2^-53; L the list length; kappa the largest (|p0|_abs + |p1|_abs + |p2|_abs) / |p2| over the list at
the start; cond the largest condition of the damped scaled systems (each V_hat_p and the reduced camera system, without
the rows of zero Jacobian columns) solved on the way.  The kernel's costs agree with the replay's to
rel = 64 u (L + kappa) (cost_start) and rel cond (cost_final); the parameters to 1e3 u cond (1 + kappa) of the largest
|R|, |t| and |X| entry.  A decision (accept, a stop) is "clear" when every replayed margin up to it exceeds 4 rel cond,
and every damped system's smallest eigenvalue exceeds 4 rel (1 + lambda): reports whose decisions are all clear are compared in full (status, iterations, rejected, costs,
R, t, X, and mask / err bit for bit against the C checker under the reported parameters).  A report whose only unclear
decision is its last convergence test must converge within two more iterations.  Each test asserts a minimum count of
fully compared reports."""
import math

import numpy as np
import pytest

from oracle import bundle as oba
from oracle import bundle_exact as bx
from oracle import creproj
from oracle.refine import rodrigues
from structure_from_motion_b200 import _native
from structure_from_motion_b200.multiview import bundle_adjust_arrays
from structure_from_motion_b200.scenes import make_multi_view_scene

pytestmark = [pytest.mark.gpu, pytest.mark.filterwarnings("ignore::RuntimeWarning")]

U = 2.0 ** -53
C_COST = 64
C_PARAM = 1e3
WORST = {}
SEEN = set()  # (status, reason) of the fully compared reports


def note(name, ratio):
    WORST[name] = max(WORST.get(name, 0.0), float(ratio))
    print(f"[worst] {name}: {WORST[name]:.3g}")


@pytest.fixture(scope="module")
def eng():
    return _native.Engine(0)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def _same(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _Rt(R, t):
    return np.concatenate([R, t[:, :, None]], axis=2)


def _perturb(R, t, X, seed, deg, tfrac, xfrac, anchor=None):
    """Every pose but view 0 rotated by `deg` and its t moved by about `tfrac` of |t| (the anchor's largest component
    kept), every point moved by about `xfrac` of its depth."""
    rng = np.random.default_rng(seed)
    R0, t0 = R.copy(), t.copy()
    for c in range(1, len(R)):
        w = rng.normal(size=3)
        R0[c] = R[c] @ rodrigues(w / np.linalg.norm(w) * np.radians(deg))
        t0[c] = t[c] + rng.normal(size=3) * tfrac * np.linalg.norm(t[c]) / np.sqrt(3)
    if anchor is not None and anchor >= 0:
        k = int(np.argmax(np.abs(t[anchor])))
        t0[anchor, k] = t[anchor, k]
    return R0, t0, X + rng.normal(size=X.shape) * xfrac * X[:, 2:] / np.sqrt(3)


class Case:
    """One problem: per-view K, the start, the tracks, threshold and gauge."""

    def __init__(self, K, R0, t0, X0, off, view, x, thr, fixed, sv):
        V = len(R0)
        self.K = np.ascontiguousarray(np.broadcast_to(np.asarray(K, dtype=np.float64), (V, 3, 3)))
        self.R0, self.t0, self.X0 = R0, t0, X0
        self.off, self.view, self.x, self.thr = np.asarray(off, np.int64), np.asarray(view, np.int32), x, thr
        self.fixed, self.sv = tuple(fixed), sv
        fm = np.zeros(V, dtype=bool)
        fm[list(fixed)] = True
        self.fmask = fm

    def run(self, eng, k):
        return bundle_adjust_arrays(self.K, self.R0, self.t0, self.X0, self.off, self.view, self.x, self.thr,
                                    fixed=self.fixed, scale_view=self.sv, max_iterations=k, engine=eng)

    def problem(self):
        return oba.problem(self.K, _Rt(self.R0, self.t0), self.X0, self.off, self.view, self.x, self.thr, self.fmask,
                           self.sv)


def _scene(n, V, seed, deg, frac, thr, fixed=(0,), sv=None, noise=0.5, outliers=0.1, pseed=None, **kw):
    K, R, t, X, off, view, x, _ = make_multi_view_scene(n, V, seed, noise_px=noise, outlier_frac=outliers, **kw)
    if sv is None:
        sv = [c for c in range(V) if c not in fixed][0] if len(fixed) == 1 and len(fixed) < V else -1
    R0, t0, X0 = _perturb(R, t, X, seed + 1 if pseed is None else pseed, deg, frac, frac, sv)
    return Case(K, R0, t0, X0, off, view, x, thr, fixed, sv)


def _check_mask(case, res):
    pt = np.repeat(np.arange(len(case.off) - 1), np.diff(case.off))
    Rt = _Rt(res.R, res.t)
    for c in range(len(case.R0)):
        sel = np.flatnonzero(case.view == c)
        if sel.size:
            m, v = creproj.reproj_exact_many(Rt[c], case.K[c], res.points[pt[sel]], case.x[sel], case.thr)
            assert np.array_equal(m, res.mask[sel]) and _same(v, res.err[sel]), c


def _status(rep):
    return {v: k for k, v in _native.REFINE_STATUS.items()}[rep.status]


def compare(case, prob, res, ex, tr, tag):
    """The kernel's report against the replay's at the same cap; returns whether the full comparison ran."""
    rep = res.report
    L, kappa = tr.n_obs, tr.kappa
    rel = C_COST * U * (L + kappa)
    floor = 1e6 * bx.COST_FLOOR * tr.floor_sum  # costs below this are rounding noise of the residuals
    assert rep.num_observations == L and rep.num_points == len(prob.points), tag
    if ex.cost_start > floor:
        note("cost_start / bound", abs(rep.cost_start - ex.cost_start) / (rel * ex.cost_start))
        assert abs(rep.cost_start - ex.cost_start) <= rel * ex.cost_start, (tag, rep.cost_start, ex.cost_start)
    cond = max(1.0, ex.cond)
    clear = 4 * rel * cond
    if ex.pivot_margin <= 4 * rel:  # a damped system rounding may find not positive definite
        return False
    if ex.min_margin > clear:
        assert (_status(rep), rep.iterations, rep.rejected) == (ex.status, ex.iterations, ex.rejected), (
            tag, rep, ex.status, ex.reason, ex.iterations, ex.rejected)
    elif ex.prior_margin > clear and ex.status == bx.CONVERGED:
        assert _status(rep) == bx.CONVERGED and ex.iterations <= rep.iterations <= ex.iterations + 2, (tag, rep, ex)
    else:
        return False
    if ex.cost_final > floor:
        cf = rel * cond * ex.cost_final
        note("cost_final / bound", abs(rep.cost_final - ex.cost_final) / cf)
        assert abs(rep.cost_final - ex.cost_final) <= cf, (tag, rep.cost_final, ex.cost_final)
    else:
        assert rep.cost_final <= floor, (tag, rep.cost_final)
    pb = C_PARAM * U * cond * (1 + kappa)
    note("R / bound", np.abs(res.R - ex.R).max() / pb)
    assert np.abs(res.R - ex.R).max() <= pb, tag
    note("t / bound", np.abs(res.t - ex.t).max() / (pb * np.abs(ex.t).max()))
    assert np.abs(res.t - ex.t).max() <= pb * np.abs(ex.t).max(), tag
    par = prob.points
    if len(par):
        xs = np.abs(ex.X[par]).max()
        note("X / bound", np.abs(res.points[par] - ex.X[par]).max() / (pb * xs))
        assert np.abs(res.points[par] - ex.X[par]).max() <= pb * xs, tag
    nonpar = np.setdiff1d(np.arange(len(case.X0)), par)
    assert _same(res.points[nonpar], case.X0[nonpar]), tag
    for c in np.flatnonzero(case.fmask):
        assert _same(res.R[c], case.R0[c]) and _same(res.t[c], case.t0[c]), (tag, c)
    _check_mask(case, res)
    SEEN.add((ex.status, ex.reason))
    return True


def trajectory(eng, case, ks, tag):
    prob = case.problem()
    tr = bx.replay(prob, max(ks))
    out = []
    for k in ks:
        res = case.run(eng, k)
        ex = bx.report_after(tr, k)
        if compare(case, prob, res, ex, tr, (tag, k)):
            out.append((k, res.report))
    print(f"{tag}: L {tr.n_obs}, F {len(prob.free)}, compared {len(out)} of {len(ks)} reports in full; "
          f"statuses {sorted({(r.status, r.iterations, r.rejected) for _, r in out})}")
    return out, tr


# ---- 1. trajectories --------------------------------------------------------------------------------------------------
def _perview_case(n, V, seed):
    """A different K per view: focal lengths from 200 to 2e4, scattered principal points, nonzero skew; noise scaled
    with the focal length."""
    _, R, t, X, off, view, _, _ = make_multi_view_scene(n, V, seed, noise_px=0.0)
    rng = np.random.default_rng(seed)
    f = rng.permutation(np.geomspace(200.0, 2e4, V))
    K = np.zeros((V, 3, 3))
    K[:, 0, 0], K[:, 1, 1] = f, f * rng.uniform(0.8, 1.25, V)
    K[:, 0, 1] = f * rng.uniform(-0.02, 0.02, V)
    K[:, 0, 2], K[:, 1, 2] = rng.uniform(-500, 2000, V), rng.uniform(-300, 1500, V)
    K[:, 2, 2] = 1.0
    pt = np.repeat(np.arange(len(X)), np.diff(off))
    p = np.einsum("mij,mj->mi", K[view], np.einsum("mij,mj->mi", R[view], X[pt]) + t[view])
    x = p[:, :2] / p[:, 2:] + rng.normal(size=(len(view), 2)) * 0.5 * (f[view] / 800.0)[:, None]
    R0, t0, X0 = _perturb(R, t, X, seed + 1, 1.0, 0.01, 0.01, 1)
    return Case(K, R0, t0, X0, off, view, np.ascontiguousarray(x), 1e6, (0,), 1)


TRAJ = {
    # 8 degrees, 10 % of t and X, threshold 1e6 px^2: many steps put points behind a view (cost +inf) or overshoot
    "rejections": (lambda: _scene(150, 6, 3, 8.0, 0.1, 1e6, pseed=4), range(1, 13)),
    "per-view K": (lambda: _perview_case(200, 6, 21), range(1, 9)),
    "fixed (2, 5), no anchor": (lambda: _scene(200, 8, 22, 2.0, 0.02, 1e4, fixed=(2, 5), sv=-1), range(1, 15)),
    "fixed (3,), anchor 5": (lambda: _scene(200, 8, 23, 2.0, 0.02, 1e4, fixed=(3,), sv=5), range(1, 9)),
    "one fixed, gauge free": (lambda: _scene(150, 6, 24, 1.0, 0.01, 1e4, fixed=(0,), sv=-1), range(1, 7)),
    "all fixed (F = 0)": (lambda: _scene(200, 5, 25, 1.0, 0.02, 1e4, fixed=(0, 1, 2, 3, 4), sv=-1), range(1, 9)),
    "noise-free": (lambda: _scene(200, 6, 26, 1.0, 0.01, 1e4, noise=0.0, outliers=0.0), range(1, 13)),
}


@pytest.mark.parametrize("name", list(TRAJ))
def test_trajectory_against_the_replay(eng, name):
    make, ks = TRAJ[name]
    case = make()
    out, tr = trajectory(eng, case, list(ks), name)
    assert len(out) >= 2, name
    if name == "rejections":
        assert max(r.rejected for _, r in out) >= 3
    if name.startswith("all fixed"):
        assert all(r.num_free_views == 0 for _, r in out)
        assert _same(case.run(eng, 1).R, case.R0)


def test_statuses_covered():
    """Across the trajectories: converged by ftol and by the cost floor, and max_iterations, each in a fully compared
    report."""
    if not SEEN:
        pytest.skip("the trajectory tests did not run")
    print("seen", sorted(SEEN))
    assert (bx.CONVERGED, "ftol") in SEEN and (bx.CONVERGED, "floor") in SEEN and (bx.MAX_ITER, "max_iter") in SEEN


# ---- 2. the first step at every panel count ---------------------------------------------------------------------------
def _panel_frees():
    """Free-view counts whose padded reduced systems have 1 .. 48 tile columns (F = floor(16 q / 3), so 6F is a
    multiple of 32 for every q divisible by 3, and 255 for 48), plus 6F = 32 k + 2 (F = 11, 27, 251)."""
    fs = sorted({min(255, 16 * q // 3) for q in range(1, 49)} | {11, 27, 251})
    return fs


def _panel_case(F, pseed):
    if F == 255:
        fixed = (128,)
    else:
        nfix = min(max(1, F // 6), 256 - F)
        fixed = tuple(sorted({2 + (k * (F + nfix)) // nfix for k in range(nfix)} - {F + nfix}))[:nfix]
        fixed = tuple(c for c in fixed if c < F + nfix) or (0,)
    V = F + len(fixed)
    deg, frac = (0.5, 0.01) if V <= 64 else (0.02, 0.001)  # close views: a far start overshoots on its first step
    return _scene(max(150, 12 * V), V, 30 + F, deg, frac, 1e4, fixed=fixed, outliers=0.05, pseed=pseed,
                  arc_deg=60.0 if V <= 40 else 120.0)


@pytest.mark.parametrize("F", _panel_frees())
def test_first_step_every_panel_count(eng, F):
    """max_iterations = k against the replay's Schur steps (refined against the full system), k the first iteration
    whose proposal is accepted (after 0 or more rejected ones, which put a weakly observed point behind a view)."""
    case = _panel_case(F, 100)
    prob = case.problem()
    assert len(prob.free) == F
    tr = bx.replay(prob, 6)
    k = next(s.iteration for s in tr.steps if s.accepted and s.iteration > 0)
    ex = bx.report_after(tr, k)
    npad = (6 * F + 31) // 32 * 32
    res = case.run(eng, k)
    assert res.report.num_free_views == F
    assert compare(case, prob, res, ex, tr, ("panels", F)), (F, ex.min_margin, ex.pivot_margin, ex.cond)
    print(f"F {F} (fixed {case.fixed[:4]}..., {len(case.fixed)} fixed): {npad // 32} panels, L {tr.n_obs}, "
          f"compared at k = {k} ({ex.rejected} rejected), cond {ex.cond:.3g}")


# ---- 3. structure edges -----------------------------------------------------------------------------------------------
def _tracks(case):
    pt = np.repeat(np.arange(len(case.off) - 1), np.diff(case.off))
    return [list(zip(case.view[pt == t].tolist(), case.x[pt == t].tolist())) for t in range(len(case.off) - 1)]


def _rebuild(case, tracks, X0):
    off = np.zeros(len(tracks) + 1, dtype=np.int64)
    np.cumsum([len(t) for t in tracks], out=off[1:])
    view = np.array([v for t in tracks for v, _ in t], dtype=np.int32)
    x = np.array([xy for t in tracks for _, xy in t], dtype=np.float64).reshape(-1, 2)
    return Case(case.K, case.R0, case.t0, np.asarray(X0, dtype=np.float64), off, view, x, case.thr, case.fixed,
                case.sv)


def _project(case, X, views, rng, noise=0.5, truth=None):
    R, t = truth if truth is not None else (case.R0, case.t0)
    out = []
    for c in views:
        p = case.K[c] @ (R[c] @ X + t[c])
        out.append((int(c), (p[:2] / p[2] + rng.normal(size=2) * noise).tolist()))
    return out


def _edge_duplicates():
    """Two observations of one track in the same free view: a diagonal S block gets both (i, j) and (j, i)."""
    case = _scene(300, 6, 40, 1.0, 0.01, 1e4)
    rng = np.random.default_rng(40)
    tr = _tracks(case)
    for t in range(0, len(tr), 3):
        if len(tr[t]) >= 2:
            v, xy = tr[t][1]
            tr[t].insert(2, (v, (np.asarray(xy) + rng.normal(size=2) * 0.3).tolist()))
    return _rebuild(case, tr, case.X0)


def _edge_track64():
    """Tracks of exactly 64 observations over 64 views (the top bit of the list mask)."""
    case = _scene(500, 64, 41, 0.05, 0.002, 1e4, arc_deg=120.0)
    rng = np.random.default_rng(41)
    tr = _tracks(case)
    Xn = np.column_stack([rng.uniform(-1, 1, 8), rng.uniform(-1, 1, 8), rng.uniform(5, 7, 8)])
    tr += [_project(case, X, range(64), rng) for X in Xn]
    return _rebuild(case, tr, np.vstack([case.X0, Xn]))


def _edge_fixed_only():
    """Tracks whose passing observations are all in the fixed views 0 and 2 (V_p with no W_hat), one more observation
    in free view 4 failing the threshold."""
    case = _scene(250, 6, 42, 1.0, 0.01, 1e4, fixed=(0, 2), sv=-1)
    rng = np.random.default_rng(42)
    tr = _tracks(case)
    Xn = np.column_stack([rng.uniform(-1, 1, 20), rng.uniform(-1, 1, 20), rng.uniform(5, 7, 20)])
    for X in Xn:
        obs = _project(case, X, (0, 2, 4), rng)
        obs[2] = (4, (np.asarray(obs[2][1]) + 400.0).tolist())
        tr.append(obs)
    return _rebuild(case, tr, np.vstack([case.X0, Xn]))


def _edge_empty():
    """Empty tracks (finite and NaN points) among the others, and free view 3 whose observations all miss the list."""
    case = _scene(250, 6, 43, 1.0, 0.01, 1e4)
    tr = _tracks(case)
    X0 = list(case.X0)
    for k in (0, 7, 100, len(tr)):
        tr.insert(k, [])
        X0.insert(k, np.array([0.1, 0.2, 5.0]) if k % 2 else np.array([np.nan, 0.0, 5.0]))
    tr = [[(v, (np.asarray(xy) + 900.0).tolist() if v == 3 else xy) for v, xy in t] for t in tr]
    return _rebuild(case, tr, np.array(X0))


def _edge_big(T, V):
    """T tracks, every one seen in all V views: view 1 holds T list observations (more than 32 chunks of 256 when
    T > 8192) and S block (1, 1) T pairs (more than 32 chunks of 32); T = 128^2 + 1 makes the cost's ordered sum take
    two partials per segment."""
    return _scene(T, V, 44 + V, 0.05, 0.002, 1e4, min_len=V, max_len=V)


EDGES = {
    "duplicate views": _edge_duplicates,
    "64-observation tracks": _edge_track64,
    "fixed-only tracks": _edge_fixed_only,
    "empty tracks, empty view": _edge_empty,
    "T = 128^2 + 1, 3 views": lambda: _edge_big(128 * 128 + 1, 3),
    "T = 129 * 128, 4 views": lambda: _edge_big(129 * 128, 4),
}


@pytest.mark.parametrize("name", list(EDGES))
def test_structure_edges(eng, name):
    """The first step and a 5-iteration trajectory against the replay."""
    case = EDGES[name]()
    out, tr = trajectory(eng, case, [1, 2, 3, 4, 5], name)
    assert out and out[0][0] == 1, name
    lens = np.diff(case.off)
    if name.startswith("64"):
        assert (lens == 64).sum() >= 8
    if name.startswith("T ="):
        T = len(case.off) - 1
        assert T > 128 * 128 and (T == 128 * 128 + 1 or T % 128 == 0)
        prob = case.problem()
        assert (prob.obs_view == 1).sum() > 32 * 256
    if name.startswith("empty"):
        prob = case.problem()
        assert not (prob.obs_view == 3).any() and (case.view == 3).any()
        res = case.run(eng, 3)
        assert np.abs(res.R[3] - oba.nearest_rotation(case.R0[3])).max() <= 1e-14 and _same(res.t[3], case.t0[3])


# ---- 4. scale edges and the re-solve path -----------------------------------------------------------------------------
DMAX = np.finfo(np.float64).max
TINY = np.finfo(np.float64).tiny


def _scaled(case, kw, kp):
    K = case.K.copy()
    K[:, :2] = np.ldexp(K[:, :2], kp)
    return Case(K, case.R0, np.ldexp(case.t0, kw), np.ldexp(case.X0, kw), case.off, case.view,
                np.ldexp(case.x, kp), np.ldexp(case.thr, 2 * kp), case.fixed, case.sv)


def _ranges(case):
    """The replay's double quantities at the start, as (log2 smallest nonzero, log2 largest, world exponent, pixel
    exponent) groups: under world x 2^k and pixels x 2^k every one of them scales by 2^(ew k) and 2^(ep k) exactly.
    Residuals (0, 1), J_c's rotation columns (0, 1) and translation columns (-1, 1), J_p (-1, 1), and their products in
    U, V, W, g_c, g_p (the sums of the exponents)."""
    prob = case.problem()
    lay = bx.layout(prob)
    ev = bx.evaluate(prob, lay, prob.R, prob.t, prob.X)
    eq = bx.equations(lay, ev)
    ec = np.array([0, 0, 0, -1, -1, -1])
    groups = []

    def add(a, ew, ep):
        a = np.abs(np.asarray(a, dtype=np.float64))
        for e in np.unique(ew):
            v = a[np.broadcast_to(ew, a.shape) == e]
            v = v[v != 0]
            if v.size:
                groups.append((math.log2(v.min()), math.log2(v.max()), int(e), ep))

    free = lay.fi >= 0
    add(ev.r, np.zeros(2, int), 1)
    add(ev.Jc[free], ec[None, None, :], 1)
    add(ev.Jp, -1, 1)
    add(eq.U, ec[:, None] + ec[None, :], 2)
    add(eq.V, -2, 2)
    add(eq.W[free], ec[:, None] - 1, 2)
    add(eq.gc, ec[None, :], 2)
    add(eq.gp, -1, 2)
    diag = [(math.log2(np.diagonal(eq.U, axis1=1, axis2=2)[:, 3:].max()), -2, 2),
            (math.log2(np.diagonal(eq.V, axis1=1, axis2=2).max()), -2, 2)]
    x = np.asarray(prob.obs_x)
    lfloor = math.log2(math.fsum((x[:, 0] ** 2).tolist() + (x[:, 1] ** 2).tolist()))
    return prob, groups, diag, math.log2(float(np.abs(ev.p[:, 2]).min())), math.log2(ev.cost), lfloor


@pytest.mark.parametrize("axis", ["world", "pixel"])
def test_scale_edges_and_the_resolve_path(eng, axis):
    """World x 2^k (t and X) or pixels x 2^k (K's first two rows, x, threshold x 4^k), k swept out to where the normal
    equations overflow.  Where the replay's double quantities at the start stay within [2^20 tiny, 2^-20 max], the
    report is bit-exact to k = 0's (the window is printed with the measured bit-exact range).  Where a diagonal sum of
    the normal equations is beyond 16 max (every summation order overflows) while p2 and the cost stay 16 times inside
    their limits, the damped system is not positive definite at every lambda: the run comes back stalled at iteration
    0 with cost_final == cost_start and the projected start, as the replay's, through the re-solve path (world scale:
    the pixel sums reach the cost floor first).  Where sum(u^2 + v^2) is beyond 16 max, the cost floor is +inf and the
    start is converged at iteration 0, as the replay's.  Where the cost is beyond 16 max or p2 under 2^-537 / 16, the
    start is nonfinite and the input is reported.  Every other k must still end (no SFM_ERR_STATE) at a cost no
    higher than the start's."""
    base = _scene(150, 6, 50, 0.05, 0.002, 16.0)
    ref = base.run(eng, 5)
    prob0, groups, diag, lp2, lcost, lfloor = _ranges(base)
    lbig = max(d for d, _, _ in diag)
    # the k at which the largest diagonal sum overflows (world: x 2^-2k, pixel: x 4^k)
    kd = (1024 - lbig) / 2
    ks = sorted(set(range(-int(kd) - 40, -int(kd) + 8)) | set(range(-520, 521, 40)) | {300, 480, 500, 510, 515}) \
        if axis == "world" else sorted(set(range(int(kd) - 6, 510)) | set(range(-520, 500, 40)) | {-500, -510})
    exact, stalled, nonfinite, floored, other = [], [], [], [], []
    for k in ks:
        kw, kp = (k, 0) if axis == "world" else (0, k)
        lo = min(a + ew * kw + ep * kp for a, _, ew, ep in groups)
        hi = max(b + ew * kw + ep * kp for _, b, ew, ep in groups)
        ldiag = max(d + ew * kw + ep * kp for d, ew, ep in diag)
        p2, cost = lp2 + kw, lcost + 2 * kp
        case = _scaled(base, kw, kp)
        res = case.run(eng, 5)  # never SFM_ERR_STATE: the host's batch loop ends
        rep = res.report
        inside = lo >= -1022 + 20 and hi <= 1024 - 20 and p2 >= -537 + 4 and cost <= 1024 - 4
        same = (_same(res.R, ref.R) and _same(res.t, np.ldexp(ref.t, kw)) and _same(res.points, np.ldexp(ref.points, kw))
                and _same(np.ldexp(ref.report.cost_final, 2 * kp), rep.cost_final)
                and (rep.iterations, rep.status, rep.rejected) == (ref.report.iterations, ref.report.status,
                                                                    ref.report.rejected))
        if same:
            exact.append(k)
        if inside:
            assert same, (axis, k)
            continue
        if cost > 1024 + 4 or p2 < -537 - 4:
            assert rep.status == "nonfinite" and _same(res.R, case.R0) and _same(res.points, case.X0), (axis, k)
            nonfinite.append(k)
        elif lfloor + 2 * kp > 1024 + 4 and p2 >= -537 + 4 and cost <= 1024 - 4:
            # sum(u^2 + v^2) overflows: the cost floor is +inf, so the start is converged before any solve
            ex = bx.report_after(bx.replay(case.problem(), 5), 5)
            assert (ex.status, ex.reason, ex.iterations) == (bx.CONVERGED, "floor", 0)
            assert (rep.status, rep.iterations, rep.rejected) == ("converged", 0, 0), (axis, k, rep)
            assert _same(rep.cost_final, rep.cost_start) and _same(res.t, case.t0) and _same(res.points, case.X0)
            floored.append(k)
        elif ldiag > 1024 + 4 and p2 >= -537 + 4 and cost <= 1024 - 4:
            prob = case.problem()
            r1 = case.run(eng, 1)
            tr = bx.replay(prob, 1)
            ex = bx.report_after(tr, 1)
            assert ex.status == bx.STALLED and ex.reason == "resolve_cap" and ex.iterations == 0
            for r in (res, r1):
                q = r.report
                assert (q.status, q.iterations, q.rejected) == ("stalled", 0, 0), (axis, k, q)
                assert _same(q.cost_final, q.cost_start)
                assert abs(q.cost_start - tr.cost_start) <= C_COST * U * (tr.n_obs + tr.kappa) * tr.cost_start
                assert _same(r.t, case.t0) and _same(r.points, case.X0)
                assert np.abs(r.R - prob.R).max() <= 1e-14
            stalled.append(k)
        else:
            other.append((k, rep.status, rep.iterations))
            assert rep.cost_final <= rep.cost_start or rep.status == "nonfinite"
    lo_k = hi_k = 0
    for k in sorted((k for k in ks if k < 0), reverse=True):
        if k not in exact:
            break
        lo_k = k
    for k in sorted(k for k in ks if k > 0):
        if k not in exact:
            break
        hi_k = k
    print(f"{axis}: bit-exact to k = 0 at every swept k in [{lo_k}, {hi_k}] (swept {ks[0]} .. {ks[-1]}); "
          f"stalled through the re-solve path at k = {stalled}; converged at the infinite cost floor at k = {floored}; "
          f"nonfinite at k = {nonfinite}; unclear at {other}")
    if axis == "world":
        assert stalled, "the re-solve path ran"
