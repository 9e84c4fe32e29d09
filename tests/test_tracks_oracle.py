"""The multi-view track oracle (oracle/tracks.py) and the track scene and layout helpers, on the CPU: the exact DLT, the
pair search's count / sum / index rule, the replayed refinement, make_multi_view_scene and tracks_from_dense."""
import mpmath
import numpy as np

from oracle import creproj
from oracle import tracks as otr
from structure_from_motion_b200.multiview import tracks_from_dense
from structure_from_motion_b200.scenes import make_multi_view_scene


def _scene(n=50, V=8, seed=0, **kw):
    K, R, t, X, off, view, x, out = make_multi_view_scene(n, V, seed, **kw)
    Rt = np.concatenate([R, t[:, :, None]], axis=2)
    return np.broadcast_to(K, (V, 3, 3)), Rt, X, off, view, x, out


def test_exact_dlt_recovers_noise_free_points():
    K, Rt, X, off, view, _, _ = _scene(20, 8, 1)
    worst = mpmath.mpf(0)
    with mpmath.workdps(otr.DPS):
        for i in range(20):
            vs = view[off[i]:off[i + 1]]
            Ps = [creproj.projection(K[c], Rt[c]) for c in vs]
            Xi = [mpmath.mpf(float(a)) for a in X[i]]
            xs = []
            for P in Ps:  # the exact projection of the exact point: noise-free to 50 digits
                p = [sum(mpmath.mpf(float(P[r][c])) * Xi[c] for c in range(3)) + mpmath.mpf(float(P[r][3])) for r in range(3)]
                xs.append((p[0] / p[2], p[1] / p[2]))
            got = otr.dlt_exact(Ps, xs)
            err = mpmath.sqrt(sum((g - e) ** 2 for g, e in zip(got, Xi))) / mpmath.sqrt(sum(e ** 2 for e in Xi))
            worst = max(worst, err)
    assert worst <= mpmath.mpf("1e-30"), worst


def test_pair_search_prefers_count():
    """An outlier observation: the winner is a pair of inliers, with every inlier passing."""
    K, Rt, X, off, view, x, _ = _scene(10, 8, 2, noise_px=0.3, min_len=5, max_len=5)
    vs, xs = view[off[0]:off[1]], x[off[0]:off[1]].copy()
    xs[2] = xs[2] + 80.0
    table = otr.pair_table(K, Rt, vs, xs, 4.0)
    w = otr.pair_search(table)
    i, j, _, cand, count, _, mask, _ = table[w]
    assert cand and count == 4 and 2 not in (i, j) and not mask[2]
    assert count == max(r[4] for r in table if r[3])


def test_pair_search_ties_go_to_the_smaller_sum():
    """All observations inliers: every pair has the same count, and the winner has the smallest sum."""
    K, Rt, X, off, view, x, _ = _scene(10, 8, 3, noise_px=0.5, min_len=4, max_len=4)
    vs, xs = view[off[0]:off[1]], x[off[0]:off[1]]
    table = otr.pair_table(K, Rt, vs, xs, 16.0)
    assert all(r[3] and r[4] == 4 for r in table)
    w = otr.pair_search(table)
    sums = [r[5] for r in table]
    assert w == int(np.argmin(sums)) and len(set(sums)) == len(sums)


def test_pair_search_equal_sums_go_to_the_lower_index():
    """Observation 2 repeats observation 1 bit for bit: pairs (0, 1) and (0, 2) have the same point, count and sum, and
    (0, 1) - the lower index - wins."""
    K, Rt, X, off, view, x, _ = _scene(10, 8, 4, noise_px=0.5, min_len=2, max_len=2)
    vs = np.array([view[off[0]], view[off[0] + 1], view[off[0] + 1]])
    xs = np.array([x[off[0]], x[off[0] + 1], x[off[0] + 1]])
    table = otr.pair_table(K, Rt, vs, xs, 4.0)
    assert (table[0][4], table[0][5]) == (table[1][4], table[1][5]) and table[0][3]
    assert otr.pair_search(table) == 0


def test_no_candidate():
    """A point behind both cameras: no pair passes its own observations."""
    K, Rt, X, off, view, x, _ = _scene(10, 8, 5, noise_px=0.0, min_len=2, max_len=2)
    vs = view[off[0]:off[1]]
    behind = []
    Xb = -np.array([0.0, 0.0, 30.0])  # far behind every camera of the arc (all look towards +z)
    for c in vs:
        p = creproj.projection(K[c], Rt[c]) @ np.append(Xb, 1.0)
        behind.append(p[:2] / p[2])
    assert otr.pair_search(otr.pair_table(K, Rt, vs, np.array(behind), 4.0)) == -1


def test_refine_replay_lowers_the_cost():
    K, Rt, X, off, view, x, _ = _scene(10, 8, 6, noise_px=1.0, min_len=6, max_len=6)
    vs, xs = view[off[0]:off[1]], x[off[0]:off[1]]
    Ps = [creproj.projection(K[c], Rt[c]) for c in vs]
    X0 = otr.dlt_svd(Ps, xs)
    Xr, c = otr.refine_replay(X0, Ps, xs)
    assert c <= otr.cost(X0, Ps, xs)
    J, r = otr.jacobian(Xr, Ps, xs), otr.residuals(Xr, Ps, xs)
    assert np.linalg.norm(J.T @ r) <= 1e-8 * np.linalg.norm(J) * np.linalg.norm(r)


def test_multi_view_scene_windows_and_outliers():
    V = 12
    K, R, t, X, off, view, x, out = make_multi_view_scene(4000, V, 7, outlier_frac=0.2)
    n = np.diff(off)
    assert n.min() == 2 and n.max() == 8 and off[0] == 0 and off[-1] == len(view) == len(x) == len(out)
    for i in range(len(n)):
        v = view[off[i]:off[i + 1]]
        assert np.array_equal(v, np.arange(v[0], v[0] + len(v))) and v[0] >= 0 and v[-1] < V
    assert abs(out.mean() - 0.2) <= 1.0 / len(out)
    # inliers reproject within the noise, with every point in front of its cameras
    Rt = np.concatenate([R, t[:, :, None]], axis=2)
    pt = np.repeat(np.arange(len(n)), n)
    for c in range(V):
        sel = (view == c) & ~out
        m, val = creproj.reproj_exact_many(Rt[c], K, X[pt[sel]], x[sel], 25.0)
        assert m.all()
    for c in range(V):
        assert np.allclose(R[c] @ R[c].T, np.eye(3), atol=1e-12) and np.linalg.det(R[c]) > 0


def test_tracks_from_dense():
    vis = np.array([[1, 0, 1, 1], [0, 0, 0, 0], [1, 1, 0, 0]], dtype=bool)
    pix = np.arange(24, dtype=np.float64).reshape(3, 4, 2)
    off, view, x = tracks_from_dense(vis, pix)
    assert off.tolist() == [0, 3, 3, 5] and view.tolist() == [0, 2, 3, 0, 1]
    assert np.array_equal(x, pix[[0, 0, 0, 2, 2], [0, 2, 3, 0, 1]])
