"""One-off fuzz of the homography paths against the oracles: random sizes (8 .. 20 000 correspondences, around the
64-record tile and the 2 048-record item), hypothesis counts (1 .. 4 097, around the 64-hypothesis item), thresholds
over nine decades and at the fixed-point edges, outlier fractions, samplers, every aggregation and selection mode, and
random cameras (fx != fy, shifted principal point, skew 0 or 3 px).

Per case: the fitter against oracle.homography.homography_4pt (validity equal, H within the conditioning-scaled
bound), the scorer and K3 against ctransfer on the GPU's own models (oracle.homography.expected_selection: counts
bit-equal, errors within 1e-12, winner among the oracle's best), the winner's mask and errors bit-equal; when a model
exists, the pose tail (decomposition against oracle.homography_pose, pass bits and counts equal to its vote, points
within 1e-6 of its triangulation) and the model scores of the winner and a fitted E bit-equal to oracle/cselect.
usage: python tools/fuzz_homography.py [cases]"""
import os
import random
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import cselect, ctransfer  # noqa: E402
from oracle import homography as oh  # noqa: E402
from oracle import homography_pose as hp  # noqa: E402
from oracle import restatement as o  # noqa: E402
from structure_from_motion_b200 import _native  # noqa: E402
from structure_from_motion_b200.scenes import make_planar_scene  # noqa: E402

SPECIAL = [float(np.nextafter(2.0 ** k, 0.0)) for k in (-3, 2, 4, 10)] + [2.0 ** k for k in (-3, 2, 4, 10)]
SPECIAL += [1e-130, 1e100, float(np.nextafter(1e100, np.inf))]


def _condition(a, b):
    na, _ = o.hartley_normalise(a)
    nb, _ = o.hartley_normalise(b)
    A = []
    for (x, y), (u, v) in zip(na, nb):
        A.append([-x, -y, -1, 0, 0, 0, u * x, u * y, u])
        A.append([0, 0, 0, -x, -y, -1, v * x, v * y, v])
    s = np.linalg.svd(np.array(A), compute_uv=False)
    return s[0] / s[7]


def _set_gap(a, b):
    return max(min(max(np.abs(Ra - Rb).max(), np.abs(ta - tb).max(), np.abs(na - nb).max(), abs(da - db) / db)
                   for Rb, tb, nb, db in b) for Ra, ta, na, da in a)


def _candidates(p):
    R = np.array(p.R).reshape(4, 3, 3)
    t, n = np.array(p.t).reshape(4, 3), np.array(p.n).reshape(4, 3)
    return [(R[i], t[i], n[i], float(p.d[i])) for i in range(1 if p.rotation_only else 4)]


def run_case(eng, k, rng):
    n = int(rng.choice([8, 9, 63, 64, 65, 500, 2047, 2048, 2049, 4097, 20000]))
    h = int(rng.choice([1, 2, 31, 63, 64, 65, 129, 1000, 4097]))
    frac = float(rng.choice([0.0, 0.3, 0.9]))
    thr = float(rng.choice(SPECIAL)) if rng.uniform() < 0.3 else float(10.0 ** rng.uniform(-4, 5))
    sampler = ["table", "device", "reference"][k % 3]
    agg = ["rms", "sum", "mean", "square"][k % 4]
    sel = ["min_error", "max_inliers", "msac"][(k // 4) % 3]
    min_extra = float(rng.choice([0, 3, 0.5 * n]))
    f = rng.uniform(500, 1500)
    K = np.array([[f, float(rng.choice([0.0, 3.0])), rng.uniform(560, 720)], [0.0, f * rng.uniform(0.9, 1.1),
                  rng.uniform(420, 540)], [0.0, 0.0, 1.0]])
    _, x1, x2, _, _ = make_planar_scene(n, frac, seed=300 + k, K=K)
    cols = (x1[:, 0], x1[:, 1], x2[:, 0], x2[:, 1])
    eng.upload_pairs(x1, x2, np.eye(3))
    if sampler == "device":
        eng.sample_device(k, h, hyp_offset=int(rng.integers(0, 1 << 20)))
        table = eng.get_table()
    else:
        if sampler == "reference":
            h = min(h, max(1, 2_000_000 // n))  # the Python shuffle costs n per row
            random.seed(k)
            table = o.python_shuffle_table(n, h)
        else:
            table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
        eng.set_table(table)
    desc = f"{k:3d} n {n:6d} h {h:5d} thr {thr:9.3e} out {frac:.1f} {sampler:9s} {agg:6s} {sel:9s} skew {K[0, 1]:.0f}"
    bad = []
    # fitter
    Hs, valid = eng.fit_homography()
    for i in range(h):
        s = table[i, :4]
        Hr, ok = oh.homography_4pt(x1[s], x2[s])
        if bool(valid[i]) != ok:
            bad.append(f"valid[{i}]")
        elif ok:
            cond = _condition(x1[s], x2[s])
            if np.max(np.abs(Hs[i] - Hr)) / np.max(np.abs(Hr)) > 1e-9 * max(1.0, cond / 1e2):
                bad.append(f"H[{i}]")
    # scorer, K3, mask
    best, mask, err, cnt, err_h = eng.ransac_homography(thr, min_extra, agg, sel, want_arrays=True)
    Hs, valid = eng.get_models()
    ref = oh.expected_selection(Hs, valid, *cols, thr, table, agg, sel, min_extra)
    if not np.array_equal(np.where(valid, cnt, -1), np.where(valid, ref["count_extra"], -1)):
        bad.append("count_extra")
    fin = np.isfinite(ref["err"])
    if not np.array_equal(np.isfinite(err_h), fin):
        bad.append("err_h finite")
    elif np.any(np.abs(err_h[fin] - ref["err"][fin]) > 1e-12 * np.abs(ref["err"][fin])):
        bad.append("err_h")
    if int(best.index) not in ref["winners"]:
        bad.append(f"winner {best.index} not in {ref['winners'][:4]}")
    if best.index < 0:
        return desc + " no model", bad
    Hw = Hs[best.index]
    m_ref, v_ref = ctransfer.transfer_exact_many(Hw, *cols, thr)
    if not (np.array_equal(mask.astype(bool), m_ref) and np.array_equal(err.view(np.int64), v_ref.view(np.int64))):
        bad.append("mask")
    # pose tail on the winner
    p, num, idx, ok, X = eng.homography_pose_and_triangulate(K, thr)
    dec = hp.decompose_homography(Hw, K)
    gpu = _candidates(p)
    if bool(p.rotation_only) != dec["rotation_only"]:
        bad.append("rotation_only")
    elif not dec["rotation_only"]:
        s = dec["sv"]
        tol = 1e-6 if min(abs(s[0] - 1.0), abs(s[2] - 1.0)) < 1e-4 else 1e-9
        if _set_gap(gpu, dec["candidates"]) > tol:
            bad.append("decomposition")
        icols = (x1[idx, 0], x1[idx, 1], x2[idx, 0], x2[idx, 1])
        bits, counts, vbest = hp.vote(gpu, K, *icols)
        if not (np.array_equal(ok, bits) and np.array_equal(np.array(p.counts), counts)):
            bad.append("vote")
        elif counts.any():
            if int(p.best) != vbest:
                bad.append("voted")
            R, t, _, _ = gpu[vbest]
            passing = (bits >> vbest) & 1
            Xo = hp.triangulate(K, R, t, *icols, passing)
            live = passing.astype(bool)
            if not np.array_equal(np.isnan(Xo), np.isnan(X)):
                bad.append("points nan")
            elif live.any() and np.max(np.abs(X[live] - Xo[live]) / np.linalg.norm(Xo[live], axis=1)[:, None]) > 1e-6:
                bad.append("points")
    # model scores of the winner and a fitted E
    eng.upload_pairs(x1, x2, K)
    eng.sample_device(k, 64)
    E, ev, _ = eng.fit()
    Ew = E[np.flatnonzero(ev)[0]] if ev.any() else None
    sc, pp = eng.model_scores(Ew, Hw, K, per_point=True)
    rs = cselect.score_models(K, x1, x2, Ew, Hw)
    if not (np.array_equal(pp, rs["per_point"], equal_nan=True) and
            (sc.fixed_e, sc.fixed_h, sc.count_e, sc.count_h, sc.model) ==
            (rs["fixed_e"], rs["fixed_h"], rs["count_e"], rs["count_h"], rs["model"])):
        bad.append("model scores")
    return desc + f" winner {best.index:5d} inliers {num:6d}", bad


def main():
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 40
    rng = np.random.default_rng(2027)
    eng = _native.get_engine(0)
    mismatches = 0
    for k in range(cases):
        desc, bad = run_case(eng, k, rng)
        mismatches += bool(bad)
        print(desc, "ok" if not bad else "MISMATCH " + ", ".join(bad), flush=True)
    print("mismatches:", mismatches)
    sys.exit(1 if mismatches else 0)


if __name__ == "__main__":
    main()
