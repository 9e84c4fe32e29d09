"""One-off fuzz of the PnP path against the oracles: random sizes (8 .. 20 000 records, around the 64-record tile and
the 2 048-record item), hypothesis counts (1 .. 4 097, around the 64-hypothesis item), thresholds over nine decades
and at the fixed-point edges, outlier fractions, the table and device samplers, every aggregation and selection mode,
and random cameras (fx != fy, shifted principal point, skew 0 or 3 px).

Per case: the scorer and K3 against oracle/creproj on the GPU's own poses (oracle.pnp.expected_selection: counts
bit-equal, errors within 1e-12, winner among the oracle's best), the winner's mask and errors bit-equal, and the fitter
of up to 4 rows against the exact P3P (validity equal and [R|t] within 1e-5 relative outside the ambiguity band: point-3 errors of two solutions within 1e-6 relative, the
collinearity sine within 0.1 % of its tolerance, or a sine below 1e-3, where float64 conditioning rules).
usage: python tools/fuzz_pnp.py [cases]"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import creproj  # noqa: E402
from oracle import pnp as op  # noqa: E402
from structure_from_motion_b200 import _native  # noqa: E402
from structure_from_motion_b200.scenes import make_pnp_scene  # noqa: E402

SPECIAL = [float(np.nextafter(2.0 ** k, 0.0)) for k in (-3, 2, 4, 10)] + [2.0 ** k for k in (-3, 2, 4, 10)]
SPECIAL += [1e-130, 1e100, float(np.nextafter(1e100, np.inf))]
AGGS = ["sum", "square", "mean", "rms"]
SELS = ["min_error", "max_inliers", "msac"]


def run_case(eng, k, rng):
    n = int(rng.choice([8, 9, 63, 64, 65, 2047, 2048, 2049, int(rng.integers(8, 20001))]))
    h = int(rng.choice([1, 63, 64, 65, 127, 128, 129, int(rng.integers(1, 4098))]))
    thr = float(rng.choice(SPECIAL)) if rng.random() < 0.3 else float(10.0 ** rng.uniform(-4, 5))
    frac = float(rng.uniform(0, 0.9))
    agg, sel = str(rng.choice(AGGS)), str(rng.choice(SELS))
    fx = float(rng.uniform(400, 1200))
    K = np.array([[fx, float(rng.choice([0.0, 3.0])), float(rng.uniform(500, 800))],
                  [0, fx * float(rng.uniform(0.9, 1.1)), float(rng.uniform(400, 560))], [0, 0, 1]])
    K_, X, x, R, t, _ = make_pnp_scene(n, frac, seed=int(rng.integers(1 << 30)), noise_px=float(rng.uniform(0, 2)), K=K)
    sampler = "device" if rng.random() < 0.5 else "table"
    desc = f"case {k}: n={n} h={h} thr={thr:.6g} frac={frac:.2f} {agg}/{sel} {sampler}"
    bad = []
    eng.upload_pnp(X, x, K)
    if sampler == "device":
        eng.sample_device(int(rng.integers(1 << 40)), h, hyp_offset=int(rng.integers(0, 1000)))
    else:
        table = np.stack([rng.choice(n, 8, replace=False) for _ in range(h)]).astype(np.int32)
        eng.set_table(table)
    best, Rt_w, mask, err, cnt, err_h = eng.ransac_pnp(thr, 0.0, agg, sel, want_arrays=True)
    table = eng.get_table()
    models, valid = eng.get_pnp_models()
    exp = op.expected_selection(models, valid, K, X, x, thr, table, agg, sel)
    if not np.array_equal(cnt, np.where(valid, exp["count_extra"], -1)):
        bad.append("count_extra")
    fin = np.isfinite(exp["err"])
    if not np.array_equal(fin, np.isfinite(err_h)) or not np.all(
            np.abs(err_h[fin] - exp["err"][fin]) <= 1e-12 * np.abs(exp["err"][fin]) + 1e-300):
        bad.append("err_h")
    if int(best.index) not in exp["winners"].tolist():
        bad.append(f"winner {best.index} not in {exp['winners'][:5]}")
    if best.index >= 0:
        if not np.array_equal(Rt_w.reshape(12), models[best.index].reshape(12)):
            bad.append("winner pose")
        m_c, v_c = creproj.reproj_exact_many(models[best.index], K, X, x, thr)
        if not np.array_equal(m_c, mask.astype(bool)) or not np.array_equal(v_c.view(np.int64), err.view(np.int64)):
            bad.append("mask/err")
    for i in rng.choice(h, min(h, 4), replace=False):
        rows = table[i][:4]
        ref, info = op.fit_pnp_exact(K, X[rows], x[rows])
        ambiguous = info["gap"] < 1e-6 or abs(info["collinear"] / op.COLLINEAR - 1) < 1e-3 or info["collinear"] < 1e-3
        if ambiguous:
            continue
        if (ref is not None) != bool(valid[i]):
            bad.append(f"validity row {i}: gpu {bool(valid[i])} oracle {ref is not None}")
        elif ref is not None and np.abs(ref - models[i]).max() > 1e-5 * (1 + np.abs(ref).max()):
            bad.append(f"pose row {i}: {np.abs(ref - models[i]).max():.3g}")
    return desc, bad


def main():
    cases = int(sys.argv[1]) if len(sys.argv) > 1 else 40
    rng = np.random.default_rng(2029)
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
