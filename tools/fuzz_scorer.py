"""One-off fuzz of K1-K3 against the exact C scorer: random sizes, thresholds, outlier fractions, variants.
Counts must be bit-equal, sums within 1e-12 relative, winner equal.  usage: python tools/fuzz_scorer.py [cases]"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from oracle import csed  # noqa: E402
from oracle import restatement as o  # noqa: E402
from structure_from_motion_b200 import _native  # noqa: E402
from structure_from_motion_b200.scenes import make_scene  # noqa: E402

cases = int(sys.argv[1]) if len(sys.argv) > 1 else 40
rng = np.random.default_rng(2026)
eng = _native.get_engine(0)
bad = 0
for k in range(cases):
    n = int(rng.choice([8, 9, 31, 64, 65, 127, 500, 2049, 4096, 7777, 20000]))
    h = int(rng.choice([1, 2, 31, 32, 33, 63, 64, 65, 129, 1000, 4097]))
    thr = float(10.0 ** rng.uniform(-9, 1))
    frac = float(rng.choice([0.0, 0.1, 0.4, 0.9]))
    variant, hpt, g = [("screen", 2, 16), ("full", 2, 16), ("screen32", 4, 8), ("auto", 2, 16), ("screen32", 2, 16)][k % 5]
    agg = ["rms", "sum", "mean", "square"][k % 4]
    K, x1, x2, *_ = make_scene(n, frac, seed=100 + k)
    nxa, nya = o.k_normalise(x1[:, 0], x1[:, 1], K)
    nxb, nyb = o.k_normalise(x2[:, 0], x2[:, 1], K)
    eng.set_score_variant(variant, hpt, g)
    eng.upload_pairs(x1, x2, K)
    eng.sample_device(k, h)
    E, valid, _ = eng.fit()
    table = eng.get_table()
    cnt, s1, s2, err = eng.score(thr, min_extra=3, aggregation=agg)
    best = eng.get_best()
    v = valid.astype(np.uint8)
    cnt_o, s1_o, s2_o = csed.score_batch(E.reshape(-1, 9), nxa, nya, nxb, nyb, thr, table=table, valid=v, nthreads=8)
    ok_cnt = np.array_equal(np.where(valid, cnt, -1), np.where(valid, cnt_o, -1))
    with np.errstate(all="ignore"):
        ok_s = np.allclose(s1[valid], s1_o[valid], rtol=1e-12, atol=0, equal_nan=True) and \
            np.allclose(s2[valid], s2_o[valid], rtol=1e-12, atol=0, equal_nan=True)
    ntot = 8 + cnt_o
    with np.errstate(all="ignore"):
        exp = {"sum": s1_o, "square": s2_o, "mean": s1_o / ntot, "rms": np.sqrt(s2_o / ntot)}[agg]
    exp = np.where((cnt_o >= 3) & valid, exp, np.inf)
    want = int(np.argmin(exp)) if np.isfinite(exp).any() else -1
    ok_w = best.index == want or (want >= 0 and best.index >= 0 and abs(exp[best.index] - exp[want]) <= 1e-12 * abs(exp[want]))
    status = "ok" if (ok_cnt and ok_s and ok_w) else "MISMATCH"
    if status != "ok":
        dc = np.flatnonzero(np.where(valid, cnt, -1) != np.where(valid, cnt_o, -1))
        with np.errstate(all="ignore"):
            r1 = np.nanmax(np.abs(s1[valid] - s1_o[valid]) / np.maximum(np.abs(s1_o[valid]), 1e-300)) if valid.any() else 0
            r2 = np.nanmax(np.abs(s2[valid] - s2_o[valid]) / np.maximum(np.abs(s2_o[valid]), 1e-300)) if valid.any() else 0
        print("     cnt", ok_cnt, "sums", ok_s, "winner", ok_w, "| count diffs at", dc[:5], cnt[dc[:5]], cnt_o[dc[:5]],
              "| max rel dS1 %.3e dS2 %.3e" % (r1, r2), "| nonfinite s1", int((~np.isfinite(s1[valid])).sum()),
              int((~np.isfinite(s1_o[valid])).sum()))
    bad += status != "ok"
    print(f"{k:3d} n {n:6d} h {h:5d} thr {thr:8.2e} out {frac:.1f} {variant:8s} hpt {hpt} {agg:6s} inl/hyp {np.maximum(cnt_o, 0).mean():9.1f} "
          f"winner {best.index:5d}/{want:5d} {status}")
eng.set_score_variant("screen")
print("mismatches:", bad)
sys.exit(1 if bad else 0)
