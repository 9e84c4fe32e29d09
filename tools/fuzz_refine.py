"""Fuzz of the least-squares refinement (sfm_set_refinement) of essential-matrix and homography winners:

  - every pair of Engine.batch_two_view / batch_two_view_homography with refinement against the single-pair call on
    that pair (upload + sample_device(seed, h, stream=pair_id0 + p) + two_view / two_view_homography): the refined
    model, the reports, the inlier list, pass bits, votes and points bit for bit, and the RANSAC side (E / H, winner,
    error) bit-equal to the same batch without refinement;
  - per refined pair: cost_final <= cost_start, model[8] == 1, an essential matrix with singular values (s, s, 0);
  - on single pairs, the final cost against scipy's Levenberg-Marquardt (oracle/refine.py) from the same start on the
    same inlier list.
Ragged batches (sizes around the 256-entry chunk and the 1 024-record tail block), thresholds over several decades plus
0, inf and NaN, every aggregation and selection mode, skewed cameras.
usage: python tools/fuzz_refine.py [cases]"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from fuzz_batch_homography import batch  # noqa: E402
from oracle import refine as O  # noqa: E402
from structure_from_motion_b200 import _native  # noqa: E402

AGGS = ["sum", "square", "mean", "rms"]
SELS = ["min_error", "max_inliers", "msac"]
SIZES = [0, 5, 8, 63, 64, 65, 255, 256, 257, 1024, 1025, 2047, 2048, 2049]
E_THRS = [1e-7, 1e-6, 1e-5, 1e-4, 0.0, float("inf"), float("nan")]
H_THRS = [0.25, 4.0, 64.0, 1e3, 0.0, float("inf"), float("nan")]
REPORT = ("cost_ransac", "cost_start", "cost_final", "num", "iterations", "status", "rejected")


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def invariants(rep, kind):
    """Messages for a report that breaks what every refinement keeps."""
    bad = []
    st = _native.REFINE_STATUS[int(rep.status)]
    m = np.array(rep.model, dtype=np.float64).reshape(3, 3)
    if st in ("no_model",):
        return bad
    if m[2, 2] != 1.0:
        bad.append("model[8] != 1")
    if st == "nonfinite":
        return bad
    if not rep.cost_final <= rep.cost_start:
        bad.append(f"cost_final {rep.cost_final} > cost_start {rep.cost_start}")
    if kind == "E":
        s = np.linalg.svd(m, compute_uv=False)
        if abs(s[0] - s[1]) > 1e-12 * s[0] or s[2] > 1e-12 * s[0]:
            bad.append(f"singular values {s}")
    return bad


def compare_batch(eng, kind, xa, xb, offsets, Ks, h, seed, pair_id0, thr, iters, agg="rms", sel="min_error",
                  min_extra=0.0):
    """Mismatch messages of a refined batch against the single-pair calls and the unrefined batch."""
    call = eng.batch_two_view if kind == "E" else eng.batch_two_view_homography
    key = "E" if kind == "E" else "H"
    r0 = call(xa, xb, offsets, Ks, h, seed, thr, min_extra, agg, sel, pair_id0=pair_id0)
    r = call(xa, xb, offsets, Ks, h, seed, thr, min_extra, agg, sel, pair_id0=pair_id0, refine_iterations=iters)
    bad = []
    for k in (key, "best_index", "best_err", "count_extra", "num_invalid"):
        if not np.array_equal(_bits(r0[k]) if r0[k].dtype == np.float64 else r0[k],
                              _bits(r[k]) if r[k].dtype == np.float64 else r[k]):
            bad.append(f"RANSAC {k} changed by the refinement")
    for p in range(len(offsets) - 1):
        lo, hi = int(offsets[p]), int(offsets[p + 1])
        s0, s1 = int(r["inlier_offsets"][p]), int(r["inlier_offsets"][p + 1])
        tag = f"{kind} pair {p} (n {hi - lo}, thr {thr}, {agg}/{sel}, iters {iters})"
        if hi - lo < 8:
            if _native.REFINE_STATUS[int(r["refine_status"][p])] != "no_model":
                bad.append(f"{tag}: a short pair is not 'no model'")
            continue
        if kind == "E":
            eng.upload_pairs(xa[lo:hi], xb[lo:hi], Ks[p])
            eng.sample_device(seed, h, stream=pair_id0 + p)
            _, _, _, ps, _, idx, ok, X = eng.two_view(thr, min_extra, agg, sel, refine_iterations=iters)
        else:
            eng.upload_pairs(xa[lo:hi], xb[lo:hi], np.eye(3))
            eng.sample_device(seed, h, stream=pair_id0 + p)
            _, _, _, ps, _, idx, ok, X = eng.two_view_homography(Ks[p], thr, min_extra, agg, sel, refine_iterations=iters)
        rep = eng.get_refinement(1)[0]
        checks = {
            "refined model": np.array_equal(_bits(np.array(rep.model)), _bits(r["refined_" + key][p].reshape(9))),
            "inliers": np.array_equal(idx, r["inlier_idx"][s0:s1]),
            "pass": np.array_equal(ok, r["pass_bits"][s0:s1]),
            "counts": np.array_equal(np.array(ps.counts), r["counts"][p]),
            "vote": int(ps.best) == int(r["pose_index"][p]),
            "points": np.array_equal(_bits(X), _bits(r["points"][s0:s1])),
        }
        for f in REPORT:
            v = getattr(rep, f)
            w = r["refine_" + ("iterations" if f == "iterations" else f)][p]
            checks[f] = _bits(v) == _bits(w) if isinstance(v, float) else int(v) == int(w)
        bad += [f"{tag}: {k} differs from the single-pair call" for k, v in checks.items() if not v]
        bad += [f"{tag}: {m}" for m in invariants(rep, kind)]
    return bad, r


def oracle_check(eng, kind, pa, pb, K, h, seed, thr, iters=100, rtol=1e-9, min_extra=0.0):
    """(messages, report, oracle cost) of a single-pair refinement against scipy's LM from the same start on the same
    inlier list (the tail's list of the unrefined call)."""
    if kind == "E":
        eng.upload_pairs(pa, pb, K)
        eng.sample_device(seed, h)
        best, _, _, _, _, idx, _, _ = eng.two_view(thr, min_extra)
        nrm = eng.get_normalised()
        eng.sample_device(seed, h)
        eng.two_view(thr, min_extra, refine_iterations=iters)
    else:
        eng.upload_pairs(pa, pb, np.eye(3))
        eng.sample_device(seed, h)
        best, _, _, _, _, idx, _, _ = eng.two_view_homography(K, thr, min_extra)
        eng.sample_device(seed, h)
        eng.two_view_homography(K, thr, min_extra, refine_iterations=iters)
    rep = eng.get_refinement(1)[0]
    bad = invariants(rep, kind)
    if best.index < 0:
        return bad, rep, None
    Er = np.array(best.E, dtype=np.float64).reshape(3, 3)
    if kind == "E":
        na, nb = nrm[idx, :2], nrm[idx, 2:]
        R0, t0 = O.pose_start(Er)
        c0 = O.e_cost(O.e_from_pose(R0, t0), na, nb)
        Eo, co, _ = O.refine_e(R0, t0, na, nb)
        Mg = np.array(rep.model).reshape(3, 3)
        dm = min(np.linalg.norm(Mg - Eo), np.linalg.norm(Mg + Eo)) / np.linalg.norm(Eo)
    else:
        c0 = O.h_cost(Er, pa[idx], pb[idx])
        Eo, co = O.refine_h(Er, pa[idx], pb[idx])
        Mg = np.array(rep.model).reshape(3, 3)
        dm = np.linalg.norm(Mg - Eo) / np.linalg.norm(Eo)
    if abs(rep.cost_start - c0) > 1e-9 * max(c0, 1e-300):
        bad.append(f"cost_start {rep.cost_start!r} vs oracle {c0!r}")
    if co > 0 and abs(rep.cost_final - co) > rtol * co:
        bad.append(f"cost_final {rep.cost_final!r} not within {rtol} of the oracle optimum {co!r}")
    return bad, rep, dict(cost=co, model=Eo, dmodel=dm)


def one_case(eng, rng, case):
    P = int(rng.integers(1, 7))
    sizes = [int(rng.choice(SIZES + [int(rng.integers(8, 4000))])) for _ in range(P)]
    kinds = [str(rng.choice(["e", "p", "r"])) for _ in range(P)]
    xa, xb, offsets, Ks = batch(sizes, kinds, 3000 + case, skew=bool(rng.integers(0, 2)))
    if offsets[-1] == 0:
        return []
    kind = str(rng.choice(["E", "H"]))
    thr = float(rng.choice(E_THRS if kind == "E" else H_THRS))
    agg, sel = str(rng.choice(AGGS)), str(rng.choice(SELS))
    h = int(rng.choice([1, 64, 200, 513]))
    iters = int(rng.choice([1, 2, 5, 20]))
    bad, _ = compare_batch(eng, kind, xa, xb, offsets, Ks, h, int(rng.integers(0, 2 ** 31)), int(rng.integers(0, 1000)),
                           thr, iters, agg, sel)
    return [f"case {case} (sizes {sizes}, kinds {''.join(kinds)}, h {h}): {m}" for m in bad]


def main(cases):
    eng = _native.Engine(_native.default_device())
    rng = np.random.default_rng(20261021)
    bad = []
    for case in range(cases):
        bad += one_case(eng, rng, case)
    for m in bad[:50]:
        print(m)
    print(f"cases: {cases}  mismatches: {len(bad)}")
    eng.close()
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main(int(sys.argv[1]) if len(sys.argv) > 1 else 40))
