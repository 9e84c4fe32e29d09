"""Fuzz of the batched homography and model-selection calls against the single-pair calls on the same pairs: random
ragged batches (empty, too short, around the 64-record tile and the 2 048-record item), general, planar and
rotation-only pairs, random skewed cameras, hypothesis counts, thresholds (including 0, < 0 and > 1e100), every
aggregation and selection mode, pair_id0 != 0.

Per case:
  - Engine.batch_two_view_homography against, for every pair p, upload_pairs(a, b, I) + sample_device(seed, h,
    stream=pair_id0 + p) + Engine.two_view_homography(Ks[p]): H, winner, counts, inlier list, pass bits, votes, the
    voted candidate, rotation flag and points, all bit for bit;
  - Engine.batch_score_models on that upload against Engine.model_scores on each pair alone, with random given /
    not-given flags, per-point errors included, bit for bit.
usage: python tools/fuzz_batch_homography.py [cases]"""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from structure_from_motion_b200 import _native  # noqa: E402
from structure_from_motion_b200.scenes import make_planar_scene, make_scene  # noqa: E402

AGGS = ["sum", "square", "mean", "rms"]
SELS = ["min_error", "max_inliers", "msac"]


def scene(kind, n, seed, K):
    """[n,2] pixel pairs of a general ("e"), planar ("p") or rotation-only ("r") scene with camera K."""
    m = max(n, 8)
    if kind == "e":
        _, x1, x2, *_ = make_scene(m, 0.2, seed, K=K)
    else:
        _, x1, x2, *_ = make_planar_scene(m, 0.2, seed, rotation_only=kind == "r", K=K)
    return x1[:n].copy(), x2[:n].copy()


def batch(sizes, kinds, seed, skew=False):
    """Concatenated pairs, offsets and per-pair cameras (random fx != fy, principal point and optional skew)."""
    rng = np.random.default_rng(seed)
    xa, xb, Ks = [], [], []
    for p, (n, k) in enumerate(zip(sizes, kinds)):
        K = np.array([[rng.uniform(600, 900), rng.uniform(0, 3) if skew else 0.0, rng.uniform(600, 680)],
                      [0.0, rng.uniform(600, 900), rng.uniform(440, 520)], [0.0, 0.0, 1.0]])
        a, b = scene(k, n, seed * 131 + p, K)
        xa.append(a), xb.append(b), Ks.append(K)
    offsets = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return np.concatenate(xa).reshape(-1, 2), np.concatenate(xb).reshape(-1, 2), offsets, np.stack(Ks)


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float64).view(np.int64)


def compare_homography(eng, xa, xb, offsets, Ks, h, seed, pair_id0, thr, min_extra=0.0, agg="rms", sel="min_error",
                       dist=50.0, rot=1e-2):
    """Mismatch messages of batch_two_view_homography against the single-pair calls (empty list: all bit-equal)."""
    r = eng.batch_two_view_homography(xa, xb, offsets, Ks, h, seed, thr, min_extra, agg, sel, dist, rot, pair_id0=pair_id0)
    bad = []
    for p in range(len(offsets) - 1):
        lo, hi = int(offsets[p]), int(offsets[p + 1])
        s0, s1 = int(r["inlier_offsets"][p]), int(r["inlier_offsets"][p + 1])
        tag = f"pair {p} (n {hi - lo}, thr {thr}, {agg}/{sel})"
        if hi - lo < 8:
            if not (r["best_index"][p] == -1 and s0 == s1 and r["pose_index"][p] == -2 and r["num_invalid"][p] == h
                    and not np.any(r["H"][p])):
                bad.append(f"{tag}: a short pair has a model or a segment")
            continue
        eng.upload_pairs(xa[lo:hi], xb[lo:hi], np.eye(3))
        eng.sample_device(seed, h, stream=pair_id0 + p)
        best, _, _, ps, _, idx, ok, X = eng.two_view_homography(Ks[p], thr, min_extra, agg, sel, dist, rot)
        checks = {
            "H": np.array_equal(_bits(np.array(best.E)), _bits(r["H"][p].reshape(9))),
            "best_index": int(best.index) == int(r["best_index"][p]),
            "best_err": _bits(best.err) == _bits(r["best_err"][p]),
            "count_extra": (int(best.count_extra) if best.index >= 0 else -1) == int(r["count_extra"][p]),
            "num_invalid": int(best.num_invalid) == int(r["num_invalid"][p]),
            "inliers": np.array_equal(idx, r["inlier_idx"][s0:s1]),
            "pass": np.array_equal(ok, r["pass_bits"][s0:s1]),
            "counts": np.array_equal(np.array(ps.counts), r["counts"][p]),
            "vote": int(ps.best) == int(r["pose_index"][p]),
            "rotation": bool(ps.rotation_only) == bool(r["rotation_only"][p]),
            "points": np.array_equal(_bits(X), _bits(r["points"][s0:s1])),
        }
        if best.index >= 0:
            b = max(int(ps.best), 0)
            checks["R"] = np.array_equal(_bits(np.array(ps.R[b])), _bits(r["R"][p].reshape(9)))
            checks["t"] = np.array_equal(_bits(np.array(ps.t[b])), _bits(r["t"][p]))
            checks["n"] = np.array_equal(_bits(np.array(ps.n[b])), _bits(r["n"][p]))
            checks["d"] = _bits(ps.d[b]) == _bits(r["d"][p])
        bad += [f"{tag}: {k} differs" for k, v in checks.items() if not v]
    return bad, r


def compare_scores(eng, xa, xb, offsets, Ks, E, H, have_e, have_h, sigma=1.0, ratio=0.45):
    """Mismatch messages of batch_score_models (on the engine's current batched upload of these pairs) against
    model_scores on each pair alone."""
    s, pp = eng.batch_score_models(E, H, have_e, have_h, sigma, ratio, per_point=True)
    bad = []
    for p in range(len(offsets) - 1):
        lo, hi = int(offsets[p]), int(offsets[p + 1])
        ge, gh = bool(have_e[p]), bool(have_h[p])
        tag = f"scores of pair {p} (n {hi - lo}, E {ge}, H {gh})"
        if not ge and not gh:
            if s[p].model != -1 or s[p].fixed_e or s[p].fixed_h or not np.isnan(pp[lo:hi]).all():
                bad.append(f"{tag}: a pair without models has scores")
            continue
        if hi == lo:
            continue  # an empty pair cannot be uploaded alone
        eng.upload_pairs(xa[lo:hi], xb[lo:hi], np.eye(3))
        r, rp = eng.model_scores(E[p] if ge else None, H[p] if gh else None, Ks[p], sigma, ratio, per_point=True)
        fields = ("score_e", "score_h", "ratio_h", "fixed_e", "fixed_h", "count_e", "count_h", "model")
        bad += [f"{tag}: {f} differs" for f in fields if getattr(r, f) != getattr(s[p], f)
                and not (isinstance(getattr(r, f), float) and _bits(getattr(r, f)) == _bits(getattr(s[p], f)))]
        if not np.array_equal(_bits(rp), _bits(pp[lo:hi])):
            bad.append(f"{tag}: per-point errors differ")
    return bad


def one_case(eng, rng, case):
    P = int(rng.integers(1, 9))
    pool = [0, 5, 7, 8, 9, 33, 63, 64, 65, 300, 1024, 1025, 2047, 2048, 2049, int(rng.integers(8, 5000))]
    sizes = [int(rng.choice(pool)) for _ in range(P)]
    kinds = [str(rng.choice(["e", "p", "r"])) for _ in range(P)]
    xa, xb, offsets, Ks = batch(sizes, kinds, 1000 + case, skew=bool(rng.integers(0, 2)))
    if offsets[-1] == 0:
        return []
    h = int(rng.choice([1, 63, 64, 65, 200, 513]))
    thr = float(rng.choice([4.0, 0.5, 25.0, 0.0, -1.0, 1e101, 2.0 ** 4, float(np.nextafter(2.0 ** 4, 0))]))
    agg, sel = str(rng.choice(AGGS)), str(rng.choice(SELS))
    min_extra = float(rng.choice([0.0, 3.0]))
    seed, pair_id0 = int(rng.integers(0, 2 ** 31)), int(rng.integers(0, 1000))
    bad, r = compare_homography(eng, xa, xb, offsets, Ks, h, seed, pair_id0, thr, min_extra, agg, sel)
    have_e = rng.integers(0, 2, P).astype(bool)
    have_h = rng.integers(0, 2, P).astype(bool)
    have_h[~have_e & ~have_h & (rng.random(P) < 0.5)] = True
    E = rng.normal(size=(P, 3, 3))
    H = np.where(r["best_index"][:, None, None] >= 0, r["H"], np.eye(3) + 0.01 * rng.normal(size=(P, 3, 3)))
    eng.batch_two_view_homography(xa, xb, offsets, Ks, 1, seed, thr, pair_id0=pair_id0)  # the batched upload again
    bad += compare_scores(eng, xa, xb, offsets, Ks, E, H, have_e, have_h, float(rng.choice([0.5, 1.0, 3.0])))
    return [f"case {case} (sizes {sizes}, kinds {''.join(kinds)}, h {h}): {m}" for m in bad]


def main(cases):
    eng = _native.Engine(_native.default_device())
    rng = np.random.default_rng(20261020)
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
