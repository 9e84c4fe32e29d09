"""Time the batched homography path and the batched essential-matrix / homography choice on one GPU.

Shape: bench.py's config4 (512 pairs x 2 000 correspondences x 2 000 device-sampler hypotheses), half general pairs
(make_scene) and half planar pairs (make_planar_scene), 40 % outliers, each pair a permutation of its scene as in
config4.  Thresholds: 1e-5 on the SED, 4 px^2 on the transfer error, RMS, minimum error, at least 600 extra inliers
(half of the 1 200 true ones: without a floor the minimum-error winner explains little more than its own sample).

Per step, one context (the engine's own stream), host clock around every call (each ends in a synchronisation):
  batch_h        Engine.batch_two_view_homography, with its stage times from sfm_get_timing (fit / score / finalise /
                 tail = mask + pose + triangulate) - the device events of one call
  batch_scores   Engine.batch_score_models on that upload (stage "score" = the k_score_models launch)
  batch_e        Engine.batch_two_view (the E side alone)
  batch_select   model_selection.batch_two_view_select_arrays (E batch + H batch + scores + host assembly)
  loop_select    the same pairs through a loop of single-pair two_view_select_arrays(sampler="device") calls
The batched H scorer's rate is P n h / (its "score" stage), next to the single-pair rate of DESIGN.md section 7a.

Prints one JSON line with the card's name, power limit and maximum SM clock read in the same run.

    python tools/time_batch_select.py [--steps 5] [--warmup 1] [--loop-pairs 512] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.time_homography import gpu_info  # noqa: E402

P, N, H, OUTLIERS, E_THR, H_THR, MIN_EXTRA = 512, 2000, 2000, 0.4, 1e-5, 4.0, 600


def scenes():
    import numpy as np

    from structure_from_motion_b200.scenes import make_planar_scene, make_scene

    gen = make_scene(N, OUTLIERS, seed=0)[:3]
    pla = make_planar_scene(N, OUTLIERS, seed=0)[:3]
    rng = np.random.default_rng(0)
    xa, xb, Ks = [], [], []
    for p in range(P):
        K, x1, x2 = gen if p % 2 == 0 else pla
        perm = rng.permutation(N)
        xa.append(x1[perm])
        xb.append(x2[perm])
        Ks.append(K)
    return np.concatenate(xa), np.concatenate(xb), np.arange(P + 1, dtype=np.int64) * N, np.stack(Ks)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--loop-pairs", type=int, default=P, help="pairs timed through the single-pair loop")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np

    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.model_selection import batch_two_view_select_arrays, two_view_select_arrays

    if _native.load_library().sfm_device_count() < 1:
        raise SystemExit("time_batch_select.py needs a CUDA device")
    eng = _native.Engine(0)
    eng.enable_timing(True)
    xa, xb, offsets, Ks = scenes()
    keys = ("batch_h", "batch_scores", "batch_e", "batch_select", "loop_select")
    wall = {k: [] for k in keys}
    stages_h, stages_s = [], []
    models = None
    for step in range(args.warmup + args.steps):
        rec = step >= args.warmup
        t0 = time.perf_counter()
        r = eng.batch_two_view_homography(xa, xb, offsets, Ks, H, 1, H_THR, MIN_EXTRA)
        t1 = time.perf_counter()
        st = eng.get_timing()[0]
        keep = r["best_index"] >= 0
        t2 = time.perf_counter()
        eng.batch_score_models(np.tile(np.eye(3), (P, 1, 1)), r["H"], np.zeros(P, bool), keep)
        t3 = time.perf_counter()
        ss = eng.get_timing()[0]
        t4 = time.perf_counter()
        eng.batch_two_view(xa, xb, offsets, Ks, H, 1, E_THR, MIN_EXTRA)
        t5 = time.perf_counter()
        eng.get_timing()
        t6 = time.perf_counter()
        sel = batch_two_view_select_arrays(xa, xb, offsets, Ks, E_THR, H_THR, H, 1, min_extra=MIN_EXTRA, engine=eng)
        t7 = time.perf_counter()
        eng.get_timing()
        t8 = time.perf_counter()
        for p in range(args.loop_pairs):
            lo, hi = offsets[p], offsets[p + 1]
            try:
                two_view_select_arrays(Ks[p], xa[lo:hi], xb[lo:hi], E_THR, H_THR, MIN_EXTRA, "rms", H, None,
                                       sampler="device", seed=p, engine=eng)
            except ValueError:
                pass
        t9 = time.perf_counter()
        eng.get_timing()
        if rec:
            for k, v in zip(keys, (t1 - t0, t3 - t2, t5 - t4, t7 - t6, t9 - t8)):
                wall[k].append(v * 1e3)
            stages_h.append(st)
            stages_s.append(ss)
            models = sel["model"]
    med = {k: float(np.median(v)) for k, v in wall.items()}
    sh = {k: float(np.median([s[k] for s in stages_h])) for k in stages_h[0]}
    score_ms = sh["score"]
    out = {
        "tool": "time_batch_select", "gpu": gpu_info(0),
        "shape": f"{P} pairs x {N} correspondences x {H} hypotheses (device sampler), half make_scene, half "
                 f"make_planar_scene, {OUTLIERS:.0%} outliers",
        "steps": args.steps,
        "wall_ms_median": med,
        "wall_ms_all": wall,
        "loop_pairs": args.loop_pairs,
        "loop_select_ms_per_512_pairs": med["loop_select"] * P / args.loop_pairs,
        "batch_h_stages_ms": {"upload": sh["upload"], "fit": sh["fit"], "score": sh["score"], "finalise": sh["select"],
                              "tail": sh["mask"] + sh["pose"] + sh["triangulate"]},
        "batch_scores_kernel_ms": float(np.median([s["score"] for s in stages_s])),
        "batch_h_scorer_evals_per_s": P * N * H / (score_ms * 1e-3) if score_ms > 0 else None,
        "single_pair_h_scorer_evals_per_s_design_7a": 0.303e12,
        "models": {m: int(np.sum(models == m)) for m in ("essential", "homography")},
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    eng.close()


if __name__ == "__main__":
    main()
