"""Accuracy of the PnP pose refinement (refine_iterations = 20) against the RANSAC pose, and the range of exact
rescaling.

* make_pnp_scene(1000, 0.4, s), 0.5 px noise, seeds 0-7, 500 hypotheses (reference sampler), min_extra 300,
  threshold 4 px^2: rotation error (degrees) and |t - t_true| of the RANSAC pose and of the refined pose.
* The three-view composition of tests/test_gpu_pnp.py (make_three_view_scene(3000, 0.2, 61)) with
  refine_iterations 0 and 20 on both stages: max |R3 - R3_true|.
* World x 2^k (t with it) and pixels / K's first two rows x 2^k (threshold x 4^k): the k for which the report is
  bit-identical after exact rescaling, swept in steps of 2 from 0 outwards until the first difference.
Writes one JSON object with the GPU's name, power limit and maximum SM clock.

    python tools/pnp_refine_accuracy.py [--out profiles/pnp_refine_accuracy_b200.json]
"""
from __future__ import annotations

import argparse
import json
import os
import random
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.time_homography import gpu_info  # noqa: E402


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np

    from oracle.refine import rodrigues
    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.pnp import ransac_pnp_arrays, refine_pnp_arrays
    from structure_from_motion_b200.scenes import make_pnp_scene, make_three_view_scene
    from structure_from_motion_b200.two_view import two_view_arrays

    eng = _native.get_engine(0)

    def rot_err(a, b):
        return float(np.degrees(np.arccos(np.clip((np.trace(a @ b.T) - 1) / 2, -1, 1))))

    rows = []
    for s in range(8):
        K, X, x, R, t, _ = make_pnp_scene(1000, 0.4, s, noise_px=0.5)
        random.seed(s)
        res = ransac_pnp_arrays(K, X, x, 4.0, 300, "rms", 500, engine=eng, refine_iterations=20)
        f = res.refinement
        rows.append({"seed": s, "rot_off_deg": rot_err(res.R, R), "rot_on_deg": rot_err(f.R, R),
                     "t_off": float(np.linalg.norm(res.t - t)), "t_on": float(np.linalg.norm(f.t - t)),
                     "status": f.status, "iterations": f.iterations, "num": f.num})
    med = {k: float(np.median([r[k] for r in rows])) for k in ("rot_off_deg", "rot_on_deg", "t_off", "t_on")}

    K, x1, x2, x3, (R2, t2), (R3, t3), Xw = make_three_view_scene(3000, 0.2, seed=61)
    three = {}
    for it in (0, 20):
        random.seed(1)
        tv = two_view_arrays(K, x1, x2, 1e-5, 1500, "rms", 200, engine=eng, refine_iterations=it)
        idx = tv.inlier_indices[tv.passing]
        random.seed(2)
        res = ransac_pnp_arrays(K, tv.points[tv.passing], x3[idx], 4.0, len(idx) // 2, "rms", 200, engine=eng,
                                refine_iterations=it)
        three[str(it)] = float(np.abs((res.refinement.R if it else res.R) - R3).max())

    K, X, x, R, t, _ = make_pnp_scene(400, 0.0, seed=31, noise_px=0.5)
    R0 = R @ rodrigues([2e-3, -1e-3, 1e-3])
    base = refine_pnp_arrays(R0, t, K, X, x, 25.0, engine=eng)

    def world_ok(k):
        sc = refine_pnp_arrays(R0, np.ldexp(t, k), K, np.ldexp(X, k), x, 25.0, engine=eng)
        return (np.array_equal(sc.R, base.R) and np.array_equal(sc.t, np.ldexp(base.t, k))
                and sc.iterations == base.iterations and sc.status == base.status and sc.num == base.num)

    def pixel_ok(k):
        Ks = K.copy()
        Ks[:2] = np.ldexp(Ks[:2], k)
        sc = refine_pnp_arrays(R0, t, Ks, X, np.ldexp(x, k), float(np.ldexp(25.0, 2 * k)), engine=eng)
        return (np.array_equal(sc.R, base.R) and np.array_equal(sc.t, base.t) and sc.iterations == base.iterations
                and sc.cost_final == np.ldexp(base.cost_final, 2 * k) and sc.num == base.num)

    def sweep(ok, sign):
        k = 0
        while abs(k) < 1100:
            k2 = k + 2 * sign
            try:
                good = ok(k2)
            except Exception:
                good = False
            if not good:
                return k, k2
            k = k2
        return k, None

    rng = {}
    for name, ok in (("world", world_ok), ("pixels", pixel_ok)):
        lo = sweep(ok, -1)
        hi = sweep(ok, +1)
        rng[name] = {"exact_from": lo[0], "first_failure_below": lo[1], "exact_to": hi[0], "first_failure_above": hi[1]}

    out = {"gpu": gpu_info(0), "scenes": rows, "median": med, "three_view_R3_maxabs": three, "scale_range": rng}
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
