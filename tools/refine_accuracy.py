"""Accuracy of the least-squares refinement (sfm_set_refinement) against the truth, on one GPU.

  essential    8 seeds of make_scene(1 000 points, 0.5 px, 40 % outliers), 500 device-sampler hypotheses, SED threshold
               1e-5, RMS, min_extra 300, selections min_error and max_inliers: median rotation error and median
               translation-direction error of two_view_arrays with refine_iterations 0 and 30, and the median inlier
               list the refinement ran on
  homography   8 seeds of make_planar_scene(1 000 points, 0.5 px, 40 %), 4 px^2, min_extra 300: median rotation and
               plane-normal errors of two_view_homography_arrays (the truth's candidate from the exact H's decomposition)
  selection    256 planar pairs (make_planar_scene(2 000, 40 %), one seed per pair) and 128 general pairs
               (make_scene(2 000, 40 %)) through batch_two_view_select_arrays (SED 1e-5, 4 px^2, min_extra 600, RMS,
               minimum error: the shape of DESIGN.md sections 7c / 7d) at 512 and 2 000 hypotheses, refine_iterations 0
               and 20: how many pairs of each kind pick H and E
(tests/test_gpu_refine.py asserts the direction of the first two.)  Prints one JSON line with the card's name, power
limit and maximum SM clock read in the same run.

    python tools/refine_accuracy.py [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tools.time_homography import gpu_info  # noqa: E402


def _rot(Ra, Rb):
    import numpy as np
    return float(np.degrees(np.arccos(np.clip((np.trace(Ra.T @ Rb) - 1.0) / 2.0, -1.0, 1.0))))


def _dir(a, b):
    import numpy as np
    a, b = a / np.linalg.norm(a), b / np.linalg.norm(b)
    return float(np.degrees(np.arccos(np.clip(abs(a @ b), 0.0, 1.0))))


def main() -> None:
    import numpy as np

    from structure_from_motion_b200 import _native
    from structure_from_motion_b200.homography import two_view_homography_arrays
    from structure_from_motion_b200.model_selection import batch_two_view_select_arrays
    from structure_from_motion_b200.scenes import make_planar_scene, make_scene
    from structure_from_motion_b200.two_view import two_view_arrays

    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    eng = _native.Engine(0)
    med = lambda v: float(np.median(v))
    rec = {"tool": "tools/refine_accuracy.py", "gpu": gpu_info(0)}

    ess = {}
    for sel in ("min_error", "max_inliers"):
        r = {0: ([], []), 30: ([], [])}
        nums = []
        for seed in range(8):
            K, x1, x2, R, t, _ = make_scene(1000, 0.4, 100 + seed, noise_px=0.5)
            for it in (0, 30):
                tv = two_view_arrays(K, x1, x2, 1e-5, 300, "rms", 500, sampler="device", seed=seed, on_degenerate="skip",
                                     selection=sel, engine=eng, refine_iterations=it)
                r[it][0].append(_rot(tv.R, R)), r[it][1].append(_dir(tv.t, t))
                if it:
                    nums.append(tv.refinement.num)
        ess[sel] = {"rotation_deg_median": {"off": med(r[0][0]), "on": med(r[30][0])},
                    "translation_dir_deg_median": {"off": med(r[0][1]), "on": med(r[30][1])},
                    "inlier_list_median": med(nums)}
    rec["essential"] = ess

    r = {0: ([], []), 30: ([], [])}
    for seed in range(8):
        K, x1, x2, H, _ = make_planar_scene(1000, 0.4, 200 + seed, noise_px=0.5)
        d = eng.decompose_homography(H, K)
        for it in (0, 30):
            hv = two_view_homography_arrays(K, x1, x2, 4.0, 300, sampler="device", seed=seed, engine=eng,
                                            max_iterations=500, refine_iterations=it)
            c = int(np.argmin([_rot(np.array(d.R[k]).reshape(3, 3), hv.R) for k in range(4)]))
            r[it][0].append(_rot(hv.R, np.array(d.R[c]).reshape(3, 3))), r[it][1].append(_dir(hv.n, np.array(d.n[c])))
    rec["homography"] = {"rotation_deg_median": {"off": med(r[0][0]), "on": med(r[30][0])},
                         "normal_deg_median": {"off": med(r[0][1]), "on": med(r[30][1])}}

    xa, xb, Ks, kinds = [], [], [], []
    for p in range(256 + 128):
        planar = p < 256
        K, x1, x2 = (make_planar_scene(2000, 0.4, seed=1000 + p) if planar else make_scene(2000, 0.4, seed=1000 + p))[:3]
        xa.append(x1), xb.append(x2), Ks.append(K), kinds.append("planar" if planar else "general")
    xa, xb = np.concatenate(xa), np.concatenate(xb)
    offsets = np.arange(len(Ks) + 1, dtype=np.int64) * 2000
    kinds = np.array(kinds)
    picks = {}
    for h in (512, 2000):
        for it in (0, 20):
            out = batch_two_view_select_arrays(xa, xb, offsets, np.stack(Ks), 1e-5, 4.0, h, 7, min_extra=600,
                                               engine=eng, refine_iterations=it)
            m = out["model"]
            picks[f"h{h}_refine{it}"] = {k: {"homography": int(np.sum((kinds == k) & (m == "homography"))),
                                             "essential": int(np.sum((kinds == k) & (m == "essential"))),
                                             "neither": int(np.sum((kinds == k) & np.equal(m, None)))}
                                         for k in ("planar", "general")}
    rec["selection"] = picks
    eng.close()
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
