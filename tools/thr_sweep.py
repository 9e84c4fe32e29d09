"""K2 time against the inlier threshold (config 3): the screen's cost grows with the survivor rate."""
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from structure_from_motion_b200 import _native  # noqa: E402
from structure_from_motion_b200.scenes import make_scene  # noqa: E402

n, h = 100_000, 65_536
K, x1, x2, *_ = make_scene(n, 0.4, seed=0)
eng = _native.get_engine(0)
eng.upload_pairs(x1, x2, K)
eng.sample_device(0, h)
eng.fit(want_E=False)
eng.enable_timing(True)
print("thr        variant   ms      evals/s     mean inliers per hypothesis")
thrs = (1.5e-8, 1.5e-7, 1.5e-6, 1.5e-5, 1.5e-4, 1.5e-3)
if "--cliff" in sys.argv:  # the two inlier-rich points and the headline, auto and two-sided only
    thrs = (1.5e-6, 1.5e-4, 1.5e-3)
for thr in thrs:
    shapes = (("auto", 2, 16), ("screen", 2, 16), ("full", 2, 16), ("screen32", 4, 8))
    if "--cliff" in sys.argv:
        shapes = (("auto", 2, 16), ("full", 2, 16))
    for v, hpt, g in shapes:
        eng.set_score_variant(v, hpt, g)
        ts = []
        for r in range(3):
            cnt, _, _, _ = eng.score(thr, 10, "rms")
            t, _ = eng.get_timing()
            ts.append(t["score"])
        print(f"{thr:8.1e}  {v:9s} hpt {hpt} {min(ts[1:]):7.3f}  {n * h / min(ts[1:]) * 1e3:.3e}   {np.maximum(cnt, 0).mean():.1f}")
